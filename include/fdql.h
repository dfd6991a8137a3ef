/*
 * fdql.h -- C ABI of libfdql.so, the B200 (sm_100a) learner hot path of franQ / FastDeepQLearning.
 *
 * The reference has no FFI: its boundary is Python duck typing (SURVEY.md section 8b).  These are the entry
 * points the Python mirror classes in fastdeepqlearning_b200/ bind with ctypes; each one names the reference
 * code it replaces (paths relative to the reference checkout).
 *
 * Conventions
 *   - every pointer is a CUDA device pointer unless its name ends in _host;
 *   - every launch goes to `stream` (a cudaStream_t passed as void*; NULL = legacy default stream);
 *   - return value 0 = FDQL_OK, negative = error; fdql_last_error() returns a thread-local message;
 *   - no exceptions cross the ABI, no allocation after fdql_arena_create (except *_host staging, sized once);
 *   - thread-compatible: one arena may be driven by one writer thread and one reader thread, each on its
 *     own stream; the caller orders writer->reader with stream/event dependencies.
 *   - all learner-visible data is fp32, the dtype franQ's TorchDataLoader casts every key to
 *     (franQ/Replay/wrappers/torch_dataloader.py:36); row indices are int64 like numpy.random.randint.
 */
#ifndef FDQL_H_
#define FDQL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDQL_OK 0
#define FDQL_EINVAL (-1)      /* bad argument (also: n_drop == 0, the reference's empty-target quirk Q8)   */
#define FDQL_ECUDA (-2)       /* a CUDA runtime call failed; message holds cudaGetErrorString               */
#define FDQL_EOVERSAMPLE (-3) /* franQ/Replay/replay_memory.py:6,50,57-58 OversampleError                   */
#define FDQL_ENOMEM (-4)

#define FDQL_MAX_KEYS 24

/* Key roles: which stored column plays which part in relabelling / returns.  NONE = gathered verbatim. */
enum {
  FDQL_ROLE_NONE = 0,
  FDQL_ROLE_REWARD = 1,
  FDQL_ROLE_TASK_DONE = 2,
  FDQL_ROLE_EPISODE_DONE = 3,
  FDQL_ROLE_EPISODE_STEP = 4,
  FDQL_ROLE_MC_RETURN = 5,
  FDQL_ROLE_ACHIEVED_GOAL = 6,
  FDQL_ROLE_DESIRED_GOAL = 7
};

/* Device reward functors R(achieved_goal, goal) -> (reward, done); the enum-dispatched stand-in for the
 * Python callable HindsightNStepReplay receives (franQ/Replay/wrappers/her.py:13,62,67). */
enum {
  FDQL_REWARD_NONE = 0,
  FDQL_REWARD_BITFLIP = 1,      /* franQ/Env/bitflip.py:143-152: all(ag==g) ? 0 : -1; done = reward==0          */
  FDQL_REWARD_ALL_GEQ = 2,      /* franQ/Env/classic_control_goal/classic_goal.py:88-93: all(ag>=g) ? 0 : -1     */
  FDQL_REWARD_FIRST_GEQ = 3,    /* classic_goal.py:306-311: done = ag[0]>=g[0]; reward = done-1                   */
  FDQL_REWARD_WEIGHTED_PNORM = 4 /* franQ/Env/eleurent_parking.py:42-55: -(sum|ag-g|*w)^p; done = reward>-thr;
                                    params = {p, thr, w[0..G)}                                                   */
};

/* fdql_sample_streams modes (which row of the episode supplies the hindsight goal) */
enum {
  FDQL_GOAL_FINAL = 0,  /* her.py:49-50  mode "final": the episode's last achieved_goal                      */
  FDQL_GOAL_RANDOM = 1, /* her.py:51-53  mode "random": any row of the episode                               */
  FDQL_GOAL_FUTURE = 2  /* HER "future" strategy (BASELINE.json configs[2]); not a reference mode            */
};

/* fdql_sample_gather option bits */
#define FDQL_OPT_EXACT_EPISODE_STEP 1u /* scan the episode prefix so relabelled episode_step equals her.py:72-83 bit for bit */
#define FDQL_OPT_EMIT_LEARNER_AUX 2u   /* also write mask / is_contiguous / upstream weight (deepQlearning.py:201-203,222-225) */
#define FDQL_OPT_CORESIDENT 4u         /* this gather runs on one stream while a loss kernel runs on another (the reference's prefetch
                                          thread, torch_dataloader.py:22-39): take ONE small block per SM whose wide keys move through
                                          cp.async staging + bulk write-back, leaving the issue slots to the loss kernel.  See
                                          fdql_set_coresident.  Shapes the lean kernel does not serve ignore the bit. */

typedef struct fdql_arena fdql_arena;

const char* fdql_last_error(void);
int fdql_version(void);

/* ---- replay arena: replaces ReplayMemory.__init__/_jit_initialize (franQ/Replay/replay_memory.py:18-35) and the
 *      AsyncReplayMemory child process (franQ/Replay/async_replay_memory.py:9-70).  One SoA slab per key in HBM;
 *      width-1 keys are packed into one 16B-aligned scalar record per row next to the episode extents. ---- */
int fdql_arena_create(int64_t capacity, int32_t n_keys, const int32_t* widths_host, const int32_t* roles_host,
                      int32_t device, fdql_arena** out);
int fdql_arena_destroy(fdql_arena* a);
/* cursor state with the reference's arithmetic: top=(top+1)%capacity, len=max(top,len)  (replay_memory.py:45-46, Q1) */
int fdql_arena_info(const fdql_arena* a, int64_t* capacity, int64_t* top, int64_t* len, int64_t* bytes);
int fdql_arena_set_cursor(fdql_arena* a, int64_t top, int64_t len);
/* raw view of one key's storage for zero-copy host-language views: element (row, c) lives at base[row*row_stride + col + c] */
int fdql_arena_key_view(const fdql_arena* a, int32_t key, float** base, int64_t* row_stride, int32_t* col);
/* internal columns: which=0 ep_start(int32 bits), 1 ep_end(int32 bits) inside the scalar record; 2 goal-agnostic reward (column 2 of
 * the 16-byte scan records); 3 the 16-byte link records (column 0).  Used for zero-copy views and for snapshot / restore. */
int fdql_arena_meta_view(const fdql_arena* a, int32_t which, float** base, int64_t* row_stride, int32_t* col);
/* discount the link records were built with (state 0: none yet, 1: gamma valid, 2: mixed -> sample-time relabelling scans the tail);
 * set != 0 writes *gamma / *state into the arena (restore of a snapshot), else reads them */
int fdql_arena_link_state(fdql_arena* a, int32_t set, double* gamma, int32_t* state);

/* ReplayMemory.add for n rows at once (replay_memory.py:38-46): src[k] is a dense [n_rows, width_k] fp32 array.
 * Rows land at top, top+1, ... modulo capacity; the cursor advances with Q1 semantics. */
int fdql_arena_append(fdql_arena* a, int64_t n_rows, const float* const* src, void* stream);
int fdql_arena_append_host(fdql_arena* a, int64_t n_rows, const float* const* src_host, void* stream);

/* The same from ONE packed host block [n_rows, row_floats] (pinned for the copy to be asynchronous): key k of row r lives at
 * packed_host[r * row_floats + key_offsets_host[k] ..].  One host-to-device copy per call instead of one per key; this is what the
 * Python mirror's add() stages rows into (Runner._replay_handler -> replay.add, franQ/Runner/runner.py:177-191).  Offsets and
 * row_floats that are multiples of 4 keep the 128-bit path.  flags: FDQL_APPEND_SQUASH_REWARDS applies the Pohlen transform of
 * franQ/Replay/wrappers/squash_rewards.py:5-7 to the reward column inside the append kernel (SquashRewards.add, :15-18).
 * The block may be reused by the host once the work enqueued on `stream` so far has completed (record an event after the call). */
#define FDQL_APPEND_SQUASH_REWARDS 1u
int fdql_arena_append_packed_host(fdql_arena* a, int64_t n_rows, const float* packed_host, int32_t row_floats,
                                  const int32_t* key_offsets_host, uint32_t flags, void* stream);

/* NStepReturn._flush + calculate_montecarlo_return (franQ/Replay/wrappers/nstep_return.py:36-48,60-72) for n_eps
 * complete episodes already in the ring: episode e occupies rows ep_begin[e] .. ep_begin[e]+ep_len[e]-1 (mod capacity).
 * Writes mc_return (if with_returns), the episode extents, and (if reward_op != NONE and the goal roles are bound)
 * the goal-agnostic reward r - R(ag, dg) (her.py:65-68) used later by sample-time relabelling. */
int fdql_commit_episodes(fdql_arena* a, int32_t n_eps, const int64_t* ep_begin, const int32_t* ep_len, double gamma,
                         int32_t with_returns, int32_t reward_op, const float* reward_params_host, int32_t n_params,
                         void* stream);

/* HindsightNStepReplay._hindsight_flush (her.py:55-95) at write time: for each episode copy rows src_begin.. to
 * dst_begin.. with desired_goal := achieved_goal[goal_row], reward/task_done/episode_step relabelled, and mc_return
 * recomputed over the whole real episode (quirk Q5).  dst rows must already be reserved with fdql_arena_reserve. */
int fdql_her_flush_episodes(fdql_arena* a, int32_t n_eps, const int64_t* src_begin, const int32_t* ep_len,
                            const int64_t* dst_begin, const int64_t* goal_row, int32_t reward_op,
                            const float* reward_params_host, int32_t n_params, double gamma, int32_t with_returns,
                            void* stream);
/* fdql_her_flush_episodes with the rewards computed beforehand (for a reward function the functors cannot express, evaluated by the
 * caller on the device before the call) instead of by a functor.  The episode arguments and the rows written are those of
 * fdql_her_flush_episodes: desired_goal := achieved_goal[goal_row], reward := (r - R(ag, dg)) + R(ag, g*) in fp64 rounded to fp32,
 * task_done := done(R(ag, g*)), episode_step re-based at every relabelled terminal (her.py:72-83), the extents of the copy, and
 * mc_return over the whole real episode (quirk Q5).
 * Packed layout: the n_rows = sum(ep_len) source rows episode after episode in the order of the episode table, each episode
 * oldest row first, so that source row j of episode e is packed row sum(ep_len[0..e)) + j.  Device arrays of n_rows each:
 *   reward[i], done[i]  R(ag_i, g*) of the row and its episode's goal g* = achieved_goal[goal_row[e]] (done: non-zero = done);
 *   reward_dg[i]        R(ag_i, dg_i), the row's reward under its own desired_goal (the goal-agnostic term of her.py:65-68).
 * Needs achieved_goal and desired_goal keys.  Reads ep_len back to the host to check sum(ep_len) == n_rows, so the call waits for the
 * work already enqueued on `stream`. */
int fdql_her_flush_episodes_given(fdql_arena* a, int32_t n_eps, const int64_t* src_begin, const int32_t* ep_len,
                                  const int64_t* dst_begin, const int64_t* goal_row, int64_t n_rows, const float* reward,
                                  const uint8_t* done, const float* reward_dg, double gamma, int32_t with_returns, void* stream);
/* advance the cursor by n rows without writing them (their content is produced by fdql_her_flush_episodes) */
int fdql_arena_reserve(fdql_arena* a, int64_t n_rows, int64_t* first_row);

/* quirk Q3 (nstep_return.py:33-34,50-57): NStepReturn._pop stores the oldest buffered row a second time, with the return
 * truncated after n_step rewards.  Copies row src_row to dst_row (reserved by the caller) and sets its mc_return to the
 * recurrence over the rewards of rows src_row .. src_row+n_step-1. */
int fdql_q3_duplicate(fdql_arena* a, int64_t src_row, int32_t n_step, int64_t dst_row, double gamma, void* stream);

/* DeepQLearning.get_losses pre-processing for discrete actions (franQ/Agent/deepQlearning.py:206-210):
 * out[r, :] = eye(n_actions)[(long)action[r]] for the n_rows rows of a gathered [T, B, 1] action column (fp32 in, fp32 out).
 * torch's indexing raises on an out-of-range action; here the row becomes all zeros and *out_of_range (device int32, may be NULL,
 * caller-zeroed) is set to 1. */
int fdql_action_onehot(int64_t n_rows, int32_t n_actions, const float* action, float* out, int32_t* out_of_range, void* stream);

/* ---- "vmap" hindsight variant (her_mode="vmap"): V virtual goals per row instead of one relabelled copy -------------------
 * The virtual columns are ordinary keys of the arena, named by their key index: virtual_goals [V+1, G] (flattened),
 * virtual_rewards [V+1], virtual_dones [V+1], virtual_mc_return [V+1] (key_returns = -1: absent); column V is the real goal.
 *
 * fdql_vmap_flush_episodes: for n_eps complete episodes already in the ring,
 *   mode bit 0  HindsightVmapWrite._hindsight_flush + _virtual_episode_calc (franQ/Replay/wrappers/her_vmap.py:30-43,66-88):
 *               virtual goal v of episode e := achieved_goal[pick_rows[e*V + v]] (the reference draws the picks with
 *               np.random.randint(0, L, V), :75), virtual_reward = (reward - R(ag, dg)) + R(ag, vg) in float32,
 *               virtual_done = (task_done and not done(R(ag, dg))) or done(R(ag, vg));
 *   mode bit 1  NStepReturnVmap._flush + _inner (franQ/Replay/wrappers/nstep_return_vmap.py:37-48,61-74): per column the
 *               recurrence G_j = fl32(r_j + G_{j+1} * gamma * m_j) in fp64, newest row first; done_quirk != 0 uses
 *               m_j = dones[j] exactly as the reference does (quirk Q7), 0 uses m_j = 1 - dones[j]. */
int fdql_vmap_flush_episodes(fdql_arena* a, int32_t n_eps, const int64_t* ep_begin, const int32_t* ep_len, const int64_t* pick_rows,
                             int32_t key_goals, int32_t key_rewards, int32_t key_dones, int32_t key_returns, int32_t reward_op,
                             const float* reward_params_host, int32_t n_params, double gamma, int32_t mode, int32_t done_quirk,
                             void* stream);
/* fdql_vmap_flush_episodes with the rewards computed beforehand instead of by a functor (see fdql_her_flush_episodes_given).  Mode bit
 * 0 must be set; bit 1 and done_quirk act as above.  Packed layout: the n_rows = sum(ep_len) rows episode after episode in the order
 * of the episode table, each oldest row first; reward and done are device grids [n_rows, V+1] (row-major; done: non-zero = done):
 *   column v < V  R(ag_i, achieved_goal[pick_rows[e*V + v]]), the row under virtual goal v of its episode;
 *   column V      R(ag_i, dg_i), the row under its own desired_goal (the term the virtual rewards and dones are rebased from).
 * virtual_reward = (reward - column V) + column v in float32, virtual_done = (task_done and not done[V]) or done[v]; column V of
 * the stored keys keeps the row's own reward and task_done as in fdql_vmap_flush_episodes.  Reads ep_len back to the host to check
 * sum(ep_len) == n_rows, so the call waits for the work already enqueued on `stream`. */
int fdql_vmap_flush_episodes_given(fdql_arena* a, int32_t n_eps, const int64_t* ep_begin, const int32_t* ep_len,
                                   const int64_t* pick_rows, int32_t key_goals, int32_t key_rewards, int32_t key_dones,
                                   int32_t key_returns, int64_t n_rows, const float* reward, const uint8_t* done, double gamma,
                                   int32_t mode, int32_t done_quirk, void* stream);

/* HindsightVmapRead.temporal_sample (franQ/Replay/wrappers/her_vmap.py:104-123) for windows (starts[b]+t) % len, t<T:
 * desired_goal [T,n,G] := virtual_goals[..., column, :], reward / task_done / mc_return [T,n,1] := the same column of
 * virtual_rewards / virtual_dones / virtual_mc_return.  Only the chosen column is read.  Outputs and aux may be NULL;
 * aux (mask [T,n,1], is_contiguous [T-1,n,1], loss weight [T-1,n,1]) follows the selected dones (deepQlearning.py:201-203,222-225). */
int fdql_vmap_select_column(const fdql_arena* a, int64_t n_windows, int32_t T, int64_t len, const int64_t* starts, int32_t column,
                            int32_t key_goals, int32_t key_rewards, int32_t key_dones, int32_t key_returns, int32_t batch_for_weight,
                            float* out_desired_goal, float* out_reward, float* out_task_done, float* out_mc_return, float* aux_mask,
                            float* aux_contig, float* aux_weight, void* stream);

/* np.random.randint(0, len-T, B) (replay_memory.py:59) + HER goal choice (her.py:48-53), drawn on the device with a
 * counter-based generator.  Parity runs inject the streams instead.  flags[b]=1 with probability relabel_prob.
 * counter_dev (may be NULL): four uint64 in device memory {draw counter, 0, ring length or 0, 0}; when given, the draw uses
 * counter + counter_dev[0] and the kernel advances it, so a captured CUDA graph draws fresh streams at every replay; a non-zero
 * counter_dev[2] replaces the ring length the launch was given (starts ~ U[0, counter_dev[2] - T)), so the same captured launch keeps
 * sampling the whole ring while it fills -- the caller stores the length there after every append. */
int fdql_sample_streams(const fdql_arena* a, int64_t n, int32_t T, int32_t goal_mode, float relabel_prob, uint64_t seed,
                        uint64_t counter, uint64_t* counter_dev, int64_t* starts, uint8_t* flags, int64_t* goal_rows,
                        void* stream);

/* fdql_sample_streams + fdql_sample_gather in one launch: the window starts, hindsight flags and goal rows are drawn inside the
 * gather kernel with the same counter-based generator (identical streams for the same seed / counter), written to starts / flags /
 * goal_rows (flags and goal_rows NULL: no relabelling) and used at once.  len is the ring's current length.  Shapes the fused kernel
 * does not serve (small batches, T > 32 with relabelling, other reward functors) run as the two separate launches. */
int fdql_sample_gather_draw(const fdql_arena* a, int64_t n_windows, int32_t T, int32_t goal_mode, float relabel_prob, uint64_t seed,
                            uint64_t counter, uint64_t* counter_dev, int64_t* starts, uint8_t* flags, int64_t* goal_rows,
                            int32_t reward_op, const float* reward_params_host, int32_t n_params, double gamma, uint32_t opts,
                            int32_t batch_for_weight, float* const* out, float* aux_mask, float* aux_contig, float* aux_weight,
                            void* stream);

/* One pass of the learner loop as ONE launch: fdql_sample_gather_draw of batch k+1 (arguments up to aux_weight, same meaning; the
 * reference does this in TorchDataLoader's prefetch thread one batch ahead, torch_dataloader.py:22-39) and fdql_tqc_loss of batch k
 * (arguments from M on, same meaning; distributional_soft_actor_critic.py:50-58,70-103) in a warp-specialised persistent kernel, one
 * block per SM: 16 loss warps + 8 gather warps with separate shared memory, named barriers and work counters.  The two halves must not
 * alias (the loss reads batch k's reward / mask / mc_return / weight while the gather writes batch k+1 into other buffers).
 * M == 0: the gather alone; n_windows == 0: the loss alone.  Shapes the fused kernel does not serve (loss tables other than 97..128
 * atoms, small batches, keys wider than the lean copy plan, other reward functors) run as the separate launches, gather then loss on
 * `stream`, with identical results.  TD pairs (T == 2) over the reference's usual record ({reward, task_done, episode_done,
 * episode_step, mc_return}, valid link records) and one long vector + up to three vectors of <= 16 floats take a build with these facts
 * compiled in; any other arena runs the general build, with identical results (tests/test_gpu_r2.py).  The fused kernel claims its
 * work from counters in a 16-slot workspace of the arena, one slot per
 * launch in turn: at most 16 fused passes of one arena may be in flight at a time (passes on one stream never are). */
int fdql_fused_pass(const fdql_arena* a, int64_t n_windows, int32_t T, int32_t goal_mode, float relabel_prob, uint64_t seed,
                    uint64_t counter, uint64_t* counter_dev, int64_t* starts, uint8_t* flags, int64_t* goal_rows, int32_t reward_op,
                    const float* reward_params_host, int32_t n_params, double gamma, uint32_t opts, int32_t batch_for_weight,
                    float* const* out, float* aux_mask, float* aux_contig, float* aux_weight, int64_t M, int32_t n_atoms, int32_t n_drop,
                    const float* next_z, const float* q_pred, const float* next_log_pi, const float* reward, const float* mask,
                    const float* mc_return, const float* grad_scale, float alpha, float loss_gamma, float* loss, float* grad_q,
                    double* stats, void* stream);

/* ReplayMemory.__getitem__ / sample (replay_memory.py:48-52,68-70): out[k] is [n, width_k]. */
int fdql_gather_rows(const fdql_arena* a, int64_t n, const int64_t* idx, float* const* out, void* stream);

/* ReplayMemory.temporal_sample/_temporal_sample_idxes (replay_memory.py:54-66) + TorchDataLoader (torch_dataloader.py:36)
 * + sample-time HER relabel with reward recompute (her.py:55-95) + return recompute (nstep_return.py:60-72), fused.
 * Window b covers rows (starts[b]+t) % len, t<T; out[k] is [T, n_windows, width_k] (time-major like the reference).
 * flags/goal_rows may be NULL (no relabelling).  aux (may be NULL unless FDQL_OPT_EMIT_LEARNER_AUX):
 *   aux_mask [T,n,1], aux_contig [T-1,n,1], aux_weight [T-1,n,1] = contig/((sum_t contig+1e-4)*batch*T). */
int fdql_sample_gather(const fdql_arena* a, int64_t n_windows, int32_t T, int64_t len, const int64_t* starts,
                       const uint8_t* flags, const int64_t* goal_rows, int32_t reward_op,
                       const float* reward_params_host, int32_t n_params, double gamma, uint32_t opts,
                       int32_t batch_for_weight, float* const* out, float* aux_mask, float* aux_contig,
                       float* aux_weight, void* stream);

/* test hook (returns the previous setting): bit 0 routes fdql_sample_gather / fdql_gather_rows through the
 * descriptor-walking kernel that serves rows wider than 128 float4; bit 1 makes the bitflip functor take the full-vector
 * relabel scan instead of the hash-assisted one; bit 2 makes the hash-assisted scan use the per-pass suffix scan for the
 * returns instead of the scan-free (Horner + one reduction) form; bit 3 routes plain and bitflip gathers through the
 * warp-per-window kernels instead of the tile kernel; bit 4: tile kernel without link records; bit 5: lean kernel wherever it can
 * serve; bits 6..10: probe switches of the gather role (probe builds, -DFDQL_PROBES, only); bit 11: fused pass without the T == 2
 * build; bit 12: without the compiled copy plan */
int fdql_debug_force_generic_gather(int on);

/* test hook (returns the previous setting): 1 routes the TQC / quantile-Huber losses through the warp-per-transition kernel
 * that serves more than 128 atoms instead of the quad kernel (4 lanes per transition) */
int fdql_debug_tqc_warp_kernel(int on);

/* Co-residency of the two hot kernels (returns the previous setting).  on != 0: the loss kernels (fdql_tqc_loss*, fdql_quantile_huber)
 * size their blocks so that every SM keeps room for one block of a gather launched with FDQL_OPT_CORESIDENT on another stream
 * (16 instead of 20 warps of the group kernel: 56 KB of shared memory and a quarter of the register file stay free). */
int fdql_set_coresident(int on);

/* DistributionalSoftActorCritic.q_loss from the MLP outputs onward + quantile_huber_loss_f, forward and backward
 * (franQ/Agent/components/distributional_soft_actor_critic.py:50-58,70,76-82,90-103): pool+sort the n_atoms target
 * atoms, keep the n_atoms-n_drop smallest, y = reward + mask*gamma*(z + alpha*(-log_pi)), quantile-Huber against
 * q_pred with tau over the concatenated atoms, + mean relu(mc_return - q_pred) when mc_return != NULL.
 *   next_z, q_pred, grad_q : [M, n_atoms]        next_log_pi (NULL = no entropy term), reward, mask, mc_return : [M]
 *   grad_scale : [M] or NULL; grad_q[m,:] = d loss[m] / d q_pred[m,:] * (grad_scale ? grad_scale[m] : 1)
 *   loss : [M];  td_target : [M, n_atoms-n_drop] or NULL;  stats : 4 doubles {sum q, sum row-var(ddof=1), #violations, M}
 *   accumulated (caller zeroes).  */
int fdql_tqc_loss(int64_t M, int32_t n_atoms, int32_t n_drop, const float* next_z, const float* q_pred,
                  const float* next_log_pi, const float* reward, const float* mask, const float* mc_return,
                  const float* grad_scale, float alpha, float gamma, float* loss, float* grad_q, float* td_target,
                  double* stats, void* stream);
/* same, with the entropy temperature read from device memory (alpha_dev[0]) at kernel time: for callers that keep
 * curr_alpha = exp(log_alpha) on the device (soft_actor_critic.py:151) and for CUDA-graph capture of the learner step */
int fdql_tqc_loss_dev_alpha(int64_t M, int32_t n_atoms, int32_t n_drop, const float* next_z, const float* q_pred,
                            const float* next_log_pi, const float* reward, const float* mask, const float* mc_return,
                            const float* grad_scale, const float* alpha_dev, float gamma, float* loss, float* grad_q,
                            float* td_target, double* stats, void* stream);

/* quantile_huber_loss_f(quantiles [M, n_quantiles], samples [M, n_samples]) -> loss [M] and d loss / d quantiles
 * (distributional_soft_actor_critic.py:90-103) for callers that built the target themselves. */
int fdql_quantile_huber(int64_t M, int32_t n_quantiles, int32_t n_samples, const float* quantiles, const float* samples,
                        const float* grad_scale, float* loss, float* grad_q, void* stream);

/* SoftActorCritic.q_loss, non-distributional variant (franQ/Agent/components/soft_actor_critic.py:63-99,134). */
int fdql_sac_min_target_loss(int64_t M, int32_t n_atoms, const float* target_z, const float* q_pred,
                             const float* next_log_pi, const float* reward, const float* mask, const float* mc_return,
                             const float* grad_scale, float alpha, float gamma, float* loss, float* grad_q,
                             double* stats, void* stream);

/* same, with the entropy temperature read from device memory (alpha_dev[0]) at kernel time: no host read of curr_alpha in the
 * learner step (soft_actor_critic.py:40,151 keeps it as a Python float), CUDA-graph capturable */
int fdql_sac_min_target_loss_dev_alpha(int64_t M, int32_t n_atoms, const float* target_z, const float* q_pred,
                                       const float* next_log_pi, const float* reward, const float* mask, const float* mc_return,
                                       const float* grad_scale, const float* alpha_dev, float gamma, float* loss, float* grad_q,
                                       double* stats, void* stream);

/* Host-buffer form of one whole pass (what a non-CUDA caller binds): streams and critic outputs come from host
 * memory (pinned for the copies to overlap), loss [ (T-1)*n ] and grad_q [ (T-1)*n, n_atoms ] go back to host memory;
 * the gathered batch stays in HBM in out[] for the device-side MLPs.  Transition m = t*n + b pairs row t (q_pred) with
 * row t+1 (reward, mask, mc_return: quirk Q10); grad_q is already scaled by the loss-reduce weight
 * contig/((sum_t contig+1e-4)*n*T) (deepQlearning.py:222-225,249).  Work is enqueued behind `stream` and joined back
 * into it; the host buffers may be reused once `stream` has been synchronised. */
int fdql_hotpath_step_host(fdql_arena* a, int64_t n_windows, int32_t T, int64_t len, const int64_t* starts_host,
                           const uint8_t* flags_host, const int64_t* goal_rows_host, int32_t reward_op,
                           const float* reward_params_host, int32_t n_params, double gamma, uint32_t opts,
                           float* const* out, int32_t n_atoms, int32_t n_drop, const float* next_z_host,
                           const float* q_pred_host, const float* next_log_pi_host, float alpha, float* loss_host,
                           float* grad_q_host, void* stream);

/* ---- prioritized experience replay: proportional PER with importance-sampling correction (Schaul, Quan, Antonoglou, Silver,
 *      "Prioritized Experience Replay", ICLR 2016).  NOT a reference mode: franQ draws every window start uniformly
 *      (replay_memory.py:59); this is an opt-in extension like FDQL_GOAL_FUTURE.
 *
 * A priority store belongs to one arena (at most one per arena; destroy it before the arena) and to one window length T.  It holds a
 * leaf q[r] = p_r^alpha (fp32) per ring row r, taken as a window start, under a 32-ary tree of fp64 sums and fp32 minima (4 + ~4/31 x
 * 12 bytes per row, plus a 4-byte claim slot per row for duplicate starts of an update: ~8.5 bytes per row, 85 MB at 1e7 rows).
 * Every node is recomputed from its children in one fixed order, never adjusted by atomics: the same call sequence gives the same tree
 * bits whatever the scheduling.
 *
 * Eligibility invariant: q[r] > 0 iff r < len - T, the start range of quirk Q2 (np.random.randint(0, len - T)).  A row gets q_max
 * (a device scalar: the running max of every leaf written, 1.0 at creation) when it is (over)written, or when it becomes eligible
 * because len grew.  The writers (fdql_arena_append and its host forms, fdql_arena_reserve and so fdql_her_flush_episodes /
 * fdql_q3_duplicate / vmap rows, fdql_arena_set_cursor) run on the writer's stream and only RECORD the rows they wrote on the host
 * side of the arena; every tree write happens on the stream of the PER calls (the reader's): the next fdql_per_sample or
 * fdql_per_update, or fdql_per_apply_pending, applies what was recorded.  While `stream` is being captured into a CUDA graph the
 * recorded rows are left for the next uncaptured call (a captured copy would re-apply them at every replay). */
typedef struct fdql_per fdql_per;

/* alpha >= 0 (priority exponent), eps > 0 (added to every |delta|), eta in [0, 1] (R2D2's max / mean mix over a window), T >= 2.
 * Rows already in the ring are activated at once. */
int fdql_per_create(fdql_arena* a, int32_t T, float alpha, float eps, float eta, fdql_per** out);
int fdql_per_destroy(fdql_per* per);
/* n windows drawn by priority, stratified: window b takes the target S (b + xi_b) / n, S the root sum, and descends to the leaf whose
 * prefix interval holds it (fp rounding past the last positive leaf is clamped to that leaf).  xi_b comes from Philox (b, counter, seed)
 * with the counter / counter_dev protocol of fdql_sample_streams (counter_dev[2] is not read: the tree holds the eligible range), or from
 * xi (device double[n] in [0, 1), may be NULL) for parity runs.  flags / goal_rows (may be NULL) follow fdql_sample_streams' hindsight
 * rules for the drawn start.  is_weight (may be NULL) [n] = (q_min / q[start])^beta with q_min the smallest positive leaf (Schaul's
 * (N P)^-beta / max w) and beta read from beta_dev[0] at kernel time (an annealed beta inside a captured graph).
 * FDQL_EOVERSAMPLE when len < 2T (under the invariant also the only case of S == 0). */
int fdql_per_sample(fdql_per* per, int64_t n, int32_t goal_mode, float relabel_prob, uint64_t seed, uint64_t counter,
                    uint64_t* counter_dev, const double* xi, const float* beta_dev, int64_t* starts, uint8_t* flags,
                    int64_t* goal_rows, float* is_weight, void* stream);
/* new priorities of n windows from the per-transition loss [T-1, n] of their transitions (a loss kernel's `loss`, m = t n + b) and the
 * gather's is_contiguous [T-1, n] (NULL: every transition counts): delta_b = eta max_t + (1 - eta) mean_t over the contiguous ones
 * (0 when none), q = (delta_b + eps)^alpha.  A non-finite loss or q writes q_max instead.  Duplicate starts: the largest b wins.
 * Leaves that are 0 (rows that are not eligible starts) stay 0. */
int fdql_per_update(fdql_per* per, int64_t n, const int64_t* starts, const float* loss, const float* contig, void* stream);
int fdql_per_apply_pending(fdql_per* per, void* stream);
/* the leaves [capacity] and q_max_dev[0] (device memory) for snapshots and tests; after writing leaves call fdql_per_rebuild */
int fdql_per_view(const fdql_per* per, float** leaves, float** q_max_dev);
/* node arrays of tree level `level` in [1, L] (level L is the root): fp64 sums and fp32 minima of positive leaves (+inf: none), n_nodes
 * of them; node i covers entries 32 i .. 32 i + 31 of the level below (level 0: the leaves).  A level past L fails with L in the
 * message.  For tests and tools. */
int fdql_per_level_view(const fdql_per* per, int32_t level, double** sums, float** mins, int64_t* n_nodes);
/* every node of the tree from the leaves */
int fdql_per_rebuild(fdql_per* per, void* stream);

/* fdql_fused_pass with prioritized starts, for the store `per` (T = per->T, the arena is per's): one call does one pass.
 *   Gather half, batch k+1 (arguments n_windows .. aux_weight, as fdql_fused_pass): the window starts are drawn from the priority tree
 *   by exactly fdql_per_sample's rules (stratified targets, xi from Philox (b, counter, seed) with the counter_dev protocol or injected,
 *   the clamp past the last positive leaf, flags / goal rows from the drawn start; counter_dev[2] is not read).  Window b covers rows
 *   start_b .. start_b + T - 1 (a drawn start is < len - T, so no window wraps; the ring's current length is not baked into the launch, and
 *   a captured pass keeps gathering the right rows while the ring grows).  It also writes is_weight [n] = (q_min / q[start])^beta with
 *   beta = beta_dev[0] (is_weight NULL: no weights, and beta_dev is not read and may be NULL) and critic_weight [T-1, n] =
 *   aux_weight * is_weight (may be NULL; needs FDQL_OPT_EMIT_LEARNER_AUX, aux_weight and is_weight).  aux_weight itself stays the uniform
 *   reduce weight: the actor and temperature losses take it unweighted.
 *   Loss half, batch k (arguments M .. stats, as fdql_fused_pass): pass batch k's critic_weight (written by the previous call) as
 *   grad_scale.  Then, in stream order after the launch that read the tree, the priorities of batch k as fdql_per_update computes them,
 *   from loss_starts (batch k's starts, written by the previous call), this call's per-transition loss and loss_contig (batch k's
 *   is_contiguous, may be NULL): M / (T - 1) windows.
 * M == 0: the gather alone, no update; n_windows == 0: the loss and the update alone.  Rows recorded by writers are applied first, on
 * `stream`, never under capture (as every PER call).
 * Staleness: the draw of batch j sees the priorities of batches <= j - 2 (batch j - 1's loss runs in the same call as batch j's draw):
 * the one-batch lag that any overlap of sampling with the loss implies.  Callers that need the priorities of batch j - 1 in draw j call
 * fdql_per_update before fdql_per_sample instead.
 * Double buffers: call k writes the gather outputs, starts, is_weight and critic_weight of batch k+1 while its loss reads those of batch
 * k, so each of them needs two sets, swapped every call.  Shapes the fused kernel does not serve run as fdql_per_sample, the co-resident
 * fdql_sample_gather on its streams, critic_weight, fdql_tqc_loss and the update, with identical results.
 * FDQL_EINVAL: NULL per, a loss half without loss_starts or loss, critic_weight without FDQL_OPT_EMIT_LEARNER_AUX; FDQL_EOVERSAMPLE as
 * fdql_per_sample. */
int fdql_fused_pass_per(fdql_per* per, int64_t n_windows, int32_t goal_mode, float relabel_prob, uint64_t seed, uint64_t counter,
                        uint64_t* counter_dev, const double* xi, const float* beta_dev, int64_t* starts, uint8_t* flags, int64_t* goal_rows,
                        float* is_weight, float* critic_weight, int32_t reward_op, const float* reward_params_host, int32_t n_params,
                        double gamma, uint32_t opts, int32_t batch_for_weight, float* const* out, float* aux_mask, float* aux_contig,
                        float* aux_weight, int64_t M, int32_t n_atoms, int32_t n_drop, const float* next_z, const float* q_pred,
                        const float* next_log_pi, const float* reward, const float* mask, const float* mc_return, const float* grad_scale,
                        float alpha, float loss_gamma, float* loss, float* grad_q, double* stats, const int64_t* loss_starts,
                        const float* loss_contig, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FDQL_H_ */
