// The "vmap" hindsight variant of the reference on the device (include/fdql.h: fdql_vmap_flush_episodes, fdql_vmap_select_column).
//   HindsightVmapWrite._hindsight_flush + _virtual_episode_calc   franQ/Replay/wrappers/her_vmap.py:30-43,66-88
//   NStepReturnVmap._flush + calculate_montecarlo_return/_inner   franQ/Replay/wrappers/nstep_return_vmap.py:37-48,61-74
//   HindsightVmapRead.temporal_sample / cleanup                    franQ/Replay/wrappers/her_vmap.py:104-123
// Storage follows the reference: every row carries V virtual goals plus its real goal ([V+1, G]) and the V+1 rewards, dones
// and returns-to-go it would have had under each of them; these are ordinary wide keys of the arena.  The reference fills them
// with a jax.vmap over goals on the host, row by row in Python; here one block per episode evaluates the L x (V+1) grid of
// reward functors in parallel and then runs the V+1 return recurrences (one thread each, exact reference arithmetic).
// At sample time the reference gathers all V+1 columns of every sampled row (2.5 KB per row at V = 32, G = 16) and keeps one;
// the select kernel reads only the chosen column (4 G + 12 bytes per row) and emits the learner aux from the selected dones.
#include "common.cuh"

namespace fdql {

struct VmapKeys {
  WideSlab goals, rewards, dones, returns;  // returns.base == nullptr: no virtual_mc_return key
  int32_t V, G;                             // virtual goals per row (the real goal is column V), goal width
};

// R(achieved_goal[row_a], goal) -> (reward, done), one thread, full vectors (the functors of goal_eval.cuh)
__device__ __forceinline__ void eval_row_thread(const RewardSpec& rs, const float* __restrict__ a, const float* __restrict__ g, int G,
                                                float& reward, bool& done) {
  if (rs.op == FDQL_REWARD_WEIGHTED_PNORM) {
    double acc = 0.0;
    for (int c = 0; c < G; ++c) acc += fabs((double)a[c] - (double)g[c]) * (double)rs.params[2 + c];
    const double r = -pow(acc, (double)rs.params[0]);
    reward = (float)r;
    done = r > -(double)rs.params[1];
    return;
  }
  bool ok = true;
  if (rs.op == FDQL_REWARD_BITFLIP) {
    for (int c = 0; c < G; ++c) ok &= a[c] == g[c];
  } else if (rs.op == FDQL_REWARD_ALL_GEQ) {
    for (int c = 0; c < G; ++c) ok &= a[c] >= g[c];
  } else {  // FDQL_REWARD_FIRST_GEQ
    ok = a[0] >= g[0];
  }
  reward = ok ? 0.f : -1.f;
  done = ok;
}

// mode bit 0: fill virtual_goals / virtual_rewards / virtual_dones (HindsightVmapWrite); bit 1: virtual_mc_return (NStepReturnVmap).
// Reward = RewardSpec evaluates R(ag, vg) and R(ag, dg) with the device functor; GivenReward loads them from the packed
// [n_rows, V+1] grid, whose column V holds R(ag, dg) (common.cuh).
template <class Reward>
__global__ void __launch_bounds__(128) vmap_flush_kernel(ArenaDev A, VmapKeys K, int32_t n_eps, const int64_t* __restrict__ ep_begin,
                                                        const int32_t* __restrict__ ep_len, const int64_t* __restrict__ pick_rows,
                                                        Reward rw, double gamma, int mode, int done_quirk) {
  constexpr bool given = kGivenReward<Reward>;
  const int ep = blockIdx.x;
  if (ep >= n_eps) return;
  const int64_t s = ep_begin[ep];
  const int L = ep_len[ep];
  const int V = K.V, G = K.G, C1 = V + 1;
  if (mode & 1) {
    int64_t p0 = 0;  // first packed row of this episode (GivenReward)
    if constexpr (given) p0 = packed_first_row(ep_len, ep);
    const WideSlab AG = A.wide[A.wide_ag], DG = A.wide[A.wide_dg];
    const int64_t* picks = pick_rows + (int64_t)ep * V;
    for (int item = threadIdx.x; item < L * C1; item += blockDim.x) {
      const int j = item / C1, v = item - j * C1;
      const int64_t row = ring_row(s, j, A.capacity);
      const float* ag = AG.base + row * (int64_t)AG.stride;
      const float* dg = DG.base + row * (int64_t)DG.stride;
      const float* rec = A.rec + row * (int64_t)A.rec_stride;
      const float r = rec[A.col_reward];
      const bool done = rec[A.col_task_done] != 0.f;
      float vr = r;
      bool vd = done;
      const float* goal = dg;  // column V: the real goal, reward and done (her_vmap.py:85-87)
      if (v < V) {
        goal = AG.base + picks[v] * (int64_t)AG.stride;
        float Rd, Rv;
        bool dd, dv;
        if constexpr (given) {
          const int64_t k = (p0 + j) * C1;
          Rd = rw.reward[k + V];
          dd = rw.done[k + V] != 0;
          Rv = rw.reward[k + v];
          dv = rw.done[k + v] != 0;
        } else {
          eval_row_thread(rw, ag, dg, G, Rd, dd);
          eval_row_thread(rw, ag, goal, G, Rv, dv);
        }
        vr = __fadd_rn(__fsub_rn(r, Rd), Rv);  // float32 like jax: (reward - desired_reward) + virtual_reward  (:34,39)
        vd = (done && !dd) || dv;              // (done and not desired_done) or virtual_done                 (:37,40)
      }
      K.rewards.base[row * (int64_t)K.rewards.stride + v] = vr;
      K.dones.base[row * (int64_t)K.dones.stride + v] = vd ? 1.f : 0.f;
      float* gout = K.goals.base + row * (int64_t)K.goals.stride + (int64_t)v * G;
      for (int c = 0; c < G; ++c) gout[c] = goal[c];
    }
    __syncthreads();
  }
  if ((mode & 2) && K.returns.base != nullptr) {
    // nstep_return_vmap.py:72-74, newest row first: G_j = fl32(r_j + G_{j+1} * gamma * m_j) in fp64, m_j = dones[j] as the
    // reference has it (quirk Q7, done_quirk != 0) or (1 - dones[j]) (returns stop at a virtual terminal)
    for (int v = threadIdx.x; v < C1; v += blockDim.x) {
      float acc = 0.f;
      for (int j = L - 1; j >= 0; --j) {
        const int64_t row = ring_row(s, j, A.capacity);
        const float r = K.rewards.base[row * (int64_t)K.rewards.stride + v];
        const bool d = K.dones.base[row * (int64_t)K.dones.stride + v] != 0.f;
        const double m = done_quirk ? (d ? 1.0 : 0.0) : (d ? 0.0 : 1.0);
        acc = j == L - 1 ? r : (float)__dadd_rn((double)r, __dmul_rn(__dmul_rn((double)acc, gamma), m));
        K.returns.base[row * (int64_t)K.returns.stride + v] = acc;
      }
    }
  }
}

// one column of the virtual keys for a [T, n] batch of windows + the learner aux from the selected dones
__global__ void __launch_bounds__(256) vmap_select_kernel(ArenaDev A, VmapKeys K, int64_t n, int32_t T, int64_t len,
                                                         const int64_t* __restrict__ starts, int32_t column, float* __restrict__ o_goal,
                                                         float* __restrict__ o_reward, float* __restrict__ o_done,
                                                         float* __restrict__ o_return, float* __restrict__ aux_mask,
                                                         float* __restrict__ aux_contig, float* __restrict__ aux_weight, float inv_bt) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const int G = K.G;
  if (o_goal != nullptr) {  // desired_goal[t, b, :] = virtual_goals[row, column, :]
    const int64_t items = (int64_t)T * n * G;
    for (int64_t i = tid; i < items; i += nthreads) {
      const int64_t tb = i / G;
      const int c = (int)(i - tb * G);
      const int64_t t = tb / n, b = tb - t * n;
      int64_t s = starts[b];
      if (s >= len) s %= len;
      const int64_t row = ring_row(s, t, len);
      o_goal[i] = __ldg(K.goals.base + row * (int64_t)K.goals.stride + (int64_t)column * G + c);
    }
  }
  for (int64_t b = tid; b < n; b += nthreads) {
    int64_t s = starts[b];
    if (s >= len) s %= len;
    float prev_step = 0.f, prev_mask = 0.f, csum = 0.f;
    for (int t = 0; t < T; ++t) {
      const int64_t row = ring_row(s, t, len);
      const float d = __ldg(K.dones.base + row * (int64_t)K.dones.stride + column);
      if (o_reward) o_reward[(int64_t)t * n + b] = __ldg(K.rewards.base + row * (int64_t)K.rewards.stride + column);
      if (o_done) o_done[(int64_t)t * n + b] = d;
      if (o_return && K.returns.base) o_return[(int64_t)t * n + b] = __ldg(K.returns.base + row * (int64_t)K.returns.stride + column);
      if (aux_mask || aux_contig || aux_weight) {
        // mask = !task_done (deepQlearning.py:201); is_contiguous[t-1] = (step[t]==step[t-1]+1) & mask[t-1] (:202-203)
        const float step = A.col_ep_step >= 0 ? __ldg(A.rec + row * (int64_t)A.rec_stride + A.col_ep_step) : 0.f;
        const float m = d != 0.f ? 0.f : 1.f;
        if (aux_mask) aux_mask[(int64_t)t * n + b] = m;
        if (t > 0) {
          const float c = (step == prev_step + 1.f && prev_mask != 0.f) ? 1.f : 0.f;
          csum += c;
          if (aux_contig) aux_contig[(int64_t)(t - 1) * n + b] = c;
          if (aux_weight) aux_weight[(int64_t)(t - 1) * n + b] = c;  // rescaled below
        }
        prev_step = step;
        prev_mask = m;
      }
    }
    if (aux_weight && T >= 2) {  // contig / ((sum_t contig + 1e-4) * B * T)  (deepQlearning.py:222-225,249)
      const float scale = inv_bt / (csum + 1e-4f);
      for (int t = 0; t < T - 1; ++t) aux_weight[(int64_t)t * n + b] *= scale;
    }
  }
}

// deepQlearning.py:206-210: action_onehot = eye(n)[action.long()] for every row of the [T, B, 1] action column
__global__ void __launch_bounds__(256) onehot_kernel(int64_t n_rows, int32_t n_actions, const float* __restrict__ action,
                                                    float* __restrict__ out, int32_t* __restrict__ bad) {
  const int64_t total = n_rows * n_actions;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / n_actions;
    const int c = (int)(i - r * n_actions);
    const int64_t a = (int64_t)__ldg(action + r);  // .long(): truncation towards zero
    if (c == 0 && (a < 0 || a >= n_actions) && bad != nullptr) atomicExch(bad, 1);
    st_stream1(out + i, a == c ? 1.f : 0.f);
  }
}

static int vmap_keys(const fdql_arena* a, int32_t key_goals, int32_t key_rewards, int32_t key_dones, int32_t key_returns, VmapKeys* out) {
  for (const int32_t key : {key_goals, key_rewards, key_dones, key_returns})
    FDQL_REQUIRE(key < 0 || key >= a->n_keys || a->key_narrow[key] < 0,
                 "key %d is stored as uint8 / int8: the virtual goal / reward / done / return keys must be fp32", key);
  auto slab = [&](int32_t key, WideSlab* w) -> bool {
    if (key < 0 || key >= a->n_keys || a->key_wide[key] < 0) return false;
    *w = a->dev.wide[a->key_wide[key]];
    return true;
  };
  memset(out, 0, sizeof(*out));
  FDQL_REQUIRE(slab(key_goals, &out->goals) && slab(key_rewards, &out->rewards) && slab(key_dones, &out->dones),
               "virtual_goals / virtual_rewards / virtual_dones must be keys of width >= 2 of this arena");
  if (key_returns >= 0) FDQL_REQUIRE(slab(key_returns, &out->returns), "virtual_mc_return must be a key of width >= 2 of this arena");
  const int C1 = out->rewards.width;
  FDQL_REQUIRE(C1 >= 2 && out->dones.width == C1 && (key_returns < 0 || out->returns.width == C1),
               "virtual_rewards / virtual_dones / virtual_mc_return must share one width V+1 >= 2");
  FDQL_REQUIRE(out->goals.width % C1 == 0, "virtual_goals width %d is not a multiple of V+1 = %d", out->goals.width, C1);
  out->V = C1 - 1;
  out->G = out->goals.width / C1;
  return FDQL_OK;
}

}  // namespace fdql

using namespace fdql;

extern "C" {

int fdql_action_onehot(int64_t n_rows, int32_t n_actions, const float* action, float* out, int32_t* out_of_range, void* stream) {
  FDQL_REQUIRE(n_rows >= 0 && n_actions >= 1, "bad sizes");
  if (n_rows == 0) return FDQL_OK;
  FDQL_REQUIRE(action != nullptr && out != nullptr, "null argument");
  int64_t blocks = (n_rows * n_actions + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  onehot_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(n_rows, n_actions, action, out, out_of_range);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int fdql_vmap_flush_episodes(fdql_arena* a, int32_t n_eps, const int64_t* ep_begin, const int32_t* ep_len, const int64_t* pick_rows,
                             int32_t key_goals, int32_t key_rewards, int32_t key_dones, int32_t key_returns, int32_t reward_op,
                             const float* reward_params_host, int32_t n_params, double gamma, int32_t mode, int32_t done_quirk,
                             void* stream) {
  FDQL_REQUIRE(a != nullptr && n_eps >= 0, "bad argument");
  if (n_eps == 0) return FDQL_OK;
  FDQL_REQUIRE(ep_begin != nullptr && ep_len != nullptr, "null episode table");
  FDQL_REQUIRE((mode & 3) != 0 && (mode & ~3) == 0, "mode: bit 0 = fill goals/rewards/dones, bit 1 = returns");
  VmapKeys K;
  int rc = vmap_keys(a, key_goals, key_rewards, key_dones, key_returns, &K);
  if (rc) return rc;
  RewardSpec rs;
  memset(&rs, 0, sizeof(rs));
  if (mode & 1) {
    FDQL_REQUIRE(pick_rows != nullptr, "the fill mode needs the rows whose achieved_goal become the virtual goals");
    FDQL_REQUIRE(a->dev.wide_ag >= 0 && a->dev.wide_dg >= 0 && a->dev.col_reward >= 0 && a->dev.col_task_done >= 0,
                 "the fill mode needs achieved_goal, desired_goal, reward and task_done keys");
    FDQL_REQUIRE(reward_op != FDQL_REWARD_NONE, "the fill mode needs a reward functor");
    FDQL_REQUIRE(a->dev.wide[a->dev.wide_ag].width == K.G && a->dev.wide[a->dev.wide_dg].width == K.G,
                 "goal width %d does not match virtual_goals (%d per goal)", a->dev.wide[a->dev.wide_ag].width, K.G);
    rc = upload_reward_spec(a, reward_op, reward_params_host, n_params, (cudaStream_t)stream, &rs);
    if (rc) return rc;
  }
  if (mode & 2) FDQL_REQUIRE(key_returns >= 0, "the returns mode needs a virtual_mc_return key");
  vmap_flush_kernel<RewardSpec><<<(unsigned)n_eps, 128, 0, (cudaStream_t)stream>>>(a->dev, K, n_eps, ep_begin, ep_len, pick_rows, rs,
                                                                                 gamma, mode, done_quirk);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int fdql_vmap_flush_episodes_given(fdql_arena* a, int32_t n_eps, const int64_t* ep_begin, const int32_t* ep_len,
                                   const int64_t* pick_rows, int32_t key_goals, int32_t key_rewards, int32_t key_dones,
                                   int32_t key_returns, int64_t n_rows, const float* reward, const uint8_t* done, double gamma,
                                   int32_t mode, int32_t done_quirk, void* stream) {
  FDQL_REQUIRE(a != nullptr && n_eps >= 0 && n_rows >= 0, "bad argument");
  FDQL_REQUIRE((mode & 1) != 0 && (mode & ~3) == 0, "mode: bit 0 (fill goals/rewards/dones from the given grid) must be set, bit 1 = returns");
  if (n_eps == 0) {
    FDQL_REQUIRE(n_rows == 0, "n_rows = %lld but there are no episodes", (long long)n_rows);
    return FDQL_OK;
  }
  FDQL_REQUIRE(ep_begin != nullptr && ep_len != nullptr, "null episode table");
  FDQL_REQUIRE(pick_rows != nullptr, "the fill mode needs the rows whose achieved_goal become the virtual goals");
  FDQL_REQUIRE(reward != nullptr && done != nullptr, "null reward or done grid");
  VmapKeys K;
  int rc = vmap_keys(a, key_goals, key_rewards, key_dones, key_returns, &K);
  if (rc) return rc;
  FDQL_REQUIRE(a->dev.wide_ag >= 0 && a->dev.wide_dg >= 0 && a->dev.col_reward >= 0 && a->dev.col_task_done >= 0,
               "the fill mode needs achieved_goal, desired_goal, reward and task_done keys");
  FDQL_REQUIRE(a->dev.wide[a->dev.wide_ag].width == K.G && a->dev.wide[a->dev.wide_dg].width == K.G,
               "goal width %d does not match virtual_goals (%d per goal)", a->dev.wide[a->dev.wide_ag].width, K.G);
  if (mode & 2) FDQL_REQUIRE(key_returns >= 0, "the returns mode needs a virtual_mc_return key");
  rc = check_packed_rows(a, n_eps, ep_len, n_rows, (cudaStream_t)stream);
  if (rc) return rc;
  const GivenReward g{reward, done, nullptr};
  vmap_flush_kernel<GivenReward><<<(unsigned)n_eps, 128, 0, (cudaStream_t)stream>>>(a->dev, K, n_eps, ep_begin, ep_len, pick_rows, g,
                                                                                  gamma, mode, done_quirk);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int fdql_vmap_select_column(const fdql_arena* a, int64_t n_windows, int32_t T, int64_t len, const int64_t* starts, int32_t column,
                            int32_t key_goals, int32_t key_rewards, int32_t key_dones, int32_t key_returns, int32_t batch_for_weight,
                            float* out_desired_goal, float* out_reward, float* out_task_done, float* out_mc_return, float* aux_mask,
                            float* aux_contig, float* aux_weight, void* stream) {
  FDQL_REQUIRE(a != nullptr && starts != nullptr, "null argument");
  FDQL_REQUIRE(T >= 1 && len >= T && len <= a->dev.capacity, "need 1 <= T <= len <= capacity (T=%d len=%lld)", T, (long long)len);
  if (n_windows <= 0) return n_windows == 0 ? FDQL_OK : FDQL_EINVAL;
  VmapKeys K;
  int rc = vmap_keys(a, key_goals, key_rewards, key_dones, key_returns, &K);
  if (rc) return rc;
  FDQL_REQUIRE(column >= 0 && column <= K.V, "column must be in [0, V] (V = the real goal), got %d", column);
  if (aux_contig || aux_weight) FDQL_REQUIRE(a->dev.col_ep_step >= 0, "is_contiguous needs an episode_step key");
  const float inv_bt = 1.f / ((float)(batch_for_weight > 0 ? batch_for_weight : (int32_t)n_windows) * (float)T);
  int64_t blocks = ((int64_t)T * n_windows * (out_desired_goal ? K.G : 1) + 255) / 256;
  const int64_t cap = (int64_t)a->num_sms * 16;
  if (blocks > cap) blocks = cap;
  vmap_select_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a->dev, K, n_windows, T, len, starts, column, out_desired_goal,
                                                                      out_reward, out_task_done, out_mc_return, aux_mask, aux_contig,
                                                                      aux_weight, inv_bt);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

}  // extern "C"
