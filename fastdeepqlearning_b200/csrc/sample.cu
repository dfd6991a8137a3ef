// Read side of the replay arena: index/goal stream sampling, row gather, and the fused
// window gather + sample-time hindsight relabel + return recompute.
//   ReplayMemory.sample / temporal_sample / __getitem__   franQ/Replay/replay_memory.py:48-70
//   TorchDataLoader fp32 cast                              franQ/Replay/wrappers/torch_dataloader.py:36
//   HindsightNStepReplay._hindsight_flush                  franQ/Replay/wrappers/her.py:55-95
//   calculate_montecarlo_return                            franQ/Replay/wrappers/nstep_return.py:60-72
//   DeepQLearning.get_losses mask / is_contiguous / reduce weights   franQ/Agent/deepQlearning.py:201-203,222-225,249
//
// One warp owns one sampled window.  Wide keys move as 128-bit vectors (a row of a key is a run of whole 32 B
// sectors, see common.cuh); the hindsight scan walks the contiguous tail of the window's episode in the
// achieved_goal slab, 32 rows per pass, and combines per-pass partial returns with a warp-shuffle scan.
#include "common.cuh"
#include "goal_eval.cuh"
#include "tqc_group.cuh"
#include "draw.cuh"

#include <atomic>

namespace fdql {

// a whole 8-float scalar record (one 32-byte sector) in ONE load instruction: a thread-per-window phase reads records of 32
// unrelated rows per warp instruction, so every separate column load costs the L1 another 32 sector look-ups
__device__ __forceinline__ void ld_rec8(const float* rec, float (&r)[8]) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7])
               : "l"(rec));
}
__device__ __forceinline__ float pick8(const float (&r)[8], int c) {  // r[c] for a run-time column without local memory
  float v = r[0];
#pragma unroll
  for (int k = 1; k < 8; ++k) v = c == k ? r[k] : v;
  return v;
}

// one window's streams: start ~ U[0, range), flag ~ Bernoulli(p) (never for rows of uncommitted episodes), goal row by mode
// (rec8: when given, the start row's scalar record is 8 floats wide and is returned whole for the caller's own use)
// record columns of the builds specialised on a window length (window_scalar_phase, TC > 0)
constexpr int kCanonReward = 0, kCanonTaskDone = 1, kCanonEpStep = 3, kCanonMcReturn = 4, kCanonScal = 5, kCanonEpStart = 5, kCanonEpEnd = 6;
// (PER: the start was drawn from the priority tree, per_descend_chunk; per_z / per_w are the last two words of the window's Philox draw)
template <int TC = 0, bool PER = false>
__device__ __forceinline__ void draw_window(const ArenaDev& A, int64_t b, int64_t range, int goal_mode, float relabel_prob, uint64_t seed,
                                            uint64_t counter, bool want_flags, int64_t& s, bool& f, int64_t& g, int& es, int& ee,
                                            float (*rec8)[8] = nullptr, int64_t per_s = 0, uint32_t per_z = 0, uint32_t per_w = 0) {
  uint4 x;
  if constexpr (PER) {
    x = make_uint4(0u, 0u, per_z, per_w);
    s = per_s;
  } else {
    x = philox4x32((uint64_t)b, counter, seed);
    const uint64_t r64 = ((uint64_t)x.x << 32) | x.y;
    s = (int64_t)__umul64hi(r64, (uint64_t)range);
  }
  f = false;
  g = s;
  es = -1;
  ee = -1;
  if (!want_flags) return;
  const float* rec = A.rec + s * (int64_t)A.rec_stride;
  if (rec8 != nullptr) {
    ld_rec8(rec, *rec8);
    es = __float_as_int(pick8(*rec8, TC > 0 ? kCanonEpStart : A.col_ep_start));
    ee = __float_as_int(pick8(*rec8, TC > 0 ? kCanonEpEnd : A.col_ep_end));
  } else {
    es = __float_as_int(__ldg(rec + A.col_ep_start));
    ee = __float_as_int(__ldg(rec + A.col_ep_end));
  }
  hindsight_pick(A.capacity, s, es, ee, x.z, x.w, goal_mode, relabel_prob, f, g);
}
// counter_dev[2] (optional, non-zero): the ring's current length, so that a captured launch keeps sampling the whole ring while it
// fills (the range len - T is otherwise baked into the launch)
__device__ __forceinline__ int64_t device_draw_range(const unsigned long long* counter_dev, int64_t range, int T) {
  if (counter_dev == nullptr) return range;
  const unsigned long long len = *reinterpret_cast<const volatile unsigned long long*>(counter_dev + 2);
  return len != 0ull ? (int64_t)len - T : range;
}
// starts ~ U[0, len-T) like np.random.randint(0, len-T, B) (replay_memory.py:59); flag ~ Bernoulli(p); goal row by mode
// over the committed extents of the start row's episode (her.py:48-53).  Uncommitted rows are never relabelled.
__global__ void __launch_bounds__(256)
sample_streams_kernel(ArenaDev A, int64_t n, int64_t range, int T, int goal_mode, float relabel_prob, uint64_t seed, uint64_t counter,
                      unsigned long long* counter_dev, int64_t* __restrict__ starts, uint8_t* __restrict__ flags,
                      int64_t* __restrict__ goal_rows) {
  counter = device_draw_counter(counter_dev, counter);
  range = device_draw_range(counter_dev, range, T);
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  int64_t s, g;
  bool f;
  int es, ee;
  draw_window(A, b, range, goal_mode, relabel_prob, seed, counter, flags != nullptr, s, f, g, es, ee);
  starts[b] = s;
  if (flags == nullptr) return;
  flags[b] = f ? 1 : 0;
  if (goal_rows) goal_rows[b] = g;
}

// ---- fused window gather -------------------------------------------------------------------------
struct GatherArgs {
  ArenaDev A;
  OutPtrs out;  // indexed by the caller's key
  const int64_t* starts;
  const uint8_t* flags;
  const int64_t* goal_rows;
  int64_t n;    // windows in the whole batch (row pitch of the time-major outputs)
  int64_t b_begin, b_end;  // slice of windows this launch handles
  int64_t len;  // modulus of the window indices (replay_memory.py:65)
  int32_t T;
  uint32_t opts;
  RewardSpec rs;
  double gamma;
  float inv_bt;  // 1 / (batch * T) for the reduce weights
  float* aux_mask;
  float* aux_contig;
  float* aux_weight;
  int32_t tile;  // tile kernel: windows per block iteration (32..256)
  // tile kernel, fused draw (draw_range > 0): the streams are drawn in the kernel exactly as sample_streams_kernel draws them
  int64_t draw_range;
  int32_t goal_mode;
  float relabel_prob;
  uint64_t seed, counter;
  unsigned long long* counter_dev;
  int64_t* starts_out;
  uint8_t* flags_out;
  int64_t* goal_out;
  int32_t dbg;       // probe switches of the lean kernel (1: no wide-key phase, 2: no scalar phase, 4: FMA loop for the scalar phase,
                     // 8: no cp.async fills, 16: no bulk write-back)
  int32_t use_link;  // tile kernel, equality rewards: link records are valid for this gamma -> O(hits) relabelled returns
  double log2_gamma, inv_gamma;
  // lean kernel: the wide keys that have an output, resolved on the host (at most kLeanMaxKeys; more take the tile kernel)
  struct LeanKey {
    const char* base;    // slab
    char* out;           // time-major output [T, n, 16 * vecs bytes]
    uint32_t stride;     // bytes between slab rows
    uint32_t vecs;       // float4 per row
    uint32_t stage_off;  // byte offset of the key inside a stage, in units of one stage window (x kLeanStageWindows in the kernel)
    int32_t is_dg;       // desired_goal: relabelled rows read the hindsight goal row's achieved_goal instead
  } lean_key[4];
  int32_t lean_nk;
  uint32_t lean_row_bytes;  // sum of 16 * vecs over the keys = bytes of one window row in a stage
  const char* lean_ag_base;
  uint32_t lean_ag_stride;
#ifdef FDQL_FUSED_ROLE_CLOCK
  unsigned long long* role_clock;
#endif
  int* lean_work_ctr;  // optional {next unclaimed chunk, blocks done}, zero at launch: chunks claimed across all blocks (see TqcArgs::work_ctr)
};
constexpr int kLeanMaxKeys = 4;

__device__ __forceinline__ double warp_suffix_scan(double v, double g, int lane) {
  // inclusive suffix scan of v with ratio g: out_l = sum_{m>=l} g^(m-l) v_m  (pairs (v, c) with c = g^(span))
  double c = g;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const double o = shfl_down_f64(v, d);
    if (lane + d < 32) v = fma(c, o, v);
    c = c * c;
  }
  return v;
}

template <int LPR, bool RELABEL>
__global__ void __launch_bounds__(256) sample_gather_kernel(const __grid_constant__ GatherArgs g) {
  extern __shared__ float smem[];
  const ArenaDev& A = g.A;
  const int lane = lane_id();
  const int wib = threadIdx.x >> 5;
  const int T = g.T;
  // per-warp scratch for the T window rows: relabelled reward, return, done flag, contiguity
  float* sm_r = smem + (size_t)wib * 4 * T;
  float* sm_g = sm_r + T;
  float* sm_d = sm_g + T;
  float* sm_c = sm_d + T;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t cap = A.capacity;
  const bool want_aux = (g.opts & FDQL_OPT_EMIT_LEARNER_AUX) != 0;

  for (int64_t b = g.b_begin + (int64_t)blockIdx.x * (blockDim.x >> 5) + wib; b < g.b_end; b += nwarps) {
    int64_t s = __ldg(g.starts + b);
    if (s >= g.len) s %= g.len;

    // ---- relabel set-up: episode extents of the start row, goal vector --------------------------
    bool relabel = false;
    int tail_last = -1;  // window-relative index of the episode's last row
    int64_t grow = 0, ep_first = 0;
    if (RELABEL) {
      if (g.flags != nullptr && __ldg(g.flags + b) != 0) {
        const float* rec = A.rec + s * (int64_t)A.rec_stride;
        const int es = __float_as_int(__ldg(rec + A.col_ep_start)), ee = __float_as_int(__ldg(rec + A.col_ep_end));
        if (es >= 0) {
          relabel = true;
          ep_first = es;
          tail_last = (int)(ee - s + (ee < s ? cap : 0));
          grow = __ldg(g.goal_rows + b);
        }
      }
    }

    // ---- wide keys: [T rows] x [vecs] float4 per key, time-major output -------------------------
    for (int w = 0; w < A.n_wide; ++w) {
      const WideSlab W = A.wide[w];
      float* __restrict__ o = g.out.p[W.key];
      if (o == nullptr) continue;
      const bool is_dg = RELABEL && relabel && w == A.wide_dg;
      const WideSlab S = is_dg ? A.wide[A.wide_ag] : W;
      const bool vec_store = (W.width & 3) == 0 && ((reinterpret_cast<uintptr_t>(o) & 15) == 0);
      const int items = T * W.vecs;
      for (int i = lane; i < items; i += 32) {
        const int t = i / W.vecs, v = i - t * W.vecs;
        int64_t row = s + t;
        if (row >= g.len) row -= g.len;
        const float* src = (is_dg && t <= tail_last) ? S.base + grow * (int64_t)S.stride : W.base + row * (int64_t)W.stride;
        const float4 x = ldg4(src + 4 * v);
        float* dst = o + ((int64_t)t * g.n + b) * W.width + 4 * v;
        if (vec_store) {
          st_stream4(dst, x);
        } else {
          const int m = min(4, W.width - 4 * v);
          const float xs[4] = {x.x, x.y, x.z, x.w};
          for (int c = 0; c < m; ++c) st_stream1(dst + c, xs[c]);
        }
      }
    }

    // ---- hindsight scan over the episode tail (her.py:62-69 + nstep_return.py:69-72, quirk Q5) ---
    int seg_first = -1;  // episode-relative index of the first row of the synthetic episode the window starts in; -1 unknown
    int j0 = 0;          // episode-relative index of the window's first row
    if (RELABEL && relabel) {
      const float4 gstar = load_goal_slice<LPR>(A, grow);
      double carry = 0.0;  // return of the first row after the chunk in flight
      const double gam = g.gamma;
      // gamma^(32-lane): weight of the carry for this lane's row
      double wcar = 1.0;
      {
        double p = gam;
        int e = 32 - lane;
        while (e) {  // <= 6 iterations
          if (e & 1) wcar *= p;
          p *= p;
          e >>= 1;
        }
      }
      for (int jb = (tail_last >> 5) << 5; jb >= 0; jb -= 32) {
        float Rg;
        bool dn;
        eval_chunk<LPR, false>(A, g.rs, s, jb, tail_last, gstar, Rg, dn);
        const int j = jb + lane;
        const bool valid = j <= tail_last;
        float rnew = 0.f;
        if (valid) rnew = (float)((double)__ldg(reinterpret_cast<const float*>(A.scan + ring_row(s, j, cap)) + 2) + (double)Rg);
        double G = warp_suffix_scan(valid ? (double)rnew : 0.0, gam, lane);
        G = fma(wcar, carry, G);
        carry = shfl_idx_f64(G, 0);
        if (valid && j < T) {
          sm_r[j] = rnew;
          sm_g[j] = (float)G;
          sm_d[j] = dn ? 1.f : 0.f;
        }
      }
      j0 = (int)(s - ep_first + (s < ep_first ? cap : 0));
      if (g.opts & FDQL_OPT_EXACT_EPISODE_STEP) {
        seg_first = 0;
        for (int jb = ((j0 - 1) >> 5) << 5; jb >= 0 && j0 > 0; jb -= 32) {
          float Rg;
          bool dn;
          eval_chunk<LPR, false>(A, g.rs, ep_first, jb, j0 - 1, gstar, Rg, dn);
          const unsigned bal = __ballot_sync(kFull, dn && (jb + lane) < j0);
          if (bal) {
            seg_first = jb + 32 - __clz(bal);
            break;
          }
        }
      }
      __syncwarp();
    }

    // ---- scalar record columns + learner aux, lane <-> window row ---------------------------------
    float contig_sum = 0.f;
    float carry_step = 0.f, carry_mask = 0.f;
    for (int tb = 0; tb < T; tb += 32) {
      const int t = tb + lane;
      const bool valid = t < T;
      int64_t row = s + (valid ? t : 0);
      if (row >= g.len) row -= g.len;
      const float* rec = A.rec + row * (int64_t)A.rec_stride;
      const bool in_ep = RELABEL && relabel && valid && t <= tail_last;
      float v_step = 0.f, v_done = 0.f;
      if (A.col_ep_step >= 0) v_step = __ldg(rec + A.col_ep_step);
      if (A.col_task_done >= 0) v_done = __ldg(rec + A.col_task_done);
      float v_rew = 0.f, v_ret = 0.f;
      if (RELABEL && relabel) {
        const bool dn = in_ep && sm_d[t] != 0.f;
        const unsigned bal = __ballot_sync(kFull, dn);
        if (in_ep) {
          v_rew = sm_r[t];
          v_ret = sm_g[t];
          v_done = dn ? 1.f : 0.f;
          const unsigned below = bal & ((1u << lane) - 1u);
          const int f = below ? (j0 + tb + 32 - __clz(below)) : seg_first;
          if (f >= 0 && A.col_ep_step >= 0)
            v_step = v_step - __ldg(A.rec + ring_row(ep_first, f, cap) * (int64_t)A.rec_stride + A.col_ep_step);
        }
        if (bal) seg_first = j0 + tb + 32 - __clz(bal);
      }
      if (valid) {
        for (int c = 0; c < A.n_scal; ++c) {
          float* o = g.out.p[A.scal_key[c]];
          if (o == nullptr) continue;
          float val;
          if (c == A.col_ep_step) val = v_step;
          else if (c == A.col_task_done) val = v_done;
          else if (in_ep && c == A.col_reward) val = v_rew;
          else if (in_ep && c == A.col_mc_return) val = v_ret;
          else val = __ldg(rec + c);
          st_stream1(o + (int64_t)t * g.n + b, val);
        }
      }
      if (want_aux) {
        // mask = !task_done (deepQlearning.py:201); is_contiguous[t] = (step[t+1]==step[t]+1) & mask[t] (:202-203)
        const float v_mask = v_done != 0.f ? 0.f : 1.f;
        if (valid && g.aux_mask) st_stream1(g.aux_mask + (int64_t)t * g.n + b, v_mask);
        const float nxt = __shfl_down_sync(kFull, v_step, 1);
        if (lane < 31 && t + 1 < T) {
          const float c = (nxt == v_step + 1.f && v_mask != 0.f) ? 1.f : 0.f;
          sm_c[t] = c;
          contig_sum += c;
        }
        const float first_step = __shfl_sync(kFull, v_step, 0);
        if (tb > 0 && lane == 0) {
          const float c = (first_step == carry_step + 1.f && carry_mask != 0.f) ? 1.f : 0.f;
          sm_c[tb - 1] = c;
          contig_sum += c;
        }
        carry_step = __shfl_sync(kFull, v_step, 31);
        carry_mask = __shfl_sync(kFull, v_mask, 31);
      }
    }
    if (want_aux) {
#pragma unroll
      for (int d = 16; d >= 1; d >>= 1) contig_sum += __shfl_xor_sync(kFull, contig_sum, d);
      __syncwarp();
      // upstream weight of q_loss[t,b] in the scalar loss: contig / ((sum_t contig + 1e-4) * B * T)  (deepQlearning.py:222-225,249)
      const float denom = contig_sum + 1e-4f;
      for (int t = lane; t < T - 1; t += 32) {
        const float c = sm_c[t];
        if (g.aux_contig) st_stream1(g.aux_contig + (int64_t)t * g.n + b, c);
        if (g.aux_weight) st_stream1(g.aux_weight + (int64_t)t * g.n + b, (c / denom) * g.inv_bt);
      }
    }
    __syncwarp();
  }
}

// =================================================================================================
// Fast path: every lane owns up to S fixed "row vectors" (one float4 of one key, or of the scalar record) and keeps the
// source / destination pointers for them in registers for the whole kernel, so a window row costs one 128-bit load and
// one 128-bit store per lane and no descriptor look-ups.  Used when a row has at most 32*S float4 (S <= 4).
//   MODE 0  plain gather
//   MODE 1  hindsight relabel, reward functor evaluated on the full goal vectors (any functor)
//   MODE 2  hindsight relabel for equality rewards (bitflip): the 16-byte scan records of the episode tail are read
//           128 rows at a time (4 independent 128-bit loads per lane), "differs" is decided by the stored 64-bit hash
//           and only hash matches are verified on the full vectors -> exact, at 16 B instead of 4*G+4 B per tail row.
// The loads of the first two window rows are issued before the relabel scan, so their latency hides behind it.
// =================================================================================================
// slot kind flags: how the lane's row vector is stored, and whether it is the desired_goal (replaced by the hindsight goal)
enum { SLOT_NONE = 0, SLOT_V4 = 1, SLOT_SCAL = 2, SLOT_PART = 4, SLOT_DG = 8 };
enum { RC_PLAIN = 0, RC_REWARD = 1, RC_TASK_DONE = 2, RC_EP_STEP = 3, RC_MC_RETURN = 4, RC_SKIP = 7 };

struct Slot {
  const float* src;  // slab base + 4*v
  float* dst;        // output base + 4*v (wide) or the scalar key's output
  uint32_t sstride;  // floats between rows of the slab
  uint32_t dwidth;   // floats between rows of the output
  uint32_t meta;     // kind flags | v << 4 | valid floats << 12
  uint32_t ovr;      // scalar columns with a role: shared-window address of the per-row override array | 1 if always applied
};

// `galt` (may be null): the hindsight goal row, read instead of the stored desired_goal by the lanes that own it
__device__ __forceinline__ float4 slot_load(const Slot& sl, int64_t row, const float* galt) {
  float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
  const float* p = sl.src + row * (int64_t)sl.sstride;
  if (galt != nullptr && (sl.meta & SLOT_DG)) p = galt + 4 * ((sl.meta >> 4) & 255u);
  if (sl.meta & SLOT_SCAL) x.x = __ldg(p);
  else if (sl.meta & (SLOT_V4 | SLOT_PART)) x = ldg4(p);
  return x;
}

__device__ __forceinline__ int ring_row32(int base, int off, int cap) {  // capacity < 2^31 (fdql_arena_create)
  const unsigned r = (unsigned)base + (unsigned)off;
  return (int)(r >= (unsigned)cap ? r - (unsigned)cap : r);
}

template <int S, int LPR, int MODE>
__global__ void __launch_bounds__(256, MODE == 1 ? 2 : 3) sample_gather_fast_kernel(const __grid_constant__ GatherArgs g) {
  constexpr bool RELABEL = MODE != 0;
  constexpr bool HASH = MODE >= 2;     // equality reward: 16-byte scan records + verified hash matches
  constexpr bool HORNER = MODE == 3;   // ... with the scan-free return recompute (host picks it when T <= 32 and gamma^-(T-1) is harmless)
  constexpr int HEAD = 2;  // window rows whose loads are issued ahead of the scan
  extern __shared__ float smem[];
  const ArenaDev& A = g.A;
  const int lane = lane_id();
  const int wib = threadIdx.x >> 5;
  const int T = g.T;
  // per-warp scratch, one entry per window row: relabelled reward, return, final task_done, final episode_step, contiguity
  float* sm_r = smem + (size_t)wib * 5 * T;
  float* sm_g = sm_r + T;
  float* sm_d = sm_g + T;
  float* sm_s = sm_d + T;
  float* sm_c = sm_s + T;
  const int64_t cap = A.capacity;
  const bool want_aux = (g.opts & FDQL_OPT_EMIT_LEARNER_AUX) != 0;

  // ---- the lane's plan -------------------------------------------------------------------------
  Slot slot[S];
#pragma unroll
  for (int k = 0; k < S; ++k) {
    int i = lane + 32 * k;
    Slot sl;
    sl.src = nullptr; sl.dst = nullptr; sl.sstride = 0; sl.dwidth = 0; sl.meta = SLOT_NONE; sl.ovr = 0;
    bool found = false;
    for (int w = 0; w < A.n_wide; ++w) {
      const int vecs = g.out.p[A.wide[w].key] != nullptr ? A.wide[w].vecs : 0;  // keys without an output take no lanes
      if (!found && i >= 0 && i < vecs) {
        found = true;
        float* o = g.out.p[A.wide[w].key];
        if (o != nullptr) {
          const int width = A.wide[w].width;
          const bool v4 = (width & 3) == 0 && ((reinterpret_cast<uintptr_t>(o) & 15) == 0);
          const bool dg = RELABEL && w == A.wide_dg;
          sl.src = A.wide[w].base + 4 * i;
          sl.dst = o + 4 * i;
          sl.sstride = A.wide[w].stride;
          sl.dwidth = width;
          sl.meta = (v4 ? SLOT_V4 : SLOT_PART) | (dg ? SLOT_DG : 0) | (i << 4) | (min(4, width - 4 * i) << 12);
        }
      }
      i -= vecs;
    }
    if (!found && i >= 0 && i < A.n_scal) {  // one lane per scalar column of the record: 4-byte load, 4-byte store
      float* o = g.out.p[A.scal_key[i]];
      if (o != nullptr) {
        sl.src = A.rec + i;
        sl.dst = o;
        sl.sstride = A.rec_stride;
        sl.dwidth = 1;
        sl.meta = SLOT_SCAL;
        if (RELABEL) {  // task_done / episode_step are final for every row of a relabelled window, reward / return inside the episode
          if (i == A.col_task_done) sl.ovr = (uint32_t)__cvta_generic_to_shared(sm_d) | 1u;
          if (i == A.col_ep_step) sl.ovr = (uint32_t)__cvta_generic_to_shared(sm_s) | 1u;
          if (i == A.col_reward) sl.ovr = (uint32_t)__cvta_generic_to_shared(sm_r);
          if (i == A.col_mc_return) sl.ovr = (uint32_t)__cvta_generic_to_shared(sm_g);
        }
      }
    }
    slot[k] = sl;
  }

  // gamma^(32-lane): weight of the carried return for this lane's row inside a 32-row pass
  double wcar = 1.0;
  if (RELABEL) {
    double p = g.gamma;
    int e = 32 - lane;
    while (e) {
      if (e & 1) wcar *= p;
      p *= p;
      e >>= 1;
    }
  }
  // MODE 2 return recompute without a scan per pass: every lane folds its rows j = lane, lane+32, ... with Horner in
  // gamma^32, one weighted warp reduction gives G_0, and G_j = gamma^-j (G_0 - sum_{i<j} gamma^i r'_i) for the window rows.
  // Used when the window fits one pass and gamma^-(T-1) is harmless in fp64; otherwise the per-pass suffix scan runs.
  double w_lane = 1.0, gamma32 = 1.0;
  if (HORNER) {
    double p = g.gamma;
    for (int e = lane; e; e >>= 1) {
      if (e & 1) w_lane *= p;
      p *= p;
    }
    double q = g.gamma;
    for (int e = 0; e < 5; ++e) q *= q;
    gamma32 = q;
  }
  const WideSlab AG = RELABEL ? A.wide[A.wide_ag] : A.wide[0];
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  const int cap32 = (int)A.capacity, len32 = (int)g.len;

  // ---- software pipeline over this warp's windows ------------------------------------------------------------------
  // While window i is processed, the stream entries of window i+2 and the episode extents of window i+1 are in flight,
  // and the rows / goal row / scan records of window i+1 are being pulled into L2 by prefetches, so that the loads of
  // the next iteration find their lines on chip instead of paying a dependent chain of DRAM round trips.
  struct Hdr {
    int32_t s, grow;
    bool flag;
  };
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t b_first = g.b_begin + (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
  auto load_hdr = [&](int64_t bi) {
    Hdr h;
    h.s = 0; h.grow = 0; h.flag = false;
    if (bi < g.b_end) {
      int64_t s64 = __ldg(g.starts + bi);
      if (s64 >= g.len) s64 %= g.len;
      h.s = (int32_t)s64;
      if (RELABEL) {
        h.flag = __ldg(g.flags + bi) != 0;
        h.grow = (int32_t)__ldg(g.goal_rows + bi);
      }
    }
    return h;
  };
  auto load_ext = [&](const Hdr& h, int& es_, int& ee_) {
    es_ = -1; ee_ = -1;
    if (RELABEL && h.flag) {
      const float* rec = A.rec + (int64_t)h.s * A.rec_stride;
      es_ = __float_as_int(__ldg(rec + A.col_ep_start));
      ee_ = __float_as_int(__ldg(rec + A.col_ep_end));
    }
  };
  auto prefetch_rows = [&](const Hdr& h) {
#pragma unroll
    for (int t = 0; t < HEAD; ++t) {
      const int row = ring_row32(h.s, t, len32);
#pragma unroll
      for (int k = 0; k < S; ++k)
        if (t < T && (slot[k].meta & 15u) != SLOT_NONE) prefetch_l2(slot[k].src + (int64_t)row * slot[k].sstride);
    }
    if (RELABEL && h.flag) {
      if (lane < AG.vecs) prefetch_l2(AG.base + (int64_t)h.grow * AG.stride + 4 * lane);
      if (HASH && lane == 0) prefetch_l2(A.scan + h.grow);
    }
  };
  auto prefetch_tail = [&](const Hdr& h, int es_, int ee_) {
    if (HASH && h.flag && es_ >= 0) {
      const int tl = ee_ - h.s + (ee_ < h.s ? cap32 : 0);
      for (int j = lane; j <= tl && j < 512; j += 32) prefetch_l2(A.scan + ring_row32(h.s, j, cap32));
    }
  };
  Hdr cur = load_hdr(b_first), nxt = load_hdr(b_first + nwarps);
  int es, ee, es_n = -1, ee_n = -1;
  load_ext(cur, es, ee);
  for (int64_t b = b_first; b < g.b_end; b += nwarps) {
    const Hdr nn = load_hdr(b + 2 * nwarps);
    load_ext(nxt, es_n, ee_n);
    prefetch_rows(nxt);
    const int s = cur.s, grow = cur.grow;
    const bool flag = cur.flag;

    bool relabel = false;
    int tail_last = -1;
    int ep_first = 0;
    if (RELABEL && flag && es >= 0) {
      relabel = true;
      ep_first = es;
      tail_last = ee - s + (ee < s ? cap32 : 0);
    }
    const float* galt = (RELABEL && relabel) ? AG.base + (int64_t)grow * AG.stride : nullptr;

    // ---- issue the loads of the head rows before the scan ------------------------------------------------------------
    float4 xh[HEAD][S];
#pragma unroll
    for (int t = 0; t < HEAD; ++t) {
      const int row = ring_row32(s, t, len32);
#pragma unroll
      for (int k = 0; k < S; ++k) {
        xh[t][k] = zero4;
        if (t < T) xh[t][k] = slot_load(slot[k], row, t <= tail_last ? galt : nullptr);
      }
    }

    // ---- hindsight scan over the episode tail (her.py:62-69 + nstep_return.py:69-72, quirk Q5) -----------------------
    int seg_first = -1, j0 = 0;
    if (RELABEL && relabel) {
      j0 = s - ep_first + (s < ep_first ? cap32 : 0);
      double carry = 0.0;
      if (HASH) {
        const float4 gsc = __ldg(A.scan + grow);
        const int gd = grow - s + (grow < s ? cap32 : 0);  // window-relative index of the goal row (may lie outside the tail)
        double acc = 0.0;  // Horner accumulator of this lane's rows
        for (int jb = (tail_last >> 7) << 7; jb >= 0; jb -= 128) {
          float4 r4[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int j = jb + 32 * u + lane;
            r4[u] = j <= tail_last ? __ldg(A.scan + ring_row32(s, j, cap32)) : zero4;
          }
#pragma unroll
          for (int u = 3; u >= 0; --u) {
            const int jbu = jb + 32 * u;
            if (jbu > tail_last) continue;
            const int j = jbu + lane;
            const bool valid = j <= tail_last;
            bool m = valid && __float_as_uint(r4[u].x) == __float_as_uint(gsc.x) && __float_as_uint(r4[u].y) == __float_as_uint(gsc.y);
            if (m) {  // hash match: the goal row itself is equal unless it holds a NaN; any other row is verified
              if (j == gd) m = (__float_as_uint(r4[u].w) & 1u) == 0u;
              else m = rows_equal(A, ring_row32(s, j, cap32), grow);
            }
            const float rnew = valid ? (float)((double)r4[u].z + (m ? 0.0 : -1.0)) : 0.f;
            if (HORNER) {
              acc = fma(acc, gamma32, (double)rnew);
              if (valid && j < T) {
                sm_r[j] = rnew;
                sm_d[j] = m ? 1.f : 0.f;
              }
            } else {
              double G = warp_suffix_scan((double)rnew, g.gamma, lane);
              G = fma(wcar, carry, G);
              carry = shfl_idx_f64(G, 0);
              if (valid && j < T) {
                sm_r[j] = rnew;
                sm_g[j] = (float)G;
                sm_d[j] = m ? 1.f : 0.f;
              }
            }
          }
        }
        if (HORNER) {
          // G_0 = sum_l gamma^l acc_l ; window row j: G_j = (G_0 - sum_{i<j} gamma^i r'_i) / gamma^j
          double tot = acc * w_lane;
#pragma unroll
          for (int d = 16; d >= 1; d >>= 1) tot += shfl_xor_f64(tot, d);
          __syncwarp();
          double pre = 0.0;  // exclusive prefix of gamma^i r'_i over the window rows
          if (T == 2) {
            pre = lane == 1 ? (double)sm_r[0] : 0.0;
          } else if (T > 2) {
            double v = (lane < T && lane <= tail_last) ? w_lane * (double)sm_r[lane] : 0.0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
              const double o = shfl_up_f64(v, d);
              if (lane >= d) v += o;
            }
            pre = shfl_up_f64(v, 1);
            if (lane == 0) pre = 0.0;
          }
          if (lane < T && lane <= tail_last) sm_g[lane] = (float)((tot - pre) / w_lane);
        }
        if (g.opts & FDQL_OPT_EXACT_EPISODE_STEP) {
          seg_first = 0;
          for (int jb = ((j0 - 1) >> 5) << 5; jb >= 0 && j0 > 0; jb -= 32) {
            const int j = jb + lane;
            const bool valid = j < j0;
            const int row = ring_row32(ep_first, valid ? j : 0, cap32);
            const float4 r = valid ? __ldg(A.scan + row) : zero4;
            bool m = valid && __float_as_uint(r.x) == __float_as_uint(gsc.x) && __float_as_uint(r.y) == __float_as_uint(gsc.y);
            if (m) {
              if (row == grow) m = (__float_as_uint(r.w) & 1u) == 0u;
              else m = rows_equal(A, row, grow);
            }
            const unsigned bal = __ballot_sync(kFull, m);
            if (bal) {
              seg_first = jb + 32 - __clz(bal);
              break;
            }
          }
        }
      } else {
        const float4 gstar = load_goal_slice<LPR>(A, grow);
        for (int jb = (tail_last >> 5) << 5; jb >= 0; jb -= 32) {
          float Rg;
          bool dn;
          eval_chunk<LPR, false>(A, g.rs, s, jb, tail_last, gstar, Rg, dn);
          const int j = jb + lane;
          const bool valid = j <= tail_last;
          float rnew = 0.f;
          if (valid) rnew = (float)((double)__ldg(reinterpret_cast<const float*>(A.scan + ring_row(s, j, cap)) + 2) + (double)Rg);
          double G = warp_suffix_scan(valid ? (double)rnew : 0.0, g.gamma, lane);
          G = fma(wcar, carry, G);
          carry = shfl_idx_f64(G, 0);
          if (valid && j < T) {
            sm_r[j] = rnew;
            sm_g[j] = (float)G;
            sm_d[j] = dn ? 1.f : 0.f;
          }
        }
        if (g.opts & FDQL_OPT_EXACT_EPISODE_STEP) {
          seg_first = 0;
          for (int jb = ((j0 - 1) >> 5) << 5; jb >= 0 && j0 > 0; jb -= 32) {
            float Rg;
            bool dn;
            eval_chunk<LPR, false>(A, g.rs, ep_first, jb, j0 - 1, gstar, Rg, dn);
            const unsigned bal = __ballot_sync(kFull, dn && (jb + lane) < j0);
            if (bal) {
              seg_first = jb + 32 - __clz(bal);
              break;
            }
          }
        }
      }
      __syncwarp();
    }

    // ---- lane <-> window row: final task_done / episode_step of every row, learner aux --------------------
    if ((RELABEL && relabel) || want_aux) {
      if (T <= 32) {  // the whole window fits one pass: no carries between passes, no staging of the contiguity bits
        const int t = lane;
        const bool valid = t < T;
        int64_t row = s + (valid ? t : 0);
        if (row >= g.len) row -= g.len;
        const float* rec = A.rec + row * (int64_t)A.rec_stride;
        float v_step = 0.f, v_done = 0.f;
        if (A.col_ep_step >= 0) v_step = __ldg(rec + A.col_ep_step);
        if (A.col_task_done >= 0) v_done = __ldg(rec + A.col_task_done);
        if (RELABEL && relabel) {
          const bool in_ep = valid && t <= tail_last;
          const bool dn = in_ep && sm_d[t] != 0.f;
          const unsigned bal = __ballot_sync(kFull, dn);
          if (in_ep) {
            v_done = dn ? 1.f : 0.f;
            const unsigned below = bal & ((1u << lane) - 1u);
            const int f = below ? (j0 + 32 - __clz(below)) : seg_first;
            if (f >= 0 && A.col_ep_step >= 0)
              v_step = v_step - __ldg(A.rec + ring_row(ep_first, f, cap) * (int64_t)A.rec_stride + A.col_ep_step);
          }
          if (valid) {
            sm_d[t] = v_done;
            sm_s[t] = v_step;
          }
        }
        if (want_aux) {
          const float v_mask = v_done != 0.f ? 0.f : 1.f;
          if (valid && g.aux_mask) st_stream1(g.aux_mask + (int64_t)t * g.n + b, v_mask);
          const float nxt = __shfl_down_sync(kFull, v_step, 1);
          const float c = (t + 1 < T && nxt == v_step + 1.f && v_mask != 0.f) ? 1.f : 0.f;
          float csum = c;
#pragma unroll
          for (int d = 16; d >= 1; d >>= 1) csum += __shfl_xor_sync(kFull, csum, d);
          if (t + 1 < T) {
            if (g.aux_contig) st_stream1(g.aux_contig + (int64_t)t * g.n + b, c);
            if (g.aux_weight) st_stream1(g.aux_weight + (int64_t)t * g.n + b, (c / (csum + 1e-4f)) * g.inv_bt);
          }
        }
        __syncwarp();
      } else {
      float contig_sum = 0.f, carry_step = 0.f, carry_mask = 0.f;
      for (int tb = 0; tb < T; tb += 32) {
        const int t = tb + lane;
        const bool valid = t < T;
        int64_t row = s + (valid ? t : 0);
        if (row >= g.len) row -= g.len;
        const float* rec = A.rec + row * (int64_t)A.rec_stride;
        float v_step = 0.f, v_done = 0.f;
        if (A.col_ep_step >= 0) v_step = __ldg(rec + A.col_ep_step);
        if (A.col_task_done >= 0) v_done = __ldg(rec + A.col_task_done);
        if (RELABEL && relabel) {
          const bool in_ep = valid && t <= tail_last;
          const bool dn = in_ep && sm_d[t] != 0.f;
          const unsigned bal = __ballot_sync(kFull, dn);
          if (in_ep) {
            v_done = dn ? 1.f : 0.f;
            const unsigned below = bal & ((1u << lane) - 1u);
            const int f = below ? (j0 + tb + 32 - __clz(below)) : seg_first;
            if (f >= 0 && A.col_ep_step >= 0)
              v_step = v_step - __ldg(A.rec + ring_row(ep_first, f, cap) * (int64_t)A.rec_stride + A.col_ep_step);
          }
          if (bal) seg_first = j0 + tb + 32 - __clz(bal);
          if (valid) {
            sm_d[t] = v_done;
            sm_s[t] = v_step;
          }
        }
        if (want_aux) {
          // mask = !task_done (deepQlearning.py:201); is_contiguous[t] = (step[t+1]==step[t]+1) & mask[t] (:202-203)
          const float v_mask = v_done != 0.f ? 0.f : 1.f;
          if (valid && g.aux_mask) st_stream1(g.aux_mask + (int64_t)t * g.n + b, v_mask);
          const float nxt = __shfl_down_sync(kFull, v_step, 1);
          if (lane < 31 && t + 1 < T) {
            const float c = (nxt == v_step + 1.f && v_mask != 0.f) ? 1.f : 0.f;
            sm_c[t] = c;
            contig_sum += c;
          }
          const float first_step = __shfl_sync(kFull, v_step, 0);
          if (tb > 0 && lane == 0) {
            const float c = (first_step == carry_step + 1.f && carry_mask != 0.f) ? 1.f : 0.f;
            sm_c[tb - 1] = c;
            contig_sum += c;
          }
          carry_step = __shfl_sync(kFull, v_step, 31);
          carry_mask = __shfl_sync(kFull, v_mask, 31);
        }
      }
      if (want_aux) {
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) contig_sum += __shfl_xor_sync(kFull, contig_sum, d);
        __syncwarp();
        // upstream weight of q_loss[t,b]: contig / ((sum_t contig + 1e-4) * B * T)  (deepQlearning.py:222-225,249)
        const float denom = contig_sum + 1e-4f;
        for (int t = lane; t < T - 1; t += 32) {
          const float c = sm_c[t];
          if (g.aux_contig) st_stream1(g.aux_contig + (int64_t)t * g.n + b, c);
          if (g.aux_weight) st_stream1(g.aux_weight + (int64_t)t * g.n + b, (c / denom) * g.inv_bt);
        }
      }
      __syncwarp();
      }
    }

    // ---- the rows: one 128-bit load + store per lane and slot -----------------------------------------------
    auto emit = [&](int t, const float4 (&x)[S]) {
      const bool in_ep = RELABEL && relabel && t <= tail_last;
      const int64_t orow = (int64_t)t * g.n + b;
#pragma unroll
      for (int k = 0; k < S; ++k) {
        const uint32_t meta = slot[k].meta;
        if (meta & SLOT_V4) st_stream4(slot[k].dst + orow * slot[k].dwidth, x[k]);
        if (meta & SLOT_SCAL) {
          float val = x[k].x;
          const uint32_t ovr = slot[k].ovr;
          if (RELABEL && relabel && ovr != 0u && ((ovr & 1u) || in_ep)) val = lds_f32((ovr & ~3u) + 4u * (uint32_t)t);
          st_stream1(slot[k].dst + orow, val);
        }
        if (meta & SLOT_PART) {
          const int m = (meta >> 12) & 15u;
          const float xs[4] = {x[k].x, x[k].y, x[k].z, x[k].w};
          float* dst = slot[k].dst + orow * slot[k].dwidth;
          for (int c = 0; c < m; ++c) st_stream1(dst + c, xs[c]);
        }
      }
    };
#pragma unroll
    for (int t = 0; t < HEAD; ++t)
      if (t < T) emit(t, xh[t]);
    for (int t = HEAD; t < T; ++t) {
      int64_t row = s + t;
      if (row >= g.len) row -= g.len;
      float4 x[S];
#pragma unroll
      for (int k = 0; k < S; ++k) x[k] = slot_load(slot[k], row, t <= tail_last ? galt : nullptr);
      emit(t, x);
    }
    prefetch_tail(nxt, es_n, ee_n);
    cur = nxt;
    es = es_n;
    ee = ee_n;
    nxt = nn;
    __syncwarp();
  }
}

// probe switches (GatherArgs.dbg) exist only in probe builds (profiles/build_variant.sh ... -DFDQL_PROBES): dead branches inside the
// hot loops cost instruction-cache lines even when they are never taken
#ifdef FDQL_PROBES
#define FDQL_DBG(g) ((g).dbg)
#else
#define FDQL_DBG(g) 0
#endif
constexpr int kTileWindows = 256;
#ifndef TILE_MINB
#define TILE_MINB 4
#endif
#ifndef TAIL_UNROLL
#define TAIL_UNROLL 4
#endif
#ifndef WIN_UNROLL
#define WIN_UNROLL 2
#endif

// Phase 1 of the tile / lean kernels for ONE window (one thread): everything scalar -- index / goal streams (drawn here when DRAW),
// episode extents, hindsight reward / task_done / episode_step, the relabelled return, every scalar key and the learner aux are
// written to the time-major outputs; returns what the wide-key phase needs (start row, goal row, last in-episode window row or -1).
// the hindsight predicate of one tail row: R(ag_j, g*) == 0  <=>  achieved_goal[row] == achieved_goal[goal_row]; `gsc` = scan record of
// the goal row, `gd` = its offset from the window start.  A hash match is verified on the full vectors, except for the goal row
// itself, which is equal unless it holds a NaN.
__device__ __forceinline__ bool scan_matches(const ArenaDev& A, int s, int grow, int cap32, const float4& gsc, int gd, int j, const float4& r) {
  bool m = __float_as_uint(r.x) == __float_as_uint(gsc.x) && __float_as_uint(r.y) == __float_as_uint(gsc.y);
  if (m) {
    if (j == gd) m = (__float_as_uint(r.w) & 1u) == 0u;
    else m = rows_equal(A, ring_row32(s, j, cap32), grow);
  }
  return m;
}
// The tail-scan form of the relabelled return for ONE window (one thread): return-to-go over the whole real episode with relabelled
// rewards (quirk Q5), newest row first, each step in fp64 and rounded to fp32 on store exactly like nstep_return.py:69-72; rows inside
// the window are written to `o_ret`.  Returns the first row of the synthetic episode the window starts in (exact mode scans the
// episode prefix, her.py:72-83), or -1.
__device__ __forceinline__ int tail_scan_window(const GatherArgs& g, int s, int grow, int tail_last, int ep_first, int j0, int T,
                                                float* o_ret, int64_t b, float4& gsc, int& gd) {
  const ArenaDev& A = g.A;
  const int cap32 = (int)A.capacity;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  gsc = __ldg(A.scan + grow);
  gd = grow - s + (grow < s ? cap32 : 0);
  float acc = 0.f;
  bool first = true;
  constexpr int UR = TAIL_UNROLL;  // scan records in flight per thread (per-thread L2 prefetches were measured slower)
  for (int jt = tail_last; jt >= 0; jt -= UR) {
    float4 r4[UR];
#pragma unroll
    for (int u = 0; u < UR; ++u) r4[u] = jt - u >= 0 ? __ldg(A.scan + ring_row32(s, jt - u, cap32)) : zero4;
#pragma unroll
    for (int u = 0; u < UR; ++u) {
      const int j = jt - u;
      if (j < 0) break;
      const bool m = scan_matches(A, s, grow, cap32, gsc, gd, j, r4[u]);
      const float rnew = (float)((double)r4[u].z + (m ? 0.0 : -1.0));
      acc = first ? rnew : (float)__dadd_rn((double)rnew, __dmul_rn((double)acc, g.gamma));
      first = false;
      if (j < T && o_ret != nullptr) st_stream1(o_ret + (int64_t)j * g.n + b, acc);
    }
  }
  int seg_first = -1;
  if (g.opts & FDQL_OPT_EXACT_EPISODE_STEP) {
    seg_first = 0;
    for (int j = j0 - 1; j >= 0; --j) {
      const int row = ring_row32(ep_first, j, cap32);
      const float4 r = __ldg(A.scan + row);
      bool m = __float_as_uint(r.x) == __float_as_uint(gsc.x) && __float_as_uint(r.y) == __float_as_uint(gsc.y);
      if (m) {
        if (row == grow) m = (__float_as_uint(r.w) & 1u) == 0u;
        else m = rows_equal(A, row, grow);
      }
      if (m) {
        seg_first = j + 1;
        break;
      }
    }
  }
  return seg_first;
}
// The same two steps as calls, for the kernels specialised on a window length (TC > 0: link records serve every window except those of
// episodes without a chain -- longer than 32767 rows --, so the scan is cold code there and stays out of the hot loop's instruction
// stream; the goal row's scan record is simply fetched again per row).
__device__ __noinline__ int tail_scan_window_cold(const GatherArgs& g, int s, int grow, int tail_last, int ep_first, int j0, int T,
                                                  float* o_ret, int64_t b) {
  float4 gsc;
  int gd;
  return tail_scan_window(g, s, grow, tail_last, ep_first, j0, T, o_ret, b, gsc, gd);
}
__device__ __noinline__ bool scan_row_matches_cold(const GatherArgs& g, int s, int grow, int t) {
  const ArenaDev& A = g.A;
  const int cap32 = (int)A.capacity;
  const float4 gsc = __ldg(A.scan + grow);
  const int gd = grow - s + (grow < s ? cap32 : 0);
  return scan_matches(A, s, grow, cap32, gsc, gd, t, __ldg(A.scan + ring_row32(s, t, cap32)));
}

// TC > 0: the window length is the compile-time constant TC, scalar records are 8 floats and the link records are valid (the launcher
// checks all three); TC = 0: everything at run time.  PER (with DRAW): the start per_s comes from the priority tree (per_descend_chunk),
// the hindsight streams from per_z / per_w, and the importance weight and the critic weight are written through `pd`.
template <bool HASH, bool DRAW, int TC = 0, bool PER = false>
__device__ __forceinline__ void window_scalar_phase(const GatherArgs& g, int64_t b, uint64_t draw_ctr, int& s_out, int& grow_out,
                                                    int& tail_out, const PerDraw* pd = nullptr, int per_s = 0, uint32_t per_z = 0,
                                                    uint32_t per_w = 0) {
  const ArenaDev& A = g.A;
  const int T = TC > 0 ? TC : g.T;
  const int cap32 = (int)A.capacity, len32 = (int)g.len;
  const bool want_aux = (g.opts & FDQL_OPT_EMIT_LEARNER_AUX) != 0;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  int64_t s64;
  bool relabel = false;
  int tail_last = -1, ep_first = 0, grow = 0;
  // 8-float scalar records (<= 6 scalar keys + the two extents) travel whole, one 256-bit load per row
  const bool vec8 = TC > 0 ? true : A.rec_stride == 8;
  // TC > 0 also fixes the record columns (the launcher checks them): the reference's transition keys in their usual order
  // {reward, task_done, episode_done, episode_step, mc_return} followed by the two episode extents -- the column picks out of the
  // 8-float record and the per-key stores then need no select chains
  const int n_scal = TC > 0 ? kCanonScal : A.n_scal;
  const int col_reward = TC > 0 ? kCanonReward : A.col_reward, col_task_done = TC > 0 ? kCanonTaskDone : A.col_task_done;
  const int col_ep_step = TC > 0 ? kCanonEpStep : A.col_ep_step, col_mc_return = TC > 0 ? kCanonMcReturn : A.col_mc_return;
  float rv0[8];
  bool have0 = false;
  if (DRAW) {  // fused draw: same generator, same streams as sample_streams_kernel
    int64_t g64;
    bool f;
    int es, ee;
    have0 = HASH && vec8;
    if constexpr (PER)  // (counter_dev[2] is not read: the tree holds the eligible range)
      draw_window<TC, true>(A, b, 0, g.goal_mode, g.relabel_prob, g.seed, draw_ctr, HASH, s64, f, g64, es, ee, have0 ? &rv0 : nullptr, per_s,
                            per_z, per_w);
    else
      draw_window<TC>(A, b, device_draw_range(g.counter_dev, g.draw_range, T), g.goal_mode, g.relabel_prob, g.seed, draw_ctr, HASH, s64, f, g64,
                      es, ee, have0 ? &rv0 : nullptr);
    if (g.starts_out) g.starts_out[b] = s64;
    if (g.flags_out) g.flags_out[b] = f ? 1 : 0;
    if (g.goal_out) g.goal_out[b] = g64;
    if (HASH && f) {
      relabel = true;
      ep_first = es;
      tail_last = ee - (int)s64 + (ee < (int)s64 ? cap32 : 0);
      grow = (int)g64;
    }
  } else {
    s64 = __ldg(g.starts + b);
    if (s64 >= g.len) s64 %= g.len;
    if (HASH && g.flags != nullptr && __ldg(g.flags + b) != 0) {
      const float* rec = A.rec + s64 * A.rec_stride;
      const int es = __float_as_int(__ldg(rec + A.col_ep_start)), ee = __float_as_int(__ldg(rec + A.col_ep_end));
      if (es >= 0) {
        relabel = true;
        ep_first = es;
        tail_last = ee - (int)s64 + (ee < (int)s64 ? cap32 : 0);
        grow = (int)__ldg(g.goal_rows + b);
      }
    }
  }
  const int s = (int)s64;
  s_out = s;
  grow_out = grow;
  tail_out = tail_last;
  float* o_ret = col_mc_return >= 0 ? g.out.p[A.scal_key[col_mc_return]] : nullptr;

  float4 gsc = zero4;
  int gd = -1;
  // ---- link path (common.cuh): the rows that hit g* are the chain of bit-identical achieved goals through the goal row, so
  // the relabelled return of window row t is GA_t + sum_{hits m >= t} gamma^(m-t); nothing is read from the rest of the tail
  bool linked = false;
  uint64_t inwin = 0;  // bit t: window row t hits the goal (link records serve windows of up to 64 rows)
  double W = 0.0;      // sum over the hits m >= 0 (relative to the window start) of gamma^m
  int seg_first = -1;  // first row of the synthetic episode the window starts in, episode-relative (exact mode)
  int j0 = 0;
  if (HASH && relabel) j0 = s - ep_first + (s < ep_first ? cap32 : 0);
  if (HASH && relabel && (TC > 0 || g.use_link)) {
    const int jg = grow - ep_first + (grow < ep_first ? cap32 : 0);
    const float4 lg = __ldg(A.link + grow);
    const int pk = __float_as_int(lg.z);
    if (pk >= 0 && jg <= j0 + tail_last) {  // a chain exists and the goal row belongs to this episode
      linked = true;
      int near_before = -0x40000000;
      if (((pk >> 30) & 1) == 0) {  // a goal holding a NaN is hit by nothing, not even by its own row
        auto visit = [&](int m) {
          if (m >= 0) {
            W += exp2((double)m * g.log2_gamma);
            if (m < T) inwin |= 1ull << m;
          } else {
            near_before = max(near_before, m);
          }
        };
        const int mg = jg - j0;
        visit(mg);
        if (mg >= 0) {  // towards the window start; the first hit before it ends the walk
          int cur = mg, d = __float_as_int(lg.w);
          while (d > 0) {
            cur -= d;
            visit(cur);
            if (cur < 0) break;
            d = __float_as_int(__ldg(A.link + ring_row32(ep_first, j0 + cur, cap32)).w);
          }
        }
        int cur = mg, d = pk & 0x7fff;
        while (d > 0) {  // towards the episode end
          cur += d;
          visit(cur);
          d = __float_as_int(__ldg(A.link + ring_row32(ep_first, j0 + cur, cap32)).z) & 0x7fff;
        }
      }
      if (g.opts & FDQL_OPT_EXACT_EPISODE_STEP) seg_first = near_before < 0 && near_before > -0x40000000 ? j0 + near_before + 1 : 0;
    }
  }
  if (HASH && relabel && !linked) {
    if constexpr (TC > 0) seg_first = tail_scan_window_cold(g, s, grow, tail_last, ep_first, j0, T, o_ret, b);
    else seg_first = tail_scan_window(g, s, grow, tail_last, ep_first, j0, T, o_ret, b, gsc, gd);
  }
  double gp = 1.0, gi = 1.0, Wsub = 0.0;  // gamma^t, gamma^-t, hits before window row t
  // forward over the window rows: scalar keys (with the hindsight overrides) and the learner aux
  float prev_step = 0.f, prev_mask = 0.f, csum = 0.f;
  for (int t = 0; t < T; ++t) {
    const int row = ring_row32(s, t, len32);
    const float* rec = A.rec + (int64_t)row * A.rec_stride;
    const bool in_ep = HASH && relabel && t <= tail_last;
    float rv[8];
    if (vec8) {
      if (t == 0 && have0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) rv[k] = rv0[k];
      } else {
        ld_rec8(rec, rv);
      }
    }
    float v_step = col_ep_step >= 0 ? (vec8 ? pick8(rv, col_ep_step) : __ldg(rec + col_ep_step)) : 0.f;
    float v_done = col_task_done >= 0 ? (vec8 ? pick8(rv, col_task_done) : __ldg(rec + col_task_done)) : 0.f;
    float v_rew = 0.f;
    if (in_ep) {
      bool m;
      if (linked) {
        const float4 lt = __ldg(A.link + ring_row32(s, t, cap32));
        m = ((inwin >> t) & 1ull) != 0ull;
        v_rew = (float)((double)lt.y + (m ? 0.0 : -1.0));
        if (o_ret != nullptr) st_stream1(o_ret + (int64_t)t * g.n + b, (float)((double)lt.x + gi * (W - Wsub)));
        if (m) Wsub += gp;
        gp *= g.gamma;
        gi *= g.inv_gamma;
      } else if constexpr (TC > 0) {  // (cold: see tail_scan_window_cold; the link record carries the same goal-agnostic reward)
        m = scan_row_matches_cold(g, s, grow, t);
        v_rew = (float)((double)__ldg(A.link + ring_row32(s, t, cap32)).y + (m ? 0.0 : -1.0));
      } else {
        const float4 r = __ldg(A.scan + ring_row32(s, t, cap32));
        m = scan_matches(A, s, grow, cap32, gsc, gd, t, r);
        v_rew = (float)((double)r.z + (m ? 0.0 : -1.0));
      }
      v_done = m ? 1.f : 0.f;
      if (seg_first >= 0 && col_ep_step >= 0)
        v_step -= __ldg(A.rec + (int64_t)ring_row32(ep_first, seg_first, cap32) * A.rec_stride + col_ep_step);
      if (m) seg_first = j0 + t + 1;
    }
    if (vec8) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        if (c >= n_scal) break;
        float* o = g.out.p[A.scal_key[c]];
        if (o == nullptr) continue;
        float val;
        if (c == col_ep_step) val = v_step;
        else if (c == col_task_done) val = v_done;
        else if (in_ep && c == col_reward) val = v_rew;
        else if (in_ep && c == col_mc_return) continue;  // written by the return recurrence above
        else val = rv[c];
        st_stream1(o + (int64_t)t * g.n + b, val);
      }
    } else {
      for (int c = 0; c < n_scal; ++c) {
        float* o = g.out.p[A.scal_key[c]];
        if (o == nullptr) continue;
        float val;
        if (c == col_ep_step) val = v_step;
        else if (c == col_task_done) val = v_done;
        else if (in_ep && c == col_reward) val = v_rew;
        else if (in_ep && c == col_mc_return) continue;  // written by the return recurrence above
        else val = __ldg(rec + c);
        st_stream1(o + (int64_t)t * g.n + b, val);
      }
    }
    if (want_aux) {
      // mask = !task_done (deepQlearning.py:201); is_contiguous[t-1] = (step[t]==step[t-1]+1) & mask[t-1] (:202-203)
      const float v_mask = v_done != 0.f ? 0.f : 1.f;
      if (g.aux_mask) st_stream1(g.aux_mask + (int64_t)t * g.n + b, v_mask);
      if (t > 0) {
        const float c = (v_step == prev_step + 1.f && prev_mask != 0.f) ? 1.f : 0.f;
        csum += c;
        if (g.aux_contig) st_stream1(g.aux_contig + (int64_t)(t - 1) * g.n + b, c);
        if (g.aux_weight && T > 2) g.aux_weight[(int64_t)(t - 1) * g.n + b] = c;  // parked, rescaled below
      }
      prev_step = v_step;
      prev_mask = v_mask;
    }
  }
  // importance weight, only when asked for (beta_dev may be NULL otherwise; critic_weight comes with is_weight); computed after the
  // window rows so that it is not live across the out-of-line tail scan
  float isw = 1.f;
  if constexpr (PER) {
    if (pd->is_weight != nullptr) {
      isw = per_is_weight(pd->P.mins[pd->P.n_levels][0], pd->P.leaves[s], pd->beta_dev[0]);
      pd->is_weight[b] = isw;
    }
  }
  if (want_aux && g.aux_weight && T >= 2) {
    // upstream weight of q_loss[t,b]: contig / ((sum_t contig + 1e-4) * B * T)  (deepQlearning.py:222-225,249)
    const float scale = g.inv_bt / (csum + 1e-4f);
    if (T == 2) {
      const float wv = csum * scale;
      st_stream1(g.aux_weight + b, wv);
      if (PER && pd->critic_weight != nullptr) st_stream1(pd->critic_weight + b, wv * isw);
    } else {
      for (int t = 0; t < T - 1; ++t) {
        float* w = g.aux_weight + (int64_t)t * g.n + b;
        const float wv = *w * scale;
        *w = wv;
        if (PER && pd->critic_weight != nullptr) pd->critic_weight[(int64_t)t * g.n + b] = wv * isw;
      }
    }
  }
}

// Prioritized draw of the windows cb0 + lane (lane < n_here) of a chunk, for the thread-per-window phase: lane w keeps window w's target
// and node, and the warp descends through the tree for one window after the other with the descent steps of per_sample_kernel
// (draw.cuh), so the starts are the same bits.  The root's children are the same for every window and are scanned once per chunk; below
// it, the children of kPerWindowsInFlight windows are loaded together before their steps.  Returns the start and the last two Philox
// words of the window (its hindsight streams).
constexpr int kPerWindowsInFlight = 8;
__device__ __forceinline__ void per_descend_chunk(const PerDraw& pd, const GatherArgs& g, int64_t cb0, int n_here, uint64_t draw_ctr,
                                                  int& s_out, uint32_t& z_out, uint32_t& w_out) {
  constexpr int U = kPerWindowsInFlight;
  const PerDev& P = pd.P;
  const int lane = lane_id();
  const int L = P.n_levels;
  const int64_t b = cb0 + min(lane, n_here - 1);
  const uint4 x = philox4x32((uint64_t)b, draw_ctr, g.seed);
  z_out = x.z;
  w_out = x.w;
  double t = per_target(P.sums[L][0], b, g.n, pd.xi != nullptr ? pd.xi[b] : per_uniform(x));
  int node;
  {  // root
    const double v = lane < P.n[L - 1] ? (L == 1 ? (double)P.leaves[lane] : P.sums[L - 1][lane]) : 0.0;
    double incl, excl;
    per_scan(v, lane, incl, excl);
    node = 0;
    for (int w = 0; w < n_here; ++w) {
      double tw = shfl_idx_f64(t, w);
      const int pick = per_pick(v, incl, excl, tw);
      if (lane == w) {
        t = tw;
        node = pick;
      }
    }
  }
  for (int l = L - 1; l >= 1; --l) {
    const int64_t n_below = P.n[l - 1];
    const double* sums = P.sums[l - 1];
    for (int w0 = 0; w0 < n_here; w0 += U) {
      int nd[U];
      double v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        nd[u] = __shfl_sync(kFull, node, min(w0 + u, n_here - 1));
        const int64_t c = 32 * (int64_t)nd[u] + lane;
        v[u] = 0.0;
        if (c < n_below) v[u] = l == 1 ? (double)__ldg(P.leaves + c) : __ldg(sums + c);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int w = w0 + u;
        if (w >= n_here) break;  // (uniform) the last group of a short chunk
        double tw = shfl_idx_f64(t, w);
        double incl, excl;
        per_scan(v[u], lane, incl, excl);
        const int pick = per_pick(v[u], incl, excl, tw);
        if (lane == w) {
          t = tw;
          node = 32 * nd[u] + pick;
        }
      }
    }
  }
  s_out = node;
}

// =================================================================================================
// Tile kernel (plain gather and equality-reward hindsight): a block owns a tile of 256 sampled windows.
//   phase 1, one THREAD per window -- everything scalar: index / goal streams, episode extents, the hindsight scan over
//     the tail's 16-byte scan records (hash match -> verified), the return recurrence in the reference's own order
//     (fp64 step, fp32 store: bit-exact mc_return), task_done / episode_step re-basing, every scalar key of the row and
//     the learner aux.  All 32 lanes of a warp work on different windows, stores are coalesced over the batch index.
//   phase 2, one WARP per window -- the wide keys: each lane owns <= S float4 of a row (row plan in registers), loads of four
//     windows are in flight before their stores; the desired_goal lanes read the hindsight goal row instead.
// The two phases meet in 12 bytes of shared memory per window (start row, goal row, last in-episode window row).
// =================================================================================================

template <int S, bool HASH, bool DRAW>
__global__ void __launch_bounds__(kTileWindows, TILE_MINB) sample_gather_tile_kernel(const __grid_constant__ GatherArgs g) {
  __shared__ int sm_s[kTileWindows], sm_grow[kTileWindows], sm_tail[kTileWindows];
  const ArenaDev& A = g.A;
  const int lane = lane_id();
  const int wib = threadIdx.x >> 5;
  const int T = g.T;
  const int len32 = (int)g.len;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

  // ---- the lane's plan for phase 2: wide keys only ---------------------------------------------------------------
  Slot slot[S];
#pragma unroll
  for (int k = 0; k < S; ++k) {
    int i = lane + 32 * k;
    Slot sl;
    sl.src = nullptr; sl.dst = nullptr; sl.sstride = 0; sl.dwidth = 0; sl.meta = SLOT_NONE; sl.ovr = 0;
    bool found = false;
    for (int w = 0; w < A.n_wide; ++w) {
      const int vecs = g.out.p[A.wide[w].key] != nullptr ? A.wide[w].vecs : 0;  // keys without an output take no lanes
      if (!found && i >= 0 && i < vecs) {
        found = true;
        float* o = g.out.p[A.wide[w].key];
        if (o != nullptr) {
          const int width = A.wide[w].width;
          const bool v4 = (width & 3) == 0 && ((reinterpret_cast<uintptr_t>(o) & 15) == 0);
          sl.src = A.wide[w].base + 4 * i;
          sl.dst = o + 4 * i;
          sl.sstride = A.wide[w].stride;
          sl.dwidth = width;
          sl.meta = (v4 ? SLOT_V4 : SLOT_PART) | ((HASH && w == A.wide_dg) ? SLOT_DG : 0) | (i << 4) | (min(4, width - 4 * i) << 12);
        }
      }
      i -= vecs;
    }
    slot[k] = sl;
  }
  const WideSlab AG = HASH ? A.wide[A.wide_ag] : A.wide[0];

  const uint64_t draw_ctr = DRAW ? device_draw_counter(g.counter_dev, g.counter) : 0;
  const int tile_w = g.tile;  // small launches use small tiles so that every SM gets work
  const int64_t n_tiles = (g.b_end - g.b_begin + tile_w - 1) / tile_w;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t b0 = g.b_begin + tile * tile_w;
    const int n_here = (int)min((int64_t)tile_w, g.b_end - b0);

    // ================= phase 1: thread <-> window =================
    if ((int)threadIdx.x < n_here) {
      int s, grow, tail_last;
      window_scalar_phase<HASH, DRAW>(g, b0 + threadIdx.x, draw_ctr, s, grow, tail_last);
      sm_s[threadIdx.x] = s;
      sm_grow[threadIdx.x] = grow;
      sm_tail[threadIdx.x] = tail_last;
    }
    __syncthreads();

    // ================= phase 2: warp <-> window, wide keys =================
    constexpr int UW = WIN_UNROLL;  // windows whose loads are in flight together
    for (int w0 = wib * UW; w0 < n_here; w0 += UW * (kTileWindows / 32)) {
      float4 x[UW][2][S];
      int sv[UW], tl[UW];
      const float* ga[UW];
#pragma unroll
      for (int u = 0; u < UW; ++u) {
        const int wi = min(w0 + u, n_here - 1);
        sv[u] = sm_s[wi];
        tl[u] = sm_tail[wi];
        ga[u] = (HASH && tl[u] >= 0) ? AG.base + (int64_t)sm_grow[wi] * AG.stride : nullptr;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const int row = ring_row32(sv[u], t, len32);
#pragma unroll
          for (int k = 0; k < S; ++k) {
            x[u][t][k] = zero4;
            if (t < T && w0 + u < n_here) x[u][t][k] = slot_load(slot[k], row, t <= tl[u] ? ga[u] : nullptr);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < UW; ++u) {
        if (w0 + u >= n_here) continue;
        const int64_t b = b0 + w0 + u;
        auto put = [&](int t, const float4 (&v)[S]) {
          const int64_t orow = (int64_t)t * g.n + b;
#pragma unroll
          for (int k = 0; k < S; ++k) {
            const uint32_t meta = slot[k].meta;
            if (meta & SLOT_V4) st_stream4(slot[k].dst + orow * slot[k].dwidth, v[k]);
            if (meta & SLOT_PART) {
              const int m = (meta >> 12) & 15u;
              const float xs[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
              float* dst = slot[k].dst + orow * slot[k].dwidth;
              for (int c = 0; c < m; ++c) st_stream1(dst + c, xs[c]);
            }
          }
        };
#pragma unroll
        for (int t = 0; t < 2; ++t)
          if (t < T) put(t, x[u][t]);
        for (int t = 2; t < T; ++t) {
          const int row = ring_row32(sv[u], t, len32);
          float4 v[S];
#pragma unroll
          for (int k = 0; k < S; ++k) v[k] = slot_load(slot[k], row, t <= tl[u] ? ga[u] : nullptr);
          put(t, v);
        }
      }
    }
    __syncthreads();
  }
}


// =================================================================================================
// Lean kernel: the tile kernel's work with the wide keys moved by the copy engines instead of through registers.
//   A warp owns a chunk of 32 consecutive windows.  Phase 1 is the same thread-per-window scalar phase (window_scalar_phase).
//   Phase 2 stages the wide keys of 16 windows x one window row in shared memory with 16-byte asynchronous copies (cp.async:
//   lane v of the warp owns float4 v of the row, the desired_goal lanes read the hindsight goal row instead) and writes every key
//   of the stage back with ONE bulk copy (cp.async.bulk shared -> global): the outputs are time-major [T, n, w], so the 16 rows
//   of a key are contiguous.  Two stages per warp are in flight while the warp runs phase 1 of its next chunk, so a block of a
//   few warps keeps as many bytes in flight as the tile kernel does with 32 warps per SM, for ~6x fewer issued instructions.
//   It can therefore run as ONE small block per SM next to the issue-bound loss kernel (FDQL_OPT_CORESIDENT), which is how the
//   reference overlaps sampling with training (torch_dataloader.py:22-39, a prefetch thread one batch ahead).
// Served: plain gathers and equality-reward hindsight, every wide key with an output a whole number of float4 and 16-byte aligned
// outputs, at most 32 float4 per row; everything else takes the tile kernel.
// =================================================================================================
constexpr int kLeanWarps = 4;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_store_s2g(void* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ bool elect_one() {  // one lane of the converged warp, known to the compiler as a single-thread region
  uint32_t pred;
  asm volatile("{\n .reg .pred p;\n elect.sync _|p, 0xffffffff;\n selp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
  return pred != 0;
}

#ifndef FDQL_LEAN_MAXVECS
#define FDQL_LEAN_MAXVECS 32
#endif
// 16-byte asynchronous copy predicated on `on` (a predicated instruction, never a branch: every basic block that holds an LDGSTS
// starts with three dummy LDS on sm_100a, so the copies of a stage want to sit in ONE block)
__device__ __forceinline__ void cp_async16_if(uint32_t dst, const void* src, bool on) {
  asm volatile("{\n .reg .pred p;\n setp.ne.u32 p, %2, 0;\n @p cp.async.cg.shared.global [%0], [%1], 16;\n}" ::"r"(dst), "l"(src),
               "r"((uint32_t)on)
               : "memory");
}
// Copy plan known at compile time (PLAN != 0): hex digits 3..0 = copy rounds of wide keys 0..3 = ceil(vecs / kParts), 0 = no such
// key; digit 4 = index of the desired_goal key + 1 (0 = none).  The fills of one key of a stage, straight-line: all rounds but the last are whole (every lane has a float4 in
// them), the last one is predicated.
template <int ROUNDS, bool HASH, bool IS_DG, int kParts, int kLeanStageWindows>
__device__ __forceinline__ void lean_fill_key(const GatherArgs& g, const int k, const unsigned row, const unsigned gw, const bool relab,
                                              const uint32_t dl, const uint32_t wl16, const uint32_t part_u, const uint32_t part16) {
  if constexpr (ROUNDS > 0) {
    const GatherArgs::LeanKey& K = g.lean_key[k];
    const char* p = K.base + (uint64_t)row * K.stride;
    if (HASH && IS_DG && relab) p = g.lean_ag_base + (uint64_t)gw * g.lean_ag_stride;  // (the plan names the desired_goal key)
    p += part16;
    const uint32_t d = wl16 * K.vecs + (dl + K.stage_off * kLeanStageWindows);
#pragma unroll
    for (int j = 0; j < ROUNDS - 1; ++j) cp_async16(d + 16u * kParts * j, p + 16 * kParts * j);
    cp_async16_if(d + 16u * kParts * (ROUNDS - 1), p + 16 * kParts * (ROUNDS - 1), (uint32_t)((ROUNDS - 1) * kParts) + part_u < K.vecs);
  }
}
// (the launcher takes a compiled plan only when T * n * 16 * vecs fits 32 bits: the output offset is then one 32 x 32 -> 64 multiply-add)
template <int ROUNDS, int kLeanStageWindows>
__device__ __forceinline__ void lean_store_key(const GatherArgs& g, const int k, const uint32_t orow, const uint32_t sb, const uint32_t nw) {
  if constexpr (ROUNDS > 0) {
    const GatherArgs::LeanKey& K = g.lean_key[k];
    const uint32_t row_bytes = 16u * K.vecs, units = nw * K.vecs;  // (units: the copy size in 16-byte units, as the instruction wants it)
    __builtin_assume(units < (1u << 20));
    bulk_store_s2g(K.out + orow * row_bytes, sb + K.stage_off * kLeanStageWindows, units << 4);
  }
}
// The kernel body as a device function (stand-alone kernel below; gather role of the fused pass kernel).  `wib`: this warp's index
// among the role's `n_warps` warps of the block (taken through a shuffle by the caller: warp-uniform for the compiler, so the stage
// bookkeeping and the bulk copies use uniform registers); `blk` / `n_blk`: the block's rank among the blocks that share the windows;
// `bar_id`: 0 = the role is the whole block, otherwise its named barrier.
// `pd` (PER builds): the starts are drawn from this priority tree (per_descend_chunk) instead of uniformly.
template <bool HASH, bool DRAW, int kLeanStageWindows, int TC = 0, int kStages = 2, int PLAN = 0, bool PER = false>
__device__ __forceinline__ void gather_lean_body(const GatherArgs& g, unsigned char* lean_smem, const int wib, const int n_warps,
                                                 const int blk, const int n_blk, const int bar_id, const PerDraw* pd = nullptr) {
  const int lane = lane_id();
  const int T = TC > 0 ? TC : g.T;  // (TC: see window_scalar_phase)
  const int len32 = (int)g.len;

  // ---- lane plan: lane = window-in-stage * kParts + part; a lane moves float4 part, part + kParts, ... of every wide key of its
  //      window, so ONE cp.async instruction serves all the windows of a stage
  constexpr int kParts = 32 / kLeanStageWindows;
  constexpr int kMaxJ = FDQL_LEAN_MAXVECS / kParts;  // a key has at most FDQL_LEAN_MAXVECS float4 per row (wider keys: tile kernel)
  const int wl = lane / kParts;
  uint32_t wl_u = (uint32_t)wl, part_u = (uint32_t)(lane % kParts), part16 = 16u * part_u;
  asm volatile("" : "+r"(wl_u), "+r"(part_u), "+r"(part16));  // held in registers (the compiler otherwise re-derives them per stage)
  const uint32_t stage_bytes = g.lean_row_bytes * kLeanStageWindows;
  // kStages stages per warp: two = the fills of one stage fly while the previous one is written back; one = a stage is filled, then
  // written back, and the other warps of the role cover its latencies (same shared memory for stages of twice the windows)
  uint32_t warp_smem = (uint32_t)__cvta_generic_to_shared(lean_smem) + (uint32_t)wib * (uint32_t)kStages * stage_bytes;
  if constexpr (PLAN != 0) asm volatile("" : "+r"(warp_smem));  // kept in a register (otherwise re-derived from the CTA id in every stage)

  const uint64_t draw_ctr = DRAW ? device_draw_counter(g.counter_dev, g.counter, wib * 32 + lane, n_blk, bar_id, n_warps * 32) : 0;
  const int64_t n_windows = g.b_end - g.b_begin;
  const int64_t n_chunks = (n_windows + 31) / 32;
  const int64_t warps_total = (int64_t)n_blk * n_warps;
  uint32_t it = 0;            // stages issued by this warp
  // the stage whose copies are in flight and whose write-back is still to be issued
  int p_t = 0, p_n = 0;
  int64_t p_b0 = 0;
  auto finish_stage = [&](uint32_t buf, int t, int64_t b0, int nw) {
    // (the caller has waited for the stage's cp.async groups)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the bulk copy engine
    __syncwarp();
    if (elect_one()) {  // one bulk copy per key: its rows are contiguous in the stage and in the time-major output
      const uint32_t sb = warp_smem + buf * stage_bytes;
      const int64_t orow = (int64_t)t * g.n + b0;
      if constexpr (PLAN != 0) {
        const uint32_t orow32 = (uint32_t)t * (uint32_t)g.n + (uint32_t)b0;
        lean_store_key<(PLAN >> 12) & 15, kLeanStageWindows>(g, 0, orow32, sb, (uint32_t)nw);
        lean_store_key<(PLAN >> 8) & 15, kLeanStageWindows>(g, 1, orow32, sb, (uint32_t)nw);
        lean_store_key<(PLAN >> 4) & 15, kLeanStageWindows>(g, 2, orow32, sb, (uint32_t)nw);
        lean_store_key<PLAN & 15, kLeanStageWindows>(g, 3, orow32, sb, (uint32_t)nw);
      } else
#pragma unroll
      for (int k = 0; k < kLeanMaxKeys; ++k) {
        if (k < g.lean_nk && !(FDQL_DBG(g) & 16)) {
          const uint32_t row_bytes = 16u * g.lean_key[k].vecs;
          bulk_store_s2g(g.lean_key[k].out + orow * (int64_t)row_bytes, sb + g.lean_key[k].stage_off * kLeanStageWindows, (uint32_t)nw * row_bytes);
        }
      }
      bulk_commit_group();
    }
  };
  int* const wctr = g.lean_work_ctr;
  int64_t chunk = (int64_t)blk * n_warps + wib;
  if (wctr != nullptr) {
    int c = 0;
    if (lane == 0) c = atomicAdd(wctr, 1);
    chunk = __shfl_sync(kFull, c, 0);
  }
  while (chunk < n_chunks) {
    int c_next = 0;  // claimed now, looked at when this chunk is done: the atomic's round trip stays off the critical path
    if (wctr != nullptr && lane == 0) c_next = atomicAdd(wctr, 1);
    const int64_t cb0 = g.b_begin + chunk * 32;
    const int n_here = (int)min((int64_t)32, g.b_end - cb0);
    int s = 0, grow = 0, tail_last = -1;
    if (FDQL_DBG(g) & 4) {  // probe: the issue load of the scalar phase (~70 warp instructions per window) as a tiny loop of dependent FMAs
      float x = (float)lane;
#ifdef FDQL_PROBE_BIGCODE  // the same issue load as straight-line code (35 KB): what the instruction cache costs the co-run
#pragma unroll
      for (int i = 0; i < 2240; ++i) x = fmaf(x, 1.0001f, 0.5f);
#else
#pragma unroll 1
      for (int i = 0; i < 2240; ++i) x = fmaf(x, 1.0001f, 0.5f);
#endif
      if (x == 12345.f) g.aux_mask[0] = x;
    }
    if constexpr (PER) {
      int per_s;
      uint32_t per_z, per_w;
      per_descend_chunk(*pd, g, cb0, n_here, draw_ctr, per_s, per_z, per_w);
      if (lane < n_here) window_scalar_phase<HASH, true, TC, true>(g, cb0 + lane, draw_ctr, s, grow, tail_last, pd, per_s, per_z, per_w);
    } else if (FDQL_DBG(g) & 2) s = (int)(((cb0 + lane) * 7919) % (len32 - T));
    else if (lane < n_here) window_scalar_phase<HASH, DRAW, TC>(g, cb0 + lane, draw_ctr, s, grow, tail_last);
    __syncwarp();
#pragma unroll 1
    for (int t = 0; t < ((FDQL_DBG(g) & 1) ? 0 : T); ++t) {
      for (int w0 = 0; w0 < n_here; w0 += kLeanStageWindows, ++it) {
        const int nw = min(kLeanStageWindows, n_here - w0);
        const uint32_t buf = kStages == 2 ? (it & 1u) : 0u;
        // the bulk write-back that read this buffer (issued one stage ago, for the stage before that) must be done reading it
        if (elect_one()) bulk_wait_group_read<0>();
        __syncwarp();
        // (registers, not shared memory: next to the loss kernel the shared-memory pipe is the busiest unit of the SM)
        // lanes past the last window of a short stage repeat that window: their slots are filled but never written back
        const int src_lane = min(w0 + (int)wl_u, n_here - 1);
        const int sw = __shfl_sync(kFull, s, src_lane);
        const int tlw = __shfl_sync(kFull, tail_last, src_lane);
        const int gw = __shfl_sync(kFull, grow, src_lane);
        unsigned row = (unsigned)sw + (unsigned)t;
        if (row >= (unsigned)len32) row -= (unsigned)len32;
        const bool relab = HASH && t <= tlw;
        const uint32_t dl = warp_smem + buf * stage_bytes + part16;
        if constexpr (PLAN != 0) {
          constexpr int kDg = ((PLAN >> 16) & 7) - 1;  // which key is desired_goal (-1: none)
          const uint32_t wl16 = 16u * wl_u;
          lean_fill_key<(PLAN >> 12) & 15, HASH, kDg == 0, kParts, kLeanStageWindows>(g, 0, row, (unsigned)gw, relab, dl, wl16, part_u, part16);
          lean_fill_key<(PLAN >> 8) & 15, HASH, kDg == 1, kParts, kLeanStageWindows>(g, 1, row, (unsigned)gw, relab, dl, wl16, part_u, part16);
          lean_fill_key<(PLAN >> 4) & 15, HASH, kDg == 2, kParts, kLeanStageWindows>(g, 2, row, (unsigned)gw, relab, dl, wl16, part_u, part16);
          lean_fill_key<PLAN & 15, HASH, kDg == 3, kParts, kLeanStageWindows>(g, 3, row, (unsigned)gw, relab, dl, wl16, part_u, part16);
        } else
#pragma unroll
        for (int k = 0; k < kLeanMaxKeys; ++k) {
          if (k < g.lean_nk) {
            const char* p = g.lean_key[k].base + (uint64_t)row * g.lean_key[k].stride;
            if (HASH && g.lean_key[k].is_dg && relab) p = g.lean_ag_base + (uint64_t)(unsigned)gw * g.lean_ag_stride;
            p += part16;
            const uint32_t d = dl + g.lean_key[k].stage_off * kLeanStageWindows + wl_u * (16u * g.lean_key[k].vecs);
            if (!(FDQL_DBG(g) & 8)) {
              // every round is one instruction predicated on "this lane has a float4 in it": no branches inside a stage, except that
              // keys of a single round skip the other slots (measured: a jump table over the round count, and rotating the rounds per
              // window so that the shared-memory writes are conflict free, both made the co-run slower)
              const uint32_t vecs = g.lean_key[k].vecs;
              if (part_u < vecs) cp_async16(d, p);
              if (vecs > (uint32_t)kParts) {  // (uniform)
#pragma unroll
                for (int j = 1; j < (kMaxJ < 4 ? kMaxJ : 4); ++j)
                  if ((uint32_t)(j * kParts) + part_u < vecs) cp_async16(d + 16u * kParts * j, p + 16 * kParts * j);
                if (vecs > (uint32_t)(4 * kParts)) {  // (uniform) a predicated-off copy still costs its issue slots: skip in blocks of four
#pragma unroll
                  for (int j = 4; j < kMaxJ; ++j)
                    if ((uint32_t)(j * kParts) + part_u < vecs) cp_async16(d + 16u * kParts * j, p + 16 * kParts * j);
                }
              }
            }
          }
        }
        cp_async_commit_group();
        if constexpr (kStages == 1) {
          cp_async_wait_group<0>();
          finish_stage(0u, t, cb0 + w0, nw);
        } else {
          if (it > 0) {  // the previous stage has had a whole stage of issue time to land
            cp_async_wait_group<1>();
            finish_stage(buf ^ 1u, p_t, p_b0, p_n);
          }
          p_t = t;
          p_b0 = cb0 + w0;
          p_n = nw;
        }
      }
    }
    chunk = wctr != nullptr ? (int64_t)__shfl_sync(kFull, c_next, 0) : chunk + warps_total;
  }
  if (kStages == 2 && it > 0) {
    cp_async_wait_group<0>();
    finish_stage((it - 1) & 1u, p_t, p_b0, p_n);
  }
  if (elect_one()) bulk_wait_group_read<0>();
  if (wctr != nullptr) {  // the last block to get here re-arms the counter for the next launch
    role_barrier(bar_id, n_warps * 32);
    if (wib == 0 && lane == 0) {
      __threadfence();
      if (atomicAdd(wctr + 1, 1) == n_blk - 1) {
        wctr[0] = 0;
        wctr[1] = 0;
        __threadfence();
      }
    }
  }
}

template <bool HASH, bool DRAW, int kLeanStageWindows>
__global__ void __launch_bounds__(kLeanWarps * 32, 5) sample_gather_lean_kernel(const __grid_constant__ GatherArgs g) {
  extern __shared__ __align__(128) unsigned char lean_smem_dyn[];
  const int wib = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
  gather_lean_body<HASH, DRAW, kLeanStageWindows>(g, lean_smem_dyn, wib, kLeanWarps, (int)blockIdx.x, (int)gridDim.x, 0);
}

// =================================================================================================
// Fused pass kernel: ONE launch per pass does what bench.py's pipelined schedule does with two -- the loss role (16 warps:
// tqc_group_body on batch k, whose critic outputs exist) and the gather role (8 warps: gather_lean_body samples, relabels and gathers
// batch k+1 into the other buffer) share every SM from the first to the last cycle of the launch.  One block per SM; the roles never
// meet (separate shared memory, separate named barriers, separate work counters).  This is the reference's prefetch thread
// (torch_dataloader.py:22-39) as warp specialisation; consecutive passes are ordered by the stream, so no events are needed.
// =================================================================================================
#ifndef FDQL_FUSED_LOSS_WARPS
#define FDQL_FUSED_LOSS_WARPS 16
#endif
#ifndef FDQL_FUSED_GATHER_WARPS
#define FDQL_FUSED_GATHER_WARPS 8
#endif
#ifndef FDQL_FUSED_STAGE_WINDOWS
#define FDQL_FUSED_STAGE_WINDOWS 8
#endif
#ifndef FDQL_FUSED_STAGES
#define FDQL_FUSED_STAGES 2
#endif
#ifndef FDQL_FUSED_PLAN
#define FDQL_FUSED_PLAN 0x44111  // the copy plan compiled into the T = 2 build of the fused pass (see gather_lean_body)
#endif
constexpr int kFusedLossWarps = FDQL_FUSED_LOSS_WARPS, kFusedGatherWarps = FDQL_FUSED_GATHER_WARPS, kFusedStageWindows = FDQL_FUSED_STAGE_WINDOWS,
              kFusedStages = FDQL_FUSED_STAGES;
#ifdef FDQL_FUSED_ROLE_CLOCK
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#endif

template <int FLAGS, bool HASH, bool DRAW, int TC = 0, int PLAN = 0>
__global__ void __launch_bounds__((kFusedLossWarps + kFusedGatherWarps) * 32, 1)
fused_pass_kernel(const __grid_constant__ GatherArgs g, const __grid_constant__ TqcArgs a) {
  extern __shared__ __align__(128) unsigned char fused_smem[];
  const int w = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
  constexpr uint32_t kLossBytes = kFusedLossWarps * GrpCfg<128>::kWarpFloatsAlias * sizeof(float);
#ifdef FDQL_FUSED_ROLE_CLOCK  // probe build: when does each role of each block end?  ({start, loss end, gather end} per block, ns)
  unsigned long long* clk = g.role_clock + 3 * blockIdx.x;
  unsigned long long* acc = g.role_clock + 3 * 256;  // {last end, gap sum, launches, loss sum, gather sum} accumulated by block 0
  unsigned long long t_start = 0;
  if (threadIdx.x == 0 || threadIdx.x == kFusedLossWarps * 32) t_start = globaltimer_ns();
  if (threadIdx.x == 0) {
    clk[0] = t_start;
    if (blockIdx.x == 0) {
      const unsigned long long le = *reinterpret_cast<volatile unsigned long long*>(acc);
      if (le != 0 && t_start > le && t_start - le < 1000000ull) {
        atomicAdd(acc + 1, t_start - le);
        atomicAdd(acc + 2, 1ull);
        const unsigned long long us = (t_start - le) / 1000ull;  // histogram of the gap in microseconds, 0..31+
        atomicAdd(acc + 8 + (us < 31ull ? us : 31ull), 1ull);
      }
    }
  }
#endif
  if (w < kFusedLossWarps) {
    tqc_group_body<128, FLAGS>(a, reinterpret_cast<float*>(fused_smem), w, kFusedLossWarps, (int)blockIdx.x, (int)gridDim.x, 1);
#ifdef FDQL_FUSED_ROLE_CLOCK
    asm volatile("bar.sync 1, %0;" ::"r"(kFusedLossWarps * 32) : "memory");
    if (threadIdx.x == 0) {
      const unsigned long long te = globaltimer_ns();
      clk[1] = te;
      atomicMax(acc, te);
      if (blockIdx.x == 0) atomicAdd(acc + 3, te - t_start);
    }
#endif
  } else {
    gather_lean_body<HASH, DRAW, kFusedStageWindows, TC, kFusedStages, PLAN>(g, fused_smem + kLossBytes, w - kFusedLossWarps, kFusedGatherWarps, (int)blockIdx.x,
                                                     (int)gridDim.x, 2);
#ifdef FDQL_FUSED_ROLE_CLOCK
    asm volatile("bar.sync 2, %0;" ::"r"(kFusedGatherWarps * 32) : "memory");
    if (threadIdx.x == kFusedLossWarps * 32) {
      const unsigned long long te = globaltimer_ns();
      clk[2] = te;
      atomicMax(acc, te);
      if (blockIdx.x == 0) atomicAdd(acc + 4, te - t_start);
    }
#endif
  }
}

// The same kernel with prioritized starts (fdql_fused_pass_per): the gather role draws from the priority tree in `pd`; the loss role is
// the same code.
template <int FLAGS, bool HASH, int TC = 0, int PLAN = 0>
__global__ void __launch_bounds__((kFusedLossWarps + kFusedGatherWarps) * 32, 1)
fused_pass_per_kernel(const __grid_constant__ GatherArgs g, const __grid_constant__ TqcArgs a, const __grid_constant__ PerDraw pd) {
  extern __shared__ __align__(128) unsigned char fused_smem[];
  const int w = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
  constexpr uint32_t kLossBytes = kFusedLossWarps * GrpCfg<128>::kWarpFloatsAlias * sizeof(float);
  if (w < kFusedLossWarps)
    tqc_group_body<128, FLAGS>(a, reinterpret_cast<float*>(fused_smem), w, kFusedLossWarps, (int)blockIdx.x, (int)gridDim.x, 1);
  else
    gather_lean_body<HASH, true, kFusedStageWindows, TC, kFusedStages, PLAN, true>(g, fused_smem + kLossBytes, w - kFusedLossWarps,
                                                                                   kFusedGatherWarps, (int)blockIdx.x, (int)gridDim.x, 2, &pd);
}

int g_tile_override = 0;
int g_tile_ctas_per_sm = 0;  // tuning hook: resident tile-kernel blocks per SM (0 = as many as fit)
int g_force_generic_gather = 0;       // tests flip this to cover the descriptor-walking kernel
int g_force_full_vector_relabel = 0;  // ... and this to cover MODE 1 with the bitflip functor

int launch_gather(const fdql_arena* a, int64_t n, int64_t b_begin, int64_t b_end, int32_t T, int64_t len, const int64_t* starts, const uint8_t* flags,
                         const int64_t* goal_rows, int32_t reward_op, const float* reward_params_host, int32_t n_params,
                         double gamma, uint32_t opts, int32_t batch_for_weight, float* const* out, float* aux_mask,
                         float* aux_contig, float* aux_weight, cudaStream_t st, const DrawSpec* draw) {
  {
    const int rc = flush_pending_invalidation(a, st);
    if (rc) return rc;
  }
  GatherArgs g;
  memset(&g, 0, sizeof(g));
  if (draw != nullptr) {
    g.draw_range = draw->range;
    g.goal_mode = draw->goal_mode;
    g.relabel_prob = draw->relabel_prob;
    g.seed = draw->seed;
    g.counter = draw->counter;
    g.counter_dev = draw->counter_dev;
    g.starts_out = draw->starts_out;
    g.flags_out = draw->flags_out;
    g.goal_out = draw->goal_out;
  }
  g.A = a->dev;
  for (int k = 0; k < a->n_keys; ++k) g.out.p[k] = out[k];
  g.starts = starts;
  g.flags = flags;
  g.goal_rows = goal_rows;
  g.n = n;
  g.b_begin = b_begin;
  g.b_end = b_end;
  g.len = len;
  g.T = T;
  g.opts = opts;
  g.gamma = gamma;
  g.inv_bt = 1.f / ((float)(batch_for_weight > 0 ? batch_for_weight : (int32_t)n) * (float)T);
  g.aux_mask = aux_mask;
  g.aux_contig = aux_contig;
  g.aux_weight = aux_weight;
  const bool relabel = draw != nullptr ? draw->flags_out != nullptr : flags != nullptr;
  int lpr = 1;
  if (relabel) {
    FDQL_REQUIRE(draw != nullptr || goal_rows != nullptr, "flags without goal_rows");
    FDQL_REQUIRE(a->dev.wide_ag >= 0 && a->dev.wide_dg >= 0, "relabelling needs achieved_goal and desired_goal keys");
    FDQL_REQUIRE(reward_op != FDQL_REWARD_NONE, "relabelling needs a reward functor");
    FDQL_REQUIRE(a->dev.wide[a->dev.wide_ag].vecs <= 32, "goal wider than 128 floats is not supported");
    int rc = upload_reward_spec(a, reward_op, reward_params_host, n_params, st, &g.rs);
    if (rc) return rc;
    lpr = lanes_per_row(a->dev.wide[a->dev.wide_ag].vecs);
  }
  const int warps_per_block = 8;
  const size_t smem = (size_t)warps_per_block * 5 * T * sizeof(float);
  FDQL_REQUIRE(smem <= 200 * 1024, "temporal_len %d too long for the per-warp window scratch", T);
  const int64_t want_blocks = (b_end - b_begin + warps_per_block - 1) / warps_per_block;
  int64_t blocks = want_blocks;
  int wide_vecs = 0;  // one lane per float4 of a wide key that has an output (+ one lane per scalar column in the warp kernels)
  for (int w = 0; w < a->dev.n_wide; ++w)
    if (out[a->dev.wide[w].key] != nullptr) wide_vecs += a->dev.wide[w].vecs;
  const int row_vecs = wide_vecs + a->dev.n_scal;
  const int slots = (row_vecs + 31) / 32;
  const int wslots = (wide_vecs + 31) / 32;
  const bool hash_ok = relabel && reward_op == FDQL_REWARD_BITFLIP && !g_force_full_vector_relabel;
  // small tail-scanning launches are latency-bound and run faster with one warp per window (measured: 4096 windows 20 us vs 29 us);
  // from ~48K windows on, the tile kernel's lower instruction count wins (262144 windows: 209 us vs 261 us)
  // link records (chain of equal achieved goals + goal-agnostic return) serve equality rewards when they were built with this
  // discount and the window fits the 64-bit hit mask; otherwise the kernels scan the episode tail
  // (the lean / fused kernels take them up to 64 window rows; the tile kernel, thread per window with T link records each, is
  // faster through the tail scan beyond 32: measured at T = 50, 16384 windows, 0.267 against 0.440 ms)
  const bool link_ok64 = hash_ok && a->link_state == 1 && a->link_gamma == gamma && gamma > 0.0 && T <= 64 && !(g_force_generic_gather & 16);
  const bool link_ok = link_ok64 && T <= 32;
  // with link records the tile kernel has no tail loop and wins from ~1K windows on (measured 4096 windows: 14.7 us vs 19.5 us per call)
  const bool big = (b_end - b_begin) >= 49152 || (link_ok && (b_end - b_begin) >= 1024) || g_tile_override != 0;
  // lean kernel (wide keys through cp.async staging + bulk write-back): asked for by FDQL_OPT_CORESIDENT (one block per SM, next to
  // the loss kernel of another stream) or by the tuning hook; needs whole-float4 keys and 16-byte aligned outputs
  bool lean_ok = wslots <= 1 && wide_vecs > 0 && (!relabel || hash_ok) && !(g_force_generic_gather & (1 | 8));
  g.lean_nk = 0;
  g.lean_row_bytes = 0;
  for (int w = 0; w < a->dev.n_wide && lean_ok; ++w) {
    float* o = out[a->dev.wide[w].key];
    if (o == nullptr) continue;
    if ((a->dev.wide[w].width & 3) != 0 || (reinterpret_cast<uintptr_t>(o) & 15) != 0 || g.lean_nk == kLeanMaxKeys ||
        a->dev.wide[w].vecs > FDQL_LEAN_MAXVECS) {
      lean_ok = false;
      break;
    }
    GatherArgs::LeanKey& K = g.lean_key[g.lean_nk++];
    K.base = reinterpret_cast<const char*>(a->dev.wide[w].base);
    K.out = reinterpret_cast<char*>(o);
    K.stride = 4u * (uint32_t)a->dev.wide[w].stride;
    K.vecs = (uint32_t)a->dev.wide[w].vecs;
    K.stage_off = g.lean_row_bytes;
    K.is_dg = (relabel && w == a->dev.wide_dg) ? 1 : 0;
    g.lean_row_bytes += 16u * K.vecs;
  }
  if (relabel && a->dev.wide_ag >= 0) {
    g.lean_ag_base = reinterpret_cast<const char*>(a->dev.wide[a->dev.wide_ag].base);
    g.lean_ag_stride = 4u * (uint32_t)a->dev.wide[a->dev.wide_ag].stride;
  }
  const bool coresident = (opts & FDQL_OPT_CORESIDENT) != 0;
  if (lean_ok && draw != nullptr && draw->fuse_tqc != nullptr) {
    // fused pass: this gather as the gather role, the given loss as the loss role of ONE launch (one block per SM).  Served: the
    // 128-atom-table group kernel with aliased partial sums and full atom slots (97..128 predicted atoms, e.g. 5 x 25) on batches
    // large enough for its one-block-per-SM form; anything else falls through to the gather alone and the caller launches the loss.
    const TqcArgs& ta = *static_cast<const TqcArgs*>(draw->fuse_tqc);
    int need = ta.n_atoms > ta.n_z ? ta.n_atoms : ta.n_z;
    if (ta.n_z - ta.n_drop + 1 > need) need = ta.n_z - ta.n_drop + 1;
    const int64_t n_groups = (ta.M + GrpCfg<128>::G - 1) / GrpCfg<128>::G;
    if (need > 64 && need <= 128 && ta.n_atoms > 96 && ta.n_atoms >= 3 * GrpCfg<128>::kRedPitch &&
        n_groups > (int64_t)2 * kFusedLossWarps * a->num_sms) {
      g.use_link = link_ok64;
      g.log2_gamma = gamma > 0.0 ? log2(gamma) : 0.0;
      g.inv_gamma = gamma > 0.0 ? 1.0 / gamma : 0.0;
      g.dbg = (g_force_generic_gather >> 6) & 31;  // probe switches, see GatherArgs.dbg (0 outside profiles/)
      TqcArgs t = ta;
      t.grp_red_alias = 1;
      // work counters of this launch: one of kFusedSlots {loss next, loss done, gather next, gather done} quadruples of the arena, taken
      // in turn (launches that share a slot are kFusedSlots launches apart; each launch leaves its slot zeroed)
      static std::atomic<unsigned> slot_turn{0};
      int* ws = a->fused_ws + 4 * (slot_turn.fetch_add(1) % kFusedSlots);
#ifdef FDQL_FUSED_ROLE_CLOCK
      g.role_clock = reinterpret_cast<unsigned long long*>(a->fused_ws + 4 * kFusedSlots);
#endif
#ifndef FDQL_FUSED_STATIC_SPLIT
      t.work_ctr = ws;
      g.lean_work_ctr = ws + 2;
#endif
      const size_t smem = (size_t)kFusedLossWarps * GrpCfg<128>::kWarpFloatsAlias * sizeof(float) +
                          (size_t)kFusedGatherWarps * kFusedStages * kFusedStageWindows * 16 * wide_vecs;
      const int flags_ = (t.mc_return ? kGrpLb : 0) | (t.stats ? kGrpStats : 0) | kGrpFull;
      if (smem <= 227 * 1024) {
#define FDQL_LAUNCH_FUSED(FLAGSV, HASHV, TCV, PLANV)                                                                        \
  do {                                                                                                                      \
    auto kern = fused_pass_kernel<FLAGSV, HASHV, true, TCV, PLANV>;                                                         \
    static size_t smem_set = 0;                                                                                             \
    if (smem_set != smem) {                                                                                                 \
      FDQL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                        \
      FDQL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)); \
      smem_set = smem;                                                                                                      \
    }                                                                                                                       \
    kern<<<(unsigned)a->num_sms, (kFusedLossWarps + kFusedGatherWarps) * 32, smem, st>>>(g, t);                             \
  } while (0)
#define FDQL_LAUNCH_FUSED_PER(FLAGSV, HASHV, TCV, PLANV)                                                                    \
  do {                                                                                                                      \
    auto kern = fused_pass_per_kernel<FLAGSV, HASHV, TCV, PLANV>;                                                           \
    static size_t smem_set = 0;                                                                                             \
    if (smem_set != smem) {                                                                                                 \
      FDQL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                        \
      FDQL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)); \
      smem_set = smem;                                                                                                      \
    }                                                                                                                       \
    kern<<<(unsigned)a->num_sms, (kFusedLossWarps + kFusedGatherWarps) * 32, smem, st>>>(g, t, *per);                       \
  } while (0)
#define FDQL_FUSED_FLAGS_OF(LAUNCH, HASHV, TCV, PLANV)               \
  do {                                                               \
    switch (flags_) {                                                \
      case 4: LAUNCH(4, HASHV, TCV, PLANV); break;                   \
      case 5: LAUNCH(5, HASHV, TCV, PLANV); break;                   \
      case 6: LAUNCH(6, HASHV, TCV, PLANV); break;                   \
      default: LAUNCH(7, HASHV, TCV, PLANV); break;                  \
    }                                                                \
  } while (0)
#define FDQL_FUSED_FLAGS(HASHV, TCV, PLANV) FDQL_FUSED_FLAGS_OF(FDQL_LAUNCH_FUSED, HASHV, TCV, PLANV)
        // TD pairs (T = 2: one transition per window, the shape the learner and the headline use) take the build with the window
        // length, the 8-float scalar record and valid link records known at compile time
        const ArenaDev& D = a->dev;
        const bool canon = D.rec_stride == 8 && D.n_scal == kCanonScal && D.col_reward == kCanonReward && D.col_task_done == kCanonTaskDone &&
                           D.col_ep_step == kCanonEpStep && D.col_mc_return == kCanonMcReturn && D.col_ep_start == kCanonEpStart &&
                           D.col_ep_end == kCanonEpEnd;
        const bool spec2 = hash_ok && T == 2 && canon && g.use_link && !(g_force_generic_gather & 2048);
        // copy plan of the gather role: rounds per wide key (hex digits), compiled for one long vector plus up to three vectors of
        // one round each (an observation next to action / goals of <= 16 floats); any other layout runs the run-time plan
        unsigned plan = 0, dg_key = 0;
        for (int k = 0; k < kLeanMaxKeys; ++k) {
          plan = (plan << 4) | (k < g.lean_nk ? (g.lean_key[k].vecs + (32 / kFusedStageWindows) - 1) / (32 / kFusedStageWindows) : 0u);
          if (k < g.lean_nk && g.lean_key[k].is_dg) dg_key = (unsigned)k + 1u;
        }
        plan |= dg_key << 16;  // (digit 4: the desired_goal key + 1, 0 = none)
        const bool out32 = (uint64_t)T * (uint64_t)n * 16u * FDQL_LEAN_MAXVECS < (1ull << 32);  // (see lean_store_key)
        const PerDraw* per = static_cast<const PerDraw*>(draw->per);
        if (per != nullptr) {  // prioritized: the T = 2 build with the compiled copy plan, else the general build (identical results)
          if (spec2 && out32 && plan == FDQL_FUSED_PLAN && !(g_force_generic_gather & 4096))
            FDQL_FUSED_FLAGS_OF(FDQL_LAUNCH_FUSED_PER, true, 2, FDQL_FUSED_PLAN);
          else if (hash_ok) FDQL_FUSED_FLAGS_OF(FDQL_LAUNCH_FUSED_PER, true, 0, 0);
          else FDQL_FUSED_FLAGS_OF(FDQL_LAUNCH_FUSED_PER, false, 0, 0);
        } else if (spec2 && out32 && plan == FDQL_FUSED_PLAN && !(g_force_generic_gather & 4096)) FDQL_FUSED_FLAGS(true, 2, FDQL_FUSED_PLAN);
        else if (spec2) FDQL_FUSED_FLAGS(true, 2, 0);
        else if (hash_ok) FDQL_FUSED_FLAGS(true, 0, 0);
        else FDQL_FUSED_FLAGS(false, 0, 0);
#undef FDQL_FUSED_FLAGS
#undef FDQL_FUSED_FLAGS_OF
#undef FDQL_LAUNCH_FUSED_PER
#undef FDQL_LAUNCH_FUSED
        FDQL_CUDA(cudaGetLastError());
#ifdef FDQL_FUSED_ROLE_CLOCK
        {
          static int calls = 0;
          cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
          cudaStreamIsCapturing(st, &cap);
          if (cap == cudaStreamCaptureStatusNone && ++calls % 97 == 0) {
            unsigned long long hc[3 * 256];
            cudaStreamSynchronize(st);
            cudaMemcpy(hc, g.role_clock, sizeof(unsigned long long) * 3 * a->num_sms, cudaMemcpyDeviceToHost);
            unsigned long long t0 = ~0ull;
            for (int b = 0; b < a->num_sms; ++b) t0 = hc[3 * b] < t0 ? hc[3 * b] : t0;
            double sl = 0, sg = 0, ml = 0, mg = 0, ss = 0;
            for (int b = 0; b < a->num_sms; ++b) {
              const double l = (double)(hc[3 * b + 1] - t0), gg = (double)(hc[3 * b + 2] - t0);
              sl += l; sg += gg; ss += (double)(hc[3 * b] - t0);
              ml = l > ml ? l : ml; mg = gg > mg ? gg : mg;
            }
            fprintf(stderr, "[role clock] start +%.1f us | loss role ends avg %.1f max %.1f us | gather role ends avg %.1f max %.1f us\n",
                    ss / a->num_sms / 1e3, sl / a->num_sms / 1e3, ml / 1e3, sg / a->num_sms / 1e3, mg / 1e3);
          }
        }
#endif
        *draw->fused = 1;
        return FDQL_OK;
      }
    }
  }
  if (draw != nullptr && draw->per != nullptr) return 1;  // prioritized starts: the fused kernel only, the caller runs the separate launches
  if (lean_ok && (coresident || (g_force_generic_gather & 32))) {
    g.use_link = link_ok64;
    g.log2_gamma = gamma > 0.0 ? log2(gamma) : 0.0;
    g.inv_gamma = gamma > 0.0 ? 1.0 / gamma : 0.0;
    const int stage_w = coresident ? 8 : 16;  // co-resident: two blocks of half-size stages per SM (eight warps in 54 KB)
    const size_t lean_smem = (size_t)kLeanWarps * 2 * stage_w * 16 * wide_vecs;
    const int64_t chunks = (b_end - b_begin + 31) / 32;
    g.dbg = (g_force_generic_gather >> 6) & 31;  // probe switches, see GatherArgs.dbg
#define FDQL_LAUNCH_LEAN(HASHV, DRAWV)                                                                                     \
  do {                                                                                                                     \
    auto kern = coresident ? sample_gather_lean_kernel<HASHV, DRAWV, 8> : sample_gather_lean_kernel<HASHV, DRAWV, 16>;     \
    static int per_sm_cached2[2] = {0, 0};                                                                                 \
    static size_t smem_cached2[2] = {0, 0};                                                                                \
    int& per_sm_cached = per_sm_cached2[coresident ? 1 : 0];                                                               \
    size_t& smem_cached = smem_cached2[coresident ? 1 : 0];                                                                \
    if (per_sm_cached == 0 || smem_cached != lean_smem) {                                                                  \
      FDQL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lean_smem));                  \
      FDQL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)); \
      FDQL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_cached, kern, kLeanWarps * 32, lean_smem));          \
      if (per_sm_cached < 1) per_sm_cached = 1;                                                                            \
      smem_cached = lean_smem;                                                                                             \
    }                                                                                                                      \
    int per_sm = coresident ? (per_sm_cached < 2 ? per_sm_cached : 2) : per_sm_cached;                                     \
    if (g_tile_ctas_per_sm > 0 && g_tile_ctas_per_sm < per_sm) per_sm = g_tile_ctas_per_sm;                                \
    int64_t blocks = (chunks + kLeanWarps - 1) / kLeanWarps;                                                               \
    if (blocks > (int64_t)a->num_sms * per_sm) blocks = (int64_t)a->num_sms * per_sm;                                      \
    kern<<<(unsigned)blocks, kLeanWarps * 32, lean_smem, st>>>(g);                                                         \
  } while (0)
    if (hash_ok) {
      if (draw != nullptr) FDQL_LAUNCH_LEAN(true, true);
      else FDQL_LAUNCH_LEAN(true, false);
    } else {
      if (draw != nullptr) FDQL_LAUNCH_LEAN(false, true);
      else FDQL_LAUNCH_LEAN(false, false);
    }
#undef FDQL_LAUNCH_LEAN
    FDQL_CUDA(cudaGetLastError());
    return FDQL_OK;
  }
  if (wslots <= 4 && (!relabel || hash_ok) && big && !(g_force_generic_gather & (1 | 8))) {
    // tile size: 256 windows when there is enough work to fill the machine, down to 32 for small batches
    int tile_w = kTileWindows;
    while (tile_w > 64 && (b_end - b_begin + tile_w - 1) / tile_w < (int64_t)a->num_sms * 3) tile_w >>= 1;
    if (g_tile_override) tile_w = g_tile_override;
    g.tile = tile_w;
    g.use_link = link_ok;
    g.log2_gamma = gamma > 0.0 ? log2(gamma) : 0.0;
    g.inv_gamma = gamma > 0.0 ? 1.0 / gamma : 0.0;
    int64_t tiles = (b_end - b_begin + tile_w - 1) / tile_w;
#define FDQL_LAUNCH_TILE(SV, HASHV)                                                                              \
  do {                                                                                                           \
    auto kern = draw != nullptr ? sample_gather_tile_kernel<SV, HASHV, true> : sample_gather_tile_kernel<SV, HASHV, false>; \
    static int per_sm_cached[2] = {0, 0};                                                                        \
    int& per_sm = per_sm_cached[draw != nullptr ? 1 : 0];                                                        \
    if (per_sm == 0) {                                                                                           \
      FDQL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kTileWindows, 0));                  \
      if (per_sm < 1) per_sm = 1;                                                                                \
    }                                                                                                            \
    const int use_per_sm = g_tile_ctas_per_sm > 0 && g_tile_ctas_per_sm < per_sm ? g_tile_ctas_per_sm : per_sm; \
    if (tiles > (int64_t)a->num_sms * use_per_sm) tiles = (int64_t)a->num_sms * use_per_sm;                      \
    kern<<<(unsigned)tiles, kTileWindows, 0, st>>>(g);                                                           \
  } while (0)
#define FDQL_TILE_S(HASHV)                                   \
  do {                                                       \
    if (wslots <= 1) FDQL_LAUNCH_TILE(1, HASHV);             \
    else if (wslots == 2) FDQL_LAUNCH_TILE(2, HASHV);        \
    else FDQL_LAUNCH_TILE(4, HASHV);                         \
  } while (0)
    if (hash_ok) FDQL_TILE_S(true);
    else FDQL_TILE_S(false);
#undef FDQL_TILE_S
#undef FDQL_LAUNCH_TILE
    FDQL_CUDA(cudaGetLastError());
    return FDQL_OK;
  }
  if (draw != nullptr) return 1;  // only the tile kernel draws; the caller falls back to sample_streams + gather
  if (slots <= 4 && !(g_force_generic_gather & 1)) {
    // persistent-style grid: as many blocks as stay resident, each warp strides over the windows
#define FDQL_LAUNCH_FAST(SV, LPRV, MODEV)                                                                              \
  do {                                                                                                                 \
    auto kern = sample_gather_fast_kernel<SV, LPRV, MODEV>;                                                            \
    if (smem > 40 * 1024) FDQL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    static int per_sm_cached = 0;                                                                                      \
    static size_t smem_cached = ~(size_t)0;                                                                            \
    if (per_sm_cached == 0 || smem_cached != smem) {                                                                   \
      FDQL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_cached, kern, warps_per_block * 32, smem));      \
      if (per_sm_cached < 1) per_sm_cached = 1;                                                                        \
      smem_cached = smem;                                                                                              \
    }                                                                                                                  \
    const int per_sm = per_sm_cached;                                                                                  \
    if (blocks > (int64_t)a->num_sms * per_sm) blocks = (int64_t)a->num_sms * per_sm;                                  \
    kern<<<(unsigned)blocks, warps_per_block * 32, smem, st>>>(g);                                                     \
  } while (0)
#define FDQL_FAST_S(LPRV, MODEV)                                            \
  do {                                                                      \
    if (slots <= 1) FDQL_LAUNCH_FAST(1, LPRV, MODEV);                       \
    else if (slots == 2) FDQL_LAUNCH_FAST(2, LPRV, MODEV);                  \
    else FDQL_LAUNCH_FAST(4, LPRV, MODEV);                                  \
  } while (0)
    if (!relabel) {
      FDQL_FAST_S(1, 0);
    } else if (reward_op == FDQL_REWARD_BITFLIP && !g_force_full_vector_relabel) {
      // scan-free return recompute when the window fits one pass and gamma^-(T-1) stays harmless in fp64
      if (T <= 32 && gamma > 0.0 && pow(gamma, (double)(T - 1)) > 1e-9 && !(g_force_generic_gather & 4)) FDQL_FAST_S(1, 3);
      else FDQL_FAST_S(1, 2);
    } else {
      switch (lpr) {
        case 1: FDQL_FAST_S(1, 1); break;
        case 2: FDQL_FAST_S(2, 1); break;
        case 4: FDQL_FAST_S(4, 1); break;
        case 8: FDQL_FAST_S(8, 1); break;
        case 16: FDQL_FAST_S(16, 1); break;
        default: FDQL_FAST_S(32, 1); break;
      }
    }
#undef FDQL_FAST_S
#undef FDQL_LAUNCH_FAST
    FDQL_CUDA(cudaGetLastError());
    return FDQL_OK;
  }
  const int64_t max_blocks = (int64_t)a->num_sms * 8;
  if (blocks > max_blocks) blocks = max_blocks;
#define FDQL_LAUNCH_GATHER(LPRV, REL)                                                                              \
  do {                                                                                                             \
    if (smem > 48 * 1024)                                                                                          \
      FDQL_CUDA(cudaFuncSetAttribute(sample_gather_kernel<LPRV, REL>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                     (int)smem));                                                                  \
    sample_gather_kernel<LPRV, REL><<<(unsigned)blocks, warps_per_block * 32, smem, st>>>(g);                      \
  } while (0)
  if (!relabel) {
    FDQL_LAUNCH_GATHER(1, false);
  } else {
    switch (lpr) {
      case 1: FDQL_LAUNCH_GATHER(1, true); break;
      case 2: FDQL_LAUNCH_GATHER(2, true); break;
      case 4: FDQL_LAUNCH_GATHER(4, true); break;
      case 8: FDQL_LAUNCH_GATHER(8, true); break;
      case 16: FDQL_LAUNCH_GATHER(16, true); break;
      default: FDQL_LAUNCH_GATHER(32, true); break;
    }
  }
#undef FDQL_LAUNCH_GATHER
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

}  // namespace fdql

using namespace fdql;

extern "C" {

int fdql_debug_force_generic_gather(int on) {
  const int old = g_force_generic_gather | (g_force_full_vector_relabel << 1);
  g_tile_override = (on >> 8) & 0x1e0;  // bits 8..16: tile size override (32/64/128/256), 0 = automatic
  g_tile_ctas_per_sm = (on >> 20) & 0xf;  // bits 20..23: resident tile-kernel blocks per SM (0 = as many as fit)
  g_force_generic_gather = on & (509 | (15 << 9));  // bit 0: descriptor-walking kernel, bit 2: per-pass suffix scan instead of Horner,
                                     // bit 3: warp-per-window kernels instead of the tile kernel, bit 4: tile kernel without link records,
                                     // bit 5: lean kernel (cp.async staging + bulk write-back) wherever it can serve,
                                     // bits 6..10: probe switches (probe builds only), bit 11: fused pass without the T = 2 build, bit 12: without the compiled copy plan
  g_force_full_vector_relabel = (on >> 1) & 1;
  return old;
}

int fdql_sample_streams(const fdql_arena* a, int64_t n, int32_t T, int32_t goal_mode, float relabel_prob, uint64_t seed,
                        uint64_t counter, uint64_t* counter_dev, int64_t* starts, uint8_t* flags, int64_t* goal_rows,
                        void* stream) {
  FDQL_REQUIRE(a != nullptr && starts != nullptr, "null argument");
  FDQL_REQUIRE(n >= 0 && T >= 0, "bad sizes");
  FDQL_REQUIRE(goal_mode >= FDQL_GOAL_FINAL && goal_mode <= FDQL_GOAL_FUTURE, "bad goal mode");
  // replay_memory.py:50,57-58: OversampleError when the ring holds fewer rows than a batch / two windows
  // (the batch-size half of the reference's check is the host mirror's: it knows the configured batch size)
  if (a->len < 1 || (T > 0 && a->len < 2 * (int64_t)T)) {
    set_error("OversampleError: ring holds %lld rows, asked for %lld windows of %d", (long long)a->len, (long long)n, T);
    return FDQL_EOVERSAMPLE;
  }
  if (n == 0) return FDQL_OK;
  const int64_t range = a->len - T;  // T==0: flat sample() over [0, len)
  FDQL_REQUIRE(range > 0, "empty start range");
  {
    const int rc = flush_pending_invalidation(a, (cudaStream_t)stream);
    if (rc) return rc;
  }
  sample_streams_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a->dev, n, range, T, goal_mode, relabel_prob,
                                                                                       seed, counter,
                                                                                       reinterpret_cast<unsigned long long*>(counter_dev),
                                                                                       starts, flags, goal_rows);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int fdql_fused_pass(const fdql_arena* a, int64_t n_windows, int32_t T, int32_t goal_mode, float relabel_prob, uint64_t seed,
                    uint64_t counter, uint64_t* counter_dev, int64_t* starts, uint8_t* flags, int64_t* goal_rows, int32_t reward_op,
                    const float* reward_params_host, int32_t n_params, double gamma, uint32_t opts, int32_t batch_for_weight,
                    float* const* out, float* aux_mask, float* aux_contig, float* aux_weight, int64_t M, int32_t n_atoms, int32_t n_drop,
                    const float* next_z, const float* q_pred, const float* next_log_pi, const float* reward, const float* mask,
                    const float* mc_return, const float* grad_scale, float alpha, float loss_gamma, float* loss, float* grad_q,
                    double* stats, void* stream) {
  FDQL_REQUIRE(a != nullptr && n_windows >= 0 && M >= 0, "bad sizes");
  FDQL_REQUIRE(n_windows == 0 || (T >= 1 && starts != nullptr && out != nullptr), "null gather argument");
  FDQL_REQUIRE((flags == nullptr) == (goal_rows == nullptr), "flags and goal_rows come together");
  FDQL_REQUIRE(n_windows == 0 || (goal_mode >= FDQL_GOAL_FINAL && goal_mode <= FDQL_GOAL_FUTURE), "bad goal mode");
  if (M > 0) {
    FDQL_REQUIRE(n_atoms >= 2 && n_atoms <= 256, "n_atoms must be in [2, 256], got %d", n_atoms);
    FDQL_REQUIRE(n_drop >= 1 && n_drop < n_atoms, "n_drop must be in [1, n_atoms); got %d", n_drop);  // quirk Q8, as fdql_tqc_loss
    FDQL_REQUIRE(next_z && q_pred && reward && mask && loss && grad_q, "null loss argument");
  }
  if (n_windows > 0 && (a->len < 1 || a->len < 2 * (int64_t)T)) {  // replay_memory.py:57-58
    set_error("OversampleError: ring holds %lld rows, asked for %lld windows of %d", (long long)a->len, (long long)n_windows, T);
    return FDQL_EOVERSAMPLE;
  }
  if (n_windows > 0 && (opts & FDQL_OPT_EMIT_LEARNER_AUX))
    FDQL_REQUIRE(a->dev.col_task_done >= 0 && a->dev.col_ep_step >= 0, "learner aux needs task_done and episode_step keys");
  TqcArgs t{M, n_atoms, n_atoms, n_drop, next_z, q_pred, next_log_pi, reward, mask, mc_return, grad_scale, alpha, loss_gamma, loss, grad_q,
            nullptr, stats, nullptr, 0};
  int fused = 0;
  if (n_windows > 0) {
    DrawSpec d{a->len - T, goal_mode, relabel_prob, seed, counter, reinterpret_cast<unsigned long long*>(counter_dev), starts, flags, goal_rows};
    if (M > 0) {
      d.fuse_tqc = &t;
      d.fused = &fused;
    }
    int rc = launch_gather(a, n_windows, 0, n_windows, T, a->len, nullptr, nullptr, nullptr, reward_op, reward_params_host, n_params, gamma,
                           opts | FDQL_OPT_CORESIDENT, batch_for_weight, out, aux_mask, aux_contig, aux_weight, (cudaStream_t)stream, &d);
    if (rc == 1) {  // shapes the drawing kernels do not serve: streams + gather as two launches
      rc = fdql_sample_streams(a, n_windows, T, goal_mode, relabel_prob, seed, counter, counter_dev, starts, flags, goal_rows, stream);
      if (rc) return rc;
      rc = launch_gather(a, n_windows, 0, n_windows, T, a->len, starts, flags, goal_rows, reward_op, reward_params_host, n_params, gamma, opts,
                         batch_for_weight, out, aux_mask, aux_contig, aux_weight, (cudaStream_t)stream);
    }
    if (rc) return rc;
  }
  if (fused || M == 0) return FDQL_OK;
  return launch_tqc(t, (cudaStream_t)stream);  // not fused: the loss as its own launch, after the gather on the same stream
}

int fdql_sample_gather_draw(const fdql_arena* a, int64_t n_windows, int32_t T, int32_t goal_mode, float relabel_prob, uint64_t seed,
                            uint64_t counter, uint64_t* counter_dev, int64_t* starts, uint8_t* flags, int64_t* goal_rows,
                            int32_t reward_op, const float* reward_params_host, int32_t n_params, double gamma, uint32_t opts,
                            int32_t batch_for_weight, float* const* out, float* aux_mask, float* aux_contig, float* aux_weight,
                            void* stream) {
  FDQL_REQUIRE(a != nullptr && starts != nullptr && out != nullptr, "null argument");
  FDQL_REQUIRE(T >= 1 && n_windows >= 0, "bad sizes");
  FDQL_REQUIRE((flags == nullptr) == (goal_rows == nullptr), "flags and goal_rows come together");
  FDQL_REQUIRE(goal_mode >= FDQL_GOAL_FINAL && goal_mode <= FDQL_GOAL_FUTURE, "bad goal mode");
  if (a->len < 1 || a->len < 2 * (int64_t)T) {  // replay_memory.py:57-58
    set_error("OversampleError: ring holds %lld rows, asked for %lld windows of %d", (long long)a->len, (long long)n_windows, T);
    return FDQL_EOVERSAMPLE;
  }
  if (n_windows == 0) return FDQL_OK;
  if (opts & FDQL_OPT_EMIT_LEARNER_AUX)
    FDQL_REQUIRE(a->dev.col_task_done >= 0 && a->dev.col_ep_step >= 0, "learner aux needs task_done and episode_step keys");
  DrawSpec d{a->len - T, goal_mode, relabel_prob, seed, counter, reinterpret_cast<unsigned long long*>(counter_dev), starts, flags, goal_rows};
  int rc = launch_gather(a, n_windows, 0, n_windows, T, a->len, nullptr, nullptr, nullptr, reward_op, reward_params_host, n_params, gamma,
                         opts, batch_for_weight, out, aux_mask, aux_contig, aux_weight, (cudaStream_t)stream, &d);
  if (rc != 1) return rc;
  // shapes the fused kernel does not serve (small batches, long windows, other reward functors): two launches
  rc = fdql_sample_streams(a, n_windows, T, goal_mode, relabel_prob, seed, counter, counter_dev, starts, flags, goal_rows, stream);
  if (rc) return rc;
  return launch_gather(a, n_windows, 0, n_windows, T, a->len, starts, flags, goal_rows, reward_op, reward_params_host, n_params, gamma, opts,
                       batch_for_weight, out, aux_mask, aux_contig, aux_weight, (cudaStream_t)stream);
}

int fdql_gather_rows(const fdql_arena* a, int64_t n, const int64_t* idx, float* const* out, void* stream) {
  FDQL_REQUIRE(a != nullptr && idx != nullptr && out != nullptr, "null argument");
  if (n <= 0) return n == 0 ? FDQL_OK : FDQL_EINVAL;
  return launch_gather(a, n, 0, n, 1, a->dev.capacity, idx, nullptr, nullptr, FDQL_REWARD_NONE, nullptr, 0, 0.0, 0, 0, out, nullptr,
                       nullptr, nullptr, (cudaStream_t)stream);
}

int fdql_sample_gather(const fdql_arena* a, int64_t n_windows, int32_t T, int64_t len, const int64_t* starts,
                       const uint8_t* flags, const int64_t* goal_rows, int32_t reward_op, const float* reward_params_host,
                       int32_t n_params, double gamma, uint32_t opts, int32_t batch_for_weight, float* const* out,
                       float* aux_mask, float* aux_contig, float* aux_weight, void* stream) {
  FDQL_REQUIRE(a != nullptr && starts != nullptr && out != nullptr, "null argument");
  FDQL_REQUIRE(T >= 1 && len >= T && len <= a->dev.capacity, "need 1 <= T <= len <= capacity (T=%d len=%lld)", T, (long long)len);
  if (n_windows <= 0) return n_windows == 0 ? FDQL_OK : FDQL_EINVAL;
  if (opts & FDQL_OPT_EMIT_LEARNER_AUX)
    FDQL_REQUIRE(a->dev.col_task_done >= 0 && a->dev.col_ep_step >= 0, "learner aux needs task_done and episode_step keys");
  return launch_gather(a, n_windows, 0, n_windows, T, len, starts, flags, goal_rows, reward_op, reward_params_host, n_params, gamma, opts,
                       batch_for_weight, out, aux_mask, aux_contig, aux_weight, (cudaStream_t)stream);
}

}  // extern "C"
