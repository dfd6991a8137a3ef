// Device-side stream drawing shared by the uniform samplers (sample.cu) and the prioritized sampler (per.cu): the counter-based
// generator, the device-resident draw counter and the hindsight half of a window's draw (flag + goal row).
#pragma once
#include "common.cuh"
#include "tqc_group.cuh"

namespace fdql {

// ---- counter-based generator (Philox4x32-10) ----------------------------------------------------
__device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
  const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
  c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
}
__device__ __forceinline__ uint4 philox4x32(uint64_t ctr_lo, uint64_t ctr_hi, uint64_t key) {
  uint32_t c0 = (uint32_t)ctr_lo, c1 = (uint32_t)(ctr_lo >> 32), c2 = (uint32_t)ctr_hi, c3 = (uint32_t)(ctr_hi >> 32);
  uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c0, c1, c2, c3, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

// The hindsight half of one window's draw, given its start row s and the extents (es, ee) of s's episode: flag ~ Bernoulli(p) from
// Philox word z (never for rows of uncommitted episodes, es < 0), goal row by mode from word w (her.py:48-53).
__device__ __forceinline__ void hindsight_pick(int64_t cap, int64_t s, int es, int ee, uint32_t z, uint32_t w, int goal_mode,
                                               float relabel_prob, bool& f, int64_t& g) {
  f = (es >= 0) && ((float)z * 2.3283064365386963e-10f < relabel_prob);
  g = s;
  if (!f) return;
  if (goal_mode == FDQL_GOAL_FINAL) {
    g = ee;
  } else if (goal_mode == FDQL_GOAL_RANDOM) {
    const int64_t L = (ee - es + (ee < es ? cap : 0)) + 1;
    g = ring_row(es, (int64_t)__umulhi(w, (uint32_t)L), cap);
  } else {  // FUTURE: a row strictly after the start row, the last row when there is none
    const int64_t m = ee - s + (ee < s ? cap : 0);
    g = m == 0 ? ee : ring_row(s, 1 + (int64_t)__umulhi(w, (uint32_t)m), cap);
  }
}

// ---- prioritized draw (per.cu; the gather role of fdql_fused_pass_per in sample.cu) --------------
constexpr int kPerMaxLevels = 8;  // 32^7 > 2^31 > capacity

// device view of a priority store (see per.cu): leaves [n[0]] under levels 1..n_levels of fp64 sums / fp32 minima
struct PerDev {
  int32_t n_levels;
  int64_t n[kPerMaxLevels];
  float* leaves;
  int32_t* owner;
  double* sums[kPerMaxLevels];
  float* mins[kPerMaxLevels];
  float* q_max;
};

// what the gather role of a prioritized fused pass needs besides GatherArgs
struct PerDraw {
  PerDev P;
  const double* xi;       // injected offsets or NULL (Philox)
  const float* beta_dev;  // importance-weight exponent, read at kernel time
  float* is_weight;       // [n] or NULL
  float* critic_weight;   // [T-1, n] = aux_weight * is_weight, or NULL
};

// xi_b from the first two Philox words: 53 random bits in [0, 1)
__device__ __forceinline__ double per_uniform(const uint4& x) { return (double)((((uint64_t)x.x << 32) | x.y) >> 11) * 0x1.0p-53; }
// stratified target of window b of n: S (b + xi_b) / n
__device__ __forceinline__ double per_target(double S, int64_t b, int64_t n, double u) { return S * (((double)b + u) / (double)n); }
// (q_min / q[s])^beta in fp64, stored as fp32
__device__ __forceinline__ float per_is_weight(float qmin, float q, float beta) { return (float)pow((double)qmin / (double)q, (double)beta); }

// One level of the descent of ONE window by one warp, in two steps so that children shared by many windows are scanned once.
// per_scan: inclusive / exclusive prefix sums of the 32 children (`v` = this lane's child, 0 past the level's end) in Kogge-Stone
// order.  That order is part of the draw: every prioritized sampler descends through these two functions, so they give the same bits.
__device__ __forceinline__ void per_scan(double v, int lane, double& incl, double& excl) {
  incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const double o = shfl_up_f64(incl, d);
    if (lane >= d) incl += o;
  }
  excl = shfl_up_f64(incl, 1);
  if (lane == 0) excl = 0.0;
}
// per_pick: the first child whose inclusive prefix exceeds the window's remaining target t (warp-uniform), or the last positive
// child when fp rounding put t past it; t loses the sum of the children before the pick.
__device__ __forceinline__ int per_pick(double v, double incl, double excl, double& t) {
  const unsigned hit = __ballot_sync(kFull, incl > t);
  int pick;
  if (hit) {
    pick = __ffs(hit) - 1;
  } else {  // fp rounding put the target past the last positive child: clamp to it
    const unsigned pos = __ballot_sync(kFull, v > 0.0);
    pick = pos ? 31 - __clz(pos) : 0;
  }
  t -= shfl_idx_f64(excl, pick);
  return pick;
}

// counter_dev (optional): {draw counter, block ticket} in device memory, so that a captured CUDA graph draws fresh streams at
// every replay.  Every block reads the counter before it takes its ticket; the block with the last ticket advances it.
// (role form: `tid` = thread index within the role, `n_blk` = blocks that take a ticket, `bar_id` / `n_threads` = the role's barrier,
// see role_barrier in tqc_group.cuh; the defaults are "the whole block of an ordinary launch")
__device__ __forceinline__ uint64_t device_draw_counter(unsigned long long* counter_dev, uint64_t counter, int tid = -1, int n_blk = 0,
                                                        int bar_id = 0, int n_threads = 0) {
  __shared__ unsigned long long sh_ctr;
  if (counter_dev == nullptr) return counter;
  if (tid < 0) {
    tid = (int)threadIdx.x;
    n_blk = (int)gridDim.x;
  }
  if (tid == 0) sh_ctr = *reinterpret_cast<volatile unsigned long long*>(counter_dev);
  role_barrier(bar_id, n_threads);
  counter += sh_ctr;
  role_barrier(bar_id, n_threads);
  if (tid == 0) {
    __threadfence();
    const unsigned long long ticket = atomicAdd(counter_dev + 1, 1ull);
    if (ticket == (unsigned long long)n_blk - 1) {
      counter_dev[1] = 0ull;
      counter_dev[0] = sh_ctr + 1ull;
      __threadfence();
    }
  }
  return counter;
}

}  // namespace fdql
