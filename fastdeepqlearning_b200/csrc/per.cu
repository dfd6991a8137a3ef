// Prioritized experience replay (proportional PER, Schaul et al. 2016, arXiv:1511.05952) over the window starts of an arena.
// Not a reference mode: franQ samples uniformly (replay_memory.py:59).  See include/fdql.h for the contract, DESIGN.md section 4.5.
//
// Store: leaves q[r] = p_r^alpha (fp32, r in [0, capacity)) under a K-ary tree, K = 32: node i of level l >= 1 covers the children
// 32 i .. 32 i + 31 of level l - 1 (level 0 = the leaves) and holds their fp64 sum and the fp32 minimum of their positive leaves
// (+inf when none).  Level L has one node, the root.  A node is always recomputed from its 32 children in one fixed order (a warp
// butterfly), never adjusted by atomics, so the same call sequence gives the same tree bits whatever the scheduling.
// One warp serves one sampled window: per level one coalesced read of the 32 children, a shuffle prefix sum, a ballot.
#include <math.h>
#include <math_constants.h>

#include "common.cuh"
#include "draw.cuh"

using fdql::kPerMaxLevels;

struct fdql_per {
  fdql_arena* a;
  int32_t T;
  float alpha, eps, eta;
  int32_t n_levels;                    // L: levels above the leaves
  int64_t n[kPerMaxLevels];            // n[0] = capacity leaves, n[l] = nodes of level l
  float* leaves;
  int32_t* owner;                      // [capacity] -1, or during fdql_per_update the largest window of the batch with this start
  double* sums[kPerMaxLevels];         // [n[l]] for l >= 1
  float* mins[kPerMaxLevels];
  float* q_max;                        // {q_max, max of the leaves written by the running update}
  int64_t applied_len;                 // ring length the eligible range was last brought up to
};

namespace fdql {

static PerDev per_dev(const fdql_per* p) {
  PerDev d;
  d.n_levels = p->n_levels;
  for (int l = 0; l < kPerMaxLevels; ++l) {
    d.n[l] = p->n[l];
    d.sums[l] = p->sums[l];
    d.mins[l] = p->mins[l];
  }
  d.leaves = p->leaves;
  d.owner = p->owner;
  d.q_max = p->q_max;
  return d;
}

// up to 4 intervals [lo, hi) of node indices of one level
struct Intervals {
  int64_t lo[4], hi[4];
  int32_t k;
  int64_t total() const {
    int64_t t = 0;
    for (int i = 0; i < k; ++i) t += hi[i] - lo[i];
    return t;
  }
};
__device__ __forceinline__ int64_t interval_item(const Intervals& iv, int64_t i) {
  int64_t r = -1;
#pragma unroll
  for (int j = 0; j < 4; ++j) {  // unrolled: constant indices keep the intervals in registers
    const int64_t w = j < iv.k ? iv.hi[j] - iv.lo[j] : 0;
    if (r < 0 && i < w) r = iv.lo[j] + i;
    i -= w;
  }
  return r;
}

// Node i of level l >= 1 from its children, by one warp: the butterfly fixes the order of the fp64 additions.
__device__ __forceinline__ void recompute_node(const PerDev& P, int l, int64_t i) {
  const int64_t c = 32 * i + lane_id();
  double s = 0.0;
  float m = CUDART_INF_F;
  if (l == 1) {
    const float v = c < P.n[0] ? P.leaves[c] : 0.f;
    s = (double)v;
    if (v > 0.f) m = v;
  } else if (c < P.n[l - 1]) {
    s = P.sums[l - 1][c];
    m = P.mins[l - 1][c];
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    s += shfl_xor_f64(s, d);
    m = fminf(m, __shfl_xor_sync(kFull, m, d));
  }
  if (lane_id() == 0) {
    P.sums[l][i] = s;
    P.mins[l][i] = m;
  }
}

// leaves of the rows in `iv` := q_max where the row is an eligible window start (r < elig_end), else 0
__global__ void __launch_bounds__(256) per_set_leaves_kernel(PerDev P, Intervals iv, int64_t total, int64_t elig_end) {
  const float qm = P.q_max[0];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = interval_item(iv, i);
    P.leaves[r] = r < elig_end ? qm : 0.f;
  }
}

// one warp per node of level l in `iv` (the intervals already mapped to level l)
__global__ void __launch_bounds__(256) per_level_kernel(PerDev P, int l, Intervals iv, int64_t total) {
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total; w += nw) recompute_node(P, l, interval_item(iv, w));
}

// one warp per updated window: node (start >> 5 l) of level l; level 1 also hands the start's owner slot back (-1), and folds the
// leaves written by this update into q_max
__global__ void __launch_bounds__(256) per_update_level_kernel(PerDev P, int l, int64_t n, const int64_t* __restrict__ starts) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (l == 1 && blockIdx.x == 0 && threadIdx.x == 0) P.q_max[0] = fmaxf(P.q_max[0], P.q_max[1]);
  if (b >= n) return;
  const int64_t s = starts[b];
  if (s < 0 || s >= P.n[0]) return;
  recompute_node(P, l, s >> (5 * l));
  if (l == 1 && lane_id() == 0) P.owner[s] = -1;
}

// what level 1 of per_update_level_kernel does besides the node when level 1 is rebuilt whole: hand the owner slots back, fold q_max
__global__ void __launch_bounds__(256) per_release_kernel(PerDev P, int64_t n, const int64_t* __restrict__ starts) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) P.q_max[0] = fmaxf(P.q_max[0], P.q_max[1]);
  if (b >= n) return;
  const int64_t s = starts[b];
  if (s >= 0 && s < P.n[0]) P.owner[s] = -1;
}

// duplicate starts in one batch: the largest window index wins
__global__ void __launch_bounds__(256) per_claim_kernel(PerDev P, int64_t n, const int64_t* __restrict__ starts) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  const int64_t s = starts[b];
  if (s >= 0 && s < P.n[0]) atomicMax(P.owner + s, (int)b);
}

// new leaf of window b: delta = eta * max_t + (1 - eta) * mean_t of the loss over its contiguous transitions (0 when none),
// q = (delta + eps)^alpha; a non-finite q takes q_max as it was before this update.  Leaves that are 0 (not an eligible start) stay 0.
__global__ void __launch_bounds__(256) per_write_leaves_kernel(PerDev P, int64_t n, int32_t Tm1, const int64_t* __restrict__ starts,
                                                               const float* __restrict__ loss, const float* __restrict__ contig,
                                                               double alpha, double eps, double eta) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n) return;
  const int64_t s = starts[b];
  if (s < 0 || s >= P.n[0] || P.owner[s] != (int)b || !(P.leaves[s] > 0.f)) return;
  float mx = -CUDART_INF_F, sum = 0.f;
  int cnt = 0;
  bool bad = false;
  for (int t = 0; t < Tm1; ++t) {
    if (contig != nullptr && contig[(int64_t)t * n + b] == 0.f) continue;
    const float v = loss[(int64_t)t * n + b];
    mx = fmaxf(mx, v);
    sum += v;
    ++cnt;
    bad |= !isfinite(v);  // (fmaxf would drop a NaN)
  }
  const double delta = cnt == 0 ? 0.0 : eta * (double)mx + (1.0 - eta) * (double)(sum / (float)cnt);
  float q = (float)pow(delta + eps, alpha);
  if (bad || !isfinite(q)) {
    q = P.q_max[0];
  } else {
    q = fmaxf(q, 1.17549435e-38f);  // an eligible leaf stays positive: (tiny)^alpha must not underflow to 0
    atomicMax(reinterpret_cast<int*>(P.q_max + 1), __float_as_int(q));  // positive floats order like their bits
  }
  P.leaves[s] = q;
}

// one warp per window: stratified target S (b + xi_b) / n, descent to the leaf whose prefix interval contains it, hindsight streams
// from the remaining Philox words, importance weight (q_min / q[s])^beta
__global__ void __launch_bounds__(256)
per_sample_kernel(PerDev P, ArenaDev A, int64_t n, int goal_mode, float relabel_prob, uint64_t seed, uint64_t counter,
                  unsigned long long* counter_dev, const double* __restrict__ xi, const float* __restrict__ beta_dev,
                  int64_t* __restrict__ starts, uint8_t* __restrict__ flags, int64_t* __restrict__ goal_rows, float* __restrict__ is_weight) {
  counter = device_draw_counter(counter_dev, counter);
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = lane_id();
  if (b >= n) return;
  const int L = P.n_levels;
  uint4 x = make_uint4(0u, 0u, 0u, 0u);
  if (xi == nullptr || flags != nullptr) x = philox4x32((uint64_t)b, counter, seed);
  const double u = xi != nullptr ? xi[b] : per_uniform(x);
  double t = per_target(P.sums[L][0], b, n, u);
  int64_t node = 0;
  for (int l = L; l >= 1; --l) {
    const int64_t c = 32 * node + lane;
    double v = 0.0;
    if (c < P.n[l - 1]) v = l == 1 ? (double)P.leaves[c] : P.sums[l - 1][c];
    double incl, excl;
    per_scan(v, lane, incl, excl);
    node = c - lane + per_pick(v, incl, excl, t);
  }
  if (lane != 0) return;
  starts[b] = node;
  if (is_weight != nullptr) is_weight[b] = per_is_weight(P.mins[L][0], P.leaves[node], beta_dev[0]);
  if (flags == nullptr) return;
  const float* rec = A.rec + node * (int64_t)A.rec_stride;
  const int es = __float_as_int(__ldg(rec + A.col_ep_start)), ee = __float_as_int(__ldg(rec + A.col_ep_end));
  bool f;
  int64_t g;
  hindsight_pick(A.capacity, node, es, ee, x.z, x.w, goal_mode, relabel_prob, f, g);
  flags[b] = f ? 1 : 0;
  if (goal_rows) goal_rows[b] = g;
}

static unsigned grid_for(int64_t threads, int num_sms) {
  int64_t blocks = (threads + 255) / 256;
  const int64_t cap = (int64_t)num_sms * 16;
  if (blocks > cap) blocks = cap;
  return (unsigned)(blocks < 1 ? 1 : blocks);
}

// recompute every node above the leaf intervals `iv` (level 0 indices), level by level
static int refresh_ancestors(const fdql_per* p, const Intervals& leaves, cudaStream_t st) {
  const PerDev D = per_dev(p);
  for (int l = 1; l <= p->n_levels; ++l) {
    Intervals iv = leaves;
    for (int j = 0; j < iv.k; ++j) {
      iv.lo[j] = leaves.lo[j] >> (5 * l);
      iv.hi[j] = ((leaves.hi[j] - 1) >> (5 * l)) + 1;
    }
    const int64_t total = iv.total();
    per_level_kernel<<<grid_for(total * 32, p->a->num_sms), 256, 0, st>>>(D, l, iv, total);
    FDQL_CUDA(cudaGetLastError());
  }
  return FDQL_OK;
}

// the rows written since the last pass and the rows whose eligibility changed with the ring length get q_max or 0.  Skipped while
// `st` is being captured: a captured copy of these host-side intervals would re-apply them at every replay.
static int apply_pending(fdql_per* p, cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  FDQL_CUDA(cudaStreamIsCapturing(st, &cs));
  if (cs != cudaStreamCaptureStatusNone) return FDQL_OK;
  Arena* a = p->a;
  const int64_t cap = a->dev.capacity;
  Intervals iv;
  iv.k = 0;
  int64_t len;
  {
    std::lock_guard<std::mutex> lk(cursor_mutex());
    len = a->len;
    auto add = [&](int64_t lo, int64_t hi) {  // at most 3 row pieces + the length interval
      if (hi <= lo) return;
      iv.lo[iv.k] = lo;
      iv.hi[iv.k] = hi;
      ++iv.k;
    };
    Intervals rows;
    rows.k = 0;
    for (int i = 0; i < a->n_per_pending; ++i) {
      const int64_t f = a->per_pending[i][0], n = a->per_pending[i][1];
      if (n >= cap) {
        rows.k = 1;
        rows.lo[0] = 0;
        rows.hi[0] = cap;
        break;
      }
      // a wrapped interval is two pieces; more than 3 pieces collapse into the whole ring
      const int64_t e = f + n;
      const int64_t pieces = e > cap ? 2 : 1;
      if (rows.k + pieces > 3) {
        rows.k = 1;
        rows.lo[0] = 0;
        rows.hi[0] = cap;
        break;
      }
      rows.lo[rows.k] = f;
      rows.hi[rows.k] = e > cap ? cap : e;
      ++rows.k;
      if (e > cap) {
        rows.lo[rows.k] = 0;
        rows.hi[rows.k] = e - cap;
        ++rows.k;
      }
    }
    a->n_per_pending = 0;
    for (int i = 0; i < rows.k; ++i) add(rows.lo[i], rows.hi[i]);
    const int64_t T = p->T;
    int64_t lo = (p->applied_len < len ? p->applied_len : len) - T, hi = (p->applied_len < len ? len : p->applied_len) - T;
    add(lo < 0 ? 0 : lo, hi < 0 ? 0 : hi);
    p->applied_len = len;
  }
  if (iv.k == 0) return FDQL_OK;
  const int64_t total = iv.total();
  per_set_leaves_kernel<<<grid_for(total, a->num_sms), 256, 0, st>>>(per_dev(p), iv, total, len - p->T);
  FDQL_CUDA(cudaGetLastError());
  return refresh_ancestors(p, iv, st);
}

// new leaves for n windows, then their ancestors.  Level l is recomputed per window (one warp each, the same node as often as windows
// share it) while the batch has fewer windows than the level has nodes, and whole (one warp per node) from there up: at 262144 windows
// over 1e7 rows that is levels 2.. (9766 nodes and fewer) instead of 262144 recomputations of each.  Either form recomputes a node from
// its children in the same order, so the tree bits do not depend on the choice, and the choice depends on n alone (capturable).
static int launch_update(const fdql_per* p, int64_t n, const int64_t* starts, const float* loss, const float* contig, cudaStream_t st) {
  const PerDev D = per_dev(p);
  const unsigned g1 = (unsigned)((n + 255) / 256), gw = (unsigned)((n + 7) / 8);
  per_claim_kernel<<<g1, 256, 0, st>>>(D, n, starts);
  per_write_leaves_kernel<<<g1, 256, 0, st>>>(D, n, p->T - 1, starts, loss, contig, (double)p->alpha, (double)p->eps, (double)p->eta);
  for (int l = 1; l <= p->n_levels; ++l) {
    if (n < p->n[l]) {
      per_update_level_kernel<<<gw, 256, 0, st>>>(D, l, n, starts);
      continue;
    }
    Intervals all;
    all.k = 1;
    all.lo[0] = 0;
    all.hi[0] = p->n[l];
    per_level_kernel<<<grid_for(p->n[l] * 32, p->a->num_sms), 256, 0, st>>>(D, l, all, p->n[l]);
    if (l == 1) per_release_kernel<<<g1, 256, 0, st>>>(D, n, starts);
  }
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

// critic_weight[t, b] = aux_weight[t, b] * is_weight[b]: what the gather role of the fused kernel writes, for the separate launches
__global__ void __launch_bounds__(256) per_critic_weight_kernel(int64_t n, int64_t total, const float* __restrict__ aux_weight,
                                                                const float* __restrict__ is_weight, float* __restrict__ critic_weight) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) critic_weight[i] = aux_weight[i] * is_weight[i % n];
}

}  // namespace fdql

using namespace fdql;

extern "C" {

int fdql_per_create(fdql_arena* a, int32_t T, float alpha, float eps, float eta, fdql_per** out) {
  FDQL_REQUIRE(a != nullptr && out != nullptr, "null argument");
  FDQL_REQUIRE(T >= 2, "T must be >= 2 (a window needs a transition to carry a priority), got %d", T);
  FDQL_REQUIRE(alpha >= 0.f && isfinite(alpha), "alpha must be a finite value >= 0, got %g", (double)alpha);
  FDQL_REQUIRE(eps > 0.f && isfinite(eps), "eps must be > 0, got %g", (double)eps);
  FDQL_REQUIRE(eta >= 0.f && eta <= 1.f, "eta must be in [0, 1], got %g", (double)eta);
  FDQL_REQUIRE(a->per == nullptr, "this arena already has a priority store");
  FDQL_CUDA(cudaSetDevice(a->device));
  fdql_per* p = new fdql_per();
  memset(p, 0, sizeof(*p));
  p->a = a;
  p->T = T;
  p->alpha = alpha;
  p->eps = eps;
  p->eta = eta;
  p->n[0] = a->dev.capacity;
  int L = 0;
  while (p->n[L] > 1 || L == 0) {
    p->n[L + 1] = (p->n[L] + 31) / 32;
    ++L;
  }
  p->n_levels = L;
  const int64_t cap = a->dev.capacity;
  bool ok = cudaMalloc(reinterpret_cast<void**>(&p->leaves), sizeof(float) * cap) == cudaSuccess &&
            cudaMalloc(reinterpret_cast<void**>(&p->owner), sizeof(int32_t) * cap) == cudaSuccess &&
            cudaMalloc(reinterpret_cast<void**>(&p->q_max), sizeof(float) * 2) == cudaSuccess;
  for (int l = 1; l <= L && ok; ++l)
    ok = cudaMalloc(reinterpret_cast<void**>(&p->sums[l]), sizeof(double) * p->n[l]) == cudaSuccess &&
         cudaMalloc(reinterpret_cast<void**>(&p->mins[l]), sizeof(float) * p->n[l]) == cudaSuccess;
  if (!ok) {
    set_error("cudaMalloc failed while allocating the priority store: %s", cudaGetErrorString(cudaGetLastError()));
    fdql_per_destroy(p);
    return FDQL_ENOMEM;
  }
  const float qm[2] = {1.f, 0.f};
  cudaMemset(p->leaves, 0, sizeof(float) * cap);
  cudaMemset(p->owner, 0xff, sizeof(int32_t) * cap);
  cudaMemcpy(p->q_max, qm, sizeof(qm), cudaMemcpyHostToDevice);
  {
    std::lock_guard<std::mutex> lk(cursor_mutex());
    a->per = p;
    a->n_per_pending = 0;
    p->applied_len = 0;  // the first pass activates [0, len - T)
  }
  Intervals all;
  all.k = 1;
  all.lo[0] = 0;
  all.hi[0] = cap;
  int rc = refresh_ancestors(p, all, 0);
  if (rc == FDQL_OK) rc = apply_pending(p, 0);
  if (rc != FDQL_OK) {
    fdql_per_destroy(p);
    return rc;
  }
  FDQL_CUDA(cudaDeviceSynchronize());
  *out = p;
  return FDQL_OK;
}

int fdql_per_destroy(fdql_per* p) {
  if (!p) return FDQL_OK;
  if (p->a) {
    std::lock_guard<std::mutex> lk(cursor_mutex());
    if (p->a->per == p) p->a->per = nullptr;
  }
  if (p->leaves) cudaFree(p->leaves);
  if (p->owner) cudaFree(p->owner);
  if (p->q_max) cudaFree(p->q_max);
  for (int l = 1; l < kPerMaxLevels; ++l) {
    if (p->sums[l]) cudaFree(p->sums[l]);
    if (p->mins[l]) cudaFree(p->mins[l]);
  }
  delete p;
  return FDQL_OK;
}

int fdql_per_apply_pending(fdql_per* p, void* stream) {
  FDQL_REQUIRE(p != nullptr, "null priority store");
  return apply_pending(p, (cudaStream_t)stream);
}

int fdql_per_rebuild(fdql_per* p, void* stream) {
  FDQL_REQUIRE(p != nullptr, "null priority store");
  Intervals all;
  all.k = 1;
  all.lo[0] = 0;
  all.hi[0] = p->n[0];
  return refresh_ancestors(p, all, (cudaStream_t)stream);
}

int fdql_per_view(const fdql_per* p, float** leaves, float** q_max_dev) {
  FDQL_REQUIRE(p != nullptr, "null priority store");
  if (leaves) *leaves = p->leaves;
  if (q_max_dev) *q_max_dev = p->q_max;
  return FDQL_OK;
}

int fdql_per_level_view(const fdql_per* p, int32_t level, double** sums, float** mins, int64_t* n_nodes) {
  FDQL_REQUIRE(p != nullptr, "null priority store");
  FDQL_REQUIRE(level >= 1 && level <= p->n_levels, "level must be in [1, %d]", p->n_levels);
  if (sums) *sums = p->sums[level];
  if (mins) *mins = p->mins[level];
  if (n_nodes) *n_nodes = p->n[level];
  return FDQL_OK;
}

int fdql_per_sample(fdql_per* p, int64_t n, int32_t goal_mode, float relabel_prob, uint64_t seed, uint64_t counter,
                    uint64_t* counter_dev, const double* xi, const float* beta_dev, int64_t* starts, uint8_t* flags,
                    int64_t* goal_rows, float* is_weight, void* stream) {
  FDQL_REQUIRE(p != nullptr && starts != nullptr, "null argument");
  FDQL_REQUIRE(n >= 0, "bad sizes");
  FDQL_REQUIRE(goal_mode >= FDQL_GOAL_FINAL && goal_mode <= FDQL_GOAL_FUTURE, "bad goal mode");
  FDQL_REQUIRE(flags != nullptr || goal_rows == nullptr, "goal_rows needs flags");
  FDQL_REQUIRE(is_weight == nullptr || beta_dev != nullptr, "importance weights need beta_dev");
  const Arena* a = p->a;
  int64_t len;
  {
    std::lock_guard<std::mutex> lk(cursor_mutex());
    len = a->len;
  }
  if (len < 2 * (int64_t)p->T) {  // with the eligibility invariant this is also the only way the root sum can be 0
    set_error("OversampleError: ring holds %lld rows, asked for %lld windows of %d", (long long)len, (long long)n, p->T);
    return FDQL_EOVERSAMPLE;
  }
  if (n == 0) return FDQL_OK;
  int rc = flush_pending_invalidation(a, (cudaStream_t)stream);
  if (rc == FDQL_OK) rc = apply_pending(p, (cudaStream_t)stream);
  if (rc) return rc;
  const unsigned blocks = (unsigned)((n + 7) / 8);
  per_sample_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(per_dev(p), a->dev, n, goal_mode, relabel_prob, seed, counter,
                                                             reinterpret_cast<unsigned long long*>(counter_dev), xi, beta_dev, starts,
                                                             flags, goal_rows, is_weight);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int fdql_per_update(fdql_per* p, int64_t n, const int64_t* starts, const float* loss, const float* contig, void* stream) {
  FDQL_REQUIRE(p != nullptr, "null priority store");
  FDQL_REQUIRE(n >= 0, "bad sizes");
  if (n == 0) return FDQL_OK;
  FDQL_REQUIRE(starts != nullptr && loss != nullptr, "null argument");
  const cudaStream_t st = (cudaStream_t)stream;
  const int rc = apply_pending(p, st);
  if (rc) return rc;
  return launch_update(p, n, starts, loss, contig, st);
}

int fdql_fused_pass_per(fdql_per* p, int64_t n_windows, int32_t goal_mode, float relabel_prob, uint64_t seed, uint64_t counter,
                        uint64_t* counter_dev, const double* xi, const float* beta_dev, int64_t* starts, uint8_t* flags, int64_t* goal_rows,
                        float* is_weight, float* critic_weight, int32_t reward_op, const float* reward_params_host, int32_t n_params,
                        double gamma, uint32_t opts, int32_t batch_for_weight, float* const* out, float* aux_mask, float* aux_contig,
                        float* aux_weight, int64_t M, int32_t n_atoms, int32_t n_drop, const float* next_z, const float* q_pred,
                        const float* next_log_pi, const float* reward, const float* mask, const float* mc_return, const float* grad_scale,
                        float alpha, float loss_gamma, float* loss, float* grad_q, double* stats, const int64_t* loss_starts,
                        const float* loss_contig, void* stream) {
  // (every check that needs no field of the store comes first)
  FDQL_REQUIRE(p != nullptr, "null priority store");
  FDQL_REQUIRE(n_windows >= 0 && M >= 0, "bad sizes");
  FDQL_REQUIRE(n_windows == 0 || (starts != nullptr && out != nullptr), "null gather argument");
  FDQL_REQUIRE((flags == nullptr) == (goal_rows == nullptr), "flags and goal_rows come together");
  FDQL_REQUIRE(n_windows == 0 || (goal_mode >= FDQL_GOAL_FINAL && goal_mode <= FDQL_GOAL_FUTURE), "bad goal mode");
  FDQL_REQUIRE(critic_weight == nullptr || (opts & FDQL_OPT_EMIT_LEARNER_AUX), "critic_weight needs FDQL_OPT_EMIT_LEARNER_AUX");
  FDQL_REQUIRE(critic_weight == nullptr || (aux_weight != nullptr && is_weight != nullptr), "critic_weight needs aux_weight and is_weight");
  FDQL_REQUIRE(is_weight == nullptr || beta_dev != nullptr, "importance weights need beta_dev");
  if (M > 0) {
    FDQL_REQUIRE(loss_starts != nullptr && loss != nullptr, "the loss half needs loss_starts and loss (the priority update reads them)");
    FDQL_REQUIRE(n_atoms >= 2 && n_atoms <= 256, "n_atoms must be in [2, 256], got %d", n_atoms);
    FDQL_REQUIRE(n_drop >= 1 && n_drop < n_atoms, "n_drop must be in [1, n_atoms); got %d", n_drop);  // quirk Q8, as fdql_tqc_loss
    FDQL_REQUIRE(next_z && q_pred && reward && mask && grad_q, "null loss argument");
  }
  const int32_t T = p->T;
  FDQL_REQUIRE(M % (T - 1) == 0, "M = %lld is not a whole number of windows of T - 1 = %d transitions", (long long)M, T - 1);
  fdql_arena* a = p->a;
  const cudaStream_t st = (cudaStream_t)stream;
  int64_t len;
  {
    std::lock_guard<std::mutex> lk(cursor_mutex());
    len = a->len;
  }
  if (n_windows > 0 && len < 2 * (int64_t)T) {  // as fdql_per_sample
    set_error("OversampleError: ring holds %lld rows, asked for %lld windows of %d", (long long)len, (long long)n_windows, T);
    return FDQL_EOVERSAMPLE;
  }
  if (n_windows > 0 && (opts & FDQL_OPT_EMIT_LEARNER_AUX))
    FDQL_REQUIRE(a->dev.col_task_done >= 0 && a->dev.col_ep_step >= 0, "learner aux needs task_done and episode_step keys");
  int rc = flush_pending_invalidation(a, st);
  if (rc == FDQL_OK) rc = apply_pending(p, st);
  if (rc) return rc;
  TqcArgs t{M, n_atoms, n_atoms, n_drop, next_z, q_pred, next_log_pi, reward, mask, mc_return, grad_scale, alpha, loss_gamma, loss, grad_q,
            nullptr, stats, nullptr, 0};
  // window modulus of the gather: the capacity, not len.  Every drawn start is < len - T, so no window wraps and the rows are the same;
  // len would be frozen into a captured launch while the tree (and so the draw) follows the ring as it grows.
  const int64_t cap = a->dev.capacity;
  int fused = 0;
  if (n_windows > 0 && M > 0) {
    PerDraw pd;
    pd.P = per_dev(p);
    pd.xi = xi;
    pd.beta_dev = beta_dev;
    pd.is_weight = is_weight;
    pd.critic_weight = critic_weight;
    DrawSpec d{len - T, goal_mode, relabel_prob, seed, counter, reinterpret_cast<unsigned long long*>(counter_dev), starts, flags, goal_rows};
    d.fuse_tqc = &t;
    d.fused = &fused;
    d.per = &pd;
    rc = launch_gather(a, n_windows, 0, n_windows, T, cap, nullptr, nullptr, nullptr, reward_op, reward_params_host, n_params, gamma,
                       opts | FDQL_OPT_CORESIDENT, batch_for_weight, out, aux_mask, aux_contig, aux_weight, st, &d);
    if (rc != FDQL_OK && rc != 1) return rc;
  }
  if (n_windows > 0 && !fused) {
    // the separate launches, with the same results: prioritized streams, the co-resident gather on them, the critic weights
    rc = fdql_per_sample(p, n_windows, goal_mode, relabel_prob, seed, counter, counter_dev, xi, beta_dev, starts, flags, goal_rows, is_weight,
                         stream);
    if (rc == FDQL_OK)
      rc = launch_gather(a, n_windows, 0, n_windows, T, cap, starts, flags, goal_rows, reward_op, reward_params_host, n_params, gamma,
                         opts | FDQL_OPT_CORESIDENT, batch_for_weight, out, aux_mask, aux_contig, aux_weight, st);
    if (rc) return rc;
    if (critic_weight != nullptr) {
      const int64_t total = (int64_t)(T - 1) * n_windows;
      per_critic_weight_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(n_windows, total, aux_weight, is_weight, critic_weight);
      FDQL_CUDA(cudaGetLastError());
    }
  }
  if (M == 0) return FDQL_OK;
  if (!fused) {
    rc = launch_tqc(t, st);
    if (rc) return rc;
  }
  // after the launch that read the tree for batch k+1: the priorities of batch k
  return launch_update(p, M / (T - 1), loss_starts, loss, loss_contig, st);
}

}  // extern "C"
