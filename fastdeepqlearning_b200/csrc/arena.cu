// Replay arena in HBM + the write path (append, episode commit, write-time hindsight flush).
// Replaces franQ/Replay/replay_memory.py:18-46 (ring), franQ/Replay/wrappers/nstep_return.py:36-72 (return-to-go at
// episode flush) and franQ/Replay/wrappers/her.py:55-95 (hindsight copy) -- see include/fdql.h for the contract.
#include <stdarg.h>
#include <stdlib.h>

#include <vector>

#include "common.cuh"
#include "goal_eval.cuh"

namespace fdql {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int upload_reward_spec(const Arena* a, int32_t op, const float* params_host, int32_t n_params, cudaStream_t st,
                       RewardSpec* out) {
  out->op = op;
  out->n_params = n_params;
  out->params = a->reward_params_dev;
  if (op == FDQL_REWARD_WEIGHTED_PNORM) {
    FDQL_REQUIRE(a->dev.wide_ag >= 0, "weighted p-norm reward needs an achieved_goal key");
    const int need = 2 + a->dev.wide[a->dev.wide_ag].width;
    FDQL_REQUIRE(params_host != nullptr && n_params == need, "weighted p-norm reward needs %d params {p, thr, w[G]}, got %d",
                 need, n_params);
    // pad weights to the slab stride with zeros so the lanes' float4 slices never read past the table
    float tmp[kMaxRewardParams + 4];
    memset(tmp, 0, sizeof(tmp));
    FDQL_REQUIRE(need <= kMaxRewardParams, "goal too wide for the reward parameter table");
    memcpy(tmp, params_host, sizeof(float) * need);
    FDQL_CUDA(cudaMemcpyAsync(a->reward_params_dev, tmp, sizeof(float) * (kMaxRewardParams + 4), cudaMemcpyHostToDevice, st));
    FDQL_CUDA(cudaStreamSynchronize(st));  // tmp is a stack buffer
  }
  return FDQL_OK;
}

// -------------------------------------------------------------------------------------------------
// append: dense [n, width] sources -> ring rows top.. (mod capacity)
// -------------------------------------------------------------------------------------------------
// src_stride: floats between consecutive source rows of every key (0: each key is a dense [n_rows, width] array).  A packed host
// block [n_rows, src_stride] holds all keys of a row side by side, src.p[k] pointing at key k's offset inside row 0.
// squash: the Pohlen transform of franQ/Replay/wrappers/squash_rewards.py:5-7, sign(r) (sqrt(|r| + 1) - 1) + 0.01 r, applied to the
// reward column on its way into the ring (evaluated in fp64 like numpy does on the Python float, stored as fp32).
__global__ void __launch_bounds__(256) append_kernel(ArenaDev A, SrcPtrs src, int64_t n_rows, int64_t top, int32_t src_stride, int32_t squash) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  for (int s = 0; s < A.n_wide; ++s) {
    const WideSlab W = A.wide[s];
    const float* __restrict__ sp = src.p[W.key];
    const int64_t items = n_rows * W.vecs;
    const int64_t rstride = src_stride > 0 ? src_stride : W.width;
    const bool vec_ok = (W.width % 4 == 0) && ((reinterpret_cast<uintptr_t>(sp) & 15) == 0) && (rstride % 4 == 0);
    for (int64_t i = tid; i < items; i += nthreads) {
      const int64_t r = i / W.vecs;
      const int v = (int)(i - r * W.vecs);
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      const float* q = sp + r * rstride + 4 * v;
      if (vec_ok) {
        x = ld_stream4(q);
      } else {
        const int n = min(4, W.width - 4 * v);
        float t[4] = {0.f, 0.f, 0.f, 0.f};
        for (int c = 0; c < n; ++c) t[c] = q[c];
        x = make_float4(t[0], t[1], t[2], t[3]);
      }
      const int64_t row = ring_row(top, r % A.capacity, A.capacity);
      *reinterpret_cast<float4*>(W.base + row * (int64_t)W.stride + 4 * v) = x;
    }
  }
  for (int64_t r = tid; r < n_rows; r += nthreads) {
    const int64_t row = ring_row(top, r, A.capacity);
    float* rec = A.rec + row * (int64_t)A.rec_stride;
    for (int c0 = 0; c0 < A.rec_stride; c0 += 4) {
      float t[4];
      for (int c = 0; c < 4; ++c) {
        const int col = c0 + c;
        float val = 0.f;
        if (col < A.n_scal) {
          val = src.p[A.scal_key[col]][src_stride > 0 ? r * (int64_t)src_stride : r];
          if (squash && col == A.col_reward) {
            const double x = (double)val;
            val = (float)(copysign(sqrt(fabs(x) + 1.0) - 1.0, x) * (x != 0.0 ? 1.0 : 0.0) + 1e-2 * x);
          }
        }
        else if (col == A.col_ep_start || col == A.col_ep_end) val = __int_as_float(-1);
        t[c] = val;
      }
      *reinterpret_cast<float4*>(rec + c0) = make_float4(t[0], t[1], t[2], t[3]);
    }
    A.scan[row] = make_float4(0.f, 0.f, 0.f, 0.f);
    A.link[row] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// -------------------------------------------------------------------------------------------------
// exact return recurrence of nstep_return.py:69-72: newest row first, each step evaluated in fp64 (unfused
// multiply then add) and rounded to fp32 on store.  One warp walks one episode from its last row to its first.
// `r` holds the rewards of rows jb+lane (zero where invalid); returns this lane's G and updates (acc, first).
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ float exact_return_chunk(float r, int jb, int L, double gamma, float& acc, bool& first) {
  float mine = 0.f;
  const int lane = lane_id();
#pragma unroll 4
  for (int i = 31; i >= 0; --i) {
    const float ri = __shfl_sync(kFull, r, i);
    if (jb + i < L) {
      acc = first ? ri : (float)__dadd_rn((double)ri, __dmul_rn((double)acc, gamma));
      first = false;
    }
    if (lane == i) mine = acc;
  }
  return mine;
}

// -------------------------------------------------------------------------------------------------
// link records of one episode (common.cuh), one warp; the scan records of the episode must be written and visible.
// -------------------------------------------------------------------------------------------------
__device__ void build_link_records(const ArenaDev& A, int64_t s, int L, double gamma) {
  const int lane = lane_id();
  // goal-agnostic return-to-go: GA_j = (ga_j - 1) + gamma * GA_{j+1}, walked from the last row in fp64
  double acc = 0.0;
  for (int jb = ((L - 1) / 32) * 32; jb >= 0; jb -= 32) {
    const int j = jb + lane;
    const bool valid = j < L;
    const int64_t row = ring_row(s, valid ? j : 0, A.capacity);
    const float ga = valid ? A.scan[row].z : 0.f;
    double mine = 0.0;
    for (int i = 31; i >= 0; --i) {
      const float gi = __shfl_sync(kFull, ga, i);
      if (jb + i < L) acc = ((double)gi - 1.0) + acc * gamma;
      if (lane == i) mine = acc;
    }
    if (valid) A.link[row] = make_float4((float)mine, ga, 0.f, 0.f);
  }
  __syncwarp();
  // chain of bit-identical achieved goals: lane <-> row j looks for the nearest later row with the same hash, verified
  const bool chain_ok = L <= 32767;
  for (int jb = 0; jb < L; jb += 32) {
    const int j = jb + lane;
    if (j >= L) continue;
    const int64_t row = ring_row(s, j, A.capacity);
    const float4 me = A.scan[row];
    const bool nan = (__float_as_uint(me.w) & 1u) != 0u;
    int next = 0;
    if (chain_ok && !nan) {
      for (int k = j + 1; k < L; ++k) {
        const int64_t rk = ring_row(s, k, A.capacity);
        const float4 o = A.scan[rk];  // written earlier in this launch: a coherent load, not ld.global.nc
        if (__float_as_uint(o.x) == __float_as_uint(me.x) && __float_as_uint(o.y) == __float_as_uint(me.y) &&
            rows_equal(A, row, rk)) {
          next = k - j;
          reinterpret_cast<int*>(A.link + rk)[3] = next;  // the successor's distance back to this row
          break;
        }
      }
    }
    reinterpret_cast<int*>(A.link + row)[2] = next | (nan ? (1 << 30) : 0) | (chain_ok ? 0 : (int)0x80000000);
  }
}

template <int LPR>
__global__ void __launch_bounds__(256)
commit_kernel(ArenaDev A, int32_t n_eps, const int64_t* __restrict__ ep_begin, const int32_t* __restrict__ ep_len,
              double gamma, int with_returns, RewardSpec rs) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = lane_id();
  if (warp >= n_eps) return;
  const int64_t s = ep_begin[warp];
  const int L = ep_len[warp];
  const int64_t e = ring_row(s, L - 1, A.capacity);
  const bool want_ga = rs.op != FDQL_REWARD_NONE && A.wide_ag >= 0 && A.wide_dg >= 0 && A.col_reward >= 0;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int jb = 0; jb < L; jb += 32) {
    const int j = jb + lane;
    const bool valid = j < L;
    const int64_t row = ring_row(s, valid ? j : 0, A.capacity);
    float* rec = A.rec + row * (int64_t)A.rec_stride;
    float Rdg = 0.f;
    bool d;
    uint64_t h = 0;
    bool has_nan = false;
    if (want_ga) eval_chunk<LPR, true>(A, rs, s, jb, L - 1, zero, Rdg, d);
    if (A.wide_ag >= 0) hash_chunk<LPR>(A, s, jb, L - 1, h, has_nan);
    if (valid) {
      rec[A.col_ep_start] = __int_as_float((int)s);
      rec[A.col_ep_end] = __int_as_float((int)e);
      const float ga = want_ga ? (float)((double)rec[A.col_reward] - (double)Rdg) : 0.f;
      A.scan[row] = make_float4(__uint_as_float((uint32_t)h), __uint_as_float((uint32_t)(h >> 32)), ga,
                                __uint_as_float(has_nan ? 1u : 0u));
    }
  }
  if (with_returns && A.col_mc_return >= 0 && A.col_reward >= 0) {
    float acc = 0.f;
    bool first = true;
    for (int jb = ((L - 1) / 32) * 32; jb >= 0; jb -= 32) {
      const int j = jb + lane;
      const bool valid = j < L;
      const int64_t row = ring_row(s, valid ? j : 0, A.capacity);
      float* rec = A.rec + row * (int64_t)A.rec_stride;
      const float r = valid ? rec[A.col_reward] : 0.f;
      const float g = exact_return_chunk(r, jb, L, gamma, acc, first);
      if (valid) rec[A.col_mc_return] = g;
    }
  }
  if (A.wide_ag >= 0) {
    __syncwarp();  // the scan records of the whole episode are in place
    build_link_records(A, s, L, gamma);
  }
}

// -------------------------------------------------------------------------------------------------
// write-time hindsight copy, her.py:55-95 (+ the inner NStepReturn flush, quirk Q5): one warp per episode.
// Reward = RewardSpec evaluates R(ag_j, g*) and R(ag_j, dg_j) with the device functor; GivenReward loads them (common.cuh).
// -------------------------------------------------------------------------------------------------
template <int LPR, class Reward>
__global__ void __launch_bounds__(256)
her_flush_kernel(ArenaDev A, int32_t n_eps, const int64_t* __restrict__ src_begin, const int32_t* __restrict__ ep_len,
                 const int64_t* __restrict__ dst_begin, const int64_t* __restrict__ goal_row, Reward rw, double gamma,
                 int with_returns) {
  constexpr bool given = kGivenReward<Reward>;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = lane_id();
  if (warp >= n_eps) return;
  const int64_t s = src_begin[warp], d0 = dst_begin[warp], grow = goal_row[warp];
  const int L = ep_len[warp];
  const int64_t dend = ring_row(d0, L - 1, A.capacity);
  float4 gstar;
  int64_t p0 = 0;  // first packed row of this episode (GivenReward)
  if constexpr (given) p0 = packed_first_row(ep_len, warp);
  else gstar = load_goal_slice<LPR>(A, grow);
  // wide keys: verbatim copy, except desired_goal := g*
  for (int w = 0; w < A.n_wide; ++w) {
    const WideSlab W = A.wide[w];
    const int items = L * W.vecs;
    for (int i = lane; i < items; i += 32) {
      const int j = i / W.vecs, v = i - j * W.vecs;
      const int64_t srow = (w == A.wide_dg) ? grow : ring_row(s, j, A.capacity);
      const WideSlab& S = (w == A.wide_dg) ? A.wide[A.wide_ag] : W;
      const float4 x = ldg4(S.base + srow * (int64_t)S.stride + 4 * v);
      *reinterpret_cast<float4*>(W.base + ring_row(d0, j, A.capacity) * (int64_t)W.stride + 4 * v) = x;
    }
  }
  // records: relabelled reward / task_done / episode_step, new extents
  int seg_first = 0;  // episode-relative index of the first row of the current synthetic episode
  for (int jb = 0; jb < L; jb += 32) {
    const int j = jb + lane;
    const bool valid = j < L;
    float Rg, Rdg = 0.f;
    bool dn, has_nan;
    uint64_t h;
    if constexpr (given) {
      Rg = valid ? rw.reward[p0 + j] : 0.f;
      dn = valid && rw.done[p0 + j] != 0;
      Rdg = valid ? rw.reward_dg[p0 + j] : 0.f;
    } else {
      bool dtmp;
      eval_chunk<LPR, false>(A, rw, s, jb, L - 1, gstar, Rg, dn);
      if (A.wide_dg >= 0) eval_chunk<LPR, true>(A, rw, s, jb, L - 1, gstar, Rdg, dtmp);
    }
    hash_chunk<LPR>(A, s, jb, L - 1, h, has_nan);  // achieved_goal is copied verbatim: same hash as the source row
    const unsigned bal = __ballot_sync(kFull, valid && dn);
    if (valid) {
      const int64_t srow = ring_row(s, j, A.capacity), drow = ring_row(d0, j, A.capacity);
      const float* rs_ = A.rec + srow * (int64_t)A.rec_stride;
      float* rd = A.rec + drow * (int64_t)A.rec_stride;
      for (int c = 0; c < A.rec_stride; c += 4)
        *reinterpret_cast<float4*>(rd + c) = *reinterpret_cast<const float4*>(rs_ + c);
      const unsigned below = bal & ((1u << lane) - 1u);
      const int f = below ? (jb + 32 - __clz(below)) : seg_first;
      const double r = A.col_reward >= 0 ? (double)rs_[A.col_reward] : 0.0;
      const float ga = (float)(r - (double)Rdg);
      if (A.col_reward >= 0) rd[A.col_reward] = (float)((r - (double)Rdg) + (double)Rg);
      if (A.col_task_done >= 0) rd[A.col_task_done] = dn ? 1.f : 0.f;
      if (A.col_ep_step >= 0) {
        const float step_f = A.rec[ring_row(s, f, A.capacity) * (int64_t)A.rec_stride + A.col_ep_step];
        rd[A.col_ep_step] = rs_[A.col_ep_step] - step_f;
      }
      rd[A.col_ep_start] = __int_as_float((int)d0);
      rd[A.col_ep_end] = __int_as_float((int)dend);
      A.scan[drow] = make_float4(__uint_as_float((uint32_t)h), __uint_as_float((uint32_t)(h >> 32)), ga,
                                 __uint_as_float(has_nan ? 1u : 0u));
      A.link[drow] = A.link[srow];  // same achieved goals and goal-agnostic rewards: same chain (distances) and GA
    }
    if (bal) seg_first = jb + 32 - __clz(bal);
  }
  __syncwarp();
  if (with_returns && A.col_mc_return >= 0 && A.col_reward >= 0) {
    float acc = 0.f;
    bool first = true;
    for (int jb = ((L - 1) / 32) * 32; jb >= 0; jb -= 32) {
      const int j = jb + lane;
      const bool valid = j < L;
      float* rd = A.rec + ring_row(d0, valid ? j : 0, A.capacity) * (int64_t)A.rec_stride;
      const float r = valid ? rd[A.col_reward] : 0.f;
      const float g = exact_return_chunk(r, jb, L, gamma, acc, first);
      if (valid) rd[A.col_mc_return] = g;
    }
  }
}

// -------------------------------------------------------------------------------------------------
// quirk Q3 (nstep_return.py:33-34,50-57): when the episode buffer reaches n_step rows the reference stores the oldest row
// once more, with the return truncated after n_step rewards, and never removes it.  One warp: copy row src -> dst, then
// run the exact recurrence over the rewards of rows src .. src+n_step-1.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) q3_duplicate_kernel(ArenaDev A, int64_t src, int32_t n_step, int64_t dst, double gamma) {
  const int lane = lane_id();
  for (int w = 0; w < A.n_wide; ++w) {
    const WideSlab W = A.wide[w];
    for (int v = lane; v < W.vecs; v += 32)
      *reinterpret_cast<float4*>(W.base + dst * (int64_t)W.stride + 4 * v) = ldg4(W.base + src * (int64_t)W.stride + 4 * v);
  }
  for (int c = lane; c < A.rec_stride; c += 32) {
    float v = A.rec[src * (int64_t)A.rec_stride + c];
    if (c == A.col_ep_start || c == A.col_ep_end) v = __int_as_float(-1);  // a lone row: never relabelled at sample time
    A.rec[dst * (int64_t)A.rec_stride + c] = v;
  }
  if (lane == 0) {
    A.scan[dst] = make_float4(0.f, 0.f, 0.f, 0.f);
    A.link[dst] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (A.col_mc_return < 0 || A.col_reward < 0) return;
  float acc = 0.f, g0 = 0.f;
  bool first = true;
  for (int jb = ((n_step - 1) / 32) * 32; jb >= 0; jb -= 32) {
    const int j = jb + lane;
    const bool valid = j < n_step;
    const float r = valid ? A.rec[ring_row(src, valid ? j : 0, A.capacity) * (int64_t)A.rec_stride + A.col_reward] : 0.f;
    const float g = exact_return_chunk(r, jb, n_step, gamma, acc, first);
    if (jb == 0) g0 = g;
  }
  __syncwarp();
  if (lane == 0) A.rec[dst * (int64_t)A.rec_stride + A.col_mc_return] = g0;
}

// The ring head has just moved over the rows before `r`.  If row r belongs to a committed episode that began before it, that
// episode has lost its first rows: the survivors r .. ep_end still carry the old extents, whose start now lies in a newer
// episode.  They become uncommitted (extents -1): never relabelled at sample time, gathered verbatim -- which is all the
// reference can do with the rows of an episode it has partly overwritten.  One block.
__global__ void __launch_bounds__(256) invalidate_survivors_kernel(ArenaDev A, int64_t r) {
  __shared__ int sh[2];
  if (threadIdx.x == 0) {
    const float* rec = A.rec + r * (int64_t)A.rec_stride;
    sh[0] = __float_as_int(rec[A.col_ep_start]);
    sh[1] = __float_as_int(rec[A.col_ep_end]);
  }
  __syncthreads();
  const int es = sh[0], ee = sh[1];
  if (es < 0 || ee < 0 || es == (int)r) return;
  const int64_t n = (int64_t)ee - r + (ee < r ? A.capacity : 0) + 1;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    float* rec = A.rec + ring_row(r, i, A.capacity) * (int64_t)A.rec_stride;
    rec[A.col_ep_start] = __int_as_float(-1);
    rec[A.col_ep_end] = __int_as_float(-1);
  }
}

// called with the range [a->top, a->top + n) that is about to be (over)written, before the cursor advances
static void note_overwrite(Arena* a, int64_t n) {
  const int64_t cap = a->dev.capacity;
  if (n <= 0 || n >= cap) {
    a->pending_inval_row = -1;
    if (n >= cap) a->rows_written = cap;
    return;
  }
  const int64_t end = a->top + n;  // one past the last written row, before the modulo
  const int64_t r = end % cap;
  // row r holds data only if the ring has been written that far before
  a->pending_inval_row = (a->rows_written >= cap || r < a->rows_written) ? r : -1;
  if (end >= cap) a->rows_written = cap;
  else if (end > a->rows_written) a->rows_written = end;
}

int flush_pending_invalidation(const Arena* ca, cudaStream_t st) {
  Arena* a = const_cast<Arena*>(ca);
  if (a->pending_inval_row < 0) return FDQL_OK;
  invalidate_survivors_kernel<<<1, 256, 0, st>>>(a->dev, a->pending_inval_row);
  a->pending_inval_row = -1;
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int check_packed_rows(const Arena* a, int32_t n_eps, const int32_t* ep_len, int64_t n_rows, cudaStream_t st) {
  std::vector<int32_t> len(n_eps);
  FDQL_CUDA(cudaMemcpyAsync(len.data(), ep_len, sizeof(int32_t) * n_eps, cudaMemcpyDeviceToHost, st));
  FDQL_CUDA(cudaStreamSynchronize(st));
  int64_t sum = 0;
  for (int e = 0; e < n_eps; ++e) {
    FDQL_REQUIRE(len[e] >= 1 && len[e] <= a->dev.capacity, "ep_len[%d] = %d is not in [1, capacity]", e, len[e]);
    sum += len[e];
  }
  FDQL_REQUIRE(sum == n_rows, "n_rows = %lld but the episodes hold %lld rows", (long long)n_rows, (long long)sum);
  return FDQL_OK;
}

std::mutex& cursor_mutex() {
  static std::mutex m;
  return m;
}

// rows [first, first + n) (mod capacity) were (over)written: their leaves of the priority store become q_max or 0 (per.cu).
// Consecutive writes coalesce into one interval; when the short list is full its last entry grows to the whole ring.
static void note_per_rows(Arena* a, int64_t first, int64_t n) {
  const int64_t cap = a->dev.capacity;
  if (a->per == nullptr || n <= 0) return;
  if (n > cap) n = cap;
  if (a->n_per_pending > 0) {
    int64_t* last = a->per_pending[a->n_per_pending - 1];
    if ((last[0] + last[1]) % cap == first) {
      last[1] = last[1] + n > cap ? cap : last[1] + n;
      return;
    }
    if (a->n_per_pending == 4) {
      last[0] = 0;
      last[1] = cap;
      return;
    }
  }
  a->per_pending[a->n_per_pending][0] = first;
  a->per_pending[a->n_per_pending][1] = n;
  ++a->n_per_pending;
}

static void advance_cursor(Arena* a, int64_t n) {
  std::lock_guard<std::mutex> lk(cursor_mutex());
  note_per_rows(a, a->top, n);
  const int64_t cap = a->dev.capacity, top = a->top;
  int64_t mx;
  if (n >= cap) mx = cap - 1;
  else if (top + n < cap) mx = top + n;
  else mx = (top <= cap - 2) ? cap - 1 : top + n - cap;
  a->top = (top + n) % cap;
  if (mx > a->len) a->len = mx;  // len = max(top, len) after every row: saturates at capacity-1 (quirk Q1)
}

}  // namespace fdql

using namespace fdql;

extern "C" {

const char* fdql_last_error(void) { return fdql::g_err; }
int fdql_version(void) { return 100; }

int fdql_arena_create(int64_t capacity, int32_t n_keys, const int32_t* widths, const int32_t* roles, int32_t device,
                      fdql_arena** out) {
  FDQL_REQUIRE(out != nullptr && widths != nullptr, "null argument");
  FDQL_REQUIRE(capacity >= 2 && capacity < (1ll << 31), "capacity must be in [2, 2^31)");
  FDQL_REQUIRE(n_keys >= 1 && n_keys <= FDQL_MAX_KEYS, "n_keys must be in [1, %d]", FDQL_MAX_KEYS);
  FDQL_CUDA(cudaSetDevice(device));
  fdql_arena* a = new fdql_arena();
  memset(static_cast<Arena*>(a), 0, sizeof(Arena));
  a->n_keys = n_keys;
  a->device = device;
  a->pending_inval_row = -1;
  ArenaDev& D = a->dev;
  D.capacity = capacity;
  D.col_reward = D.col_task_done = D.col_ep_done = D.col_ep_step = D.col_mc_return = -1;
  D.wide_ag = D.wide_dg = -1;
  for (int k = 0; k < n_keys; ++k) {
    const int w = widths[k], role = roles ? roles[k] : FDQL_ROLE_NONE;
    if (w < 1) {
      set_error("key %d has width %d", k, w);
      delete a;
      return FDQL_EINVAL;
    }
    a->widths[k] = w;
    a->roles[k] = role;
    a->key_wide[k] = a->key_col[k] = -1;
    const bool goal = role == FDQL_ROLE_ACHIEVED_GOAL || role == FDQL_ROLE_DESIRED_GOAL;
    if (w == 1 && !goal) {
      const int c = D.n_scal++;
      D.scal_key[c] = k;
      a->key_col[k] = c;
      if (role == FDQL_ROLE_REWARD) D.col_reward = c;
      if (role == FDQL_ROLE_TASK_DONE) D.col_task_done = c;
      if (role == FDQL_ROLE_EPISODE_DONE) D.col_ep_done = c;
      if (role == FDQL_ROLE_EPISODE_STEP) D.col_ep_step = c;
      if (role == FDQL_ROLE_MC_RETURN) D.col_mc_return = c;
    } else {
      const int s = D.n_wide++;
      D.wide[s].width = w;
      D.wide[s].stride = (w + 3) / 4 * 4;
      D.wide[s].vecs = D.wide[s].stride / 4;
      D.wide[s].key = k;
      a->key_wide[k] = s;
      if (role == FDQL_ROLE_ACHIEVED_GOAL) D.wide_ag = s;
      if (role == FDQL_ROLE_DESIRED_GOAL) D.wide_dg = s;
    }
  }
  if (D.wide_ag >= 0 && D.wide_dg >= 0 && D.wide[D.wide_ag].width != D.wide[D.wide_dg].width) {
    set_error("achieved_goal and desired_goal widths differ");
    delete a;
    return FDQL_EINVAL;
  }
  D.col_ep_start = D.n_scal;
  D.col_ep_end = D.n_scal + 1;
  D.rec_stride = (D.n_scal + 2 + 3) / 4 * 4;
  size_t total = 0;
  auto alloc = [&](float** p, size_t n_floats) -> bool {
    const size_t b = n_floats * sizeof(float);
    if (cudaMalloc(reinterpret_cast<void**>(p), b) != cudaSuccess) return false;
    cudaMemset(*p, 0, b);
    total += b;
    return true;
  };
  bool ok = true;
  for (int s = 0; s < D.n_wide && ok; ++s) ok = alloc(&D.wide[s].base, (size_t)capacity * D.wide[s].stride);
  ok = ok && alloc(&D.rec, (size_t)capacity * D.rec_stride);
  ok = ok && alloc(reinterpret_cast<float**>(&D.scan), (size_t)capacity * 4);
  ok = ok && alloc(reinterpret_cast<float**>(&D.link), (size_t)capacity * 4);
  ok = ok && alloc(&a->reward_params_dev, kMaxRewardParams + 4);
  ok = ok && alloc(reinterpret_cast<float**>(&a->fused_ws), 4 * kFusedSlots + 2048);  // (+ 8 KB for probe builds)
  if (!ok) {
    set_error("cudaMalloc failed while allocating the arena (%zu bytes so far): %s", total,
              cudaGetErrorString(cudaGetLastError()));
    fdql_arena_destroy(a);
    return FDQL_ENOMEM;
  }
  cudaDeviceGetAttribute(&a->num_sms, cudaDevAttrMultiProcessorCount, device);
  a->bytes = (int64_t)total;
  FDQL_CUDA(cudaDeviceSynchronize());
  *out = a;
  return FDQL_OK;
}

int fdql_arena_destroy(fdql_arena* a) {
  if (!a) return FDQL_OK;
  for (int s = 0; s < a->dev.n_wide; ++s)
    if (a->dev.wide[s].base) cudaFree(a->dev.wide[s].base);
  if (a->dev.rec) cudaFree(a->dev.rec);
  if (a->dev.scan) cudaFree(a->dev.scan);
  if (a->dev.link) cudaFree(a->dev.link);
  if (a->reward_params_dev) cudaFree(a->reward_params_dev);
#ifdef FDQL_FUSED_ROLE_CLOCK
  if (a->fused_ws) {
    unsigned long long h[40];
    cudaDeviceSynchronize();
    cudaMemcpy(h, reinterpret_cast<unsigned long long*>(a->fused_ws + 4 * kFusedSlots) + 3 * 256, sizeof(h), cudaMemcpyDeviceToHost);
    if (h[2]) fprintf(stderr, "[role clock] %llu launches: gap between launches (last role end -> next block 0 start) avg %.2f us; block 0 loss role %.1f us, gather role %.1f us\n",
                      h[2], (double)h[1] / h[2] / 1e3, (double)h[3] / (h[2] + 1) / 1e3, (double)h[4] / (h[2] + 1) / 1e3);
    if (h[2]) {
      fprintf(stderr, "[role clock] gap histogram (us: launches):");
      for (int i = 0; i < 32; ++i)
        if (h[8 + i]) fprintf(stderr, " %d:%llu", i, h[8 + i]);
      fprintf(stderr, "\n");
    }
  }
#endif
  if (a->fused_ws) cudaFree(a->fused_ws);
  if (a->stage_dev) cudaFree(a->stage_dev);
  if (a->step_dev) cudaFree(a->step_dev);
  if (a->step_sync_ready) {
    for (int i = 0; i < 3; ++i) cudaStreamDestroy(a->step_streams[i]);
    for (int i = 0; i < 8; ++i) cudaEventDestroy(a->step_events[i]);
    for (int i = 0; i < a->n_slice_events; ++i) cudaEventDestroy(a->slice_events[i]);
    free(a->slice_events);
  }
  delete a;
  return FDQL_OK;
}

int fdql_arena_info(const fdql_arena* a, int64_t* capacity, int64_t* top, int64_t* len, int64_t* bytes) {
  FDQL_REQUIRE(a != nullptr, "null arena");
  if (capacity) *capacity = a->dev.capacity;
  if (top) *top = a->top;
  if (len) *len = a->len;
  if (bytes) *bytes = a->bytes;
  return FDQL_OK;
}

int fdql_arena_set_cursor(fdql_arena* a, int64_t top, int64_t len) {
  FDQL_REQUIRE(a != nullptr, "null arena");
  FDQL_REQUIRE(top >= 0 && top < a->dev.capacity && len >= 0 && len <= a->dev.capacity, "cursor out of range");
  std::lock_guard<std::mutex> lk(cursor_mutex());  // a length change moves the priority store's eligible range (per.cu)
  a->top = top;
  a->len = len;
  a->pending_inval_row = -1;
  if (len + 1 > a->rows_written) a->rows_written = len + 1 > a->dev.capacity ? a->dev.capacity : len + 1;
  return FDQL_OK;
}

int fdql_arena_key_view(const fdql_arena* a, int32_t key, float** base, int64_t* row_stride, int32_t* col) {
  FDQL_REQUIRE(a != nullptr && key >= 0 && key < a->n_keys, "bad key");
  if (a->key_wide[key] >= 0) {
    const WideSlab& W = a->dev.wide[a->key_wide[key]];
    *base = W.base;
    *row_stride = W.stride;
    *col = 0;
  } else {
    *base = a->dev.rec;
    *row_stride = a->dev.rec_stride;
    *col = a->key_col[key];
  }
  return FDQL_OK;
}

int fdql_arena_link_state(fdql_arena* a, int32_t set, double* gamma, int32_t* state) {
  FDQL_REQUIRE(a != nullptr && gamma != nullptr && state != nullptr, "null argument");
  if (set) {
    FDQL_REQUIRE(*state >= 0 && *state <= 2, "bad link state");
    a->link_gamma = *gamma;
    a->link_state = *state;
  } else {
    *gamma = a->link_gamma;
    *state = a->link_state;
  }
  return FDQL_OK;
}

int fdql_arena_meta_view(const fdql_arena* a, int32_t which, float** base, int64_t* row_stride, int32_t* col) {
  FDQL_REQUIRE(a != nullptr && which >= 0 && which <= 3, "bad meta column");
  if (which == 2) {
    *base = reinterpret_cast<float*>(a->dev.scan);
    *row_stride = 4;
    *col = 2;
  } else if (which == 3) {
    *base = reinterpret_cast<float*>(a->dev.link);
    *row_stride = 4;
    *col = 0;
  } else {
    *base = a->dev.rec;
    *row_stride = a->dev.rec_stride;
    *col = which == 0 ? a->dev.col_ep_start : a->dev.col_ep_end;
  }
  return FDQL_OK;
}

int fdql_arena_append(fdql_arena* a, int64_t n_rows, const float* const* src, void* stream) {
  FDQL_REQUIRE(a != nullptr && src != nullptr, "null argument");
  FDQL_REQUIRE(n_rows >= 0 && n_rows <= a->dev.capacity, "n_rows must be in [0, capacity]");
  if (n_rows == 0) return FDQL_OK;
  SrcPtrs sp;
  for (int k = 0; k < a->n_keys; ++k) {
    FDQL_REQUIRE(src[k] != nullptr, "source pointer for key %d is null", k);
    sp.p[k] = src[k];
  }
  int64_t widest = 1;
  for (int s = 0; s < a->dev.n_wide; ++s) widest = widest > a->dev.wide[s].vecs ? widest : a->dev.wide[s].vecs;
  int64_t blocks = (n_rows * widest + 255) / 256;
  const int64_t cap_blocks = (int64_t)a->num_sms * 8;
  if (blocks > cap_blocks) blocks = cap_blocks;
  note_overwrite(a, n_rows);
  { int rc = flush_pending_invalidation(a, (cudaStream_t)stream); if (rc) return rc; }
  append_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a->dev, sp, n_rows, a->top, a->append_src_stride, a->append_squash);
  FDQL_CUDA(cudaGetLastError());
  advance_cursor(a, n_rows);
  return FDQL_OK;
}

int fdql_arena_append_packed_host(fdql_arena* a, int64_t n_rows, const float* packed_host, int32_t row_floats,
                                  const int32_t* key_offsets_host, uint32_t flags, void* stream) {
  FDQL_REQUIRE(a != nullptr && packed_host != nullptr && key_offsets_host != nullptr, "null argument");
  FDQL_REQUIRE(n_rows >= 0 && n_rows <= a->dev.capacity, "n_rows must be in [0, capacity]");
  FDQL_REQUIRE(row_floats >= 1, "bad row size");
  if (n_rows == 0) return FDQL_OK;
  for (int k = 0; k < a->n_keys; ++k)
    FDQL_REQUIRE(key_offsets_host[k] >= 0 && key_offsets_host[k] + a->widths[k] <= row_floats, "key %d does not fit the packed row", k);
  if (flags & FDQL_APPEND_SQUASH_REWARDS) FDQL_REQUIRE(a->dev.col_reward >= 0, "squashed rewards need a reward key");
  const size_t need = (size_t)n_rows * row_floats * sizeof(float);
  if (need > a->stage_bytes) {
    FDQL_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (a->stage_dev) cudaFree(a->stage_dev);
    a->stage_dev = nullptr;
    a->stage_bytes = 0;
    FDQL_CUDA(cudaMalloc(&a->stage_dev, need));
    a->stage_bytes = need;
  }
  // ONE host-to-device copy for the whole block; the append kernel then reads the keys with the packed row stride
  FDQL_CUDA(cudaMemcpyAsync(a->stage_dev, packed_host, need, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  const float* dev_ptrs[FDQL_MAX_KEYS];
  for (int k = 0; k < a->n_keys; ++k) dev_ptrs[k] = static_cast<const float*>(a->stage_dev) + key_offsets_host[k];
  a->append_src_stride = row_floats;
  a->append_squash = (flags & FDQL_APPEND_SQUASH_REWARDS) ? 1 : 0;
  const int rc = fdql_arena_append(a, n_rows, dev_ptrs, stream);
  a->append_src_stride = 0;
  a->append_squash = 0;
  return rc;
}

int fdql_arena_append_host(fdql_arena* a, int64_t n_rows, const float* const* src_host, void* stream) {
  FDQL_REQUIRE(a != nullptr && src_host != nullptr, "null argument");
  FDQL_REQUIRE(n_rows >= 0 && n_rows <= a->dev.capacity, "n_rows must be in [0, capacity]");
  if (n_rows == 0) return FDQL_OK;
  size_t need = 0;
  for (int k = 0; k < a->n_keys; ++k) need += ((size_t)n_rows * a->widths[k] * sizeof(float) + 255) / 256 * 256;
  if (need > a->stage_bytes) {
    FDQL_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (a->stage_dev) cudaFree(a->stage_dev);
    a->stage_dev = nullptr;
    a->stage_bytes = 0;
    FDQL_CUDA(cudaMalloc(&a->stage_dev, need));
    a->stage_bytes = need;
  }
  const float* dev_ptrs[FDQL_MAX_KEYS];
  size_t off = 0;
  for (int k = 0; k < a->n_keys; ++k) {
    const size_t b = (size_t)n_rows * a->widths[k] * sizeof(float);
    float* d = reinterpret_cast<float*>(static_cast<char*>(a->stage_dev) + off);
    FDQL_CUDA(cudaMemcpyAsync(d, src_host[k], b, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    dev_ptrs[k] = d;
    off += (b + 255) / 256 * 256;
  }
  return fdql_arena_append(a, n_rows, dev_ptrs, stream);
}

int fdql_q3_duplicate(fdql_arena* a, int64_t src_row, int32_t n_step, int64_t dst_row, double gamma, void* stream) {
  FDQL_REQUIRE(a != nullptr, "null arena");
  FDQL_REQUIRE(src_row >= 0 && src_row < a->dev.capacity && dst_row >= 0 && dst_row < a->dev.capacity, "row out of range");
  FDQL_REQUIRE(n_step >= 1 && n_step <= a->dev.capacity, "bad n_step");
  { int rc = flush_pending_invalidation(a, (cudaStream_t)stream); if (rc) return rc; }
  q3_duplicate_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(a->dev, src_row, n_step, dst_row, gamma);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int fdql_arena_reserve(fdql_arena* a, int64_t n_rows, int64_t* first_row) {
  FDQL_REQUIRE(a != nullptr && n_rows >= 0 && n_rows <= a->dev.capacity, "bad reserve");
  if (first_row) *first_row = a->top;
  note_overwrite(a, n_rows);  // no stream here: the survivors are invalidated by the next call that has one
  advance_cursor(a, n_rows);
  return FDQL_OK;
}

#define FDQL_DISPATCH_LPR(lpr, ...)                     \
  switch (lpr) {                                        \
    case 1: { constexpr int LPR = 1; __VA_ARGS__; } break;   \
    case 2: { constexpr int LPR = 2; __VA_ARGS__; } break;   \
    case 4: { constexpr int LPR = 4; __VA_ARGS__; } break;   \
    case 8: { constexpr int LPR = 8; __VA_ARGS__; } break;   \
    case 16: { constexpr int LPR = 16; __VA_ARGS__; } break; \
    default: { constexpr int LPR = 32; __VA_ARGS__; } break; \
  }

int fdql_commit_episodes(fdql_arena* a, int32_t n_eps, const int64_t* ep_begin, const int32_t* ep_len, double gamma,
                         int32_t with_returns, int32_t reward_op, const float* reward_params_host, int32_t n_params,
                         void* stream) {
  FDQL_REQUIRE(a != nullptr && n_eps >= 0, "bad argument");
  if (n_eps == 0) return FDQL_OK;
  FDQL_REQUIRE(ep_begin != nullptr && ep_len != nullptr, "null episode table");
  RewardSpec rs;
  int rc = upload_reward_spec(a, reward_op, reward_params_host, n_params, (cudaStream_t)stream, &rs);
  if (rc) return rc;
  rc = flush_pending_invalidation(a, (cudaStream_t)stream);
  if (rc) return rc;
  int lpr = 1;
  if (a->dev.wide_ag >= 0) {
    FDQL_REQUIRE(a->dev.wide[a->dev.wide_ag].vecs <= 32, "goal wider than 128 floats is not supported");
    lpr = lanes_per_row(a->dev.wide[a->dev.wide_ag].vecs);
  }
  const unsigned blocks = (unsigned)(((int64_t)n_eps * 32 + 255) / 256);
  if (a->link_state == 0) {
    a->link_gamma = gamma;
    a->link_state = 1;
  } else if (a->link_state == 1 && a->link_gamma != gamma) {
    a->link_state = 2;  // mixed discounts: sample-time relabelling falls back to the tail scan
  }
  FDQL_DISPATCH_LPR(lpr, (commit_kernel<LPR><<<blocks, 256, 0, (cudaStream_t)stream>>>(a->dev, n_eps, ep_begin, ep_len, gamma,
                                                                                         with_returns, rs)));
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int fdql_her_flush_episodes(fdql_arena* a, int32_t n_eps, const int64_t* src_begin, const int32_t* ep_len,
                            const int64_t* dst_begin, const int64_t* goal_row, int32_t reward_op,
                            const float* reward_params_host, int32_t n_params, double gamma, int32_t with_returns,
                            void* stream) {
  FDQL_REQUIRE(a != nullptr && n_eps >= 0, "bad argument");
  if (n_eps == 0) return FDQL_OK;
  FDQL_REQUIRE(src_begin && ep_len && dst_begin && goal_row, "null episode table");
  FDQL_REQUIRE(a->dev.wide_ag >= 0, "hindsight flush needs an achieved_goal key");
  FDQL_REQUIRE(reward_op != FDQL_REWARD_NONE, "hindsight flush needs a reward functor");
  FDQL_REQUIRE(a->dev.wide[a->dev.wide_ag].vecs <= 32, "goal wider than 128 floats is not supported");
  RewardSpec rs;
  int rc = upload_reward_spec(a, reward_op, reward_params_host, n_params, (cudaStream_t)stream, &rs);
  if (rc) return rc;
  rc = flush_pending_invalidation(a, (cudaStream_t)stream);
  if (rc) return rc;
  const int lpr = lanes_per_row(a->dev.wide[a->dev.wide_ag].vecs);
  const unsigned blocks = (unsigned)(((int64_t)n_eps * 32 + 255) / 256);
  FDQL_DISPATCH_LPR(lpr, (her_flush_kernel<LPR, RewardSpec><<<blocks, 256, 0, (cudaStream_t)stream>>>(
                             a->dev, n_eps, src_begin, ep_len, dst_begin, goal_row, rs, gamma, with_returns)));
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int fdql_her_flush_episodes_given(fdql_arena* a, int32_t n_eps, const int64_t* src_begin, const int32_t* ep_len,
                                  const int64_t* dst_begin, const int64_t* goal_row, int64_t n_rows, const float* reward,
                                  const uint8_t* done, const float* reward_dg, double gamma, int32_t with_returns, void* stream) {
  FDQL_REQUIRE(a != nullptr && n_eps >= 0 && n_rows >= 0, "bad argument");
  if (n_eps == 0) {
    FDQL_REQUIRE(n_rows == 0, "n_rows = %lld but there are no episodes", (long long)n_rows);
    return FDQL_OK;
  }
  FDQL_REQUIRE(src_begin && ep_len && dst_begin && goal_row, "null episode table");
  FDQL_REQUIRE(reward && done && reward_dg, "null reward, done or reward_dg array");
  FDQL_REQUIRE(a->dev.wide_ag >= 0 && a->dev.wide_dg >= 0, "hindsight flush needs achieved_goal and desired_goal keys");
  FDQL_REQUIRE(a->dev.wide[a->dev.wide_ag].vecs <= 32, "goal wider than 128 floats is not supported");
  int rc = check_packed_rows(a, n_eps, ep_len, n_rows, (cudaStream_t)stream);
  if (rc) return rc;
  rc = flush_pending_invalidation(a, (cudaStream_t)stream);
  if (rc) return rc;
  const GivenReward g{reward, done, reward_dg};
  const int lpr = lanes_per_row(a->dev.wide[a->dev.wide_ag].vecs);
  const unsigned blocks = (unsigned)(((int64_t)n_eps * 32 + 255) / 256);
  FDQL_DISPATCH_LPR(lpr, (her_flush_kernel<LPR, GivenReward><<<blocks, 256, 0, (cudaStream_t)stream>>>(
                             a->dev, n_eps, src_begin, ep_len, dst_begin, goal_row, g, gamma, with_returns)));
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

}  // extern "C"
