// Shared device/host definitions for libfdql.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <type_traits>

#include "../../include/fdql.h"

namespace fdql {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ---- error plumbing ---------------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define FDQL_CUDA(call)                                                                       \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      fdql::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return FDQL_ECUDA;                                                                      \
    }                                                                                         \
  } while (0)
#define FDQL_REQUIRE(cond, ...)        \
  do {                                 \
    if (!(cond)) {                     \
      fdql::set_error(__VA_ARGS__);    \
      return FDQL_EINVAL;              \
    }                                  \
  } while (0)

// ---- arena layout in HBM ----------------------------------------------------------------------
// Wide keys (width >= 2, and goal keys of any width): one slab [capacity, stride], stride = width rounded up
// to 4 floats so that every row starts 16B-aligned and is moved with 128-bit loads.
// Width-1 keys: packed side by side into one record per row, [capacity, rec_stride], followed by two int32
// columns holding the episode extents (first/last row of the row's episode, -1 until committed).
// scan: [capacity] 16-byte scan record per row, written when the row's episode is committed:
//   .x/.y  64-bit hash of the row's achieved_goal (-0 folded into +0, so equal vectors have equal hashes)
//   .z     goal-agnostic reward r - R(ag, dg) (her.py:65-68)
//   .w     bit 0: the achieved_goal holds a NaN (never equal to anything)
// Episode scans read it as one contiguous run of 16 B per row; for equality rewards the hash decides "differs" exactly
// and only hash matches are verified against the full vectors.
// link: [capacity] 16-byte link record per row, written with the scan record (equality rewards only need THIS at sample time):
//   .x  goal-agnostic return-to-go  GA_j = sum_{m>=j} gamma^(m-j) (ga_m - 1)  over the rest of the real episode (fp64 sum, fp32 store)
//   .y  the goal-agnostic reward ga_j again (so that a window row needs one record, not two)
//   .z  int: bits 0-14 distance to the NEXT row of the episode with a bit-identical achieved_goal (0 = none; verified on the full
//            vectors when the chain is built), bit 30: the row's achieved_goal holds a NaN (equal to nothing), bit 31: no chain
//            (episode longer than 32767 rows)
//   .w  int: distance to the PREVIOUS such row (0 = none)
// Under an equality reward R(ag, g*) = 0 iff ag == g*, so the rows that hit a hindsight goal g* = achieved_goal[goal_row] are exactly
// the chain through goal_row, and the relabelled return is GA_t + sum_{hits m >= t} gamma^(m-t): O(hits) instead of O(tail).
struct WideSlab {
  float* base;
  int32_t stride;  // floats, multiple of 4
  int32_t width;   // floats
  int32_t key;     // caller's key index
  int32_t vecs;    // stride / 4
};

struct ArenaDev {
  int64_t capacity;
  int32_t n_wide, n_scal, rec_stride, pad0;
  WideSlab wide[FDQL_MAX_KEYS];
  float* rec;
  float4* scan;
  float4* link;
  int32_t scal_key[FDQL_MAX_KEYS];  // record column -> caller's key index
  int32_t col_ep_start, col_ep_end;
  int32_t col_reward, col_task_done, col_ep_done, col_ep_step, col_mc_return;  // record column or -1
  int32_t wide_ag, wide_dg;                                                    // index into wide[] or -1
};

struct OutPtrs {
  float* p[FDQL_MAX_KEYS];
};
struct SrcPtrs {
  const float* p[FDQL_MAX_KEYS];
};

constexpr int kMaxRewardParams = 2 + 128;
constexpr int kFusedSlots = 16;
struct RewardSpec {
  int32_t op;
  int32_t n_params;
  const float* params;  // device copy of {p, thr, w...} for WEIGHTED_PNORM, else unused
};

// ---- small device helpers ---------------------------------------------------------------------
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
// streaming (evict-first) 128-bit load/store for data touched once per launch
__device__ __forceinline__ float4 ld_stream4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float ld_stream1(const float* p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void st_stream4(float* p, const float4& v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_stream1(float* p, float v) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

__device__ __forceinline__ int64_t ring_row(int64_t base, int64_t off, int64_t cap) {
  int64_t r = base + off;
  return r >= cap ? r - cap : r;
}

__device__ __forceinline__ double shfl_down_f64(double v, int d) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_down_sync(kFull, lo, d);
  hi = __shfl_down_sync(kFull, hi, d);
  return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_idx_f64(double v, int src) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_sync(kFull, lo, src);
  hi = __shfl_sync(kFull, hi, src);
  return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_xor_f64(double v, int m) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_xor_sync(kFull, lo, m);
  hi = __shfl_xor_sync(kFull, hi, m);
  return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_up_f64(double v, int d) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_up_sync(kFull, lo, d);
  hi = __shfl_up_sync(kFull, hi, d);
  return __hiloint2double(hi, lo);
}

// host-side view of an arena (definition shared by the translation units)
struct Arena {
  ArenaDev dev;
  int32_t n_keys;
  int32_t widths[FDQL_MAX_KEYS];
  int32_t roles[FDQL_MAX_KEYS];
  int32_t key_wide[FDQL_MAX_KEYS];  // key -> index in dev.wide or -1
  int32_t key_col[FDQL_MAX_KEYS];   // key -> record column or -1
  int64_t top, len, bytes;
  int32_t device;
  float* reward_params_dev;  // kMaxRewardParams floats
  int* fused_ws;             // 4 * kFusedSlots zeroed ints: work counters of fdql_fused_pass launches (sample.cu)
  // staging for *_host entry points (allocated lazily, grown only when a larger call arrives)
  void* stage_dev;
  size_t stage_bytes;
  void* step_dev;  // fdql_hotpath_step_host: streams, critic outputs, aux, loss, grad
  size_t step_bytes;
  cudaStream_t step_streams[3];
  cudaEvent_t step_events[8];
  cudaEvent_t* slice_events;  // two per slice of fdql_hotpath_step_host (copies landed, kernels done), grown on demand
  int n_slice_events;
  int step_sync_ready;
  double link_gamma;    // discount the link records were built with
  int link_state;       // 0: none yet, 1: link_gamma valid, 2: episodes were committed with different discounts (links unusable)
  int num_sms;
  int32_t append_src_stride, append_squash;  // set around fdql_arena_append by the packed host form (see arena.cu)
  int64_t rows_written;        // rows [0, rows_written) of the ring have held data (capacity once it has wrapped)
  int64_t pending_inval_row;   // first row behind the write head whose episode may have lost its beginning (-1: none); see arena.cu
  // prioritized replay (per.cu): the arena's priority store, if one was created, and the ring intervals {first row, rows} written since
  // its last activation pass.  Writers only record them here (under cursor_mutex()); the PER calls apply them on their own stream.
  ::fdql_per* per;
  int64_t per_pending[4][2];
  int32_t n_per_pending;
};

int flush_pending_invalidation(const Arena* a, cudaStream_t st);
// serialises the host cursor (top, len) and the pending priority intervals between a writer thread and the PER calls of a reader
std::mutex& cursor_mutex();

int upload_reward_spec(const Arena* a, int32_t op, const float* params_host, int32_t n_params, cudaStream_t st,
                       RewardSpec* out);

// Reward source of the write-time flush kernels (her_flush_kernel, vmap_flush_kernel): either a RewardSpec, whose functor the kernel
// evaluates on the goals in the ring, or a GivenReward, whose per-row results a caller computed beforehand and packed episode after
// episode in the order of the episode table (fdql_her_flush_episodes_given, fdql_vmap_flush_episodes_given).
struct GivenReward {
  const float* reward;     // R(ag_i, goal): [n_rows] (hindsight flush) or [n_rows, V+1] (vmap fill)
  const uint8_t* done;     // done of the same pairs, non-zero = done
  const float* reward_dg;  // R(ag_i, dg_i) [n_rows] (hindsight flush; the vmap fill reads column V of `reward` instead)
};
template <class Reward>
constexpr bool kGivenReward = std::is_same<Reward, GivenReward>::value;

// First packed row of episode e in a GivenReward: the sum of ep_len[0 .. e), summed by the calling warp (all 32 lanes active).
__device__ __forceinline__ int64_t packed_first_row(const int32_t* __restrict__ ep_len, int e) {
  long long s = 0;
  for (int i = threadIdx.x & 31; i < e; i += 32) s += ep_len[i];
  for (int m = 16; m >= 1; m >>= 1) s += __shfl_xor_sync(kFull, s, m);
  return s;
}

// Host check of a *_given call: reads the device table ep_len[n_eps] back (synchronising `st`) and requires every length in
// [1, capacity] and their sum equal to n_rows, the rows of the packed arrays.
int check_packed_rows(const Arena* a, int32_t n_eps, const int32_t* ep_len, int64_t n_rows, cudaStream_t st);

}  // namespace fdql

struct fdql_arena;
namespace fdql {
// fused draw of the index / goal streams inside the gather (tile kernel only); the drawn streams are also written out
struct DrawSpec {
  int64_t range;
  int32_t goal_mode;
  float relabel_prob;
  uint64_t seed, counter;
  unsigned long long* counter_dev;
  int64_t* starts_out;
  uint8_t* flags_out;
  int64_t* goal_out;
  // fused pass (fdql_fused_pass): when set and the shape allows it, the gather is launched as the gather role of the fused pass
  // kernel together with this loss (a TqcArgs of tqc_group.cuh) and *fused is set to 1; otherwise the gather launches alone
  const void* fuse_tqc = nullptr;
  int* fused = nullptr;
  // prioritized fused pass (fdql_fused_pass_per): the starts come from this priority tree (a PerDraw of draw.cuh); only the fused
  // kernel draws them -- any shape it does not serve returns 1 with nothing launched
  const void* per = nullptr;
};
// returns FDQL_OK, an error, or (with draw != nullptr) 1 when this shape is not served by the fused kernel (nothing launched)
int launch_gather(const fdql_arena* a, int64_t n, int64_t b_begin, int64_t b_end, int32_t T, int64_t len, const int64_t* starts,
                  const uint8_t* flags, const int64_t* goal_rows, int32_t reward_op, const float* reward_params_host,
                  int32_t n_params, double gamma, uint32_t opts, int32_t batch_for_weight, float* const* out, float* aux_mask,
                  float* aux_contig, float* aux_weight, cudaStream_t st, const DrawSpec* draw = nullptr);
}

struct fdql_arena : fdql::Arena {};
