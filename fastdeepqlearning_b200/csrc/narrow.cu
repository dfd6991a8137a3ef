// Narrow keys (uint8 / int8 storage, common.cuh NarrowSlab): the gather that widens their rows to fp32 next to the fp32 gathers, the
// row copies of the write-time hindsight flush and of quirk Q3, and the append.  franQ's ring keeps each array's numpy dtype
// (franQ/Replay/replay_memory.py:23-35) and its TorchDataLoader casts to fp32 on the way out (torch_dataloader.py:36); these kernels
// do the same with the cast in registers.  A narrow row moves as whole 16-byte chunks (a row's stride is a multiple of 16 bytes).
#include "common.cuh"

namespace fdql {

constexpr int kNarrowThreads = 256;

__device__ __forceinline__ uint4 ld_stream_u4(const uint8_t* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// the four bytes of w as exact fp32 values: zero extension (uint8) or sign extension (int8)
__device__ __forceinline__ float4 widen4(uint32_t w, bool sgn) {
  if (sgn)
    return make_float4(__int2float_rn((int)(w << 24) >> 24), __int2float_rn((int)(w << 16) >> 24), __int2float_rn((int)(w << 8) >> 24),
                       __int2float_rn((int)w >> 24));
  return make_float4(__uint2float_rn(w & 0xffu), __uint2float_rn((w >> 8) & 0xffu), __uint2float_rn((w >> 16) & 0xffu),
                     __uint2float_rn(w >> 24));
}

struct NarrowGatherArgs {
  NarrowSet N;
  float* out[FDQL_MAX_KEYS];  // by narrow slab index; NULL: not gathered
  const int64_t* starts;
  int64_t n;               // windows of the whole batch (row pitch of the time-major outputs)
  int64_t b_begin, b_end;  // windows of this launch
  int64_t len;             // window modulus, as the fp32 gather of the same call
  int32_t T;
};

// the float4 of output words w = 4 bytes of the row as exact fp32 values: a 128-bit store where it is whole and aligned, else a scalar
// tail (e: its first element)
__device__ __forceinline__ void widen_store_word(uint32_t w, float* __restrict__ dst, int e, int width, bool sgn, bool vec) {
  const float4 f = widen4(w, sgn);
  if (vec && e + 4 <= width) {
    st_stream4(dst + e, f);
  } else {
    const float fs[4] = {f.x, f.y, f.z, f.w};
    for (int m = 0; m < 4 && e + m < width; ++m) st_stream1(dst + e + m, fs[m]);
  }
}

// G threads per (window, t) row, G from the widest row: 1 for rows of one chunk (bit-flip states), 4 up to 4 chunks, a warp up to 64
// chunks, a block above (image rows: 1764 chunks at 84x84x4).  Rows are taken t-major so that neighbouring groups write neighbouring
// output rows.  Each thread loads up to kU chunks (16 B each, streaming) before it stores any.  With G >= 4 the GW = min(G, 32) lanes
// that loaded GW consecutive chunks (4 GW words) then store them as 4 rounds of GW consecutive float4 -- lane s of round r widens word
// GW r + s, fetched by warp shuffles -- so that every store instruction writes one contiguous run instead of 16 B every 64 B.
template <int G>
__global__ void __launch_bounds__(kNarrowThreads) narrow_gather_kernel(const __grid_constant__ NarrowGatherArgs g) {
  constexpr int kU = 4;
  constexpr int kGroups = kNarrowThreads / G;
  constexpr int GW = G < 32 ? G : 32;
  const int64_t n_groups = (int64_t)gridDim.x * kGroups;
  const int64_t group = (int64_t)blockIdx.x * kGroups + threadIdx.x / G;
  const int sub = threadIdx.x % G;
  const int lane = lane_id();
  const int s = lane & (GW - 1);          // lane within the GW exchanging lanes
  const int lane0 = lane & ~(GW - 1);     // their first lane
  const unsigned mask = GW == 32 ? kFull : (((1u << GW) - 1u) << lane0);
  const int64_t nb = g.b_end - g.b_begin;
  const int64_t rows = nb * g.T;
  for (int k = 0; k < g.N.n; ++k) {
    float* __restrict__ o = g.out[k];
    if (o == nullptr) continue;
    const NarrowSlab S = g.N.s[k];
    const int chunks = S.stride >> 4;
    const bool sgn = S.dtype == FDQL_DTYPE_I8;
    const bool vec = (S.width & 3) == 0 && (reinterpret_cast<uintptr_t>(o) & 15) == 0;
    for (int64_t i = group; i < rows; i += n_groups) {
      const int t = (int)(i / nb);
      const int64_t b = g.b_begin + (i - (int64_t)t * nb);
      const int64_t row = ring_row(window_start(__ldg(g.starts + b), g.len), t, g.len);
      const uint8_t* src = S.base + row * (int64_t)S.stride;
      float* dst = o + ((int64_t)t * g.n + b) * S.width;
      for (int c0 = 0; c0 < chunks; c0 += kU * G) {  // (the same trip count for the whole group)
        uint4 x[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const int c = c0 + u * G + sub;
          x[u] = c < chunks ? ld_stream_u4(src + 16 * c) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          if constexpr (G == 1) {
            if (c0 + u < chunks) {
              const uint32_t words[4] = {x[u].x, x[u].y, x[u].z, x[u].w};
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (16 * (c0 + u) + 4 * q < S.width) widen_store_word(words[q], dst, 16 * (c0 + u) + 4 * q, S.width, sgn, vec);
            }
          } else {
            const int cw = c0 + u * G + (sub & ~(GW - 1));  // first chunk of the exchanging lanes
            if (cw >= chunks) continue;                      // (uniform over them)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const int from = lane0 + (GW / 4) * r + (s >> 2);
              const uint32_t w0 = __shfl_sync(mask, x[u].x, from), w1 = __shfl_sync(mask, x[u].y, from);
              const uint32_t w2 = __shfl_sync(mask, x[u].z, from), w3 = __shfl_sync(mask, x[u].w, from);
              const int q = s & 3;
              const uint32_t w = q == 0 ? w0 : q == 1 ? w1 : q == 2 ? w2 : w3;
              const int e = 16 * cw + 4 * (GW * r + s);
              if (e < S.width) widen_store_word(w, dst, e, S.width, sgn, vec);
            }
          }
        }
      }
    }
  }
}

// one block column per episode (blockIdx.x), blockIdx.y splitting its chunks; with src_begin == NULL the single row src_row -> dst_row
__global__ void __launch_bounds__(kNarrowThreads)
narrow_copy_kernel(NarrowSet N, const int64_t* __restrict__ src_begin, const int32_t* __restrict__ ep_len,
                   const int64_t* __restrict__ dst_begin, int64_t src_row, int64_t dst_row) {
  int64_t s = src_row, d = dst_row;
  int L = 1;
  if (src_begin != nullptr) {
    s = src_begin[blockIdx.x];
    d = dst_begin[blockIdx.x];
    L = ep_len[blockIdx.x];
  }
  const int64_t step = (int64_t)gridDim.y * blockDim.x;
  for (int k = 0; k < N.n; ++k) {
    const NarrowSlab S = N.s[k];
    const int chunks = S.stride >> 4;
    const int64_t items = (int64_t)L * chunks;
    for (int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; i < items; i += step) {
      const int j = (int)(i / chunks), c = (int)(i - (int64_t)j * chunks);
      const uint4 x = ld_stream_u4(S.base + ring_row(s, j, N.capacity) * (int64_t)S.stride + 16 * c);
      *reinterpret_cast<uint4*>(S.base + ring_row(d, j, N.capacity) * (int64_t)S.stride + 16 * c) = x;
    }
  }
}

struct NarrowSrc {
  const uint8_t* p[FDQL_MAX_KEYS];  // by narrow slab index
};

// source row r of slab k at src.p[k] + r * row_bytes (row_bytes 0: dense, the slab's width); 16-byte loads where the source allows,
// bytes for the rest.  The padding bytes of a ring row (past width) are written as zeros.
__global__ void __launch_bounds__(kNarrowThreads)
narrow_append_kernel(NarrowSet N, NarrowSrc src, int64_t n_rows, int64_t row_bytes, int64_t top) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  for (int k = 0; k < N.n; ++k) {
    const NarrowSlab S = N.s[k];
    const uint8_t* __restrict__ sp = src.p[k];
    const int chunks = S.stride >> 4;
    const int64_t rs = row_bytes > 0 ? row_bytes : S.width;
    const bool vec_ok = (rs % 16) == 0 && (reinterpret_cast<uintptr_t>(sp) & 15) == 0;
    const int64_t items = n_rows * chunks;
    for (int64_t i = tid; i < items; i += nthreads) {
      const int64_t r = i / chunks;
      const int c = (int)(i - r * chunks);
      const uint8_t* q = sp + r * rs + 16 * c;
      uint4 x;
      if (vec_ok && 16 * c + 16 <= S.width) {
        x = ld_stream_u4(q);
      } else {
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        const int m = min(16, S.width - 16 * c);
        for (int e = 0; e < m; ++e) w[e >> 2] |= (uint32_t)q[e] << (8 * (e & 3));
        x = make_uint4(w[0], w[1], w[2], w[3]);
      }
      const int64_t row = ring_row(top, r % N.capacity, N.capacity);
      *reinterpret_cast<uint4*>(S.base + row * (int64_t)S.stride + 16 * c) = x;
    }
  }
}

static int64_t persistent_blocks(const Arena* a, int64_t want) {
  const int64_t cap = (int64_t)a->num_sms * (2048 / kNarrowThreads);
  return want < 1 ? 1 : (want > cap ? cap : want);
}

int launch_narrow_gather(const Arena* a, int64_t n, int64_t b_begin, int64_t b_end, int32_t T, int64_t len, const int64_t* starts,
                         float* const* out, cudaStream_t st) {
  if (a->narrow.n == 0 || b_end <= b_begin) return FDQL_OK;
  NarrowGatherArgs g;
  memset(&g, 0, sizeof(g));
  g.N = a->narrow;
  int widest = 0;
  for (int k = 0; k < a->narrow.n; ++k) {
    g.out[k] = out[a->narrow.s[k].key];
    if (g.out[k] != nullptr && a->narrow.s[k].stride / 16 > widest) widest = a->narrow.s[k].stride / 16;
  }
  if (widest == 0) return FDQL_OK;
  FDQL_REQUIRE(starts != nullptr, "the narrow gather needs the window starts");
  g.starts = starts;
  g.n = n;
  g.b_begin = b_begin;
  g.b_end = b_end;
  g.len = len;
  g.T = T;
  const int64_t rows = (b_end - b_begin) * (int64_t)T;
#define FDQL_LAUNCH_NARROW(GV)                                                                                          \
  narrow_gather_kernel<GV><<<(unsigned)persistent_blocks(a, (rows + kNarrowThreads / GV - 1) / (kNarrowThreads / GV)), \
                             kNarrowThreads, 0, st>>>(g)
  if (widest <= 1) FDQL_LAUNCH_NARROW(1);
  else if (widest <= 4) FDQL_LAUNCH_NARROW(4);
  else if (widest <= 64) FDQL_LAUNCH_NARROW(32);
  else FDQL_LAUNCH_NARROW(256);
#undef FDQL_LAUNCH_NARROW
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int launch_narrow_copy(const Arena* a, int32_t n_eps, const int64_t* src_begin, const int32_t* ep_len, const int64_t* dst_begin,
                       int64_t src_row, int64_t dst_row, cudaStream_t st) {
  if (a->narrow.n == 0 || n_eps <= 0) return FDQL_OK;
  const dim3 grid((unsigned)n_eps, src_begin != nullptr ? 4u : 1u);
  narrow_copy_kernel<<<grid, kNarrowThreads, 0, st>>>(a->narrow, src_begin, ep_len, dst_begin, src_row, dst_row);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

int launch_narrow_append(const Arena* a, int64_t n_rows, const void* const* src, int64_t src_row_bytes, int64_t top, cudaStream_t st) {
  if (a->narrow.n == 0 || n_rows <= 0) return FDQL_OK;
  NarrowSrc sp;
  int64_t widest = 1;
  for (int k = 0; k < a->narrow.n; ++k) {
    sp.p[k] = static_cast<const uint8_t*>(src[a->narrow.s[k].key]);
    widest = a->narrow.s[k].stride / 16 > widest ? a->narrow.s[k].stride / 16 : widest;
  }
  narrow_append_kernel<<<(unsigned)persistent_blocks(a, (n_rows * widest + kNarrowThreads - 1) / kNarrowThreads), kNarrowThreads, 0,
                         st>>>(a->narrow, sp, n_rows, src_row_bytes, top);
  FDQL_CUDA(cudaGetLastError());
  return FDQL_OK;
}

}  // namespace fdql
