// Octree depth-wise convolution, fp32, with its two backward kernels: the native form of the
// reference's `dwconv.core` extension (libs/dwconv/csrc/dwconv.cu, pybind.cpp:10-14).
//   k_dwconv           : out[i,c] = sum_k w[k,c] * data[neigh[i,k],c]      (dwconv.cu:25-42)
//                        (called with the inverse table it is the input gradient)
//   k_dwconv_inverse   : ineigh[neigh[i,k],k] = i, -1 elsewhere            (dwconv.cu:74-85)
//   k_dwconv_wgrad     : per-chunk partials of dw[k,c] = sum_i grad[i,c] * data[neigh[i,k],c]
//   k_dwconv_wgrad_fold: fixed-order sum of the partials                   (dwconv.cu:45-72)
// Neighbour tables are int32 or int64 [rows, K], 1 <= K <= 27; entries outside [0, n_in) are
// empty taps.  These kernels serve training-side callers; the embedding forward uses k_cpe_ln
// (layers.cu), whose bf16 operands and fused LayerNorm are a different contract.
#include "common.cuh"

namespace hfl {

namespace {

constexpr int kMaxTaps = 27;
constexpr int kWgradChunks = 512;      // target number of row chunks of the weight gradient
constexpr int kWgradMinRows = 64;      // least rows per chunk
constexpr int kWgradWarps = 8;         // warps per weight-gradient block

__device__ __forceinline__ void zero(float& a) { a = 0.f; }
__device__ __forceinline__ void zero(float2& a) { a = make_float2(0.f, 0.f); }
__device__ __forceinline__ void zero(float4& a) { a = make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void fma_v(float& a, float w, float x) { a = fmaf(w, x, a); }
__device__ __forceinline__ void fma_v(float2& a, float2 w, float2 x) {
  a.x = fmaf(w.x, x.x, a.x); a.y = fmaf(w.y, x.y, a.y);
}
__device__ __forceinline__ void fma_v(float4& a, float4 w, float4 x) {
  a.x = fmaf(w.x, x.x, a.x); a.y = fmaf(w.y, x.y, a.y);
  a.z = fmaf(w.z, x.z, a.z); a.w = fmaf(w.w, x.w, a.w);
}
__device__ __forceinline__ void add_v(float2& a, float2 b) { a.x += b.x; a.y += b.y; }
__device__ __forceinline__ void add_v(float& a, float b) { a += b; }

// lane k < K: entry k of row r as a data row (-1: empty tap, row out of range or lane >= K)
template <typename IdxT>
__device__ __forceinline__ int32_t load_taps(const IdxT* __restrict__ neigh, int64_t r, int64_t n_rows, int K,
                                             int lane, int64_t n_in) {
  if (r >= n_rows || lane >= K) return -1;
  const IdxT e = __ldg(neigh + r * K + lane);
  return (e >= 0 && (int64_t)e < n_in) ? (int32_t)e : -1;
}

// ---------------------------------------------------------------------------
// Forward / input gradient.  One warp per output row; a lane owns NV vectors of W = sizeof(T)/4
// channels per pass over the row (vector j of a pass: column cb + 32 j + lane, coalesced).  The
// row's entries are read once (lane k holds tap k) and broadcast by shuffle, only the occupied taps
// are visited, TAPS of them at a time so that their gathers are in flight together, and the next
// row's entries are requested before this row's gathers.  Each channel accumulates from 0.f in
// ascending tap order with fmaf -- the order of the reference kernel (dwconv.cu:30-41).
// ---------------------------------------------------------------------------
template <typename T, int NV, typename IdxT>
__global__ void __launch_bounds__(256)
k_dwconv(const float* __restrict__ data, const IdxT* __restrict__ neigh, const float* __restrict__ w,
         int64_t n_out, int64_t n_in, int K, int C, float* __restrict__ out) {
  constexpr int TAPS = 4;
  const int lane = threadIdx.x & 31;
  const int CV = C / (int)(sizeof(T) / 4);
  const T* __restrict__ dv = reinterpret_cast<const T*>(data);
  const T* __restrict__ wv = reinterpret_cast<const T*>(w);
  T* __restrict__ ov = reinterpret_cast<T*>(out);
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  int32_t my_next = load_taps(neigh, warp0, n_out, K, lane, n_in);
  for (int64_t r = warp0; r < n_out; r += nwarps) {
    const int32_t my = my_next;
    my_next = load_taps(neigh, r + nwarps, n_out, K, lane, n_in);
    const unsigned occupied = __ballot_sync(0xffffffffu, my >= 0);
    for (int cb = 0; cb < CV; cb += 32 * NV) {
      T acc[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) zero(acc[v]);
      unsigned todo = occupied;
      while (todo) {
        int k[TAPS];
        T a[TAPS][NV];
#pragma unroll
        for (int u = 0; u < TAPS; ++u) {
          k[u] = __ffs(todo) - 1;              // -1 once the set is exhausted (warp-uniform)
          todo &= todo - 1;
          const int32_t e = __shfl_sync(0xffffffffu, my, k[u] & 31);
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const int cv = cb + 32 * v + lane;
            if (k[u] >= 0 && cv < CV) a[u][v] = dv[(int64_t)e * CV + cv];
          }
        }
#pragma unroll
        for (int u = 0; u < TAPS; ++u) {
          if (k[u] < 0) break;
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const int cv = cb + 32 * v + lane;
            if (cv < CV) fma_v(acc[v], __ldg(wv + k[u] * CV + cv), a[u][v]);
          }
        }
      }
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int cv = cb + 32 * v + lane;
        if (cv < CV) ov[r * CV + cv] = acc[v];
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Inverse table: out is pre-filled with -1; a (j,k) hit by several rows keeps the largest row.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void atomic_max(int32_t* p, int32_t v) { atomicMax(p, v); }
__device__ __forceinline__ void atomic_max(int64_t* p, int64_t v) {
  atomicMax(reinterpret_cast<long long*>(p), (long long)v);
}

template <typename IdxT>
__global__ void __launch_bounds__(256)
k_dwconv_inverse(const IdxT* __restrict__ neigh, int64_t total, int K, int64_t n_data, IdxT* __restrict__ out) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const IdxT e = __ldg(neigh + t);
    if (e >= 0 && (int64_t)e < n_data) {
      const int64_t i = t / K;
      atomic_max(out + (int64_t)e * K + (t - i * K), (IdxT)i);
    }
  }
}

// ---------------------------------------------------------------------------
// Weight gradient, deterministic without float atomics.  Block (x, y) owns rows
// [x R, (x+1) R) and vector columns [32 y, 32 y + 32) (vectors of W = sizeof(T)/4 channels);
// R depends on n only (dwconv_wgrad_rows), never on the SM count, so every launch on every GPU
// adds the same products in the same order.  Warp w takes rows x R + w, + kWgradWarps, ... and
// keeps its [K] column partials in registers; the warps are folded in warp order through shared
// memory and the block writes ws[x][k][c].  k_dwconv_wgrad_fold then sums the chunks: warp q of a
// fold block takes chunks q, q + 8, ... in order, and the 8 warp sums are added in warp order.
// ---------------------------------------------------------------------------
template <typename T, typename IdxT>
__global__ void __launch_bounds__(kWgradWarps * 32)
k_dwconv_wgrad(const float* __restrict__ grad, const float* __restrict__ data, const IdxT* __restrict__ neigh,
               int64_t n, int64_t n_in, int K, int C, int64_t rows_per_chunk, float* __restrict__ ws) {
  constexpr int GROUP = 9;                     // gathers issued together
  __shared__ T s_acc[kMaxTaps * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int CV = C / (int)(sizeof(T) / 4);
  const int cv = blockIdx.y * 32 + lane;
  const bool col = cv < CV;
  const T* __restrict__ gv = reinterpret_cast<const T*>(grad);
  const T* __restrict__ dv = reinterpret_cast<const T*>(data);
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_chunk;
  const int64_t r1 = min(n, r0 + rows_per_chunk);
  T acc[kMaxTaps];
#pragma unroll
  for (int k = 0; k < kMaxTaps; ++k) zero(acc[k]);
  int32_t my_next = load_taps(neigh, r0 + warp, r1, K, lane, n_in);
  for (int64_t r = r0 + warp; r < r1; r += kWgradWarps) {
    const int32_t my = my_next;
    my_next = load_taps(neigh, r + kWgradWarps, r1, K, lane, n_in);
    T g;
    zero(g);
    if (col) g = gv[r * CV + cv];
#pragma unroll
    for (int k0 = 0; k0 < kMaxTaps; k0 += GROUP) {
      int32_t e[GROUP];
      T x[GROUP];
#pragma unroll
      for (int u = 0; u < GROUP; ++u) {
        e[u] = __shfl_sync(0xffffffffu, my, k0 + u);     // -1 for k >= K (lanes >= K hold -1)
        if (e[u] >= 0 && col) x[u] = dv[(int64_t)e[u] * CV + cv];
      }
#pragma unroll
      for (int u = 0; u < GROUP; ++u)
        if (e[u] >= 0 && col) fma_v(acc[k0 + u], g, x[u]);
    }
  }
  for (int w = 0; w < kWgradWarps; ++w) {
    if (warp == w) {
#pragma unroll
      for (int k = 0; k < kMaxTaps; ++k) {
        if (k < K) {
          if (w == 0) s_acc[k * 32 + lane] = acc[k];
          else add_v(s_acc[k * 32 + lane], acc[k]);
        }
      }
    }
    __syncthreads();
  }
  T* __restrict__ wsv = reinterpret_cast<T*>(ws) + (int64_t)blockIdx.x * K * CV;
  for (int i = threadIdx.x; i < K * 32; i += blockDim.x) {
    const int k = i >> 5, c = blockIdx.y * 32 + (i & 31);
    if (c < CV) wsv[(int64_t)k * CV + c] = s_acc[i];
  }
}

__global__ void __launch_bounds__(256)
k_dwconv_wgrad_fold(const float* __restrict__ ws, int64_t chunks, int64_t KC, float* __restrict__ dw) {
  __shared__ float s[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * 32 + lane;
  float acc = 0.f;
  if (i < KC)
    for (int64_t p = warp; p < chunks; p += 8) acc += __ldg(ws + p * KC + i);
  s[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && i < KC) {
    float t = s[0][lane];
#pragma unroll
    for (int q = 1; q < 8; ++q) t += s[q][lane];
    dw[i] = t;
  }
}

int64_t dwconv_wgrad_rows(int64_t n) {
  int64_t r = ceil_div(ceil_div(n, kWgradChunks), kWgradWarps) * kWgradWarps;
  return r < kWgradMinRows ? kWgradMinRows : r;
}

bool aligned(const void* p, size_t a) { return ((uintptr_t)p % a) == 0; }

template <typename IdxT>
int launch_dwconv(const float* data, const IdxT* neigh, const float* w, int64_t n_out, int64_t n_in, int32_t K,
                  int32_t C, float* out, cudaStream_t st) {
  const int grid = grid_for(n_out * 32, 256, kSMs * 16);
  const bool vec4 = C % 4 == 0 && aligned(data, 16) && aligned(w, 16) && aligned(out, 16);
  if (vec4 && C <= 128)
    HFL_LAUNCH((k_dwconv<float4, 1, IdxT><<<grid, 256, 0, st>>>(data, neigh, w, n_out, n_in, K, C, out)));
  else if (vec4)
    HFL_LAUNCH((k_dwconv<float4, 2, IdxT><<<grid, 256, 0, st>>>(data, neigh, w, n_out, n_in, K, C, out)));
  else if (C <= 32)
    HFL_LAUNCH((k_dwconv<float, 1, IdxT><<<grid, 256, 0, st>>>(data, neigh, w, n_out, n_in, K, C, out)));
  else
    HFL_LAUNCH((k_dwconv<float, 4, IdxT><<<grid, 256, 0, st>>>(data, neigh, w, n_out, n_in, K, C, out)));
  return HFL_OK;
}

template <typename IdxT>
int launch_wgrad(const float* grad, const float* data, const IdxT* neigh, int64_t n, int64_t n_in, int32_t K,
                 int32_t C, float* ws, cudaStream_t st) {
  const int64_t rows = dwconv_wgrad_rows(n), chunks = ceil_div(n, rows);
  const bool vec2 = C % 2 == 0 && aligned(grad, 8) && aligned(data, 8);
  const dim3 grid((unsigned)chunks, (unsigned)ceil_div(vec2 ? C / 2 : C, 32));
  if (vec2)
    HFL_LAUNCH((k_dwconv_wgrad<float2, IdxT><<<grid, kWgradWarps * 32, 0, st>>>(grad, data, neigh, n, n_in, K, C,
                                                                                rows, ws)));
  else
    HFL_LAUNCH((k_dwconv_wgrad<float, IdxT><<<grid, kWgradWarps * 32, 0, st>>>(grad, data, neigh, n, n_in, K, C,
                                                                               rows, ws)));
  return HFL_OK;
}

}  // namespace
}  // namespace hfl

using namespace hfl;

extern "C" {

int hfl_dwconv(const float* data, const void* neigh, int32_t neigh_i64, const float* w, int64_t n_out,
               int64_t n_in, int32_t K, int32_t C, float* out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(K >= 1 && K <= kMaxTaps && C >= 1, "K must be in [1, 27] and C >= 1");
  HFL_CHECK_ARG(C < (1 << 22), "C must be below 4194304");
  HFL_CHECK_ARG(n_out >= 0 && n_in >= 0, "negative row count");
  HFL_CHECK_ARG(n_out < (1ll << 31) && n_in < (1ll << 31), "row indices must fit 32 bits");
  if (n_out == 0) return HFL_OK;
  HFL_CHECK_ARG(neigh && w && out && (data || n_in == 0), "null argument");
  if (neigh_i64)
    return launch_dwconv(data, (const int64_t*)neigh, w, n_out, n_in, K, C, out, st);
  return launch_dwconv(data, (const int32_t*)neigh, w, n_out, n_in, K, C, out, st);
}

int hfl_dwconv_inverse(const void* neigh, int32_t neigh_i64, int64_t n_rows, int64_t n_data, int32_t K,
                       void* ineigh_out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(K >= 1 && K <= kMaxTaps, "K must be in [1, 27]");
  HFL_CHECK_ARG(n_rows >= 0 && n_data >= 0, "negative row count");
  HFL_CHECK_ARG(n_rows < (1ll << 31) && n_data < (1ll << 31), "row indices must fit 32 bits");
  if (n_data == 0) return HFL_OK;
  HFL_CHECK_ARG(ineigh_out && (neigh || n_rows == 0), "null argument");
  const size_t eb = neigh_i64 ? 8 : 4;
  HFL_CUDA(cudaMemsetAsync(ineigh_out, 0xff, (size_t)n_data * K * eb, st));     // every entry -1
  if (n_rows == 0) return HFL_OK;
  const int64_t total = n_rows * K;
  const int grid = grid_for(total, 256);
  if (neigh_i64)
    HFL_LAUNCH((k_dwconv_inverse<int64_t><<<grid, 256, 0, st>>>((const int64_t*)neigh, total, K, n_data,
                                                                 (int64_t*)ineigh_out)));
  else
    HFL_LAUNCH((k_dwconv_inverse<int32_t><<<grid, 256, 0, st>>>((const int32_t*)neigh, total, K, n_data,
                                                                 (int32_t*)ineigh_out)));
  return HFL_OK;
}

int64_t hfl_dwconv_wgrad_workspace_bytes(int64_t n, int32_t K, int32_t C) {
  if (n <= 0 || K < 1 || K > kMaxTaps || C < 1) return 0;
  return (int64_t)align_up((size_t)ceil_div(n, dwconv_wgrad_rows(n)) * K * C * sizeof(float));
}

int hfl_dwconv_wgrad(const float* grad, const float* data, const void* neigh, int32_t neigh_i64, int64_t n,
                     int64_t n_in, int32_t K, int32_t C, float* dw, void* ws, int64_t ws_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(K >= 1 && K <= kMaxTaps && C >= 1, "K must be in [1, 27] and C >= 1");
  HFL_CHECK_ARG(C < (1 << 22), "C must be below 4194304");
  HFL_CHECK_ARG(n >= 0 && n_in >= 0, "negative row count");
  HFL_CHECK_ARG(n < (1ll << 31) && n_in < (1ll << 31), "row indices must fit 32 bits");
  HFL_CHECK_ARG(dw, "null argument");
  if (n == 0) {                                  // no rows: the gradient is zero
    HFL_CUDA(cudaMemsetAsync(dw, 0, (size_t)K * C * sizeof(float), st));
    return HFL_OK;
  }
  HFL_CHECK_ARG(grad && neigh && (data || n_in == 0), "null argument");
  const int64_t need = hfl_dwconv_wgrad_workspace_bytes(n, K, C);
  if (!ws || ws_bytes < need)
    return fail(HFL_ERR_WORKSPACE, "dwconv weight-gradient workspace too small (%s%lld bytes needed)", "",
                (long long)need);
  HFL_CHECK_ARG(aligned(ws, 16), "workspace must be 16-byte aligned");
  int rc = neigh_i64 ? launch_wgrad(grad, data, (const int64_t*)neigh, n, n_in, K, C, (float*)ws, st)
                     : launch_wgrad(grad, data, (const int32_t*)neigh, n, n_in, K, C, (float*)ws, st);
  if (rc != HFL_OK) return rc;
  const int64_t KC = (int64_t)K * C;
  HFL_LAUNCH((k_dwconv_wgrad_fold<<<(unsigned)ceil_div(KC, 32), 256, 0, st>>>(
      (const float*)ws, ceil_div(n, dwconv_wgrad_rows(n)), KC, dw)));
  return HFL_OK;
}

}  // extern "C"
