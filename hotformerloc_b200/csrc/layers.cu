// Warp-per-row gather / reduce kernels of the hot path (HBM- / L2-bound; SURVEY.md
// section 8 rows a5, a8 (first conv), a9, a12, a15):
//   k_stem_conv    : InputFeature('P') + OctreeConv 3^3 (3 -> 32) + LayerNorm + ReLU
//   k_cpe_ln       : x += LN(dwconv27(x)) [libs/dwconv/csrc/dwconv.cu:25-42 + CPE norm]
//                    fused with the block's pre-attention LayerNorm (bf16 GEMM operand)
//   k_ln_rows      : LayerNorm of gathered rows -> bf16 (relay-token / mixer operand)
//   k_rt_init      : relay-token init (masked window mean) + ADaPE window statistics
//                    + ADaPE fc1 (9 -> C, GELU)
//   k_pool_*       : attention pooling: column softmax statistics + weighted token sum
//   k_mixer_tail   : Mixer channel_proj / row_proj + L2 normalisation
// The residual stream is fp32 (x) with a bf16 shadow (xb) that feeds gathers and GEMMs.
// "hat" layout (hierarchical attention): K window tokens preceded by their relay token,
//   row(token t) = t + t / K + 1,  row(RT of window w) = w * (K + 1).
#include <stdlib.h>
#include <type_traits>

#include "common.cuh"
#include "ptx.cuh"

namespace hfl {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float gelu(float v) {
  return 0.5f * v * (1.0f + erff(v * 0.70710678118654752f));
}
// acc_lo += w.lo * a.lo, acc_hi += w.hi * a.hi for packed bf16 pairs: mixed-precision FMA (fp32 accumulate; the
// bf16 product is exact in fp32, so this equals fmaf on the converted values) -- no unpack instructions
__device__ __forceinline__ void fma_bf16_pair(float& lo, float& hi, uint32_t w, uint32_t a) {
  asm("{\n\t.reg .b16 wl, wh, al, ah;\n\tmov.b32 {wl, wh}, %2;\n\tmov.b32 {al, ah}, %3;\n\t"
      "fma.rn.f32.bf16 %0, wl, al, %0;\n\tfma.rn.f32.bf16 %1, wh, ah, %1;\n\t}"
      : "+f"(lo), "+f"(hi)
      : "r"(w), "r"(a));
}
__device__ __forceinline__ int64_t hat_row(int64_t t, int K) { return K ? t + t / K + 1 : t; }

template <int V>
__device__ __forceinline__ void load_bf16(const __nv_bfloat16* p, float (&v)[V]) {
  if constexpr (V == 8) {
    uint4 u = *reinterpret_cast<const uint4*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int j = 0; j < 4; ++j) { float2 f = __bfloat1622float2(h[j]); v[2 * j] = f.x; v[2 * j + 1] = f.y; }
  } else {
    uint2 u = *reinterpret_cast<const uint2*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int j = 0; j < 2; ++j) { float2 f = __bfloat1622float2(h[j]); v[2 * j] = f.x; v[2 * j + 1] = f.y; }
  }
}
template <int V>
__device__ __forceinline__ void store_bf16(__nv_bfloat16* p, const float (&v)[V]) {
  uint32_t w[V / 2];
#pragma unroll
  for (int j = 0; j < V / 2; ++j) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    w[j] = *reinterpret_cast<uint32_t*>(&h);
  }
  if constexpr (V == 8) *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  else *reinterpret_cast<uint2*>(p) = make_uint2(w[0], w[1]);
}
template <int V>
__device__ __forceinline__ void load_f32(const float* p, float (&v)[V]) {
#pragma unroll
  for (int j = 0; j < V / 4; ++j) {
    float4 f = reinterpret_cast<const float4*>(p)[j];
    v[4 * j] = f.x; v[4 * j + 1] = f.y; v[4 * j + 2] = f.z; v[4 * j + 3] = f.w;
  }
}
template <int V>
__device__ __forceinline__ void store_f32(float* p, const float (&v)[V]) {
#pragma unroll
  for (int j = 0; j < V / 4; ++j)
    reinterpret_cast<float4*>(p)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
// LayerNorm of a C = 32*V vector distributed over a warp (lane owns V contiguous channels)
template <int V>
__device__ __forceinline__ void warp_ln(float (&v)[V], const float* g, const float* b, int c0,
                                        float eps) {
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < V; ++j) s += v[j];
  const float mean = warp_sum(s) / (32.f * V);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < V; ++j) { float d = v[j] - mean; q += d * d; }
  const float rstd = rsqrtf(warp_sum(q) / (32.f * V) + eps);
  float gg[V], bb[V];
  load_f32<V>(g + c0, gg);
  load_f32<V>(b + c0, bb);
#pragma unroll
  for (int j = 0; j < V; ++j) v[j] = (v[j] - mean) * rstd * gg[j] + bb[j];
}

// Same with gamma / beta in shared memory in a "planar" layout: the V channels of a lane are split
// into V/4 planes of [32 lanes][4 floats], so every LDS.128 of a warp covers 512 contiguous bytes
// (a lane-major [lane][V] layout makes 32-byte lane strides: 2-way bank conflicts at V = 8).
template <int V>
__device__ __forceinline__ int planar_index(int c) {      // channel -> float index in the planar layout
  const int lane = c / V, j = c % V;
  return ((j >> 2) * 32 + lane) * 4 + (j & 3);
}
template <int V>
__device__ __forceinline__ void load_planar(const float* base, int lane, float (&v)[V]) {
#pragma unroll
  for (int jj = 0; jj < V / 4; ++jj) {
    const float4 f = *reinterpret_cast<const float4*>(base + (jj * 32 + lane) * 4);
    v[4 * jj] = f.x; v[4 * jj + 1] = f.y; v[4 * jj + 2] = f.z; v[4 * jj + 3] = f.w;
  }
}
template <int V>
__device__ __forceinline__ void warp_ln_planar(float (&v)[V], const float* g, const float* b, int lane,
                                               float eps) {
  // One reduction round for both moments (the two butterfly chains interleave): the CPE kernel is
  // bound by the latency of its per-row dependency chain, of which the four serial warp reductions of
  // the two-pass form were a quarter.  Sums are taken relative to this lane-0 element (shifted
  // moments), so the variance does not cancel when |mean| >> std.
  const float shift = __shfl_sync(0xffffffffu, v[0], 0);
  float s = 0.f, q = 0.f;
#pragma unroll
  for (int j = 0; j < V; ++j) { const float d = v[j] - shift; s += d; q = fmaf(d, d, q); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  const float inv_n = 1.f / (32.f * V);
  const float ms = s * inv_n;
  const float mean = shift + ms;
  const float rstd = rsqrtf(fmaxf(q * inv_n - ms * ms, 0.f) + eps);
  float gg[V], bb[V];
  load_planar<V>(g, lane, gg);
  load_planar<V>(b, lane, bb);
#pragma unroll
  for (int j = 0; j < V; ++j) v[j] = (v[j] - mean) * rstd * gg[j] + bb[j];
}

// ---------------------------------------------------------------------------
// stem: first OctreeConv (Cin = 3) on CUDA cores, one warp per leaf, lane = out channel
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_stem_conv(const float* __restrict__ leaf_pts, const int32_t* __restrict__ ne, int64_t n,
            float pscale, const float* __restrict__ w /*[81][32]*/, const float* __restrict__ g,
            const float* __restrict__ b, __nv_bfloat16* __restrict__ out) {
  __shared__ float sw[81 * 32];
  for (int i = threadIdx.x; i < 81 * 32; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp0; i < n; i += nwarps) {
    const int32_t my = lane < 27 ? __ldg(ne + i * 27 + lane) : -1;
    float fx = 0.f, fy = 0.f, fz = 0.f;
    if (my >= 0) {
      fx = leaf_pts[3 * (int64_t)my] * pscale - 1.0f;
      fy = leaf_pts[3 * (int64_t)my + 1] * pscale - 1.0f;
      fz = leaf_pts[3 * (int64_t)my + 2] * pscale - 1.0f;
    }
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 27; ++k) {
      const float x = __shfl_sync(0xffffffffu, fx, k);
      const float y = __shfl_sync(0xffffffffu, fy, k);
      const float z = __shfl_sync(0xffffffffu, fz, k);
      acc += x * sw[(3 * k) * 32 + lane] + y * sw[(3 * k + 1) * 32 + lane] + z * sw[(3 * k + 2) * 32 + lane];
    }
    const float mean = warp_sum(acc) * (1.f / 32.f);
    const float d = acc - mean;
    const float rstd = rsqrtf(warp_sum(d * d) * (1.f / 32.f) + 1e-5f);
    const float y = fmaxf(d * rstd * g[lane] + b[lane], 0.f);
    out[i * 32 + lane] = __float2bfloat16(y);
  }
}

// ---------------------------------------------------------------------------
// CPE + LayerNorm fusion.  One warp per row of the (hat or plain) layout.
// ---------------------------------------------------------------------------
struct CpeParams {
  float* x;                    // [rows, C] fp32 residual stream (updated in place)
  const __nv_bfloat16* xb;     // [rows, C] bf16 shadow (gather source, not modified)
  const int32_t* ne;           // [n, 27] neighbour table, token index space
  const __nv_bfloat16* w;      // [27, C] depth-wise weights (bf16: one 16 B load per lane and tap)
  const float *g_cpe, *b_cpe;  // CPE LayerNorm
  const float *g1, *b1;        // block norm1 (NULL: skip)
  __nv_bfloat16* y1;           // [rows, C] LN1(x) bf16 (NULL: skip)
  float* cpe_out;              // [n, C] when non-NULL: write LN(dwconv(x)) only, token-compact
  int64_t n, rows;             // real tokens, layout rows
  int K;                       // 0 = plain layout, else hat layout window size
};

template <int V>
__global__ void __launch_bounds__(256, 4) k_cpe_ln(const CpeParams p) {
  const int lane = threadIdx.x & 31;
  const int C = 32 * V, c0 = lane * V;
  // tap weights stay bf16 in smem: the kernel is bound by L1/shared-memory wavefronts (ncu: l1tex
  // 88 %), and a bf16 tap row costs 4 wavefronts per warp instead of 8; plus the four LayerNorm vectors
  __shared__ __align__(16) __nv_bfloat16 s_w[27 * 32 * V];
  __shared__ __align__(16) float s_ln[4 * 32 * V];
  for (int i = threadIdx.x; i < 27 * C; i += blockDim.x) s_w[i] = p.w[i];
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    const int q = planar_index<V>(i);
    s_ln[q] = p.g_cpe[i];
    s_ln[C + q] = p.b_cpe[i];
    s_ln[2 * C + q] = p.y1 ? p.g1[i] : 0.f;
    s_ln[3 * C + q] = p.y1 ? p.b1[i] : 0.f;
  }
  __syncthreads();
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  // token behind a layout row (-1: relay token / padding row) and its neighbour-table entry.
  // All row / token indices fit 32 bits (checked by the launcher): the divisions by the runtime
  // window size are 32-bit and happen once per row, never inside the tap loop.
  const uint32_t K = (uint32_t)p.K, n32 = (uint32_t)p.n;
  auto row_token = [&](int64_t r) -> int32_t {
    if (r >= p.rows) return -1;
    uint32_t t = (uint32_t)r;
    if (K) {
      const uint32_t w = t / (K + 1), s = t - w * (K + 1);
      if (s == 0) return -1;
      t = w * K + s - 1;
    }
    return t < n32 ? (int32_t)t : -1;
  };
  // lane k < 27 holds the LAYOUT ROW of neighbour k of the token (-1: empty)
  auto load_ne = [&](int32_t t) -> int32_t {
    int32_t ni = (t >= 0 && lane < 27) ? __ldg(p.ne + (int64_t)t * 27 + lane) : -1;
    if (K && ni >= 0) ni += (int32_t)((uint32_t)ni / K) + 1;
    return ni;
  };
  using Raw = typename std::conditional<V == 8, uint4, uint2>::type;
  constexpr int TAPS = 4;                    // gathers in flight per warp
  // the dependent chain per row is  ne -> gathers -> LN -> x;  the neighbour entries of the NEXT
  // row and the x row of THIS row are requested before the tap loop so that only the gathers'
  // latency is left on the chain.  (A chunked row schedule -- 64 consecutive rows per CTA for L1
  // reuse between Morton neighbours -- was measured: no change, the grid-strided one is kept.)
  int32_t t_next = row_token(warp0);
  int32_t my_next = load_ne(t_next);
  for (int64_t r = warp0; r < p.rows; r += nwarps) {
    const int32_t t = t_next;
    const int32_t my = my_next;
    t_next = row_token(r + nwarps);
    my_next = load_ne(t_next);
    float xv[V];
    if (!p.cpe_out) load_f32<V>(p.x + r * C + c0, xv);
    if (t >= 0) {
      float acc[V];
#pragma unroll
      for (int j = 0; j < V; ++j) acc[j] = 0.f;
      // visit only the occupied neighbours (about a third of the 27 taps on lidar surfaces),
      // TAPS at a time so that their gathers overlap; taps are accumulated in ascending order
      unsigned todo = __ballot_sync(0xffffffffu, my >= 0);
      while (todo) {
        int k[TAPS];
        Raw a[TAPS];
#pragma unroll
        for (int u = 0; u < TAPS; ++u) {
          k[u] = __ffs(todo) - 1;              // -1 once the set is exhausted (warp-uniform)
          todo &= todo - 1;
          const int32_t nrow = __shfl_sync(0xffffffffu, my, k[u] & 31);
          if (k[u] >= 0) a[u] = *reinterpret_cast<const Raw*>(p.xb + (int64_t)nrow * C + c0);
        }
#pragma unroll
        for (int u = 0; u < TAPS; ++u) {
          if (k[u] < 0) break;
          const Raw wr = *reinterpret_cast<const Raw*>(s_w + k[u] * C + c0);
          const uint32_t* aw = reinterpret_cast<const uint32_t*>(&a[u]);
          const uint32_t* ww = reinterpret_cast<const uint32_t*>(&wr);
#pragma unroll
          for (int j = 0; j < V / 2; ++j)       // bf16 x bf16 + fp32 in one instruction each (FHFMA.BF16, exact product)
            fma_bf16_pair(acc[2 * j], acc[2 * j + 1], ww[j], aw[j]);
        }
      }
      warp_ln_planar<V>(acc, s_ln, s_ln + C, lane, 1e-5f);
      if (p.cpe_out) {
        store_f32<V>(p.cpe_out + (int64_t)t * C + c0, acc);
        continue;
      }
#pragma unroll
      for (int j = 0; j < V; ++j) xv[j] += acc[j];
      store_f32<V>(p.x + r * C + c0, xv);
    } else {
      if (p.cpe_out) continue;               // relay token or padding row: no CPE
    }
    if (p.y1) {
      warp_ln_planar<V>(xv, s_ln + 2 * C, s_ln + 3 * C, lane, 1e-5f);
      store_bf16<V>(p.y1 + r * C + c0, xv);
    }
  }
}

// LayerNorm of gathered fp32 rows -> compact bf16 rows
template <int V>
__global__ void __launch_bounds__(256)
k_ln_rows(const float* __restrict__ x, const int32_t* __restrict__ rows, int64_t m,
          const float* __restrict__ g, const float* __restrict__ b, __nv_bfloat16* __restrict__ y) {
  const int lane = threadIdx.x & 31;
  const int C = 32 * V, c0 = lane * V;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp0; i < m; i += nwarps) {
    const int64_t r = rows ? (int64_t)__ldg(rows + i) : i;
    float v[V];
    load_f32<V>(x + r * C + c0, v);
    warp_ln<V>(v, g, b, c0, 1e-5f);
    store_bf16<V>(y + i * C + c0, v);
  }
}

// ---------------------------------------------------------------------------
// relay-token initialisation + ADaPE statistics / fc1, one warp per window
// ---------------------------------------------------------------------------
struct RtInitParams {
  float* x;                  // hat layout [n_win*(K+1), C]; RT rows written
  const float* src;          // NULL: average x's own token rows; else token-compact [n, C]
  const short4* xyzb;        // [n_win*K] token table
  int64_t n, n_win;
  int K, depth, mode;        // mode: 0 none, 3 pos, 6 var, 9 cov
  const float *w1, *b1;      // ADaPE fc1 [C, mode], [C]
  __nv_bfloat16* h;          // [n_win, C] GELU(fc1(stats)) bf16 (fc2 runs on the tensor cores)
  float* stats_out;          // [n_win, 9] optional (tests)
};

template <int V>
__global__ void __launch_bounds__(256) k_rt_init(const RtInitParams p) {
  const int lane = threadIdx.x & 31;
  const int C = 32 * V, c0 = lane * V;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const float cs = ldexpf(1.0f, 1 - p.depth);
  for (int64_t w = warp0; w < p.n_win; w += nwarps) {
    const int64_t t0 = w * p.K;
    const short id0 = p.xyzb[t0].w;
    // ---- masked mean of the window's token features ----
    float acc[V];
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = 0.f;
    int cnt = 0;
    for (int s = 0; s < p.K; ++s) {
      if (p.xyzb[t0 + s].w != id0) continue;                 // warp-uniform
      ++cnt;
      float v[V];
      if (p.src) {
        if (t0 + s < p.n) load_f32<V>(p.src + (t0 + s) * C + c0, v);
        else {
#pragma unroll
          for (int j = 0; j < V; ++j) v[j] = 0.f;
        }
      } else {
        load_f32<V>(p.x + (w * (p.K + 1) + 1 + s) * C + c0, v);
      }
#pragma unroll
      for (int j = 0; j < V; ++j) acc[j] += v[j];
    }
    const float inv = 1.0f / (float)cnt;
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] *= inv;
    store_f32<V>(p.x + w * (p.K + 1) * C + c0, acc);
    if (p.mode == 0) continue;
    // ---- window statistics of the node centres (models/octree.py:285-344) ----
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (int s = lane; s < p.K; s += 32) {
      const short4 q = p.xyzb[t0 + s];
      if (q.w != id0) continue;
      const bool real = t0 + s < p.n;
      sx += real ? q.x * cs - 1.0f : 0.f;
      sy += real ? q.y * cs - 1.0f : 0.f;
      sz += real ? q.z * cs - 1.0f : 0.f;
    }
    const float fc = fmaxf((float)cnt, 1.0f);
    const float mx = warp_sum(sx) / fc, my = warp_sum(sy) / fc, mz = warp_sum(sz) / fc;
    float cv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int s = lane; s < p.K; s += 32) {
      const short4 q = p.xyzb[t0 + s];
      if (q.w != id0) continue;
      const bool real = t0 + s < p.n;
      const float dx = (real ? q.x * cs - 1.0f : 0.f) - mx;
      const float dy = (real ? q.y * cs - 1.0f : 0.f) - my;
      const float dz = (real ? q.z * cs - 1.0f : 0.f) - mz;
      cv[0] += dx * dx; cv[1] += dx * dy; cv[2] += dx * dz;
      cv[3] += dy * dy; cv[4] += dy * dz; cv[5] += dz * dz;
    }
    const float den = fmaxf((float)cnt - 1.0f, 1.0f);
    const float okf = cnt >= 2 ? 1.0f : 0.0f;
    float st[9];
    st[0] = mx; st[1] = my; st[2] = mz;
#pragma unroll
    for (int j = 0; j < 6; ++j) st[3 + j] = warp_sum(cv[j]) / den * okf;
    if (p.mode == 6) { st[4] = st[6]; st[5] = st[8]; }      // 'var': diagonal only
    if (p.stats_out && lane < 9) {
      float v = st[0];
#pragma unroll
      for (int j = 1; j < 9; ++j) v = lane == j ? st[j] : v;
      p.stats_out[w * 9 + lane] = v;
    }
    float hv[V];
#pragma unroll
    for (int j = 0; j < V; ++j) {
      float a = p.b1[c0 + j];
      for (int i = 0; i < p.mode; ++i) a += p.w1[(c0 + j) * p.mode + i] * st[i];
      hv[j] = gelu(a);
    }
    store_bf16<V>(p.h + w * C + c0, hv);
  }
}

__global__ void k_hat_rows(int32_t* __restrict__ out, int64_t n, int K, int32_t offset) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (int32_t)hat_row(i, K) + offset;
}
__global__ void k_remap_hat(const int32_t* __restrict__ in, int32_t* __restrict__ out, int64_t n,
                            int K) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t v = in[i];
    out[i] = v < 0 ? -1 : (int32_t)hat_row(v, K);
  }
}
__global__ void k_f32_to_bf16(const float* __restrict__ in, __nv_bfloat16* __restrict__ out,
                              int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16(in[i]);
}

// ---------------------------------------------------------------------------
// attention pooling (models/layers/salsa.py:25-55 restricted to each submap's tokens)
//   logits [rows, ldl] fp32 come from the tcgen05 GEMM x . query^T (hat rows)
//   pass 1: per (submap, query) max and sum of exp over the submap's tokens
//   pass 2: out[b, q, :] = sum_t softmax_t * x[t, :]
// ---------------------------------------------------------------------------
struct PoolParams {
  const float* logits;   // [rows, ldl]
  const float* x;        // [rows, C] fp32 features, hat layout (unused by the MMA path)
  const __nv_bfloat16* xb; // [rows, C] bf16 shadow of the features
  const int32_t* tok_off; // [B+1] token offsets of the submaps at this level
  float* stat;           // [B, kq, 2] (max, 1/sum) in log2 domain
  float* out;            // [B, ktot, C]; this level's queries start at q_off
  int B, kq, ldl, K, C, ktot, q_off;
  float scale;
};

__global__ void __launch_bounds__(256) k_pool_stats(const PoolParams p) {
  // grid: (B, ceil(kq/32)); lane = one query column (a warp reads 32 consecutive logits of a token row: one
  // 128-byte line), the 8 warps stride over the submap's tokens with an ONLINE (max, sum) per column -- one
  // coalesced pass over the logits instead of two strided ones -- and are merged through shared memory
  const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = blockIdx.y * 32 + lane;
  const bool ok = q < p.kq;
  const int64_t t0 = p.tok_off[b], t1 = p.tok_off[b + 1];
  const float sc = p.scale * 1.4426950408889634f;
  const uint32_t K = (uint32_t)p.K;
  float m = -INFINITY, s = 0.f;
  // four tokens in flight per warp
  for (int64_t t = t0 + warp * 4; t < t1; t += 32) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t tt = t + u;
      const bool in = ok && tt < t1;
      const int64_t row = in ? (K ? tt + (int64_t)((uint32_t)tt / K) + 1 : tt) : 0;
      v[u] = in ? __ldg(p.logits + row * p.ldl + q) * sc : -INFINITY;
    }
    const float mn = fmaxf(fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])), m);
    if (mn > -INFINITY) {
      s = s * exp2f(m - mn) + exp2f(v[0] - mn) + exp2f(v[1] - mn) + exp2f(v[2] - mn) + exp2f(v[3] - mn);
      m = mn;
    }
  }
  __shared__ float sm[8][32], ss[8][32];
  sm[warp][lane] = m;
  ss[warp][lane] = s;
  __syncthreads();
  if (warp == 0 && ok) {
    float M = -INFINITY;
#pragma unroll
    for (int w = 0; w < 8; ++w) M = fmaxf(M, sm[w][lane]);
    float S = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) S += sm[w][lane] > -INFINITY ? ss[w][lane] * exp2f(sm[w][lane] - M) : 0.f;
    p.stat[((size_t)b * p.kq + q) * 2] = M;
    p.stat[((size_t)b * p.kq + q) * 2 + 1] = S > 0.f ? 1.0f / S : 0.f;
  }
}

// pass 2 on the tensor cores: out[q, c] = sum_t P[t, q] * x[t, c] is a (queries x tokens) x
// (tokens x channels) product.  CTA = (submap, group of <= 80 queries); 8 warps x 32 channels;
// per 64-token tile the CTA builds P (bf16, already normalised) in smem and streams the bf16
// feature rows through a cp.async double buffer; mma.sync m16n8k16, fp32 accumulators.
constexpr int PM_Q = 80;                  // queries per CTA (5 m-tiles)
constexpr int PM_T = 64;                  // tokens per tile
constexpr int PM_PP = 72;                 // sP pitch (bf16): 144 B rows, conflict-free ldmatrix
constexpr int PM_XP = 264;                // sX pitch (bf16): 528 B rows
constexpr int PM_SMEM = PM_Q * PM_PP * 2 + 2 * PM_T * PM_XP * 2 + PM_Q * 8 + PM_T * 8;

__global__ void __launch_bounds__(256) k_pool_mma(const PoolParams p) {
  extern __shared__ __align__(16) uint8_t psm[];
  __nv_bfloat16* sP = reinterpret_cast<__nv_bfloat16*>(psm);                         // [80][72]
  __nv_bfloat16* sX = reinterpret_cast<__nv_bfloat16*>(psm + PM_Q * PM_PP * 2);      // [2][64][264]
  float* sM = reinterpret_cast<float*>(psm + PM_Q * PM_PP * 2 + 2 * PM_T * PM_XP * 2);
  float* sI = sM + PM_Q;
  int64_t* sRow = reinterpret_cast<int64_t*>(sI + PM_Q);                              // [64]
  const int b = blockIdx.x, qbase = blockIdx.y * PM_Q;
  const int nq = min(PM_Q, p.kq - qbase);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const int64_t t0 = p.tok_off[b], t1 = p.tok_off[b + 1];
  const float sc = p.scale * 1.4426950408889634f;
  for (int q = threadIdx.x; q < PM_Q; q += 256) {
    const bool ok = q < nq;
    sM[q] = ok ? p.stat[((size_t)b * p.kq + qbase + q) * 2] : 0.f;
    sI[q] = ok ? p.stat[((size_t)b * p.kq + qbase + q) * 2 + 1] : 0.f;
  }
  float acc[5][4][4];
#pragma unroll
  for (int m = 0; m < 5; ++m)
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[m][n][e] = 0.f;
  const uint32_t sX_u = ptx::smem_u32(sX), sP_u = ptx::smem_u32(sP);
  const int n_tiles = (int)((t1 - t0 + PM_T - 1) / PM_T);

  auto stage_x = [&](int tile, int buf) {
    // 64 rows x 512 B = 2048 x 16 B chunks, 8 per thread; rows beyond the submap are zero-filled
    const int64_t tb = t0 + (int64_t)tile * PM_T;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int ch = threadIdx.x + 256 * i;
      const int tt = ch >> 5, c16 = ch & 31;
      const bool ok = tb + tt < t1;
      const int64_t row = ok ? hat_row(tb + tt, p.K) : 0;
      ptx::cp_async16(sX_u + (uint32_t)((buf * PM_T + tt) * PM_XP * 2 + c16 * 16),
                      p.xb + row * p.C + c16 * 8, ok ? 16u : 0u);
    }
    ptx::cp_async_commit();
  };
  if (n_tiles > 0) stage_x(0, 0);
  for (int tile = 0; tile < n_tiles; ++tile) {
    const int buf = tile & 1;
    const int64_t tb = t0 + (int64_t)tile * PM_T;
    __syncthreads();                                   // previous tile's sP / sX[buf^1] readers done
    if (tile + 1 < n_tiles) stage_x(tile + 1, buf ^ 1);
    if (threadIdx.x < PM_T) sRow[threadIdx.x] = tb + threadIdx.x < t1 ? hat_row(tb + threadIdx.x, p.K) : -1;
    __syncthreads();
    // ---- P tile (normalised softmax weights), bf16, [query][token] ----
    for (int i = threadIdx.x; i < PM_T * PM_Q; i += 256) {
      const int tt = i / PM_Q, q = i - tt * PM_Q;
      const int64_t row = sRow[tt];
      float pv = 0.f;
      if (row >= 0 && q < nq)
        pv = exp2f(p.logits[row * p.ldl + qbase + q] * sc - sM[q]) * sI[q];
      sP[q * PM_PP + tt] = __float2bfloat16(pv);
    }
    if (tile + 1 < n_tiles) ptx::cp_async_wait<1>(); else ptx::cp_async_wait<0>();
    __syncthreads();
    // ---- acc += P^T-tile x X-tile ----
#pragma unroll
    for (int ks = 0; ks < PM_T / 16; ++ks) {
      uint32_t bfr[2][4];
      const int mi = lane >> 3;
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2) {
        const int trow = ks * 16 + (mi & 1) * 8 + (lane & 7);
        const int col = warp * 32 + h2 * 16 + (mi >> 1) * 8;
        ptx::ldmatrix_x4_trans(bfr[h2], sX_u + (uint32_t)(((buf * PM_T + trow) * PM_XP + col) * 2));
      }
#pragma unroll
      for (int m = 0; m < 5; ++m) {
        uint32_t afr[4];
        const int arow = m * 16 + (mi & 1) * 8 + (lane & 7);
        const int acol = ks * 16 + (mi >> 1) * 8;
        ptx::ldmatrix_x4(afr, sP_u + (uint32_t)((arow * PM_PP + acol) * 2));
#pragma unroll
        for (int n = 0; n < 4; ++n) {
          uint32_t bb[2] = {bfr[n >> 1][(n & 1) * 2], bfr[n >> 1][(n & 1) * 2 + 1]};
          ptx::mma16816(acc[m][n], afr, bb);
        }
      }
    }
  }
#pragma unroll
  for (int m = 0; m < 5; ++m) {
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      const int c = warp * 32 + n * 8 + 2 * t4;
      const int q0 = m * 16 + g, q1 = q0 + 8;
      if (q0 < nq) {
        float* o = p.out + ((size_t)b * p.ktot + p.q_off + qbase + q0) * p.C + c;
        o[0] = acc[m][n][0]; o[1] = acc[m][n][1];
      }
      if (q1 < nq) {
        float* o = p.out + ((size_t)b * p.ktot + p.q_off + qbase + q1) * p.C + c;
        o[0] = acc[m][n][2]; o[1] = acc[m][n][3];
      }
    }
  }
}

// Mixer tail (salsa.py:103-111) + F.normalize (hotformerloc.py:55-56); one CTA per submap
struct TailParams {
  const float* x;          // [B, kin, C]
  const float *wc, *bc;    // channel_proj [kout, kin], [kout]
  const float *wr, *br;    // row_proj [od, C], [od]
  float* out;              // [B, kout*od]
  int kin, kout, C, od, normalize;
};
__global__ void __launch_bounds__(256) k_mixer_tail(const TailParams p) {
  extern __shared__ float sh[];
  float* sy = sh;                       // [kout][C]
  float* sd = sh + p.kout * p.C;        // [kout*od]
  __shared__ float red[8];
  const int b = blockIdx.x, c = threadIdx.x;     // C == blockDim.x
  const float* xb = p.x + (size_t)b * p.kin * p.C;
  for (int o = 0; o < p.kout; ++o) {
    float a = p.bc[o];
    for (int t = 0; t < p.kin; ++t) a += p.wc[o * p.kin + t] * xb[t * p.C + c];
    sy[o * p.C + c] = a;
  }
  __syncthreads();
  const int nout = p.kout * p.od;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int e = warp; e < nout; e += (blockDim.x >> 5)) {
    const int o = e / p.od, d = e % p.od;
    float a = 0.f;
    for (int cc = lane; cc < p.C; cc += 32) a += p.wr[d * p.C + cc] * sy[o * p.C + cc];
    a = warp_sum(a);
    if (lane == 0) sd[e] = a + p.br[d];
  }
  __syncthreads();
  float ss = 0.f;
  for (int e = threadIdx.x; e < nout; e += blockDim.x) ss += sd[e] * sd[e];
  ss = warp_sum(ss);
  if (lane == 0) red[warp] = ss;
  __syncthreads();
  float tot = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
  const float inv = p.normalize ? 1.0f / fmaxf(sqrtf(tot), 1e-12f) : 1.0f;
  for (int e = threadIdx.x; e < nout; e += blockDim.x) p.out[(size_t)b * nout + e] = sd[e] * inv;
}

// PyramidOctGeM (pooling.py:87-103): per-submap generalised mean over a level's tokens
__global__ void __launch_bounds__(256)
k_gem_pool(const float* __restrict__ x, const int32_t* __restrict__ tok_off, int K, int C,
           float pw, float eps, float* __restrict__ out, int ld_out, int col_off) {
  // grid: (B); thread = channel (strided)
  const int b = blockIdx.x;
  const int64_t t0 = tok_off[b], t1 = tok_off[b + 1];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f;
    for (int64_t t = t0; t < t1; ++t) a += powf(fmaxf(x[hat_row(t, K) * C + c], eps), pw);
    const float cnt = fmaxf((float)(t1 - t0), 1.0f);
    out[(size_t)b * ld_out + col_off + c] = powf(a / cnt, 1.0f / pw);
  }
}

// PyramidOctGeM head (pooling.py:78-84, 98-99): Linear(no bias) + eval-mode BatchNorm1d
// (+ F.normalize); fp32, one CTA per submap, thread = output feature.
__global__ void __launch_bounds__(256)
k_gem_head(const float* __restrict__ pooled, int in_dim, const float* __restrict__ w,
           const float* __restrict__ bn_g, const float* __restrict__ bn_b,
           const float* __restrict__ bn_mean, const float* __restrict__ bn_var, float bn_eps,
           int out_dim, int normalize, float* __restrict__ out) {
  extern __shared__ float gh[];
  float* sx = gh;                 // [in_dim]
  __shared__ float red[8];
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < in_dim; i += blockDim.x) sx[i] = pooled[(size_t)b * in_dim + i];
  __syncthreads();
  float ss = 0.f;
  float val[4];                   // out_dim <= 4 * blockDim
  int nv = 0;
  for (int o = threadIdx.x; o < out_dim; o += blockDim.x, ++nv) {
    float a = 0.f;
    for (int i = 0; i < in_dim; ++i) a = fmaf(w[(size_t)o * in_dim + i], sx[i], a);
    a = (a - bn_mean[o]) * rsqrtf(bn_var[o] + bn_eps) * bn_g[o] + bn_b[o];
    val[nv] = a;
    ss += a * a;
  }
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
  const float inv = normalize ? 1.0f / fmaxf(sqrtf(tot), 1e-12f) : 1.0f;
  nv = 0;
  for (int o = threadIdx.x; o < out_dim; o += blockDim.x, ++nv) out[(size_t)b * out_dim + o] = val[nv] * inv;
}

}  // namespace hfl

using namespace hfl;

#define ROWS_GRID(n) grid_for((int64_t)(n) * 32, 256, kSMs * 16)

extern "C" {

int hfl_stem_conv(const float* leaf_pts, const int32_t* ne, int64_t n, int32_t depth,
                  const float* w, const float* g, const float* b, void* out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (n == 0) return HFL_OK;
  HFL_CHECK_ARG(leaf_pts && ne && w && g && b && out, "null argument");
  HFL_LAUNCH((k_stem_conv<<<ROWS_GRID(n), 256, 0, st>>>(leaf_pts, ne, n, ldexpf(1.0f, 1 - depth), w, g, b, (__nv_bfloat16*)out)));
  return HFL_OK;
}

int hfl_cpe_ln(float* x, const void* xb, const int32_t* ne, const void* w, const float* g_cpe,
               const float* b_cpe, const float* g1, const float* b1, void* y1, float* cpe_out,
               int64_t n, int64_t rows, int32_t C, int32_t K, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (rows == 0) return HFL_OK;
  HFL_CHECK_ARG(x && xb && ne && w && g_cpe && b_cpe, "null argument");
  HFL_CHECK_ARG(C == 128 || C == 256, "C must be 128 or 256");
  HFL_CHECK_ARG(!y1 || (g1 && b1), "norm1 parameters missing");
  HFL_CHECK_ARG(rows < (1ll << 31) && n < (1ll << 31) && K >= 0, "row / token indices must fit 32 bits");
  CpeParams p{x, (const __nv_bfloat16*)xb, ne, (const __nv_bfloat16*)w, g_cpe, b_cpe, g1, b1, (__nv_bfloat16*)y1, cpe_out, n, rows, K};
  if (C == 128) HFL_LAUNCH((k_cpe_ln<4><<<ROWS_GRID(rows), 256, 0, st>>>(p)));
  else HFL_LAUNCH((k_cpe_ln<8><<<ROWS_GRID(rows), 256, 0, st>>>(p)));
  return HFL_OK;
}

int hfl_ln_rows(const float* x, const int32_t* rows, int64_t m, int32_t C, const float* g,
                const float* b, void* y, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (m == 0) return HFL_OK;
  HFL_CHECK_ARG(x && g && b && y, "null argument");
  HFL_CHECK_ARG(C == 128 || C == 256, "C must be 128 or 256");
  if (C == 128) HFL_LAUNCH((k_ln_rows<4><<<ROWS_GRID(m), 256, 0, st>>>(x, rows, m, g, b, (__nv_bfloat16*)y)));
  else HFL_LAUNCH((k_ln_rows<8><<<ROWS_GRID(m), 256, 0, st>>>(x, rows, m, g, b, (__nv_bfloat16*)y)));
  return HFL_OK;
}

int hfl_rt_init(float* x, const float* src, const int16_t* xyzb, int64_t n, int64_t n_win,
                int32_t K, int32_t C, int32_t depth, int32_t mode, const float* w1,
                const float* b1, void* h, float* stats_out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_win == 0) return HFL_OK;
  HFL_CHECK_ARG(x && xyzb, "null argument");
  HFL_CHECK_ARG(C == 128 || C == 256, "C must be 128 or 256");
  HFL_CHECK_ARG(mode == 0 || ((mode == 3 || mode == 6 || mode == 9) && w1 && b1 && h), "bad ADaPE mode");
  RtInitParams p{x, src, (const short4*)xyzb, n, n_win, K, depth, mode, w1, b1, (__nv_bfloat16*)h, stats_out};
  if (C == 128) HFL_LAUNCH((k_rt_init<4><<<ROWS_GRID(n_win), 256, 0, st>>>(p)));
  else HFL_LAUNCH((k_rt_init<8><<<ROWS_GRID(n_win), 256, 0, st>>>(p)));
  return HFL_OK;
}

int hfl_hat_rows(int32_t* out, int64_t n, int32_t K, int32_t offset, void* stream_) {
  if (n == 0) return HFL_OK;
  HFL_LAUNCH((k_hat_rows<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream_>>>(out, n, K, offset)));
  return HFL_OK;
}
int hfl_remap_hat(const int32_t* in, int32_t* out, int64_t n, int32_t K, void* stream_) {
  if (n == 0) return HFL_OK;
  HFL_LAUNCH((k_remap_hat<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream_>>>(in, out, n, K)));
  return HFL_OK;
}
int hfl_f32_to_bf16(const float* in, void* out, int64_t n, void* stream_) {
  if (n == 0) return HFL_OK;
  HFL_LAUNCH((k_f32_to_bf16<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream_>>>(in, (__nv_bfloat16*)out, n)));
  return HFL_OK;
}

int hfl_attn_pool(const float* logits, const float* x, const void* xb, const int32_t* tok_off,
                  float* stat, float* out, int32_t B, int32_t kq, int32_t ldl, int32_t K, int32_t C,
                  int32_t ktot, int32_t q_off, float scale, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (B == 0 || kq == 0) return HFL_OK;     // empty problem: no zero-sized grid
  HFL_CHECK_ARG(logits && xb && tok_off && stat && out, "null argument");
  HFL_CHECK_ARG(C == 256, "C must be 256");
  PoolParams p{logits, x, (const __nv_bfloat16*)xb, tok_off, stat, out, B, kq, ldl, K, C, ktot, q_off, scale};
  HFL_LAUNCH((k_pool_stats<<<dim3(B, (kq + 31) / 32), 256, 0, st>>>(p)));
  HFL_ENSURE_SMEM(PM_SMEM, k_pool_mma);
  HFL_LAUNCH((k_pool_mma<<<dim3(B, (kq + PM_Q - 1) / PM_Q), 256, PM_SMEM, st>>>(p)));
  return HFL_OK;
}

int hfl_mixer_tail(const float* x, const float* wc, const float* bc, const float* wr,
                   const float* br, float* out, int32_t B, int32_t kin, int32_t kout, int32_t C,
                   int32_t od, int32_t normalize, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (B == 0) return HFL_OK;
  HFL_CHECK_ARG(x && wc && bc && wr && br && out, "null argument");
  HFL_CHECK_ARG(C == 256 || C == 128, "C must equal the CTA size (128/256)");
  TailParams p{x, wc, bc, wr, br, out, kin, kout, C, od, normalize};
  const int smem = (kout * C + kout * od) * 4;
  if (smem > 48 * 1024) HFL_ENSURE_SMEM(smem, k_mixer_tail);
  HFL_LAUNCH((k_mixer_tail<<<B, C, smem, st>>>(p)));
  return HFL_OK;
}

int hfl_gem_pool(const float* x, const int32_t* tok_off, int32_t B, int32_t K, int32_t C, float pw,
                 float eps, float* out, int32_t ld_out, int32_t col_off, void* stream_) {
  if (B == 0) return HFL_OK;
  HFL_CHECK_ARG(x && tok_off && out, "null argument");
  HFL_LAUNCH((k_gem_pool<<<B, 256, 0, (cudaStream_t)stream_>>>(x, tok_off, K, C, pw, eps, out, ld_out, col_off)));
  return HFL_OK;
}

int hfl_gem_head(const float* pooled, int32_t B, int32_t in_dim, const float* w, const float* bn_g,
                 const float* bn_b, const float* bn_mean, const float* bn_var, float bn_eps,
                 int32_t out_dim, int32_t normalize, float* out, void* stream_) {
  if (B == 0) return HFL_OK;
  HFL_CHECK_ARG(pooled && w && bn_g && bn_b && bn_mean && bn_var && out, "null argument");
  HFL_CHECK_ARG(out_dim <= 1024 && in_dim * 4 <= 48 * 1024, "head too large");
  HFL_LAUNCH((k_gem_head<<<B, 256, in_dim * 4, (cudaStream_t)stream_>>>(pooled, in_dim, w, bn_g, bn_b, bn_mean, bn_var, bn_eps, out_dim, normalize, out)));
  return HFL_OK;
}

}  // extern "C"
