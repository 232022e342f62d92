// Attention pooling over ragged per-submap token segments with its backward, fp32 (training side): the
// AdaptivePooling of the reference's PyramidAttnPoolWrapper (pooling.py:183-233, salsa.py:25-55) without the
// padded (B, Nmax, C) features and the (B, N, N) mask.  For segment b = tokens [off[b], off[b+1]) of x [n, C],
// queries Q [k, C] and s = C^-0.5:
//   S[b,q,t] = s Q[q].x[t],   out[b,q] = sum_t softmax_t(S[b,q,.]) x[t],   lse[b,q] = log sum_t exp(S[b,q,t])
// An empty segment gives out = 0, lse = -inf and no gradient.  fp32 FMA throughout (no TF32).
//   k_apool_plan    : chunk table: segment b owns chunks [first[b], first[b+1]) of kChunk tokens each
//   k_apool_fwd     : CTA = (chunk, group of 32 queries): online softmax over 32-token tiles -> partial (m, l, o)
//   k_apool_merge   : warp = (b, q): folds the partials of b's chunks in chunk order -> out, lse
//   k_apool_delta   : D[b,q] = dout[b,q].out[b,q]
//   k_apool_bwd_dx  : CTA = 32-token tile of one chunk, all queries: dx = sum_q p dout[b,q] + s sum_q dS Q[q]
//   k_apool_bwd_dq  : CTA = (chunk, group of 32 queries): per-chunk partial dQ = s sum_t dS x[t]
//   k_apool_dq_fold : dQ = the chunk partials summed in a fixed order
// Every output element is a fixed-order fp32 sum, and the chunk partition depends on (off, k, C) only: results are
// bit-identical run to run, without float atomics.  The backward recomputes S from x, Q and lse (nothing of size
// B k Nmax is kept), at 14 k C FLOPs per token (S and dP once for dx and once for dQ).
#include "common.cuh"

namespace hfl {

namespace {

constexpr int kChunk = 1024;    // tokens per chunk (a chunk never crosses a segment boundary)
constexpr int kTile = 32;       // tokens per tile
constexpr int kQG = 32;         // queries per group
constexpr int kThreads = 256;   // 8 warps; warp w owns rows 4w .. 4w+3 of every 32-row tile
constexpr int kMaxK = 256;
constexpr int kMaxC = 512;
constexpr int kMaxB = 1 << 24;

// Segment b clamped into [0, n]; a decreasing pair is empty.
__device__ __forceinline__ void seg_range(const int64_t* __restrict__ off, int b, int64_t n, int64_t& s, int64_t& e) {
  s = min(max(__ldg(off + b), (int64_t)0), n);
  e = min(max(__ldg(off + b + 1), s), n);
}

// Chunk c of the plan: its segment b, first token t0 and end t1 (t0 < t1).
__device__ __forceinline__ void chunk_range(const int64_t* __restrict__ off, const int* __restrict__ first, int B,
                                            int64_t n, int c, int& b, int64_t& t0, int64_t& t1) {
  int lo = 0, hi = B;                       // first[lo] <= c < first[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(first + mid) <= c) lo = mid; else hi = mid;
  }
  b = lo;
  int64_t s, e;
  seg_range(off, b, n, s, e);
  t0 = s + (int64_t)(c - __ldg(first + b)) * kChunk;
  t1 = min(e, t0 + kChunk);
}

// rows [r0, r0 + valid) of a row-major [*, C] matrix into dst[rows][C + 4], rows >= valid zero.
__device__ __forceinline__ void load_rows(const float* __restrict__ src, int64_t r0, int valid, int rows, int C,
                                          float* dst) {
  const int C4 = C >> 2, LD4 = (C + 4) >> 2;
  for (int i = threadIdx.x; i < rows * C4; i += blockDim.x) {
    const int r = i / C4, c = i - r * C4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < valid) v = __ldg(reinterpret_cast<const float4*>(src + (r0 + r) * C) + c);
    reinterpret_cast<float4*>(dst)[r * LD4 + c] = v;
  }
}

// s[i] = A[4w + i] . X[lane] for i < 4 (A, X in smem with row stride C + 4: the float4 reads of X by a
// quarter warp hit 32 distinct banks, the reads of A are broadcasts).  With G, also g[i] = G[4w + i] . X[lane].
template <bool kTwo>
__device__ __forceinline__ void dot4(const float* A, const float* G, const float* X, int C, int w, int lane,
                                     float s[4], float g[4]) {
  const int LD = C + 4;
  const float* a = A + 4 * w * LD;
  const float* gg = kTwo ? G + 4 * w * LD : nullptr;
  const float* xr = X + lane * LD;
#pragma unroll
  for (int i = 0; i < 4; ++i) s[i] = g[i] = 0.f;
  for (int c = 0; c < C; c += 4) {
    const float4 xv = *reinterpret_cast<const float4*>(xr + c);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 av = *reinterpret_cast<const float4*>(a + i * LD + c);
      s[i] = fmaf(av.x, xv.x, s[i]); s[i] = fmaf(av.y, xv.y, s[i]);
      s[i] = fmaf(av.z, xv.z, s[i]); s[i] = fmaf(av.w, xv.w, s[i]);
      if (kTwo) {
        const float4 gv = *reinterpret_cast<const float4*>(gg + i * LD + c);
        g[i] = fmaf(gv.x, xv.x, g[i]); g[i] = fmaf(gv.y, xv.y, g[i]);
        g[i] = fmaf(gv.z, xv.z, g[i]); g[i] = fmaf(gv.w, xv.w, g[i]);
      }
    }
  }
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// acc[i][j] += sum_t P[4w + i][t] V[t][lane + 32 j] over the 32 tokens of a tile (P [32][32], V [32][C + 4]);
// channel slots j >= cv are idle.
template <int CVM>
__device__ __forceinline__ void accum_pv(const float* P, const float* V, int C, int cv, int w, int lane,
                                         float acc[4][CVM]) {
  const int LD = C + 4;
  const float* p = P + 4 * w * kTile;
#pragma unroll 2
  for (int t = 0; t < kTile; t += 4) {
    float pv[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 v = *reinterpret_cast<const float4*>(p + i * kTile + t);
      pv[i][0] = v.x; pv[i][1] = v.y; pv[i][2] = v.z; pv[i][3] = v.w;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float* vr = V + (t + u) * LD + lane;
#pragma unroll
      for (int j = 0; j < CVM; ++j) {
        if (j < cv) {
          const float xv = vr[32 * j];
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[i][j] = fmaf(pv[i][u], xv, acc[i][j]);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Plan: first[b] = sum_{b' < b} ceil(len_b' / kChunk), capped at cap (the workspace's chunk capacity, which
// well-formed offsets never reach); first[B] = the chunk count.  One CTA, block scan in rounds of 1024.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
k_apool_plan(const int64_t* __restrict__ off, int64_t n, int B, int64_t cap, int* __restrict__ first) {
  __shared__ int64_t s[1024];
  int64_t carry = 0;
  for (int base = 0; base < B; base += 1024) {
    const int b = base + threadIdx.x;
    int64_t v = 0;
    if (b < B) {
      int64_t s0, e0;
      seg_range(off, b, n, s0, e0);
      v = ceil_div(e0 - s0, kChunk);
    }
    s[threadIdx.x] = v;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
      const int64_t t = threadIdx.x >= d ? s[threadIdx.x - d] : 0;
      __syncthreads();
      s[threadIdx.x] += t;
      __syncthreads();
    }
    if (b < B) first[b] = (int)min(carry + s[threadIdx.x] - v, cap);
    carry += s[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) first[B] = (int)min(carry, cap);
}

// ---------------------------------------------------------------------------
// Forward.  blockIdx.x = chunk, blockIdx.y = query group.  Smem: Q rows of the group and the x tile
// [32][C + 4], P [32][32].  Warp w owns queries 4w .. 4w+3 in both the score and the P.x phase, so the running
// max / sum and the rescaling stay in registers and P is exchanged only within the warp.
// ---------------------------------------------------------------------------
template <int CVM>
__global__ void __launch_bounds__(kThreads)
k_apool_fwd(const float* __restrict__ x, const int64_t* __restrict__ off, const float* __restrict__ Q,
            const int* __restrict__ first, int64_t n, int B, int k, int C, float scale, float* __restrict__ part_ml,
            float* __restrict__ part_o) {
  extern __shared__ __align__(16) float smem[];
  const int LD = C + 4, cv = C >> 5;
  float* s_q = smem;
  float* s_x = s_q + kQG * LD;
  float* s_p = s_x + kTile * LD;
  const int c = blockIdx.x;
  if (c >= __ldg(first + B)) return;
  int b;
  int64_t t0, t1;
  chunk_range(off, first, B, n, c, b, t0, t1);
  const int q0 = blockIdx.y * kQG, kq = min(kQG, k - q0);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  load_rows(Q, q0, kq, kQG, C, s_q);
  float m[4], l[4], acc[4][CVM];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m[i] = -INFINITY;
    l[i] = 0.f;
#pragma unroll
    for (int j = 0; j < CVM; ++j) acc[i][j] = 0.f;
  }
  for (int64_t tt = t0; tt < t1; tt += kTile) {
    const int nt = (int)min((int64_t)kTile, t1 - tt);
    __syncthreads();                              // the previous tile's readers are done
    load_rows(x, tt, nt, kTile, C, s_x);
    __syncthreads();
    float s[4], unused[4];
    dot4<false>(s_q, nullptr, s_x, C, w, lane, s, unused);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float si = lane < nt ? s[i] * scale : -INFINITY;
      const float mn = fmaxf(m[i], warp_max(si));  // finite: the tile has a token
      const float corr = expf(m[i] - mn);
      const float p = expf(si - mn);
      l[i] = l[i] * corr + warp_sum(p);
      m[i] = mn;
      s_p[(4 * w + i) * kTile + lane] = p;
#pragma unroll
      for (int j = 0; j < CVM; ++j) acc[i][j] *= corr;
    }
    __syncwarp();
    accum_pv<CVM>(s_p, s_x, C, cv, w, lane, acc);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int q = 4 * w + i;
    if (q >= kq) continue;
    const int64_t r = (int64_t)c * k + q0 + q;
    float* o = part_o + r * C + lane;
#pragma unroll
    for (int j = 0; j < CVM; ++j)
      if (j < cv) o[32 * j] = acc[i][j];
    if (lane == 0) {
      part_ml[2 * r] = m[i];
      part_ml[2 * r + 1] = l[i];
    }
  }
}

// One warp per (b, q); the partials of b's chunks folded in chunk order.
__global__ void __launch_bounds__(256)
k_apool_merge(const int* __restrict__ first, const float* __restrict__ part_ml, const float* __restrict__ part_o,
              int B, int k, int C, float* __restrict__ out, float* __restrict__ lse) {
  const int64_t pair = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pair >= (int64_t)B * k) return;
  const int b = (int)(pair / k), q = (int)(pair - (int64_t)b * k);
  const int c0 = __ldg(first + b), c1 = __ldg(first + b + 1);
  float* o = out + pair * C;
  if (c0 >= c1) {                                 // empty segment
    for (int ch = lane; ch < C; ch += 32) o[ch] = 0.f;
    if (lane == 0) lse[pair] = -INFINITY;
    return;
  }
  float M = -INFINITY;
  for (int c = c0; c < c1; ++c) M = fmaxf(M, __ldg(part_ml + 2 * ((int64_t)c * k + q)));
  float L = 0.f;
  for (int c = c0; c < c1; ++c) {
    const int64_t r = (int64_t)c * k + q;
    L = fmaf(__ldg(part_ml + 2 * r + 1), expf(__ldg(part_ml + 2 * r) - M), L);
  }
  const float inv = 1.f / L;
  for (int ch = lane; ch < C; ch += 32) {
    float v = 0.f;
    for (int c = c0; c < c1; ++c) {
      const int64_t r = (int64_t)c * k + q;
      v = fmaf(__ldg(part_o + r * C + ch), expf(__ldg(part_ml + 2 * r) - M), v);
    }
    o[ch] = v * inv;
  }
  if (lane == 0) lse[pair] = M + logf(L);
}

// ---------------------------------------------------------------------------
// Backward
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_apool_delta(const float* __restrict__ out, const float* __restrict__ dout, int64_t pairs, int C,
              float* __restrict__ D) {
  const int64_t pair = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pair >= pairs) return;
  float v = 0.f;
  for (int ch = lane; ch < C; ch += 32) v = fmaf(__ldg(dout + pair * C + ch), __ldg(out + pair * C + ch), v);
  v = warp_sum(v);
  if (lane == 0) D[pair] = v;
}

// p and s dS of queries 4w+i (i < 4) of a group for token lane: zero for padding queries / tokens.
__device__ __forceinline__ void probs(const float s[4], const float dp[4], const float* __restrict__ lse,
                                      const float* __restrict__ D, int64_t row0, int q, int k, bool tok_ok,
                                      float scale, float p[4], float ds[4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    p[i] = ds[i] = 0.f;
    if (tok_ok && q + i < k) {
      p[i] = expf(s[i] * scale - __ldg(lse + row0 + q + i));
      ds[i] = scale * (p[i] * (dp[i] - __ldg(D + row0 + q + i)));
    }
  }
}

// blockIdx.x = chunk, blockIdx.y = 32-token tile of the chunk.  For each query group: Q and dout rows into smem,
// warp w computes p and s dS for queries 4w+i and token lane into the shared [32][32] tiles, then every thread
// adds sum_q p dout + s dS Q into its dx rows 4w+u (u < 4), channels lane + 32 j.
template <int CVM>
__global__ void __launch_bounds__(kThreads)
k_apool_bwd_dx(const float* __restrict__ x, const int64_t* __restrict__ off, const float* __restrict__ Q,
               const float* __restrict__ lse, const float* __restrict__ D, const float* __restrict__ dout,
               const int* __restrict__ first, int64_t n, int B, int k, int C, float scale, float* __restrict__ dx) {
  extern __shared__ __align__(16) float smem[];
  const int LD = C + 4, cv = C >> 5;
  float* s_x = smem;
  float* s_q = s_x + kTile * LD;
  float* s_g = s_q + kQG * LD;
  float* s_p = s_g + kQG * LD;                    // [query][token]
  float* s_ds = s_p + kQG * kTile;
  const int c = blockIdx.x;
  if (c >= __ldg(first + B)) return;
  int b;
  int64_t t0, t1;
  chunk_range(off, first, B, n, c, b, t0, t1);
  const int64_t tt = t0 + (int64_t)blockIdx.y * kTile;
  if (tt >= t1) return;
  const int nt = (int)min((int64_t)kTile, t1 - tt);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row0 = (int64_t)b * k;
  load_rows(x, tt, nt, kTile, C, s_x);
  float acc[4][CVM];
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int j = 0; j < CVM; ++j) acc[u][j] = 0.f;
  for (int q0 = 0; q0 < k; q0 += kQG) {
    const int kq = min(kQG, k - q0);
    __syncthreads();                              // the previous group's readers are done
    load_rows(Q, q0, kq, kQG, C, s_q);
    load_rows(dout, row0 + q0, kq, kQG, C, s_g);
    __syncthreads();
    float s[4], dp[4], p[4], ds[4];
    dot4<true>(s_q, s_g, s_x, C, w, lane, s, dp);
    probs(s, dp, lse, D, row0, q0 + 4 * w, k, lane < nt, scale, p, ds);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      s_p[(4 * w + i) * kTile + lane] = p[i];
      s_ds[(4 * w + i) * kTile + lane] = ds[i];
    }
    __syncthreads();
    for (int q = 0; q < kq; ++q) {
      const float4 p4 = *reinterpret_cast<const float4*>(s_p + q * kTile + 4 * w);
      const float4 d4 = *reinterpret_cast<const float4*>(s_ds + q * kTile + 4 * w);
      const float pu[4] = {p4.x, p4.y, p4.z, p4.w}, du[4] = {d4.x, d4.y, d4.z, d4.w};
      const float* gr = s_g + q * LD + lane;
      const float* qr = s_q + q * LD + lane;
#pragma unroll
      for (int j = 0; j < CVM; ++j) {
        if (j < cv) {
          const float gv = gr[32 * j], qv = qr[32 * j];
#pragma unroll
          for (int u = 0; u < 4; ++u) acc[u][j] = fmaf(du[u], qv, fmaf(pu[u], gv, acc[u][j]));
        }
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int t = 4 * w + u;
    if (t >= nt) continue;
    float* o = dx + (tt + t) * C + lane;
#pragma unroll
    for (int j = 0; j < CVM; ++j)
      if (j < cv) o[32 * j] = acc[u][j];
  }
}

// blockIdx.x = chunk, blockIdx.y = query group: the chunk's partial dQ rows of the group,
// s sum_t dS[q,t] x[t] over the chunk's tiles in token order.
// C > 256 runs one CTA per SM anyway (202 KB of smem): the whole register file keeps it spill-free.  0 = no minimum.
template <int CVM>
__global__ void __launch_bounds__(kThreads, CVM == 16 ? 1 : 0)
k_apool_bwd_dq(const float* __restrict__ x, const int64_t* __restrict__ off, const float* __restrict__ Q,
               const float* __restrict__ lse, const float* __restrict__ D, const float* __restrict__ dout,
               const int* __restrict__ first, int64_t n, int B, int k, int C, float scale,
               float* __restrict__ part_dq) {
  extern __shared__ __align__(16) float smem[];
  const int LD = C + 4, cv = C >> 5;
  float* s_q = smem;
  float* s_g = s_q + kQG * LD;
  float* s_x = s_g + kQG * LD;
  float* s_ds = s_x + kTile * LD;
  const int c = blockIdx.x;
  if (c >= __ldg(first + B)) return;
  int b;
  int64_t t0, t1;
  chunk_range(off, first, B, n, c, b, t0, t1);
  const int q0 = blockIdx.y * kQG, kq = min(kQG, k - q0);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row0 = (int64_t)b * k;
  load_rows(Q, q0, kq, kQG, C, s_q);
  load_rows(dout, row0 + q0, kq, kQG, C, s_g);
  float acc[4][CVM];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < CVM; ++j) acc[i][j] = 0.f;
  for (int64_t tt = t0; tt < t1; tt += kTile) {
    const int nt = (int)min((int64_t)kTile, t1 - tt);
    __syncthreads();
    load_rows(x, tt, nt, kTile, C, s_x);
    __syncthreads();
    float s[4], dp[4], p[4], ds[4];
    dot4<true>(s_q, s_g, s_x, C, w, lane, s, dp);
    probs(s, dp, lse, D, row0, q0 + 4 * w, k, lane < nt, scale, p, ds);
#pragma unroll
    for (int i = 0; i < 4; ++i) s_ds[(4 * w + i) * kTile + lane] = ds[i];
    __syncwarp();
    accum_pv<CVM>(s_ds, s_x, C, cv, w, lane, acc);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int q = 4 * w + i;
    if (q >= kq) continue;
    float* o = part_dq + ((int64_t)c * k + q0 + q) * C + lane;
#pragma unroll
    for (int j = 0; j < CVM; ++j)
      if (j < cv) o[32 * j] = acc[i][j];
  }
}

// dQ[i] = sum over the chunks of part_dq[chunk][i]: warp p sums chunks p, p + 8, ... in order, then the eight
// warp sums are added in warp order.
__global__ void __launch_bounds__(256)
k_apool_dq_fold(const float* __restrict__ part_dq, const int* __restrict__ first, int B, int64_t kc,
                float* __restrict__ dq) {
  __shared__ float s[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * 32 + lane;
  const int chunks = __ldg(first + B);
  float acc = 0.f;
  if (i < kc)
    for (int p = warp; p < chunks; p += 8) acc += __ldg(part_dq + (int64_t)p * kc + i);
  s[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && i < kc) {
    float t = s[0][lane];
#pragma unroll
    for (int q = 1; q < 8; ++q) t += s[q][lane];
    dq[i] = t;
  }
}

bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

int64_t max_chunks(int64_t n, int B) { return ceil_div(n, kChunk) + B; }

size_t first_bytes(int B) { return align_up((size_t)(B + 1) * sizeof(int)); }

size_t fwd_smem(int C) { return (size_t)((kQG + kTile) * (C + 4) + kQG * kTile) * sizeof(float); }
size_t dx_smem(int C) { return (size_t)((kTile + 2 * kQG) * (C + 4) + 2 * kQG * kTile) * sizeof(float); }
size_t dq_smem(int C) { return (size_t)((2 * kQG + kTile) * (C + 4) + kQG * kTile) * sizeof(float); }

int check_shape(int64_t n, int B, int k, int C) {
  HFL_CHECK_ARG(k >= 1 && k <= kMaxK, "k must be in [1, 256]");
  HFL_CHECK_ARG(C >= 32 && C <= kMaxC && C % 32 == 0, "C must be a multiple of 32 in [32, 512]");
  HFL_CHECK_ARG(B >= 1 && B <= kMaxB, "B must be in [1, 2^24]");
  HFL_CHECK_ARG(n >= 0 && n < (1ll << 31), "n must be in [0, 2^31)");
  return HFL_OK;
}

template <int CVM>
int launch_fwd(const float* x, const int64_t* off, const float* Q, const int* first, int64_t n, int B, int k, int C,
               float scale, float* part_ml, float* part_o, cudaStream_t st) {
  const dim3 grid((unsigned)max_chunks(n, B), (unsigned)ceil_div(k, kQG));
  HFL_ENSURE_SMEM(fwd_smem(C), k_apool_fwd<CVM>);
  HFL_LAUNCH((k_apool_fwd<CVM><<<grid, kThreads, fwd_smem(C), st>>>(x, off, Q, first, n, B, k, C, scale, part_ml,
                                                                     part_o)));
  return HFL_OK;
}

template <int CVM>
int launch_bwd(const float* x, const int64_t* off, const float* Q, const float* lse, const float* D,
               const float* dout, const int* first, int64_t n, int B, int k, int C, float scale, float* dx,
               float* part_dq, cudaStream_t st) {
  const unsigned chunks = (unsigned)max_chunks(n, B);
  HFL_ENSURE_SMEM(dx_smem(C), k_apool_bwd_dx<CVM>);
  HFL_LAUNCH((k_apool_bwd_dx<CVM><<<dim3(chunks, kChunk / kTile), kThreads, dx_smem(C), st>>>(
      x, off, Q, lse, D, dout, first, n, B, k, C, scale, dx)));
  HFL_ENSURE_SMEM(dq_smem(C), k_apool_bwd_dq<CVM>);
  HFL_LAUNCH((k_apool_bwd_dq<CVM><<<dim3(chunks, (unsigned)ceil_div(k, kQG)), kThreads, dq_smem(C), st>>>(
      x, off, Q, lse, D, dout, first, n, B, k, C, scale, part_dq)));
  return HFL_OK;
}

}  // namespace
}  // namespace hfl

using namespace hfl;

extern "C" {

int64_t hfl_attn_pool_train_fwd_workspace_bytes(int64_t n, int32_t B, int32_t k, int32_t C) {
  if (n < 0 || B < 1 || B > kMaxB || k < 1 || k > kMaxK || C < 32 || C > kMaxC || C % 32) return 0;
  const int64_t rows = max_chunks(n, B) * k;
  return (int64_t)(first_bytes(B) + align_up((size_t)rows * 2 * sizeof(float)) +
                   align_up((size_t)rows * C * sizeof(float)));
}

int64_t hfl_attn_pool_train_bwd_workspace_bytes(int64_t n, int32_t B, int32_t k, int32_t C) {
  if (n < 0 || B < 1 || B > kMaxB || k < 1 || k > kMaxK || C < 32 || C > kMaxC || C % 32) return 0;
  return (int64_t)(first_bytes(B) + align_up((size_t)B * k * sizeof(float)) +
                   align_up((size_t)max_chunks(n, B) * k * C * sizeof(float)));
}

int hfl_attn_pool_train_fwd(const float* x, const int64_t* offsets, const float* Q, int64_t n, int32_t B, int32_t k,
                            int32_t C, float* out, float* lse, void* ws, int64_t ws_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const int rc = check_shape(n, B, k, C);
  if (rc != HFL_OK) return rc;
  HFL_CHECK_ARG(offsets && Q && out && lse && (x || n == 0), "null argument");
  HFL_CHECK_ARG(aligned16(Q) && (n == 0 || aligned16(x)), "x and Q must be 16-byte aligned");
  const int64_t need = hfl_attn_pool_train_fwd_workspace_bytes(n, B, k, C);
  if (!ws || ws_bytes < need)
    return fail(HFL_ERR_WORKSPACE, "attention pooling forward workspace too small (%s%lld bytes needed)", "",
                (long long)need);
  HFL_CHECK_ARG(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  const int64_t rows = max_chunks(n, B) * k;
  int* first = (int*)ws;
  float* part_ml = (float*)((char*)ws + first_bytes(B));
  float* part_o = (float*)((char*)part_ml + align_up((size_t)rows * 2 * sizeof(float)));
  const float scale = (float)(1.0 / sqrt((double)C));
  HFL_LAUNCH((k_apool_plan<<<1, 1024, 0, st>>>(offsets, n, B, max_chunks(n, B), first)));
  const int cv = C / 32;
  const int r = cv <= 4 ? launch_fwd<4>(x, offsets, Q, first, n, B, k, C, scale, part_ml, part_o, st)
              : cv <= 8 ? launch_fwd<8>(x, offsets, Q, first, n, B, k, C, scale, part_ml, part_o, st)
                        : launch_fwd<16>(x, offsets, Q, first, n, B, k, C, scale, part_ml, part_o, st);
  if (r != HFL_OK) return r;
  HFL_LAUNCH((k_apool_merge<<<(unsigned)ceil_div((int64_t)B * k, 8), 256, 0, st>>>(first, part_ml, part_o, B, k, C,
                                                                                  out, lse)));
  return HFL_OK;
}

int hfl_attn_pool_train_bwd(const float* x, const int64_t* offsets, const float* Q, const float* out,
                            const float* lse, const float* dout, int64_t n, int32_t B, int32_t k, int32_t C,
                            float* dx, float* dQ, void* ws, int64_t ws_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const int rc = check_shape(n, B, k, C);
  if (rc != HFL_OK) return rc;
  HFL_CHECK_ARG(offsets && Q && out && lse && dout && dQ && (n == 0 || (x && dx)), "null argument");
  HFL_CHECK_ARG(aligned16(Q) && (n == 0 || (aligned16(x) && aligned16(dout))), "x, Q and dout must be 16-byte aligned");
  const int64_t need = hfl_attn_pool_train_bwd_workspace_bytes(n, B, k, C);
  if (!ws || ws_bytes < need)
    return fail(HFL_ERR_WORKSPACE, "attention pooling backward workspace too small (%s%lld bytes needed)", "",
                (long long)need);
  HFL_CHECK_ARG(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  int* first = (int*)ws;
  float* D = (float*)((char*)ws + first_bytes(B));
  float* part_dq = (float*)((char*)D + align_up((size_t)B * k * sizeof(float)));
  const float scale = (float)(1.0 / sqrt((double)C));
  HFL_LAUNCH((k_apool_plan<<<1, 1024, 0, st>>>(offsets, n, B, max_chunks(n, B), first)));
  HFL_LAUNCH((k_apool_delta<<<(unsigned)ceil_div((int64_t)B * k, 8), 256, 0, st>>>(out, dout, (int64_t)B * k, C, D)));
  const int cv = C / 32;
  const int r = cv <= 4 ? launch_bwd<4>(x, offsets, Q, lse, D, dout, first, n, B, k, C, scale, dx, part_dq, st)
              : cv <= 8 ? launch_bwd<8>(x, offsets, Q, lse, D, dout, first, n, B, k, C, scale, dx, part_dq, st)
                        : launch_bwd<16>(x, offsets, Q, lse, D, dout, first, n, B, k, C, scale, dx, part_dq, st);
  if (r != HFL_OK) return r;
  const int64_t kc = (int64_t)k * C;
  HFL_LAUNCH((k_apool_dq_fold<<<(unsigned)ceil_div(kc, 32), 256, 0, st>>>(part_dq, first, B, kc, dQ)));
  return HFL_OK;
}

}  // extern "C"
