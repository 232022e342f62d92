// Relay-token self-attention core with its backward, fp32 (training side): the part of the reference's
// RTAttention.forward between qkv and proj (hotformerloc_backbone.py:83-119) with the mask of
// models/octree.py:229-265, over the ragged per-submap RT sequences instead of concat_and_pad_rt /
// unpad_and_split_rt (relay_token_utils.py:12-79).  Sequence b = packed rows [cu[b], cu[b+1]); for head h
// (head dim 16) and rows i, j of one sequence:
//   s_ij = 0.25 q_i.k_j + (ids[i] == ids[j] ? 0 : -1000)
//   o[i, 16h+e] = sum_j softmax_j(s_i.) v_j[e],        lse[i, h] = log sum_j exp(s_ij)
// The reference pads every sequence to (B, Nmax) with slots whose id matches no RT (not even the padding
// windows' id B), so every padding slot carries -1000 against every real RT.  Row i's own key has bias 0,
// so a padding slot's weight is exp(-1000 + O(|q||k|)) relative to it, which is exactly 0 in fp32 (and in
// fp64): attention over the ragged sequence equals the padded one at every real row, and the padding slots
// get no gradient.  No [B, H, Nmax, Nmax] tensor exists: the forward keeps lse, the backward recomputes p.
//   k_rt_plan : sanitised offsets (each cu entry clamped into [0, T], never below the previous one) and the
//               tile table: sequence b owns tiles [first[b], first[b+1]) of kTile rows
//   k_rt_fwd  : CTA = (tile of query rows, head), thread = query row; online softmax over smem key tiles
//   k_rt_dq   : same partition; D_i = dO_i.o_i, p = exp(s - lse_i), dq_i = 0.25 sum_j p (dO_i.v_j - D_i) k_j
//   k_rt_dkv  : CTA = (tile of key rows, head), thread = key row; dk_j = 0.25 sum_i dS_ij q_i and
//               dv_j = sum_i p_ij dO_i over the queries of the key's own sequence, in ascending i
// Every output element is a fixed-order fp32 sum in one thread (no float atomics, no TF32): o, lse and dqkv
// are bit-identical run to run.  The grid is sized by the bound ceil(T / kTile) + B on the tile count, so
// no host max_len is needed and a sequence may have any length from 0 to T.
#include "common.cuh"

namespace hfl {

namespace {

constexpr int kHd = 16;                 // head dim (C = 16 H)
constexpr int kMaxHeads = 16;
constexpr int kTile = 128;              // query (or key) rows per CTA = threads per CTA
constexpr int kKT = 128;                // keys (or queries) staged in shared memory per step
constexpr int kMaxB = 1 << 24;
constexpr float kScale = 0.25f;         // 16^-0.5 (a power of two: scaling q first is exact)
constexpr float kMaskBias = -1000.f;    // the reference's additive mask value (not -inf)

struct RtArgs {
  const float* qkv;                     // [T, 3C]
  const void* ids;                      // [T] int32 / int64
  const int* off;                       // [B + 1] sanitised offsets (workspace)
  const int* first;                     // [B + 1] tile table (workspace)
  int B, H, ids_i64;
};

__device__ __forceinline__ long long load_id(const RtArgs& a, int64_t r) {
  return a.ids_i64 ? (long long)__ldg((const long long*)a.ids + r) : (long long)__ldg((const int*)a.ids + r);
}

__device__ __forceinline__ void load16(const float* __restrict__ p, float v[kHd]) {
  const float4* p4 = reinterpret_cast<const float4*>(p);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float4 t = __ldg(p4 + c);
    v[4 * c] = t.x; v[4 * c + 1] = t.y; v[4 * c + 2] = t.z; v[4 * c + 3] = t.w;
  }
}

__device__ __forceinline__ void store16(float* p, const float v[kHd], float s) {
  float4* p4 = reinterpret_cast<float4*>(p);
#pragma unroll
  for (int c = 0; c < 4; ++c) p4[c] = make_float4(v[4 * c] * s, v[4 * c + 1] * s, v[4 * c + 2] * s, v[4 * c + 3] * s);
}

__device__ __forceinline__ float dot16(const float a[kHd], const float* b) {
  float d = 0.f;
#pragma unroll
  for (int e = 0; e < kHd; ++e) d = fmaf(a[e], b[e], d);
  return d;
}

// Tile c of the plan: its rows [r0, r1) (r0 < r1) and its sequence's rows [s, e).
__device__ __forceinline__ void tile_range(const RtArgs& a, int c, int& r0, int& r1, int& s, int& e) {
  int lo = 0, hi = a.B;                 // first[lo] <= c < first[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(a.first + mid) <= c) lo = mid; else hi = mid;
  }
  s = __ldg(a.off + lo);
  e = __ldg(a.off + lo + 1);
  r0 = s + (c - __ldg(a.first + lo)) * kTile;
  r1 = min(e, r0 + kTile);
}

// Columns [col, col + 16) of rows [j0, j0 + n) of a row-major matrix with ld floats per row into
// dst[kKT][16]; rows >= n are left as they are (never read).
__device__ __forceinline__ void stage16(const float* __restrict__ src, int64_t ld, int col, int j0, int n,
                                        float* dst) {
  float4* d4 = reinterpret_cast<float4*>(dst);
  for (int t = threadIdx.x; t < n * 4; t += blockDim.x) {
    const int r = t >> 2, c = t & 3;
    d4[t] = __ldg(reinterpret_cast<const float4*>(src + (int64_t)(j0 + r) * ld + col) + c);
  }
}

// ---------------------------------------------------------------------------
// Plan (one CTA of 1024 threads).  off[b] = min(max_{b' <= b} clamp(cu[b'], 0, T), T) for b <= B: a
// decreasing pair is an empty sequence, an entry above T cuts its sequence at T, and sequences never
// overlap.  first[b] = sum_{b' < b} ceil(len_b' / kTile), capped at cap (the grid's tile capacity
// ceil(T / kTile) + B, which the sanitised offsets never exceed); first[B] = the tile count.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
k_rt_plan(const int* __restrict__ cu, int T, int B, int cap, int* __restrict__ off, int* __restrict__ first) {
  __shared__ int s[1024];
  int carry = 0;                        // running max of the clamped entries so far
  for (int base = 0; base <= B; base += 1024) {
    const int b = base + threadIdx.x;
    s[threadIdx.x] = b <= B ? min(max(__ldg(cu + b), 0), T) : 0;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
      const int t = threadIdx.x >= d ? s[threadIdx.x - d] : 0;
      __syncthreads();
      s[threadIdx.x] = max(s[threadIdx.x], t);
      __syncthreads();
    }
    if (b <= B) off[b] = max(carry, s[threadIdx.x]);
    carry = max(carry, s[1023]);
    __syncthreads();
  }
  int tiles = 0;                        // off[] written above by this block: visible after the barrier
  for (int base = 0; base < B; base += 1024) {
    const int b = base + threadIdx.x;
    const int v = b < B ? (int)ceil_div(off[b + 1] - off[b], kTile) : 0;
    s[threadIdx.x] = v;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
      const int t = threadIdx.x >= d ? s[threadIdx.x - d] : 0;
      __syncthreads();
      s[threadIdx.x] += t;
      __syncthreads();
    }
    if (b < B) first[b] = min(tiles + s[threadIdx.x] - v, cap);
    tiles += s[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) first[B] = min(tiles, cap);
}

// ---------------------------------------------------------------------------
// Forward.  blockIdx.x = tile, blockIdx.y = head.  Shared: k, v [kKT][16] and ids [kKT] of the current key
// block of the tile's sequence.  Thread i holds 0.25 q_i and its output row in registers.  The minimum of
// 4 CTAs per SM gives ptxas a 128-register budget (left alone it picks 64 and spills).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kTile, 4)
k_rt_fwd(RtArgs a, float* __restrict__ o, float* __restrict__ lse) {
  __shared__ __align__(16) float s_k[kKT * kHd];
  __shared__ __align__(16) float s_v[kKT * kHd];
  __shared__ long long s_id[kKT];
  const int c = blockIdx.x, h = blockIdx.y;
  if (c >= __ldg(a.first + a.B)) return;
  int r0, r1, s, e;
  tile_range(a, c, r0, r1, s, e);
  const int C = kHd * a.H;
  const int64_t ld = 3 * C;
  const int i = r0 + threadIdx.x;
  const bool row = i < r1;
  float q[kHd], acc[kHd];
#pragma unroll
  for (int t = 0; t < kHd; ++t) q[t] = acc[t] = 0.f;
  long long id_i = 0;
  if (row) {
    load16(a.qkv + i * ld + h * kHd, q);
#pragma unroll
    for (int t = 0; t < kHd; ++t) q[t] *= kScale;
    id_i = load_id(a, i);
  }
  float m = -INFINITY, l = 0.f;
  for (int j0 = s; j0 < e; j0 += kKT) {
    const int nk = min(kKT, e - j0);
    __syncthreads();                    // the previous block's readers are done
    stage16(a.qkv, ld, C + h * kHd, j0, nk, s_k);
    stage16(a.qkv, ld, 2 * C + h * kHd, j0, nk, s_v);
    for (int t = threadIdx.x; t < nk; t += blockDim.x) s_id[t] = load_id(a, j0 + t);
    __syncthreads();
    if (!row) continue;
    constexpr int U = 8;
    for (int u0 = 0; u0 < nk; u0 += U) {
      float sc[U];
      float tmax = -INFINITY;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int j = u0 + u;
        sc[u] = -INFINITY;
        if (j < nk) sc[u] = dot16(q, s_k + j * kHd) + (id_i == s_id[j] ? 0.f : kMaskBias);
        tmax = fmaxf(tmax, sc[u]);
      }
      const float mn = fmaxf(m, tmax);
      const float corr = expf(m - mn);
      l *= corr;
#pragma unroll
      for (int t = 0; t < kHd; ++t) acc[t] *= corr;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int j = u0 + u;
        if (j < nk) {
          const float p = expf(sc[u] - mn);
          l += p;
          const float* vj = s_v + j * kHd;
#pragma unroll
          for (int t = 0; t < kHd; ++t) acc[t] = fmaf(p, vj[t], acc[t]);
        }
      }
      m = mn;
    }
  }
  if (!row) return;
  store16(o + (int64_t)i * C + h * kHd, acc, 1.f / l);   // l >= 1: row i's own key has bias 0
  lse[(int64_t)i * a.H + h] = m + logf(l);
}

// ---------------------------------------------------------------------------
// Backward, query rows.  Same partition and staging as the forward.  Thread i: D_i = dO_i.o_i (kept in
// the workspace for the key pass), then dq_i = 0.25 sum_j p_ij (dO_i.v_j - D_i) k_j in ascending j.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kTile)
k_rt_dq(RtArgs a, const float* __restrict__ o, const float* __restrict__ lse, const float* __restrict__ dout,
        float* __restrict__ D, float* __restrict__ dqkv) {
  __shared__ __align__(16) float s_k[kKT * kHd];
  __shared__ __align__(16) float s_v[kKT * kHd];
  __shared__ long long s_id[kKT];
  const int c = blockIdx.x, h = blockIdx.y;
  if (c >= __ldg(a.first + a.B)) return;
  int r0, r1, s, e;
  tile_range(a, c, r0, r1, s, e);
  const int C = kHd * a.H;
  const int64_t ld = 3 * C;
  const int i = r0 + threadIdx.x;
  const bool row = i < r1;
  float q[kHd], g[kHd], dq[kHd];
#pragma unroll
  for (int t = 0; t < kHd; ++t) q[t] = g[t] = dq[t] = 0.f;
  long long id_i = 0;
  float Di = 0.f, lse_i = 0.f;
  if (row) {
    float ov[kHd];
    load16(a.qkv + i * ld + h * kHd, q);
    load16(dout + (int64_t)i * C + h * kHd, g);
    load16(o + (int64_t)i * C + h * kHd, ov);
#pragma unroll
    for (int t = 0; t < kHd; ++t) {
      q[t] *= kScale;
      Di = fmaf(g[t], ov[t], Di);
    }
    D[(int64_t)i * a.H + h] = Di;
    lse_i = __ldg(lse + (int64_t)i * a.H + h);
    id_i = load_id(a, i);
  }
  for (int j0 = s; j0 < e; j0 += kKT) {
    const int nk = min(kKT, e - j0);
    __syncthreads();
    stage16(a.qkv, ld, C + h * kHd, j0, nk, s_k);
    stage16(a.qkv, ld, 2 * C + h * kHd, j0, nk, s_v);
    for (int t = threadIdx.x; t < nk; t += blockDim.x) s_id[t] = load_id(a, j0 + t);
    __syncthreads();
    if (!row) continue;
    for (int j = 0; j < nk; ++j) {
      const float* kj = s_k + j * kHd;
      const float p = expf(dot16(q, kj) + (id_i == s_id[j] ? 0.f : kMaskBias) - lse_i);
      const float ds = p * (dot16(g, s_v + j * kHd) - Di);
#pragma unroll
      for (int t = 0; t < kHd; ++t) dq[t] = fmaf(ds, kj[t], dq[t]);
    }
  }
  if (row) store16(dqkv + i * ld + h * kHd, dq, kScale);
}

// ---------------------------------------------------------------------------
// Backward, key rows.  blockIdx.x = tile of key rows, blockIdx.y = head.  Shared: 0.25 q, dO [kKT][16],
// lse, D and ids of the current block of the sequence's queries.  Thread j holds k_j, v_j and its dk, dv
// rows; p is recomputed as exp(s - lse_i) with the forward's score arithmetic.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kTile)
k_rt_dkv(RtArgs a, const float* __restrict__ lse, const float* __restrict__ D, const float* __restrict__ dout,
         float* __restrict__ dqkv) {
  __shared__ __align__(16) float s_q[kKT * kHd];
  __shared__ __align__(16) float s_g[kKT * kHd];
  __shared__ float s_lse[kKT];
  __shared__ float s_D[kKT];
  __shared__ long long s_id[kKT];
  const int c = blockIdx.x, h = blockIdx.y;
  if (c >= __ldg(a.first + a.B)) return;
  int r0, r1, s, e;
  tile_range(a, c, r0, r1, s, e);
  const int C = kHd * a.H;
  const int64_t ld = 3 * C;
  const int j = r0 + threadIdx.x;
  const bool row = j < r1;
  float k[kHd], v[kHd], dk[kHd], dv[kHd];
#pragma unroll
  for (int t = 0; t < kHd; ++t) k[t] = v[t] = dk[t] = dv[t] = 0.f;
  long long id_j = 0;
  if (row) {
    load16(a.qkv + j * ld + C + h * kHd, k);
    load16(a.qkv + j * ld + 2 * C + h * kHd, v);
    id_j = load_id(a, j);
  }
  for (int i0 = s; i0 < e; i0 += kKT) {
    const int nq = min(kKT, e - i0);
    __syncthreads();
    stage16(a.qkv, ld, h * kHd, i0, nq, s_q);
    stage16(dout, C, h * kHd, i0, nq, s_g);
    for (int t = threadIdx.x; t < nq; t += blockDim.x) {
      s_lse[t] = __ldg(lse + (int64_t)(i0 + t) * a.H + h);
      s_D[t] = D[(int64_t)(i0 + t) * a.H + h];
      s_id[t] = load_id(a, i0 + t);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nq * kHd; t += blockDim.x) s_q[t] *= kScale;   // as the forward's q
    __syncthreads();
    if (!row) continue;
    for (int r = 0; r < nq; ++r) {
      const float* qi = s_q + r * kHd;
      const float* gi = s_g + r * kHd;
      float sc = 0.f, dp = 0.f;
#pragma unroll
      for (int t = 0; t < kHd; ++t) {
        sc = fmaf(qi[t], k[t], sc);     // the forward's operand order: fmaf(q, k, acc)
        dp = fmaf(gi[t], v[t], dp);
      }
      const float p = expf(sc + (s_id[r] == id_j ? 0.f : kMaskBias) - s_lse[r]);
      const float ds = p * (dp - s_D[r]);
#pragma unroll
      for (int t = 0; t < kHd; ++t) {
        dk[t] = fmaf(ds, qi[t], dk[t]);
        dv[t] = fmaf(p, gi[t], dv[t]);
      }
    }
  }
  if (!row) return;
  store16(dqkv + j * ld + C + h * kHd, dk, 1.f);   // q was staged as 0.25 q: dk already carries the scale
  store16(dqkv + j * ld + 2 * C + h * kHd, dv, 1.f);
}

bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

int64_t max_tiles(int64_t T, int B) { return ceil_div(T, kTile) + B; }

size_t table_bytes(int B) { return align_up((size_t)(B + 1) * sizeof(int)); }

int check_shape(int64_t T, int B, int H) {
  HFL_CHECK_ARG(H >= 1 && H <= kMaxHeads, "num_heads must be in [1, 16] (C = 16 num_heads)");
  HFL_CHECK_ARG(B >= 1 && B <= kMaxB, "B must be in [1, 2^24]");
  HFL_CHECK_ARG(T >= 0 && T * 3 * kHd * H < (1ll << 31) && max_tiles(T, B) < (1ll << 31),
                "T must be >= 0 with T * 3C below 2^31");
  return HFL_OK;
}

// Argument checks shared by the forward and the backward, then the plan launch; fills a.
int setup(const float* qkv, const int32_t* cu, const void* ids, int32_t ids_i64, int32_t B, int64_t T, int32_t H,
          void* ws, int64_t ws_bytes, RtArgs& a, cudaStream_t st) {
  const int rc = check_shape(T, B, H);
  if (rc != HFL_OK) return rc;
  HFL_CHECK_ARG(cu && (T == 0 || (qkv && ids)), "null argument");
  HFL_CHECK_ARG(T == 0 || aligned16(qkv), "qkv must be 16-byte aligned");
  const int64_t need = hfl_rt_attn_train_workspace_bytes(T, B, H);
  if (!ws || ws_bytes < need)
    return fail(HFL_ERR_WORKSPACE, "relay-token attention workspace too small (%s%lld bytes needed)", "",
                (long long)need);
  HFL_CHECK_ARG(((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  int* off = (int*)ws;
  int* first = (int*)((char*)ws + table_bytes(B));
  a = RtArgs{qkv, ids, off, first, B, H, ids_i64 != 0};
  HFL_LAUNCH((k_rt_plan<<<1, 1024, 0, st>>>(cu, (int)T, B, (int)max_tiles(T, B), off, first)));
  return HFL_OK;
}

}  // namespace
}  // namespace hfl

using namespace hfl;

extern "C" {

int64_t hfl_rt_attn_train_workspace_bytes(int64_t T, int32_t B, int32_t H) {
  if (T < 0 || B < 1 || B > kMaxB || H < 1 || H > kMaxHeads) return 0;
  return (int64_t)(2 * table_bytes(B) + align_up((size_t)T * H * sizeof(float)));
}

int hfl_rt_attn_train_fwd(const float* qkv, const int32_t* cu, const void* ids, int32_t ids_i64, int32_t B,
                          int64_t T, int32_t H, float* o, float* lse, void* ws, int64_t ws_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(T == 0 || (o && lse), "null argument");
  HFL_CHECK_ARG(T == 0 || aligned16(o), "o must be 16-byte aligned");
  RtArgs a;
  const int rc = setup(qkv, cu, ids, ids_i64, B, T, H, ws, ws_bytes, a, st);
  if (rc != HFL_OK || T == 0) return rc;
  HFL_LAUNCH((k_rt_fwd<<<dim3((unsigned)max_tiles(T, B), (unsigned)H), kTile, 0, st>>>(a, o, lse)));
  return HFL_OK;
}

int hfl_rt_attn_train_bwd(const float* qkv, const int32_t* cu, const void* ids, int32_t ids_i64, const float* o,
                          const float* lse, const float* dout, int32_t B, int64_t T, int32_t H, float* dqkv, void* ws,
                          int64_t ws_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(T == 0 || (o && lse && dout && dqkv), "null argument");
  HFL_CHECK_ARG(T == 0 || (aligned16(o) && aligned16(dout) && aligned16(dqkv)),
                "o, dout and dqkv must be 16-byte aligned");
  RtArgs a;
  const int rc = setup(qkv, cu, ids, ids_i64, B, T, H, ws, ws_bytes, a, st);
  if (rc != HFL_OK || T == 0) return rc;
  float* D = (float*)((char*)ws + 2 * table_bytes(B));
  const dim3 grid((unsigned)max_tiles(T, B), (unsigned)H);
  HFL_LAUNCH((k_rt_dq<<<grid, kTile, 0, st>>>(a, o, lse, dout, D, dqkv)));
  HFL_LAUNCH((k_rt_dkv<<<grid, kTile, 0, st>>>(a, lse, D, dout, dqkv)));
  return HFL_OK;
}

}  // extern "C"
