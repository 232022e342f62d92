// Octree window attention core with its backward, fp32 (training side): the part of the reference's
// OctreeAttention.forward from qkv to before proj (octformer_backbone.py:52-93), with the relative
// position bias (octformer_layers.py:156-170), the submap mask and, for H-OSA, the relay token at
// window position 0 (hotformerloc_backbone.py:197-236).  For window n, head h, queries i, keys j:
//   s[i,j] = (q_i . k_j) * 0.25 + (ids_i == ids_j ? 0 : -1000) + sum_a table[clamp(x_ia - x_ja) + bnd + a num, h]
//   o_i    = sum_j softmax_j(s)[i,j] v_j,           lse_i = log sum_j exp(s[i,j])
// (head dim 16; with hat = 1 the relay token's row and column get no bias).  No (N_win, H, L, L)
// tensor is ever written: the forward keeps lse, the backward recomputes S from qkv and lse.
//   k_wattn_fwd    : one CTA per (window, head), one thread per query row, online softmax in tiles of 8 keys
//   k_wattn_absmax : max|v| and max|dO| (fix the fixed-point scale of the table gradient)
//   k_wattn_bwd    : one CTA per (window chunk, head); dq by rows, dk / dv by columns through the P and
//                    dS tiles in shared memory, table gradient in exact int64 fixed point
//   k_wattn_dtable : fixed point -> fp32 table gradient
// Every dq / dk / dv element is a fixed-order fp32 sum in one thread, and integer addition is
// associative, so dqkv and the table gradient are bit-identical run to run without float atomics.
#include "common.cuh"

namespace hfl {

namespace {

constexpr int kHd = 16;                 // head dim (C = 16 H)
constexpr int kMaxL = 128;
constexpr int kMaxHeads = 16;
constexpr int kMaxBnd = 1 << 20;
constexpr float kScale = 0.25f;         // 16^-0.5
constexpr float kMaskBias = -1000.f;    // the reference's additive mask value (not -inf)
constexpr int kBwdCtas = 4096;          // target CTAs of the backward (partition by shape only)
constexpr int kSmemTableBytes = 32 * 1024;

struct WinArgs {
  const float* qkv;                     // [n_win, L, 3C]
  const void* xyz;                      // [n_win, L - hat, 3] int32 / int64 (unused without table)
  const void* ids;                      // [n_win, L] int32 / int64
  const float* table;                   // [3 num, H] or NULL
  int64_t n_win;
  int L, H, hat, bnd, xyz_i64, ids_i64;
};

__device__ __forceinline__ long long load_idx(const void* p, int i64, int64_t k) {
  return i64 ? (long long)__ldg((const long long*)p + k) : (long long)__ldg((const int*)p + k);
}

// Window n's ids and token coordinates into shared memory (xs[t*3+a] for window token t = pos - hat).
__device__ __forceinline__ void load_window_idx(const WinArgs& a, int64_t n, long long* s_id, long long* s_xs) {
  for (int t = threadIdx.x; t < a.L; t += blockDim.x) s_id[t] = load_idx(a.ids, a.ids_i64, n * a.L + t);
  if (a.table) {
    const int K3 = (a.L - a.hat) * 3;
    for (int t = threadIdx.x; t < K3; t += blockDim.x) s_xs[t] = load_idx(a.xyz, a.xyz_i64, n * K3 + t);
  }
}

// Rows [0, L) of window n, columns [col, col + 16) of qkv, into dst[L][16].
__device__ __forceinline__ void load_head(const float* __restrict__ src, int64_t row0, int64_t ld, int col, int L,
                                          float* dst) {
  float4* d4 = reinterpret_cast<float4*>(dst);
  for (int t = threadIdx.x; t < L * 4; t += blockDim.x) {
    const int r = t >> 2, c = t & 3;
    d4[t] = __ldg(reinterpret_cast<const float4*>(src + (row0 + r) * ld + col) + c);
  }
}

// Table rows of pair (i, j) for the three axes; false when the pair takes no bias (no table, or
// the relay token's row or column).
__device__ __forceinline__ bool rpe_bins(const WinArgs& a, const long long* s_xs, const long long* xi, int i, int j,
                                         int bin[3]) {
  if (!a.table || (a.hat && (i == 0 || j == 0))) return false;
  const int num = 2 * a.bnd + 1;
  const long long* xj = s_xs + (j - a.hat) * 3;
#pragma unroll
  for (int ax = 0; ax < 3; ++ax) {
    long long d = xi[ax] - xj[ax];
    d = d < -a.bnd ? -a.bnd : (d > a.bnd ? a.bnd : d);
    bin[ax] = (int)d + a.bnd + ax * num;
  }
  return true;
}

__device__ __forceinline__ float score(const WinArgs& a, const float q[kHd], const float* kj, long long id_i,
                                       long long id_j, bool has_bias, const int bin[3], int h) {
  float d = 0.f;
#pragma unroll
  for (int e = 0; e < kHd; ++e) d = fmaf(q[e], kj[e], d);
  float b = id_i == id_j ? 0.f : kMaskBias;
  if (has_bias) {
    const float r = __ldg(a.table + (int64_t)bin[0] * a.H + h) + __ldg(a.table + (int64_t)bin[1] * a.H + h) +
                    __ldg(a.table + (int64_t)bin[2] * a.H + h);
    b += r;
  }
  return d * kScale + b;
}

__device__ __forceinline__ void row_coords(const WinArgs& a, const long long* s_xs, int i, long long xi[3]) {
  const bool tok = a.table && i >= a.hat;
#pragma unroll
  for (int ax = 0; ax < 3; ++ax) xi[ax] = tok ? s_xs[(i - a.hat) * 3 + ax] : 0;
}

// ---------------------------------------------------------------------------
// Forward.  blockIdx.x = n H + h; blockDim = L rounded up to a warp.  Shared: k, v [L][16], ids [L],
// coordinates [L - hat][3].  Thread i holds q_i and its output row in registers.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kMaxL)
k_wattn_fwd(WinArgs a, float* __restrict__ o, float* __restrict__ lse) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int L = a.L, H = a.H, C = kHd * H;
  long long* s_id = reinterpret_cast<long long*>(smem);
  long long* s_xs = s_id + L;
  float* s_k = reinterpret_cast<float*>(s_xs + 3 * L);
  float* s_v = s_k + L * kHd;
  const int64_t n = blockIdx.x / H;
  const int h = blockIdx.x - (int)(n * H);
  const int64_t row0 = n * L;
  load_head(a.qkv, row0, 3 * C, C + h * kHd, L, s_k);
  load_head(a.qkv, row0, 3 * C, 2 * C + h * kHd, L, s_v);
  load_window_idx(a, n, s_id, s_xs);
  __syncthreads();
  const int i = threadIdx.x;
  if (i >= L) return;
  float q[kHd], acc[kHd];
  const float4* q4 = reinterpret_cast<const float4*>(a.qkv + (row0 + i) * 3 * C + h * kHd);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float4 t = __ldg(q4 + c);
    q[4 * c] = t.x; q[4 * c + 1] = t.y; q[4 * c + 2] = t.z; q[4 * c + 3] = t.w;
  }
#pragma unroll
  for (int e = 0; e < kHd; ++e) acc[e] = 0.f;
  long long xi[3];
  row_coords(a, s_xs, i, xi);
  const long long id_i = s_id[i];
  float m = -INFINITY, l = 0.f;
  constexpr int T = 8;
  for (int j0 = 0; j0 < L; j0 += T) {
    float s[T];
    float tmax = -INFINITY;
#pragma unroll
    for (int u = 0; u < T; ++u) {
      const int j = j0 + u;
      s[u] = -INFINITY;
      if (j < L) {
        int bin[3];
        const bool hb = rpe_bins(a, s_xs, xi, i, j, bin);
        s[u] = score(a, q, s_k + j * kHd, id_i, s_id[j], hb, bin, h);
      }
      tmax = fmaxf(tmax, s[u]);
    }
    const float mn = fmaxf(m, tmax);
    const float corr = expf(m - mn);
    l *= corr;
#pragma unroll
    for (int e = 0; e < kHd; ++e) acc[e] *= corr;
#pragma unroll
    for (int u = 0; u < T; ++u) {
      const int j = j0 + u;
      if (j < L) {
        const float p = expf(s[u] - mn);
        l += p;
        const float* vj = s_v + j * kHd;
#pragma unroll
        for (int e = 0; e < kHd; ++e) acc[e] = fmaf(p, vj[e], acc[e]);
      }
    }
    m = mn;
  }
  const float inv = 1.f / l;
  float4* o4 = reinterpret_cast<float4*>(o + (row0 + i) * C + h * kHd);
#pragma unroll
  for (int c = 0; c < 4; ++c)
    o4[c] = make_float4(acc[4 * c] * inv, acc[4 * c + 1] * inv, acc[4 * c + 2] * inv, acc[4 * c + 3] * inv);
  lse[(n * H + h) * L + i] = m + logf(l);
}

// ---------------------------------------------------------------------------
// Table gradient in fixed point.  Contribution dS (the gradient of s[i,j]) is added as
// round(dS 2^e) to an int64 per (bin, head); integer sums do not depend on order.  Range: with
// |v|, |dO| <= Mv, Md, |dP| = |dO_i . v_j| <= 16 Md Mv and |D_i| <= 16 Md Mv, so
// sum_j |dS_ij| = sum_j p_ij |dP_ij - D_i| <= 32 Md Mv per query row, and one bin of one head
// collects at most N_win L such rows: |bin| <= B = N_win L 32 Md Mv.  e = 61 - ceil(log2 B) keeps
// |bin| 2^e <= 2^61, plus at most N_win L^2 / 2 < 2^45 from the roundings: no int64 overflow.  Each
// rounding is <= 2^-e-1 <= B 2^-62 in absolute terms.
// ---------------------------------------------------------------------------
// v added to the int64 kept as (lo, hi) 32-bit words of a shared table: native 32-bit shared
// atomics (a 64-bit shared add is a CAS loop), the carry out of lo goes into hi.  The pair holds the
// exact sum modulo 2^64 whatever the order of the adds.
__device__ __forceinline__ void add_fx_shared(unsigned* w, long long v) {
  const unsigned lo = (unsigned)v;
  unsigned hi = (unsigned)((unsigned long long)v >> 32);
  const unsigned old = atomicAdd(w, lo);
  hi += (old + lo < old);
  if (hi) atomicAdd(w + 1, hi);
}

// 32-bit words of the shared (lo, hi) table, rounded up to 16 bytes: the float4 tiles follow it.
__host__ __device__ __forceinline__ int acc_words(int num3) { return (2 * num3 + 3) & ~3; }

__device__ __forceinline__ int fx_exponent(const unsigned* mx, int64_t n_win, int L) {
  const double M = (double)__uint_as_float(mx[0]) * (double)__uint_as_float(mx[1]);
  const double B = (double)n_win * L * 32.0 * M;
  if (!(B > 0.0) || isinf(B)) return 0;       // all zero (any exponent is exact) or non-finite inputs
  int e;
  frexp(B, &e);                               // B < 2^e
  return 61 - e;
}

// mx[0] = max|v| over the v columns of qkv, mx[1] = max|dO| (nonnegative floats order as their bits).
__global__ void __launch_bounds__(256)
k_wattn_absmax(const float* __restrict__ qkv, const float* __restrict__ dout, int64_t rows, int C,
               unsigned* __restrict__ mx) {
  unsigned bv = 0u, bd = 0u;                  // |x| as bits: NaN and inf compare above every finite value
  const int64_t total = rows * C;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / C;
    const int c = (int)(t - r * C);
    bv = max(bv, __float_as_uint(__ldg(qkv + r * 3 * C + 2 * C + c)) & 0x7fffffffu);
    bd = max(bd, __float_as_uint(__ldg(dout + t)) & 0x7fffffffu);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    bv = max(bv, __shfl_xor_sync(0xffffffffu, bv, off));
    bd = max(bd, __shfl_xor_sync(0xffffffffu, bd, off));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(mx, bv);
    atomicMax(mx + 1, bd);
  }
}

// ---------------------------------------------------------------------------
// Backward.  blockIdx.x = chunk H + h; the chunk is windows [chunk W, chunk W + W), W from the shapes
// only.  Per window: rows pass (thread i) recomputes s, p = exp(s - lse_i), dP = dO_i . v_j,
// dS = p (dP - D_i) with D_i = dO_i . o_i, stores P and dS (row stride L + 1: conflict-free column
// reads) and accumulates dq_i; the columns pass (thread j) sums dk_j = 0.25 sum_i dS_ij q_i and
// dv_j = sum_i P_ij dO_i in ascending i.  The table gradient goes to a shared int64 table of the head
// (flushed once per CTA with global integer atomics), or straight to the workspace's int64 table when
// it does not fit in kSmemTableBytes.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kMaxL)
k_wattn_bwd(WinArgs a, const float* __restrict__ o, const float* __restrict__ lse, const float* __restrict__ dout,
            int64_t win_per_cta, int table_in_smem, unsigned long long* __restrict__ ws_acc,
            const unsigned* __restrict__ mx, float* __restrict__ dqkv) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int L = a.L, H = a.H, C = kHd * H, LP = L + 1;
  const int num3 = a.table ? 3 * (2 * a.bnd + 1) : 0;
  unsigned* s_acc = reinterpret_cast<unsigned*>(smem);                // [num3][2] (lo, hi)
  long long* s_id = reinterpret_cast<long long*>(s_acc + (table_in_smem ? acc_words(num3) : 0));
  long long* s_xs = s_id + L;
  float* s_q = reinterpret_cast<float*>(s_xs + 3 * L);
  float* s_k = s_q + L * kHd;
  float* s_v = s_k + L * kHd;
  float* s_do = s_v + L * kHd;
  float* s_p = s_do + L * kHd;
  float* s_ds = s_p + L * LP;
  const int64_t chunk = blockIdx.x / H;
  const int h = blockIdx.x - (int)(chunk * H);
  const int64_t n0 = chunk * win_per_cta;
  const int64_t n1 = min(a.n_win, n0 + win_per_cta);
  double fx_scale = 0.0;
  if (a.table) {
    fx_scale = ldexp(1.0, fx_exponent(mx, a.n_win, L));
    if (table_in_smem)
      for (int t = threadIdx.x; t < 2 * num3; t += blockDim.x) s_acc[t] = 0u;
  }
  const int i = threadIdx.x;
  for (int64_t n = n0; n < n1; ++n) {
    const int64_t row0 = n * L;
    load_head(a.qkv, row0, 3 * C, h * kHd, L, s_q);
    load_head(a.qkv, row0, 3 * C, C + h * kHd, L, s_k);
    load_head(a.qkv, row0, 3 * C, 2 * C + h * kHd, L, s_v);
    load_head(dout, row0, C, h * kHd, L, s_do);
    load_window_idx(a, n, s_id, s_xs);
    __syncthreads();
    if (i < L) {
      float q[kHd], g[kHd], dq[kHd];
      float D = 0.f;
      const float4* o4 = reinterpret_cast<const float4*>(o + (row0 + i) * C + h * kHd);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float4 t = __ldg(o4 + c);
        const float oe[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = 4 * c + u;
          q[e] = s_q[i * kHd + e];
          g[e] = s_do[i * kHd + e];
          dq[e] = 0.f;
          D = fmaf(g[e], oe[u], D);
        }
      }
      const float lse_i = __ldg(lse + (n * H + h) * L + i);
      long long xi[3];
      row_coords(a, s_xs, i, xi);
      const long long id_i = s_id[i];
      for (int j = 0; j < L; ++j) {
        int bin[3];
        const bool hb = rpe_bins(a, s_xs, xi, i, j, bin);
        const float* kj = s_k + j * kHd;
        const float p = expf(score(a, q, kj, id_i, s_id[j], hb, bin, h) - lse_i);
        const float* vj = s_v + j * kHd;
        float dp = 0.f;
#pragma unroll
        for (int e = 0; e < kHd; ++e) dp = fmaf(g[e], vj[e], dp);
        const float ds = p * (dp - D);
        s_p[i * LP + j] = p;
        s_ds[i * LP + j] = ds;
#pragma unroll
        for (int e = 0; e < kHd; ++e) dq[e] = fmaf(ds, kj[e], dq[e]);
        if (hb) {
          const long long f = __double2ll_rn((double)ds * fx_scale);
          if (f && table_in_smem) {
#pragma unroll
            for (int ax = 0; ax < 3; ++ax) add_fx_shared(s_acc + 2 * bin[ax], f);
          } else if (f) {
#pragma unroll
            for (int ax = 0; ax < 3; ++ax) atomicAdd(ws_acc + (int64_t)bin[ax] * H + h, (unsigned long long)f);
          }
        }
      }
      float4* d4 = reinterpret_cast<float4*>(dqkv + (row0 + i) * 3 * C + h * kHd);
#pragma unroll
      for (int c = 0; c < 4; ++c)
        d4[c] = make_float4(dq[4 * c] * kScale, dq[4 * c + 1] * kScale, dq[4 * c + 2] * kScale,
                            dq[4 * c + 3] * kScale);
    }
    __syncthreads();
    if (i < L) {
      const int j = i;
      float dk[kHd], dv[kHd];
#pragma unroll
      for (int e = 0; e < kHd; ++e) dk[e] = dv[e] = 0.f;
      for (int r = 0; r < L; ++r) {
        const float ds = s_ds[r * LP + j], p = s_p[r * LP + j];
#pragma unroll
        for (int e = 0; e < kHd; ++e) {
          dk[e] = fmaf(ds, s_q[r * kHd + e], dk[e]);
          dv[e] = fmaf(p, s_do[r * kHd + e], dv[e]);
        }
      }
      float4* k4 = reinterpret_cast<float4*>(dqkv + (row0 + j) * 3 * C + C + h * kHd);
      float4* v4 = reinterpret_cast<float4*>(dqkv + (row0 + j) * 3 * C + 2 * C + h * kHd);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        k4[c] = make_float4(dk[4 * c] * kScale, dk[4 * c + 1] * kScale, dk[4 * c + 2] * kScale,
                            dk[4 * c + 3] * kScale);
        v4[c] = make_float4(dv[4 * c], dv[4 * c + 1], dv[4 * c + 2], dv[4 * c + 3]);
      }
    }
    __syncthreads();
  }
  if (table_in_smem && a.table)
    for (int t = threadIdx.x; t < num3; t += blockDim.x) {
      const unsigned long long v = ((unsigned long long)s_acc[2 * t + 1] << 32) | s_acc[2 * t];
      if (v) atomicAdd(ws_acc + (int64_t)t * H + h, v);
    }
}

__global__ void __launch_bounds__(256)
k_wattn_dtable(const unsigned long long* __restrict__ ws_acc, const unsigned* __restrict__ mx, int64_t n_win,
               int L, int64_t total, float* __restrict__ dtable) {
  const bool finite = mx[0] < 0x7f800000u && mx[1] < 0x7f800000u;
  const double inv = ldexp(1.0, -fx_exponent(mx, n_win, L));
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x)
    dtable[t] = finite ? (float)((double)(long long)ws_acc[t] * inv) : __uint_as_float(0x7fc00000u);
}

bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

int threads_for(int L) { return (int)ceil_div(L, 32) * 32; }

size_t fwd_smem(int L) { return (size_t)L * 4 * sizeof(long long) + (size_t)2 * L * kHd * sizeof(float); }

bool table_fits_smem(int bnd) { return (size_t)3 * (2 * bnd + 1) * sizeof(unsigned long long) <= kSmemTableBytes; }

size_t bwd_smem(int L, int bnd, int has_table) {
  const size_t tab = has_table && table_fits_smem(bnd) ? (size_t)acc_words(3 * (2 * bnd + 1)) * sizeof(unsigned) : 0;
  return tab + (size_t)L * 4 * sizeof(long long) + (size_t)4 * L * kHd * sizeof(float) +
         (size_t)2 * L * (L + 1) * sizeof(float);
}

size_t acc_bytes(int H, int bnd) { return align_up((size_t)3 * (2 * bnd + 1) * H * sizeof(unsigned long long)); }

int check_common(const WinArgs& a) {
  HFL_CHECK_ARG(a.H >= 1 && a.H <= kMaxHeads, "num_heads must be in [1, 16] (C = 16 num_heads)");
  HFL_CHECK_ARG(a.L >= 1 && a.L <= kMaxL, "L must be in [1, 128]");
  HFL_CHECK_ARG(a.hat == 0 || a.hat == 1, "hat must be 0 or 1");
  HFL_CHECK_ARG(a.bnd >= 0 && a.bnd <= kMaxBnd, "bnd must be in [0, 1048576]");
  HFL_CHECK_ARG(a.n_win >= 0, "negative window count");
  HFL_CHECK_ARG(a.n_win * a.H < (1ll << 31), "n_win * num_heads must be below 2^31");
  if (a.n_win == 0) return HFL_OK;
  HFL_CHECK_ARG(a.qkv && a.ids, "null argument");
  HFL_CHECK_ARG(!a.table || a.L == a.hat || a.xyz, "xyz is required with a table");
  HFL_CHECK_ARG(aligned16(a.qkv), "qkv must be 16-byte aligned");
  return HFL_OK;
}

}  // namespace
}  // namespace hfl

using namespace hfl;

extern "C" {

int hfl_window_attn_train_fwd(const float* qkv, const void* xyz, int32_t xyz_i64, const void* ids, int32_t ids_i64,
                              const float* rpe_table, int64_t n_win, int32_t L, int32_t H, int32_t hat, int32_t bnd,
                              float* o, float* lse, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const WinArgs a{qkv, xyz, ids, rpe_table, n_win, L, H, hat, bnd, xyz_i64 != 0, ids_i64 != 0};
  const int rc = check_common(a);
  if (rc != HFL_OK || n_win == 0) return rc;
  HFL_CHECK_ARG(o && lse, "null argument");
  HFL_CHECK_ARG(aligned16(o), "o must be 16-byte aligned");
  HFL_LAUNCH((k_wattn_fwd<<<(unsigned)(n_win * H), threads_for(L), fwd_smem(L), st>>>(a, o, lse)));
  return HFL_OK;
}

int64_t hfl_window_attn_train_bwd_workspace_bytes(int32_t H, int32_t bnd, int32_t has_rpe) {
  if (!has_rpe || H < 1 || H > kMaxHeads || bnd < 0 || bnd > kMaxBnd) return 0;
  return (int64_t)(acc_bytes(H, bnd) + 256);
}

int hfl_window_attn_train_bwd(const float* qkv, const void* xyz, int32_t xyz_i64, const void* ids, int32_t ids_i64,
                              const float* rpe_table, const float* o, const float* lse, const float* dout,
                              int64_t n_win, int32_t L, int32_t H, int32_t hat, int32_t bnd, float* dqkv,
                              float* drpe_table, void* ws, int64_t ws_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const WinArgs a{qkv, xyz, ids, rpe_table, n_win, L, H, hat, bnd, xyz_i64 != 0, ids_i64 != 0};
  const int rc = check_common(a);
  if (rc != HFL_OK) return rc;
  HFL_CHECK_ARG(!rpe_table || drpe_table, "null argument");
  const int64_t n_tab = rpe_table ? (int64_t)3 * (2 * bnd + 1) * H : 0;
  if (n_win == 0) {                              // no windows: the table gradient is zero
    if (n_tab) HFL_CUDA(cudaMemsetAsync(drpe_table, 0, (size_t)n_tab * sizeof(float), st));
    return HFL_OK;
  }
  HFL_CHECK_ARG(o && lse && dout && dqkv, "null argument");
  HFL_CHECK_ARG(aligned16(o) && aligned16(dout) && aligned16(dqkv), "o, dout and dqkv must be 16-byte aligned");
  const int64_t need = hfl_window_attn_train_bwd_workspace_bytes(H, bnd, rpe_table != nullptr);
  if (need && (!ws || ws_bytes < need))
    return fail(HFL_ERR_WORKSPACE, "window attention backward workspace too small (%s%lld bytes needed)", "",
                (long long)need);
  HFL_CHECK_ARG(!need || ((uintptr_t)ws & 255) == 0, "workspace must be 256-byte aligned");
  unsigned long long* ws_acc = (unsigned long long*)ws;
  unsigned* mx = need ? (unsigned*)((char*)ws + acc_bytes(H, bnd)) : nullptr;
  if (need) {
    HFL_CUDA(cudaMemsetAsync(ws, 0, (size_t)need, st));
    const int C = kHd * H;
    HFL_LAUNCH((k_wattn_absmax<<<grid_for(n_win * L * C, 256, kSMs * 8), 256, 0, st>>>(qkv, dout, n_win * L, C,
                                                                                       mx)));
  }
  const int64_t chunks = min(n_win, ceil_div(kBwdCtas, H));
  const int64_t per = ceil_div(n_win, chunks);
  const int in_smem = rpe_table && table_fits_smem(bnd);
  const size_t smem = bwd_smem(L, bnd, rpe_table != nullptr);
  HFL_ENSURE_SMEM(smem, k_wattn_bwd);
  HFL_LAUNCH((k_wattn_bwd<<<(unsigned)(ceil_div(n_win, per) * H), threads_for(L), smem, st>>>(
      a, o, lse, dout, per, in_smem, ws_acc, mx, dqkv)));
  if (n_tab)
    HFL_LAUNCH((k_wattn_dtable<<<grid_for(n_tab, 256), 256, 0, st>>>(ws_acc, mx, n_win, L, n_tab, drpe_table)));
  return HFL_OK;
}

}  // extern "C"
