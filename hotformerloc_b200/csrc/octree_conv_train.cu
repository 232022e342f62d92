// Octree convolution with backward, fp32 without TF32: the training-side form of ocnn.nn.OctreeConv for
// the two shapes of the model, 3x3x3 stride 1 (PatchEmbed convs / proj) and 2x2x2 stride 2 (the
// downsamples), both nempty.
//   k_oconv_fwd        : out[i,:] = sum_k sum_c data[neigh[i,k],c] W[k,c,:] over the occupied taps
//                        (called with the inverse table and W[k]^T it is the input gradient)
//   k_oconv_wgrad      : per-chunk partials of dW[k] = sum_i data[neigh[i,k]]^T (x) dout[i]
//   k_oconv_wgrad_fold : fixed-order sum of the partials
// Tables are (rows, K) int32 or int64, K in {8, 27}; an entry outside [0, n_in) is an empty tap.
//
// Work follows the occupied (row, tap) pairs, not a tile's tap union: an octree table is sparse in a
// way no dense tile sees (Oxford rows hold ~1 occupied tap of 27, almost always the centre one).  For
// each tile of kTM output rows and each tap k the block compacts the rows that have tap k into a list
// of m_k rows and runs only that product, in warp steps of LR = 32 / LC rows.  Executed FMAs of the
// forward are therefore sum over (tile, k) of ceil(m_k / LR) LR Cin TN ceil(Cout / TN), TN = 16 LC
// (tools/octree_conv_train_bench.py evaluates this rule on real tables).  The weight gradient
// contracts over the compacted rows exactly: its executed FMAs are the pairs times
// ceil(Cin / TI) TI ceil(Cout / TO) TO.
//
// Rounding (what tests/test_octree_conv_gpu.py holds each element to, (s + 2) 2^-24 sum |terms|):
//   forward / input gradient: each tap's product is one fmaf chain over the Cin channels in ascending
//     order, started from 0, and the taps are added into the output element in ascending k, so the
//     longest chain into an element is s = Cin + K (Cin the reduced width: Cout of the forward for the
//     input gradient).
//   weight gradient: a thread sums its group's rows of one chunk in row order (at most R = rows per
//     chunk terms), the G row groups of a block are added in group order, then the chunks in chunk
//     order: s = R + G + chunks <= R + 32 + chunks.
// Every output element is a fixed-order sum owned by one thread, without float atomics, over a
// partition that depends on (n, K, Cin, Cout) only: results are bit-identical across runs and GPUs,
// and int32 and int64 tables give the same bits.
#include "common.cuh"

namespace hfl {

namespace {

constexpr int kTM = 128;             // output rows per forward tile
constexpr int kKC = 32;              // input channels per shared-memory stage
constexpr int kMaxK = 27;
constexpr int kMaxC = 256;
constexpr int kWRows = 64;           // rows per weight-gradient sub-tile
constexpr int kWMinRows = 256;       // least rows per weight-gradient chunk
constexpr int kWMaxChunks = 1024;
constexpr int64_t kWMaxWsFloats = 1ll << 25;   // workspace cap: 128 MiB of partials

__device__ __forceinline__ void outer4(float* acc, float a, float4 d) {
  acc[0] = fmaf(a, d.x, acc[0]); acc[1] = fmaf(a, d.y, acc[1]);
  acc[2] = fmaf(a, d.z, acc[2]); acc[3] = fmaf(a, d.w, acc[3]);
}

__device__ __forceinline__ int32_t tap_entry(int64_t e, int64_t n_in) {
  return (e >= 0 && e < n_in) ? (int32_t)e : -1;
}

// Block-wide stable compaction of the NR = 32 NW rows whose entry is >= 0: s_src[j] = entry, s_row[j] =
// row; returns m (every thread).  Warps >= NW only take part in the barriers.
template <int NW>
__device__ __forceinline__ int compact_rows(int32_t e, int* s_cnt, int32_t* s_src, int32_t* s_row) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned bal = 0;
  if (warp < NW) {
    bal = __ballot_sync(0xffffffffu, e >= 0);
    if (lane == 0) s_cnt[warp] = __popc(bal);
  }
  __syncthreads();
  int m = 0, off = 0;
#pragma unroll
  for (int q = 0; q < NW; ++q) {
    const int c = s_cnt[q];
    if (q < warp) off += c;
    m += c;
  }
  if (warp < NW && e >= 0) {
    const int j = off + __popc(bal & ((1u << lane) - 1u));
    s_src[j] = e;
    s_row[j] = warp * 32 + lane;
  }
  return m;
}

template <int LC>
struct FwdSmem {
  static constexpr int TN = 16 * LC;
  static constexpr size_t acc = (size_t)kTM * TN;            // floats
  static constexpr size_t a = (size_t)kKC * (kTM + 1);       // floats, [ci][j], padded
  static constexpr size_t b = (size_t)kKC * TN;              // floats, [ci][c]
  static constexpr size_t nb = (size_t)kTM * kMaxK;          // int32
  static constexpr size_t bytes = (acc + a + b + nb + 2 * kTM + 4) * 4;
};

// ---------------------------------------------------------------------------
// Forward / input gradient.  Block (x, y): output rows [x kTM, (x+1) kTM), columns [y TN, (y+1) TN).
// Warp w, lane = lr LC + lc: compacted rows p PASS + w LR + lr (p < NP) and the 16 columns
// 4 (q LC + lc) + t (q, t < 4) of the block's TN, so the four float4 reads of a W stage are each one
// contiguous 16 LC-byte line across the lanes.  Per tap: compact, then for each stage of kKC input
// channels gather the m rows (A, transposed) and W[k] (B) into shared memory and accumulate in
// registers; the tap's product is then added into the block's fp32 accumulator tile s_acc by the
// compacted row's original row (one thread per element: no races, fixed order).
// ---------------------------------------------------------------------------
template <int LC, bool VEC, typename IdxT>
__global__ void __launch_bounds__(256, 2)
k_oconv_fwd(const float* __restrict__ data, const IdxT* __restrict__ neigh, const float* __restrict__ w,
            int64_t n_out, int64_t n_in, int K, int Cin, int Cout, float* __restrict__ out) {
  using S = FwdSmem<LC>;
  constexpr int TN = S::TN, LR = 32 / LC, PASS = 8 * LR, NP = kTM / PASS;
  extern __shared__ __align__(16) float smem[];
  float* s_acc = smem;
  float* s_a = s_acc + S::acc;
  float* s_b = s_a + S::a;
  int32_t* s_nb = reinterpret_cast<int32_t*>(s_b + S::b);
  int32_t* s_src = s_nb + S::nb;
  int32_t* s_row = s_src + kTM;
  int* s_cnt = s_row + kTM;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lr = lane / LC, lc = lane % LC;
  const int64_t r0 = (int64_t)blockIdx.x * kTM;
  const int col0 = blockIdx.y * TN;
  const int rows = (int)min((int64_t)kTM, n_out - r0);

  for (int i = tid; i < kTM * TN; i += 256) s_acc[i] = 0.f;
  for (int i = tid; i < rows * K; i += 256) s_nb[i] = tap_entry((int64_t)__ldg(neigh + r0 * K + i), n_in);

  for (int k = 0; k < K; ++k) {
    __syncthreads();                  // s_nb written / the previous tap is done with s_src, s_row, s_cnt
    const int32_t e = (warp < kTM / 32 && tid < rows) ? s_nb[tid * K + k] : -1;
    const int m = compact_rows<kTM / 32>(e, s_cnt, s_src, s_row);
    if (m == 0) continue;
    int np = 0;                       // passes with rows for this warp (warp-uniform)
#pragma unroll
    for (int p = 0; p < NP; ++p) np += (p * PASS + warp * LR < m);
    float acc[NP][16];
#pragma unroll
    for (int p = 0; p < NP; ++p)
#pragma unroll
      for (int c = 0; c < 16; ++c) acc[p][c] = 0.f;
    const float* wk = w + (int64_t)k * Cin * Cout;
    for (int ci0 = 0; ci0 < Cin; ci0 += kKC) {
      const int kc = min(kKC, Cin - ci0);
      __syncthreads();                // compaction visible / the previous stage's reads are done
      if (VEC) {
        for (int i = tid; i < m * (kKC / 4); i += 256) {
          const int j = i / (kKC / 4), c4 = (i % (kKC / 4)) * 4;
          if (c4 < kc) {
            const float4 v = *reinterpret_cast<const float4*>(data + (int64_t)s_src[j] * Cin + ci0 + c4);
            s_a[(c4 + 0) * (kTM + 1) + j] = v.x;
            s_a[(c4 + 1) * (kTM + 1) + j] = v.y;
            s_a[(c4 + 2) * (kTM + 1) + j] = v.z;
            s_a[(c4 + 3) * (kTM + 1) + j] = v.w;
          }
        }
        for (int i = tid; i < kc * (TN / 4); i += 256) {
          const int ci = i / (TN / 4), c = (i % (TN / 4)) * 4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (col0 + c < Cout) v = __ldg(reinterpret_cast<const float4*>(wk + (int64_t)(ci0 + ci) * Cout + col0 + c));
          *reinterpret_cast<float4*>(s_b + ci * TN + c) = v;
        }
      } else {
        for (int i = tid; i < m * kKC; i += 256) {
          const int j = i / kKC, ci = i % kKC;
          if (ci < kc) s_a[ci * (kTM + 1) + j] = data[(int64_t)s_src[j] * Cin + ci0 + ci];
        }
        for (int i = tid; i < kc * TN; i += 256) {
          const int ci = i / TN, c = i % TN;
          s_b[ci * TN + c] = (col0 + c < Cout) ? __ldg(wk + (int64_t)(ci0 + ci) * Cout + col0 + c) : 0.f;
        }
      }
      __syncthreads();
      if (np > 0) {
#pragma unroll 2
        for (int ci = 0; ci < kc; ++ci) {
          float4 b[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) b[q] = *reinterpret_cast<const float4*>(s_b + ci * TN + 4 * (q * LC + lc));
#pragma unroll
          for (int p = 0; p < NP; ++p) {
            if (p < np) {
              const float a = s_a[ci * (kTM + 1) + p * PASS + warp * LR + lr];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                acc[p][4 * q + 0] = fmaf(a, b[q].x, acc[p][4 * q + 0]);
                acc[p][4 * q + 1] = fmaf(a, b[q].y, acc[p][4 * q + 1]);
                acc[p][4 * q + 2] = fmaf(a, b[q].z, acc[p][4 * q + 2]);
                acc[p][4 * q + 3] = fmaf(a, b[q].w, acc[p][4 * q + 3]);
              }
            }
          }
        }
      }
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const int j = p * PASS + warp * LR + lr;
      if (p < np && j < m) {
        float* dst = s_acc + s_row[j] * TN;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4* d4 = reinterpret_cast<float4*>(dst + 4 * (q * LC + lc));
          float4 v = *d4;
          v.x += acc[p][4 * q + 0]; v.y += acc[p][4 * q + 1]; v.z += acc[p][4 * q + 2]; v.w += acc[p][4 * q + 3];
          *d4 = v;
        }
      }
    }
  }
  __syncthreads();
  if (VEC) {
    for (int i = tid; i < rows * (TN / 4); i += 256) {
      const int r = i / (TN / 4), c = (i % (TN / 4)) * 4;
      if (col0 + c < Cout)
        *reinterpret_cast<float4*>(out + (r0 + r) * Cout + col0 + c) = *reinterpret_cast<const float4*>(s_acc + r * TN + c);
    }
  } else {
    for (int i = tid; i < rows * TN; i += 256) {
      const int r = i / TN, c = i % TN;
      if (col0 + c < Cout) out[(r0 + r) * Cout + col0 + c] = s_acc[r * TN + c];
    }
  }
}

// ---------------------------------------------------------------------------
// Weight gradient.  Block (x, y, z): chunk x of R rows, tap y, output tile z of TI input x TO output
// channels.  The NT = TI TO / 16 threads of a row group own 4 x 4 elements each; the G = 256 / NT
// groups take the compacted rows g, g + G, ... of every kWRows sub-tile, and are folded in group order
// through shared memory.  ws[x][y][ci][co] holds the chunk's partial; k_oconv_wgrad_fold adds the
// chunks in order.
// ---------------------------------------------------------------------------
template <int TI, int TO, typename IdxT>
__global__ void __launch_bounds__(256)
k_oconv_wgrad(const float* __restrict__ data, const IdxT* __restrict__ neigh, const float* __restrict__ dout,
              int64_t n, int64_t n_in, int K, int Cin, int Cout, int64_t rows_per_chunk, float* __restrict__ ws) {
  constexpr int NT = (TI / 4) * (TO / 4), G = 256 / NT;
  static_assert(G * NT == 256 && G <= 32, "tile");
  __shared__ __align__(16) float s_buf[kWRows * (TI + TO) > G * TI * TO ? kWRows * (TI + TO) : G * TI * TO];
  __shared__ int32_t s_src[kWRows], s_row[kWRows];
  __shared__ int s_cnt[kWRows / 32];
  float* s_a = s_buf;                       // [j][TI]
  float* s_d = s_buf + kWRows * TI;         // [j][TO]
  const int tid = threadIdx.x, g = tid / NT, t = tid % NT;
  const int ti = t % (TI / 4), to = t / (TI / 4);
  const int k = blockIdx.y;
  const int n_co = (Cout + TO - 1) / TO;
  const int ci0 = (blockIdx.z / n_co) * TI, co0 = (blockIdx.z % n_co) * TO;
  const int64_t c0 = (int64_t)blockIdx.x * rows_per_chunk;
  const int64_t c1 = min(n, c0 + rows_per_chunk);
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;

  for (int64_t rb = c0; rb < c1; rb += kWRows) {
    __syncthreads();                  // the previous sub-tile's reads are done
    const int32_t e = (tid < kWRows && rb + tid < c1) ? tap_entry((int64_t)__ldg(neigh + (rb + tid) * K + k), n_in) : -1;
    const int m = compact_rows<kWRows / 32>(e, s_cnt, s_src, s_row);
    if (m == 0) continue;
    __syncthreads();
    for (int i = tid; i < m * TI; i += 256) {
      const int j = i / TI, c = i % TI;
      s_a[i] = (ci0 + c < Cin) ? __ldg(data + (int64_t)s_src[j] * Cin + ci0 + c) : 0.f;
      (void)j;
    }
    for (int i = tid; i < m * TO; i += 256) {
      const int j = i / TO, c = i % TO;
      s_d[i] = (co0 + c < Cout) ? __ldg(dout + (rb + s_row[j]) * Cout + co0 + c) : 0.f;
    }
    __syncthreads();
#pragma unroll 1
    for (int j = g; j < m; j += G) {
      const float4 a = *reinterpret_cast<const float4*>(s_a + j * TI + 4 * ti);
      const float4 d = *reinterpret_cast<const float4*>(s_d + j * TO + 4 * to);
      outer4(acc[0], a.x, d);
      outer4(acc[1], a.y, d);
      outer4(acc[2], a.z, d);
      outer4(acc[3], a.w, d);
    }
  }
  if (G > 1) {
    __syncthreads();
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) s_buf[(g * NT + t) * 16 + x * 4 + y] = acc[x][y];
    __syncthreads();
  }
  if (g == 0) {
    float* dst = ws + ((int64_t)blockIdx.x * K + k) * Cin * Cout;
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const int ci = ci0 + 4 * ti + x;
#pragma unroll
      for (int y = 0; y < 4; ++y) {
        const int co = co0 + 4 * to + y;
        float v = acc[x][y];
        if (G > 1) {
          v = s_buf[t * 16 + x * 4 + y];
#pragma unroll
          for (int q = 1; q < G; ++q) v += s_buf[(q * NT + t) * 16 + x * 4 + y];
        }
        if (ci < Cin && co < Cout) dst[(int64_t)ci * Cout + co] = v;
      }
    }
  }
}

__global__ void __launch_bounds__(256)
k_oconv_wgrad_fold(const float* __restrict__ ws, int64_t chunks, int64_t total, float* __restrict__ dw) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  float v = 0.f;
  for (int64_t p = 0; p < chunks; ++p) v += __ldg(ws + p * total + i);
  dw[i] = v;
}

// Row chunks of the weight gradient: a function of (n, K, Cin, Cout) only.
int64_t wgrad_chunks(int64_t n, int K, int Cin, int Cout) {
  int64_t c = ceil_div(n, kWMinRows);
  const int64_t cap = kWMaxWsFloats / ((int64_t)K * Cin * Cout);
  if (c > cap) c = cap;
  if (c > kWMaxChunks) c = kWMaxChunks;
  return c < 1 ? 1 : c;
}

bool aligned16(const void* p) { return ((uintptr_t)p % 16) == 0; }

template <int LC, bool VEC, typename IdxT>
int launch_fwd_lc(const float* data, const IdxT* neigh, const float* w, int64_t n_out, int64_t n_in, int K, int Cin,
                  int Cout, float* out, cudaStream_t st) {
  const size_t smem = FwdSmem<LC>::bytes;
  HFL_ENSURE_SMEM(smem, k_oconv_fwd<LC, VEC, IdxT>);
  const dim3 grid((unsigned)ceil_div(n_out, kTM), (unsigned)ceil_div(Cout, FwdSmem<LC>::TN));
  HFL_LAUNCH((k_oconv_fwd<LC, VEC, IdxT><<<grid, 256, smem, st>>>(data, neigh, w, n_out, n_in, K, Cin, Cout, out)));
  return HFL_OK;
}

template <bool VEC, typename IdxT>
int launch_fwd_vec(const float* data, const IdxT* neigh, const float* w, int64_t n_out, int64_t n_in, int K, int Cin,
                   int Cout, float* out, cudaStream_t st) {
  if (Cout <= 32) return launch_fwd_lc<2, VEC>(data, neigh, w, n_out, n_in, K, Cin, Cout, out, st);
  if (Cout <= 64) return launch_fwd_lc<4, VEC>(data, neigh, w, n_out, n_in, K, Cin, Cout, out, st);
  return launch_fwd_lc<8, VEC>(data, neigh, w, n_out, n_in, K, Cin, Cout, out, st);
}

template <typename IdxT>
int launch_fwd(const float* data, const IdxT* neigh, const float* w, int64_t n_out, int64_t n_in, int K, int Cin,
               int Cout, float* out, cudaStream_t st) {
  const bool vec = Cin % 4 == 0 && Cout % 4 == 0 && aligned16(data) && aligned16(w) && aligned16(out);
  if (vec) return launch_fwd_vec<true>(data, neigh, w, n_out, n_in, K, Cin, Cout, out, st);
  return launch_fwd_vec<false>(data, neigh, w, n_out, n_in, K, Cin, Cout, out, st);
}

template <int TI, int TO, typename IdxT>
int launch_wgrad_tile(const float* data, const IdxT* neigh, const float* dout, int64_t n, int64_t n_in, int K,
                      int Cin, int Cout, int64_t chunks, float* ws, cudaStream_t st) {
  const int64_t rows = ceil_div(n, chunks);
  const dim3 grid((unsigned)chunks, (unsigned)K, (unsigned)(ceil_div(Cin, TI) * ceil_div(Cout, TO)));
  HFL_LAUNCH((k_oconv_wgrad<TI, TO, IdxT><<<grid, 256, 0, st>>>(data, neigh, dout, n, n_in, K, Cin, Cout, rows, ws)));
  return HFL_OK;
}

template <typename IdxT>
int launch_wgrad(const float* data, const IdxT* neigh, const float* dout, int64_t n, int64_t n_in, int K, int Cin,
                 int Cout, int64_t chunks, float* ws, cudaStream_t st) {
  if (Cin <= 4)
    return Cout <= 32 ? launch_wgrad_tile<4, 32>(data, neigh, dout, n, n_in, K, Cin, Cout, chunks, ws, st)
                      : launch_wgrad_tile<4, 64>(data, neigh, dout, n, n_in, K, Cin, Cout, chunks, ws, st);
  if (Cin <= 32)
    return Cout <= 32 ? launch_wgrad_tile<32, 32>(data, neigh, dout, n, n_in, K, Cin, Cout, chunks, ws, st)
                      : launch_wgrad_tile<32, 64>(data, neigh, dout, n, n_in, K, Cin, Cout, chunks, ws, st);
  return Cout <= 32 ? launch_wgrad_tile<64, 32>(data, neigh, dout, n, n_in, K, Cin, Cout, chunks, ws, st)
                    : launch_wgrad_tile<64, 64>(data, neigh, dout, n, n_in, K, Cin, Cout, chunks, ws, st);
}

int check_shape(int64_t n_out, int64_t n_in, int32_t K, int32_t Cin, int32_t Cout) {
  HFL_CHECK_ARG(K == 8 || K == 27, "K must be 8 or 27");
  HFL_CHECK_ARG(Cin >= 1 && Cin <= kMaxC && Cout >= 1 && Cout <= kMaxC, "Cin and Cout must be in [1, 256]");
  HFL_CHECK_ARG(n_out >= 0 && n_in >= 0, "negative row count");
  HFL_CHECK_ARG(n_out < (1ll << 31) && n_in < (1ll << 31), "row indices must fit 32 bits");
  return HFL_OK;
}

}  // namespace
}  // namespace hfl

using namespace hfl;

extern "C" {

int hfl_octree_conv_train_fwd(const float* data, const void* neigh, int32_t neigh_i64, const float* w, int64_t n_out,
                              int64_t n_in, int32_t K, int32_t Cin, int32_t Cout, float* out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const int rc = check_shape(n_out, n_in, K, Cin, Cout);
  if (rc != HFL_OK) return rc;
  if (n_out == 0) return HFL_OK;
  HFL_CHECK_ARG(neigh && w && out && (data || n_in == 0), "null argument");
  if (neigh_i64) return launch_fwd(data, (const int64_t*)neigh, w, n_out, n_in, K, Cin, Cout, out, st);
  return launch_fwd(data, (const int32_t*)neigh, w, n_out, n_in, K, Cin, Cout, out, st);
}

int64_t hfl_octree_conv_train_wgrad_workspace_bytes(int64_t n, int32_t K, int32_t Cin, int32_t Cout) {
  if (n <= 0 || (K != 8 && K != 27) || Cin < 1 || Cin > kMaxC || Cout < 1 || Cout > kMaxC) return 0;
  return (int64_t)align_up((size_t)wgrad_chunks(n, K, Cin, Cout) * K * Cin * Cout * sizeof(float));
}

int hfl_octree_conv_train_wgrad(const float* data, const void* neigh, int32_t neigh_i64, const float* dout, int64_t n,
                                int64_t n_in, int32_t K, int32_t Cin, int32_t Cout, float* dw, void* ws,
                                int64_t ws_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const int rc = check_shape(n, n_in, K, Cin, Cout);
  if (rc != HFL_OK) return rc;
  HFL_CHECK_ARG(dw, "null argument");
  const int64_t total = (int64_t)K * Cin * Cout;
  if (n == 0) {                                  // no rows: the gradient is zero
    HFL_CUDA(cudaMemsetAsync(dw, 0, (size_t)total * sizeof(float), st));
    return HFL_OK;
  }
  HFL_CHECK_ARG(neigh && dout && (data || n_in == 0), "null argument");
  const int64_t need = hfl_octree_conv_train_wgrad_workspace_bytes(n, K, Cin, Cout);
  if (!ws || ws_bytes < need)
    return fail(HFL_ERR_WORKSPACE, "octree conv weight-gradient workspace too small (%s%lld bytes needed)", "",
                (long long)need);
  HFL_CHECK_ARG(aligned16(ws), "workspace must be 16-byte aligned");
  const int64_t chunks = wgrad_chunks(n, K, Cin, Cout);
  const int r = neigh_i64
      ? launch_wgrad(data, (const int64_t*)neigh, dout, n, n_in, K, Cin, Cout, chunks, (float*)ws, st)
      : launch_wgrad(data, (const int32_t*)neigh, dout, n, n_in, K, Cin, Cout, chunks, (float*)ws, st);
  if (r != HFL_OK) return r;
  HFL_LAUNCH((k_oconv_wgrad_fold<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>((const float*)ws, chunks, total, dw)));
  return HFL_OK;
}

}  // extern "C"
