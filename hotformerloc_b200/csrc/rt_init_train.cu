// Relay-token initialisation with its backward, fp32 (training side): RelayTokenInitialiser.forward
// (hotformerloc_backbone.py:345-363) and OctreeT.compute_window_stats (models/octree.py:285-344) over the
// windows of K consecutive padded rows of a pyramid level.  For window w, rows t = wK + s (s < K) of the
// int16x4 token table (x, y, z, submap; padding rows (0, 0, 0, B)):
//   valid(t) = submap(t) == submap(wK)          cnt_w = #valid rows (>= 1: the first row is valid)
//   rt[w]    = (sum over valid t of src[t]) / cnt_w,  with src[t] = 0 for the padding rows t >= n
// so an all-padding window (id B throughout, cnt = K) gives 0, as the reference's zero-padded mean does.
// ADaPE statistics (no gradient) of the node centres p = xyz 2^(1-depth) - 1, set to 0 at padding rows after
// the rescale: mean mu = sum p / max(cnt, 1), then with Bessel's correction den = max(cnt - 1, 1) and the
// guard ok = (cnt >= 2): 'var' (mode 6) mu | diag / den ok, 'cov' (mode 9) mu | upper triangle xx xy xz yy yz zz.
//   k_rtinit_fwd : CTA = window, thread = channel; rt is a fixed-order sum over s, then one division
//   k_rtinit_bwd : CTA = window, thread = channel; grad_src[t] = grad_rt[w] / cnt_w at valid rows, else 0.
//                  Each row lies in exactly one window, so the backward is a gather: no atomics.
// Results are bit-identical run to run.
#include "common.cuh"

namespace hfl {

namespace {

constexpr int kMaxC = 512;
constexpr int kMaxK = 4096;
constexpr int kMaxWindowsPerGrid = 148 * 64;   // grid-stride beyond this

__device__ __forceinline__ float warp_sum(float v) {   // the butterfly of layers.cu's inference kernel
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(kMaxC) k_rtinit_fwd(const float* __restrict__ src, const short4* __restrict__ xyzb,
                                                      int64_t n, int64_t n_win, int K, int C, int depth, int mode,
                                                      float* __restrict__ rt, float* __restrict__ stats) {
  const int c = threadIdx.x;
  const float cs = ldexpf(1.0f, 1 - depth);
  for (int64_t w = blockIdx.x; w < n_win; w += gridDim.x) {
    const int64_t t0 = w * K;
    const short id0 = xyzb[t0].w;
    float acc = 0.f;
    int cnt = 0;
    for (int s = 0; s < K; ++s) {
      const int64_t t = t0 + s;
      if (xyzb[t].w != id0) continue;                        // uniform across the CTA
      ++cnt;
      if (t < n) acc += __ldg(src + t * C + c);
    }
    rt[w * C + c] = acc / (float)cnt;
    if (mode == 0 || c >= 32) continue;
    // ---- window statistics, warp 0 ----
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (int s = c; s < K; s += 32) {
      const short4 q = xyzb[t0 + s];
      if (q.w != id0 || t0 + s >= n) continue;               // padding rows are 0 after the rescale
      sx += q.x * cs - 1.0f;
      sy += q.y * cs - 1.0f;
      sz += q.z * cs - 1.0f;
    }
    const float fc = fmaxf((float)cnt, 1.0f);
    const float mx = warp_sum(sx) / fc, my = warp_sum(sy) / fc, mz = warp_sum(sz) / fc;
    float cv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int s = c; s < K; s += 32) {
      const short4 q = xyzb[t0 + s];
      if (q.w != id0) continue;
      const bool real = t0 + s < n;
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
    if (mode == 6) { st[4] = st[6]; st[5] = st[8]; }        // 'var': the diagonal only
    if (c < mode) {
      float v = st[0];
#pragma unroll
      for (int j = 1; j < 9; ++j) v = c == j ? st[j] : v;
      stats[w * mode + c] = v;
    }
  }
}

__global__ void __launch_bounds__(kMaxC) k_rtinit_bwd(const float* __restrict__ grad_rt, const short4* __restrict__ xyzb,
                                                      int64_t n, int64_t n_win, int K, int C,
                                                      float* __restrict__ grad_src) {
  const int c = threadIdx.x;
  for (int64_t w = blockIdx.x; w < n_win; w += gridDim.x) {
    const int64_t t0 = w * K;
    if (t0 >= n) break;                                      // windows from here on hold only padding rows
    const short id0 = xyzb[t0].w;
    int cnt = 0;
    for (int s = 0; s < K; ++s) cnt += xyzb[t0 + s].w == id0;
    const float g = __ldg(grad_rt + w * C + c) / (float)cnt;
    const int64_t end = t0 + K < n ? t0 + K : n;
    for (int64_t t = t0; t < end; ++t) grad_src[t * C + c] = xyzb[t].w == id0 ? g : 0.f;
  }
}

int check_common(const void* xyzb, int64_t n, int64_t n_win, int32_t K, int32_t C) {
  HFL_CHECK_ARG(C >= 32 && C <= kMaxC && C % 32 == 0, "C must be a multiple of 32 in [32, 512]");
  HFL_CHECK_ARG(K >= 1 && K <= kMaxK, "K must be in [1, 4096]");
  HFL_CHECK_ARG(n >= 0 && n_win >= 0, "n and n_win must be non-negative");
  HFL_CHECK_ARG(n_win <= ((int64_t)1 << 40) / K, "n_win too large");
  HFL_CHECK_ARG(n <= n_win * K, "n must be at most n_win * K (every row in a window)");
  HFL_CHECK_ARG(n_win == 0 || xyzb, "null xyzb");
  HFL_CHECK_ARG(((uintptr_t)xyzb & 7) == 0, "xyzb must be 8-byte aligned");
  return HFL_OK;
}

}  // namespace
}  // namespace hfl

using namespace hfl;

extern "C" {

int hfl_rt_init_train_fwd(const float* src, const int16_t* xyzb, int64_t n, int64_t n_win, int32_t K, int32_t C,
                          int32_t depth, int32_t mode, float* rt_out, float* stats_out, void* stream_) {
  const int rc = check_common(xyzb, n, n_win, K, C);
  if (rc != HFL_OK) return rc;
  HFL_CHECK_ARG(mode == 0 || mode == 3 || mode == 6 || mode == 9, "mode must be 0, 3, 6 or 9");
  HFL_CHECK_ARG(depth >= 0 && depth <= 15, "depth must be in [0, 15]");
  if (n_win == 0) return HFL_OK;
  HFL_CHECK_ARG(rt_out && (n == 0 || src), "null argument");
  HFL_CHECK_ARG(mode == 0 || stats_out, "stats_out is required when mode != 0");
  const int grid = (int)(n_win < kMaxWindowsPerGrid ? n_win : kMaxWindowsPerGrid);
  HFL_LAUNCH((k_rtinit_fwd<<<grid, C, 0, (cudaStream_t)stream_>>>(src, (const short4*)xyzb, n, n_win, K, C, depth,
                                                                   mode, rt_out, stats_out)));
  return HFL_OK;
}

int hfl_rt_init_train_bwd(const float* grad_rt, const int16_t* xyzb, int64_t n, int64_t n_win, int32_t K, int32_t C,
                          float* grad_src, void* stream_) {
  const int rc = check_common(xyzb, n, n_win, K, C);
  if (rc != HFL_OK) return rc;
  if (n == 0) return HFL_OK;                                 // n > 0 implies n_win > 0
  HFL_CHECK_ARG(grad_rt && grad_src, "null argument");
  const int64_t used = (n + K - 1) / K;                      // windows that hold a row of src
  const int grid = (int)(used < kMaxWindowsPerGrid ? used : kMaxWindowsPerGrid);
  HFL_LAUNCH((k_rtinit_bwd<<<grid, C, 0, (cudaStream_t)stream_>>>(grad_rt, (const short4*)xyzb, n, n_win, K, C,
                                                                   grad_src)));
  return HFL_OK;
}

}  // extern "C"
