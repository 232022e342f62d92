// Batched octree construction on the device (SURVEY.md section 8 rows a1-a4, a6).
//
// One pass over the whole batch replaces the reference's per-submap
// ocnn Octree.build_octree + merge_octrees + construct_all_neigh:
//   quantise -> Morton -> LSD radix sort of (submap<<3D | morton) with the point
//   index as payload (stable => points of a leaf stay in input order) ->
//   unique -> per depth: parent keys / children / all-node index -> neighbours.
// All integer results are bit-exact against the reference (tests/test_octree_gpu.py).
// Everything is HBM-bound integer work: coalesced streaming kernels, grids sized
// from row capacities, the actual row counts are read from device memory so the
// build never synchronises with the host.
#include "common.cuh"

namespace hfl {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

// ---------------------------------------------------------------------------
// Morton helpers (x most significant of each bit triple)
// ---------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t spread3(uint64_t x) {
  x &= 0x1fffff;
  x = (x | x << 32) & 0x1f00000000ffffull;
  x = (x | x << 16) & 0x1f0000ff0000ffull;
  x = (x | x << 8) & 0x100f00f00f00f00full;
  x = (x | x << 4) & 0x10c30c30c30c30c3ull;
  x = (x | x << 2) & 0x1249249249249249ull;
  return x;
}
__host__ __device__ __forceinline__ uint32_t compact3(uint64_t x) {
  x &= 0x1249249249249249ull;
  x = (x ^ (x >> 2)) & 0x10c30c30c30c30c3ull;
  x = (x ^ (x >> 4)) & 0x100f00f00f00f00full;
  x = (x ^ (x >> 8)) & 0x1f0000ff0000ffull;
  x = (x ^ (x >> 16)) & 0x1f00000000ffffull;
  x = (x ^ (x >> 32)) & 0x1fffff;
  return (uint32_t)x;
}
__host__ __device__ __forceinline__ uint64_t morton3(uint32_t x, uint32_t y, uint32_t z) {
  return (spread3(x) << 2) | (spread3(y) << 1) | spread3(z);
}

// ---------------------------------------------------------------------------
// 1. quantise + key
// ---------------------------------------------------------------------------
__global__ void k_quantize(const float* __restrict__ pts, const int32_t* __restrict__ off,
                           int64_t n, int B, int D, uint64_t* __restrict__ keys,
                           uint32_t* __restrict__ vals) {
  const float scale = (float)(1 << (D - 1));
  const uint32_t cmask = (1u << D) - 1;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = B;  // largest b with off[b] <= i
    while (hi - lo > 1) {
      int mid = (lo + hi) >> 1;
      if ((int64_t)__ldg(off + mid) <= i) lo = mid; else hi = mid;
    }
    // (p + 1) * 2^(D-1) in fp32, no FMA contraction, then truncate toward zero
    float fx = __fmul_rn(__fadd_rn(pts[3 * i + 0], 1.0f), scale);
    float fy = __fmul_rn(__fadd_rn(pts[3 * i + 1], 1.0f), scale);
    float fz = __fmul_rn(__fadd_rn(pts[3 * i + 2], 1.0f), scale);
    uint32_t x = (uint32_t)__float2int_rz(fx) & cmask;
    uint32_t y = (uint32_t)__float2int_rz(fy) & cmask;
    uint32_t z = (uint32_t)__float2int_rz(fz) & cmask;
    keys[i] = ((uint64_t)lo << (3 * D)) | morton3(x, y, z);
    vals[i] = (uint32_t)i;
  }
}

// ---------------------------------------------------------------------------
// 2. LSD radix sort, 8-bit digits, stable.  Tile = 4096 keys per block.
// ---------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_ITEMS = 16;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;

__global__ void __launch_bounds__(RS_THREADS)
k_rs_hist(const uint64_t* __restrict__ keys, int64_t n, int shift, uint32_t* __restrict__ hist,
          int nblk) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  int64_t base = (int64_t)blockIdx.x * RS_TILE;
#pragma unroll
  for (int it = 0; it < RS_ITEMS; ++it) {
    int64_t i = base + it * RS_THREADS + threadIdx.x;
    if (i < n) atomicAdd(&h[(keys[i] >> shift) & 255], 1u);
  }
  __syncthreads();
  hist[(size_t)threadIdx.x * nblk + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of `m` uint32 in place, one block of 1024 threads
__global__ void __launch_bounds__(1024) k_scan_u32(uint32_t* __restrict__ a, int64_t m) {
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t base = 0; base < m; base += 1024 * 4) {
    int64_t i0 = base + (int64_t)threadIdx.x * 4;
    uint32_t v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = (i0 + j < m) ? a[i0 + j] : 0u;
    uint32_t t = v[0] + v[1] + v[2] + v[3];
    uint32_t inc = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += u;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      uint32_t w = wsum[lane];
      uint32_t winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t u = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += u;
      }
      wsum[lane] = winc - w;  // exclusive
    }
    __syncthreads();
    uint32_t carry = carry_s;
    uint32_t ex = carry + wsum[warp] + inc - t;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (i0 + j < m) a[i0 + j] = ex;
      ex += v[j];
    }
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = carry + wsum[warp] + inc;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(RS_THREADS)
k_rs_scatter(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ vals, int64_t n,
             int shift, const uint32_t* __restrict__ offs, int nblk,
             uint64_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out) {
  __shared__ uint32_t base[256];
  __shared__ uint32_t cnt[RS_THREADS / 32][256];
  __shared__ uint32_t pre[RS_THREADS / 32][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  base[threadIdx.x] = offs[(size_t)threadIdx.x * nblk + blockIdx.x];
#pragma unroll
  for (int w = 0; w < RS_THREADS / 32; ++w) cnt[w][threadIdx.x] = 0;
  __syncthreads();
  int64_t tile = (int64_t)blockIdx.x * RS_TILE;
  for (int it = 0; it < RS_ITEMS; ++it) {
    int64_t i = tile + it * RS_THREADS + threadIdx.x;
    bool valid = i < n;
    uint64_t k = valid ? keys[i] : 0;
    uint32_t v = valid ? vals[i] : 0;
    uint32_t digit = valid ? (uint32_t)((k >> shift) & 255) : 256u;
    unsigned peers = __match_any_sync(0xffffffffu, digit);
    int rank = __popc(peers & ((1u << lane) - 1));
    if (valid && rank == 0) cnt[warp][digit] = __popc(peers);
    __syncthreads();
    {
      uint32_t run = base[threadIdx.x];
#pragma unroll
      for (int w = 0; w < RS_THREADS / 32; ++w) {
        uint32_t c = cnt[w][threadIdx.x];
        pre[w][threadIdx.x] = run;
        cnt[w][threadIdx.x] = 0;
        run += c;
      }
      base[threadIdx.x] = run;
    }
    __syncthreads();
    if (valid) {
      uint32_t pos = pre[warp][digit] + rank;
      keys_out[pos] = k;
      vals_out[pos] = v;
    }
  }
}

// ---------------------------------------------------------------------------
// 3. segmented "unique" over a sorted key array whose length lives on the device
//    flag[i] = (i == 0) || (key[i] >> SH) != (key[i-1] >> SH);  id = incl_scan(flag) - 1
// ---------------------------------------------------------------------------
constexpr int SC_THREADS = 512;
constexpr int SC_ITEMS = 8;
constexpr int SC_TILE = SC_THREADS * SC_ITEMS;

__device__ __forceinline__ uint32_t block_excl_scan_512(uint32_t t, uint32_t* wsum, uint32_t& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = t;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = (lane < SC_THREADS / 32) ? wsum[lane] : 0;
    uint32_t winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t u = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += u;
    }
    if (lane < SC_THREADS / 32) wsum[lane] = winc - w;
    if (lane == 31) wsum[32] = winc;
  }
  __syncthreads();
  total = wsum[32];
  return wsum[warp] + inc - t;
}

// pass 1: number of flags per tile
__global__ void __launch_bounds__(SC_THREADS)
k_uniq_count(const uint64_t* __restrict__ key, const int32_t* __restrict__ n_ptr, int64_t n_imm,
             int sh, uint32_t* __restrict__ bsum) {
  __shared__ uint32_t wsum[33];
  const int64_t n = n_ptr ? (int64_t)*n_ptr : n_imm;
  int64_t i0 = (int64_t)blockIdx.x * SC_TILE + (int64_t)threadIdx.x * SC_ITEMS;
  uint32_t t = 0;
  if (i0 < n) {
    uint64_t prev = (i0 > 0) ? (key[i0 - 1] >> sh) : ~0ull;
#pragma unroll
    for (int j = 0; j < SC_ITEMS; ++j) {
      if (i0 + j < n) {
        uint64_t c = key[i0 + j] >> sh;
        t += (i0 + j == 0) || (c != prev);
        prev = c;
      }
    }
  }
  uint32_t total;
  block_excl_scan_512(t, wsum, total);
  if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

// pass 2: exclusive scan of the tile sums (<= a few thousand) + publish the total
__global__ void __launch_bounds__(1024)
k_uniq_scan(uint32_t* __restrict__ bsum, const int32_t* __restrict__ n_ptr, int64_t n_imm,
            int32_t* __restrict__ total_out) {
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t carry_s;
  const int64_t n = n_ptr ? (int64_t)*n_ptr : n_imm;
  const int64_t m = (n + SC_TILE - 1) / SC_TILE;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t base = 0; base < m; base += 1024) {
    int64_t i = base + threadIdx.x;
    uint32_t t = (i < m) ? bsum[i] : 0u;
    uint32_t inc = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += u;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      uint32_t w = wsum[lane];
      uint32_t winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t u = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += u;
      }
      wsum[lane] = winc - w;
    }
    __syncthreads();
    uint32_t carry = carry_s;
    if (i < m) bsum[i] = carry + wsum[warp] + inc - t;
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = carry + wsum[warp] + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total_out = (int32_t)carry_s;
}

// pass 3 (leaf level): sorted point keys -> leaf nodes
__global__ void __launch_bounds__(SC_THREADS)
k_uniq_leaf(const uint64_t* __restrict__ key, const uint32_t* __restrict__ sorted_idx, int64_t n,
            const uint32_t* __restrict__ bsum, uint64_t* __restrict__ nkey,
            int32_t* __restrict__ leaf_start, int32_t* __restrict__ point_leaf) {
  __shared__ uint32_t wsum[33];
  int64_t i0 = (int64_t)blockIdx.x * SC_TILE + (int64_t)threadIdx.x * SC_ITEMS;
  uint32_t f[SC_ITEMS];
  uint64_t kk[SC_ITEMS];
  uint32_t t = 0;
  if (i0 < n) {
    uint64_t prev = (i0 > 0) ? key[i0 - 1] : ~0ull;
#pragma unroll
    for (int j = 0; j < SC_ITEMS; ++j) {
      f[j] = 0;
      if (i0 + j < n) {
        kk[j] = key[i0 + j];
        f[j] = (i0 + j == 0) || (kk[j] != prev);
        prev = kk[j];
        t += f[j];
      }
    }
  }
  uint32_t total;
  uint32_t ex = block_excl_scan_512(t, wsum, total) + bsum[blockIdx.x];
  if (i0 < n) {
#pragma unroll
    for (int j = 0; j < SC_ITEMS; ++j) {
      if (i0 + j < n) {
        ex += f[j];              // inclusive count => id = ex - 1
        uint32_t id = ex - 1;
        if (f[j]) {
          nkey[id] = kk[j];
          leaf_start[id] = (int32_t)(i0 + j);
        }
        if (point_leaf) point_leaf[sorted_idx[i0 + j]] = (int32_t)id;
      }
    }
  }
}

// pass 3 (inner level d -> d-1): node keys -> parent keys, nidx[d], children[d]
__global__ void __launch_bounds__(SC_THREADS)
k_uniq_parent(const uint64_t* __restrict__ key, const int32_t* __restrict__ n_ptr,
              const uint32_t* __restrict__ bsum, uint64_t* __restrict__ pkey,
              int32_t* __restrict__ nidx, int32_t* __restrict__ children) {
  __shared__ uint32_t wsum[33];
  const int64_t n = *n_ptr;
  int64_t i0 = (int64_t)blockIdx.x * SC_TILE + (int64_t)threadIdx.x * SC_ITEMS;
  uint32_t f[SC_ITEMS];
  uint64_t kk[SC_ITEMS];
  uint32_t t = 0;
  if (i0 < n) {
    uint64_t prev = (i0 > 0) ? (key[i0 - 1] >> 3) : ~0ull;
#pragma unroll
    for (int j = 0; j < SC_ITEMS; ++j) {
      f[j] = 0;
      if (i0 + j < n) {
        kk[j] = key[i0 + j];
        f[j] = (i0 + j == 0) || ((kk[j] >> 3) != prev);
        prev = kk[j] >> 3;
        t += f[j];
      }
    }
  }
  uint32_t total;
  uint32_t ex = block_excl_scan_512(t, wsum, total) + bsum[blockIdx.x];
  if (i0 < n) {
#pragma unroll
    for (int j = 0; j < SC_ITEMS; ++j) {
      if (i0 + j < n) {
        ex += f[j];
        uint32_t pid = ex - 1;
        if (f[j]) pkey[pid] = kk[j] >> 3;
        int32_t a = (int32_t)((pid << 3) | (uint32_t)(kk[j] & 7));
        nidx[i0 + j] = a;
        children[a] = (int32_t)(i0 + j);
      }
    }
  }
}

__global__ void k_fill_children(int32_t* __restrict__ c, const int32_t* __restrict__ n_ptr,
                                int64_t mul) {
  const int64_t n = (int64_t)(*n_ptr) * mul;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    c[i] = -1;
}

// full-depth level: children[F][nkey] = i ; nidx = nkey
__global__ void k_full_level(const uint64_t* __restrict__ key, const int32_t* __restrict__ n_ptr,
                             int32_t* __restrict__ nidx, int32_t* __restrict__ children) {
  const int64_t n = *n_ptr;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    int32_t a = (int32_t)key[i];
    nidx[i] = a;
    children[a] = (int32_t)i;
  }
}

// depths below full_depth: complete grids
__global__ void k_grid_level(int64_t n, uint64_t* __restrict__ key, int32_t* __restrict__ nidx,
                             int32_t* __restrict__ children) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    key[i] = (uint64_t)i;
    nidx[i] = (int32_t)i;
    children[i] = (int32_t)i;
  }
}

// leaf means: sequential fp32 sum in input order (stable sort), then / count
__global__ void k_leaf_mean(const float* __restrict__ pts, const uint32_t* __restrict__ sorted_idx,
                            const int32_t* __restrict__ leaf_start,
                            const int32_t* __restrict__ n_leaf_ptr, int64_t n_points, int D,
                            float* __restrict__ out) {
  const int64_t nl = *n_leaf_ptr;
  const float scale = (float)(1 << (D - 1));
  for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < nl;
       l += (int64_t)gridDim.x * blockDim.x) {
    int64_t s = leaf_start[l];
    int64_t e = (l + 1 < nl) ? (int64_t)leaf_start[l + 1] : n_points;
    float ax = 0.f, ay = 0.f, az = 0.f;
    for (int64_t j = s; j < e; ++j) {
      int64_t p = sorted_idx[j];
      ax = __fadd_rn(ax, __fmul_rn(__fadd_rn(pts[3 * p + 0], 1.0f), scale));
      ay = __fadd_rn(ay, __fmul_rn(__fadd_rn(pts[3 * p + 1], 1.0f), scale));
      az = __fadd_rn(az, __fmul_rn(__fadd_rn(pts[3 * p + 2], 1.0f), scale));
    }
    float c = (float)(e - s);
    out[3 * l + 0] = __fdiv_rn(ax, c);
    out[3 * l + 1] = __fdiv_rn(ay, c);
    out[3 * l + 2] = __fdiv_rn(az, c);
  }
}

// per (depth, submap) node counts by binary search on the sorted keys
struct CountArgs {
  const uint64_t* nkey[HFL_MAX_DEPTH + 1];
};
__global__ void k_counts(CountArgs a, int D, int F, int B, int32_t* __restrict__ counts) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (D + 1) * B) return;
  int d = t / B, b = t % B;
  int32_t* row = counts + (size_t)d * (B + 2);
  if (d < F) {
    row[b] = 1 << (3 * d);
    if (b == 0) { row[B] = B << (3 * d); row[B + 1] = B << (3 * d); }
    return;
  }
  const int64_t n = row[B];
  const uint64_t* k = a.nkey[d];
  uint64_t lo_key = (uint64_t)b << (3 * d), hi_key = (uint64_t)(b + 1) << (3 * d);
  int64_t lo = 0, hi = n;
  while (lo < hi) { int64_t m = (lo + hi) >> 1; if (k[m] < lo_key) lo = m + 1; else hi = m; }
  int64_t s = lo;
  hi = n;
  while (lo < hi) { int64_t m = (lo + hi) >> 1; if (k[m] < hi_key) lo = m + 1; else hi = m; }
  row[b] = (int32_t)(lo - s);
  if (b == 0) row[B + 1] = (d == F) ? (B << (3 * d)) : 8 * counts[(size_t)(d - 1) * (B + 2) + B];
}

// ---------------------------------------------------------------------------
// import of an ocnn octree (all-node keys / children per depth -> the tables above)
// ---------------------------------------------------------------------------
// pass 1: non-empty nodes (children >= 0) per tile; pass 2 is k_uniq_scan
__global__ void __launch_bounds__(SC_THREADS)
k_import_count(const int32_t* __restrict__ ch, int64_t n, uint32_t* __restrict__ bsum) {
  __shared__ uint32_t wsum[33];
  const int64_t i0 = (int64_t)blockIdx.x * SC_TILE + (int64_t)threadIdx.x * SC_ITEMS;
  uint32_t t = 0;
#pragma unroll
  for (int j = 0; j < SC_ITEMS; ++j)
    if (i0 + j < n) t += ch[i0 + j] >= 0;
  uint32_t total;
  block_excl_scan_512(t, wsum, total);
  if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

// pass 3, depth d: all-node i with children value c.  The compact key of node i follows from its
// position alone (d <= F: i; d > F: the parent's compact key << 3 | i & 7), so nkey never holds an
// input value; the input key is only compared with it (invariant K).  Entries are scattered by
// their in-order rank r, never by c: c must equal r (invariant C) and a rank >= nn is dropped, so
// every written index is in range whatever the input.  children_out keeps c only where it is that
// rank, otherwise -1, and ranks the input leaves unfilled get node 0: the neighbour kernels index
// through these tables before the host has seen the status.
__global__ void __launch_bounds__(SC_THREADS)
k_import_level(const int32_t* __restrict__ ch, const int64_t* __restrict__ keys, int64_t n,
               int64_t nn, int d, int F, const uint64_t* __restrict__ pkey,
               const uint32_t* __restrict__ bsum, const int32_t* __restrict__ total_ptr,
               uint64_t* __restrict__ nkey, int32_t* __restrict__ nidx,
               int32_t* __restrict__ children_out, int32_t* __restrict__ nn_out,
               int32_t* __restrict__ status) {
  __shared__ uint32_t wsum[33];
  const int64_t i0 = (int64_t)blockIdx.x * SC_TILE + (int64_t)threadIdx.x * SC_ITEMS;
  int32_t c[SC_ITEMS];
  uint32_t t = 0;
#pragma unroll
  for (int j = 0; j < SC_ITEMS; ++j) {
    c[j] = (i0 + j < n) ? ch[i0 + j] : -1;
    t += c[j] >= 0;
  }
  uint32_t tot;
  uint32_t r = block_excl_scan_512(t, wsum, tot) + bsum[blockIdx.x];
  const uint64_t mmask = (1ull << (3 * d)) - 1;
  bool bad_c = false, bad_k = false;
#pragma unroll
  for (int j = 0; j < SC_ITEMS; ++j) {
    const int64_t i = i0 + j;
    if (i < n) {
      const uint64_t ck = d <= F ? (uint64_t)i : (pkey[i >> 3] << 3) | (uint64_t)(i & 7);
      bad_k |= (uint64_t)keys[i] != (((ck >> (3 * d)) << 48) | (ck & mmask));
      int32_t out = -1;
      if (c[j] >= 0) {
        if ((int64_t)r < nn) {
          nidx[r] = (int32_t)i;
          nkey[r] = ck;
          if ((uint32_t)c[j] == r) out = c[j];
        }
        bad_c |= out < 0;
        ++r;
      } else {
        bad_c |= c[j] != -1;
      }
      children_out[i] = out;
    }
  }
  const int64_t total = *total_ptr;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    *nn_out = (int32_t)nn;
    bad_c |= total != nn;
  }
  for (int64_t q = total + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nn;
       q += (int64_t)gridDim.x * blockDim.x) {
    nidx[q] = 0;
    nkey[q] = 0;
  }
  if (bad_c || bad_k) {
    atomicOr(status, (bad_c ? HFL_IMPORT_BAD_CHILDREN : 0) | (bad_k ? HFL_IMPORT_BAD_KEYS : 0));
    atomicOr(status + 1, 1 << d);
  }
}

// ---------------------------------------------------------------------------
// neighbours
// ---------------------------------------------------------------------------
__device__ __forceinline__ void lut_pc(int c, int k, int& lp, int& lc) {
  // child position c in {0..7} (x-major bits), offset k in 0..26 (x-major)
  int sx = ((c >> 2) & 1) + 2 + (k / 9) - 1;
  int sy = ((c >> 1) & 1) + 2 + ((k / 3) % 3) - 1;
  int sz = (c & 1) + 2 + (k % 3) - 1;
  lp = (sx >> 1) * 9 + (sy >> 1) * 3 + (sz >> 1);
  lc = (sx & 1) * 4 + (sy & 1) * 2 + (sz & 1);
}

__global__ void k_neigh_grid(int d, int B, int32_t* __restrict__ grid) {
  const int64_t cells = 1ll << (3 * d);
  const int64_t total = cells * B * 27;
  const int lim = 1 << d;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int k = (int)(t % 27);
    int64_t node = t / 27;
    int64_t b = node / cells, cell = node % cells;
    int x = (int)compact3((uint64_t)cell >> 2) + (k / 9) - 1;
    int y = (int)compact3((uint64_t)cell >> 1) + ((k / 3) % 3) - 1;
    int z = (int)compact3((uint64_t)cell) + (k % 3) - 1;
    bool ok = x >= 0 && y >= 0 && z >= 0 && x < lim && y < lim && z < lim;
    grid[t] = ok ? (int32_t)(b * cells + (int64_t)morton3(x, y, z)) : -1;
  }
}

__global__ void k_neigh_from_grid(const int32_t* __restrict__ grid, const int32_t* __restrict__ nidx,
                                  const int32_t* __restrict__ children,
                                  const int32_t* __restrict__ n_ptr, int32_t* __restrict__ na,
                                  int32_t* __restrict__ ne) {
  const int64_t total = (int64_t)(*n_ptr) * 27;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = t / 27;
    int k = (int)(t % 27);
    int32_t r = grid[(int64_t)nidx[i] * 27 + k];
    na[t] = r;
    if (ne) ne[t] = r < 0 ? -1 : children[r];
  }
}

// rows = non-empty nodes (nidx != null) or all nodes (nidx == null)
__global__ void k_neigh_child(const int32_t* __restrict__ na_parent,
                              const int32_t* __restrict__ children_parent,
                              const int32_t* __restrict__ children,
                              const int32_t* __restrict__ nidx, const int32_t* __restrict__ n_ptr,
                              int64_t mul, int32_t* __restrict__ na, int32_t* __restrict__ ne) {
  const int64_t total = (int64_t)(*n_ptr) * mul * 27;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = t / 27;
    int k = (int)(t % 27);
    int64_t a = nidx ? (int64_t)nidx[i] : i;
    int64_t p = a >> 3;
    int c = (int)(a & 7);
    int lp, lc;
    lut_pc(c, k, lp, lc);
    int32_t q = na_parent[p * 27 + lp];
    int32_t pn = q < 0 ? -1 : children_parent[q];
    int32_t r = pn < 0 ? -1 : pn * 8 + lc;
    if (na) na[t] = r;
    if (ne) ne[t] = r < 0 ? -1 : children[r];
  }
}

__global__ void k_full_keys(const uint64_t* __restrict__ pkey, int d, int F, int B,
                            const int32_t* __restrict__ n_parent_ptr, int64_t* __restrict__ out) {
  if (d <= F) {
    const int64_t cells = 1ll << (3 * d), total = cells * B;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x)
      out[i] = ((i / cells) << 48) | (i % cells);
    return;
  }
  const int64_t total = (int64_t)(*n_parent_ptr) * 8;
  const uint64_t mmask = (1ull << (3 * (d - 1))) - 1;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    uint64_t pk = pkey[i >> 3];
    uint64_t b = pk >> (3 * (d - 1)), m = pk & mmask;
    out[i] = (int64_t)((b << 48) | (m << 3) | (uint64_t)(i & 7));
  }
}

__global__ void k_tokens(const uint64_t* __restrict__ nkey, const int32_t* __restrict__ n_ptr, int d,
                         int B, int64_t n_pad, short4* __restrict__ out) {
  const int64_t n = *n_ptr;
  const uint64_t mmask = (1ull << (3 * d)) - 1;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_pad;
       i += (int64_t)gridDim.x * blockDim.x) {
    short4 v;
    if (i < n) {
      uint64_t k = nkey[i];
      uint64_t m = k & mmask;
      v.x = (short)compact3(m >> 2);
      v.y = (short)compact3(m >> 1);
      v.z = (short)compact3(m);
      v.w = (short)(k >> (3 * d));
    } else {
      v.x = v.y = v.z = 0;
      v.w = (short)B;
    }
    out[i] = v;
  }
}

// ---------------------------------------------------------------------------
// workspace layout
// ---------------------------------------------------------------------------
struct BuildWs {
  uint64_t *keysA, *keysB;
  uint32_t *valsA, *valsB;
  int32_t* leaf_start;
  uint32_t* hist;
  uint32_t* bsum;
  size_t bytes;
};

static BuildWs carve(char* base, int64_t n, int B, int D) {
  (void)B; (void)D;
  BuildWs w;
  size_t o = 0;
  auto take = [&](size_t bytes) { char* p = base ? base + o : nullptr; o += align_up(bytes); return p; };
  int64_t nblk = ceil_div(n, RS_TILE);
  w.keysA = (uint64_t*)take(8 * n);
  w.keysB = (uint64_t*)take(8 * n);
  w.valsA = (uint32_t*)take(4 * n);
  w.valsB = (uint32_t*)take(4 * n);
  w.leaf_start = (int32_t*)take(4 * (n + 1));
  w.hist = (uint32_t*)take(4 * 256 * nblk);
  w.bsum = (uint32_t*)take(4 * (ceil_div(n, SC_TILE) + 1));
  w.bytes = o;
  return w;
}

}  // namespace hfl

using namespace hfl;

extern "C" {

const char* hfl_last_error_string(void) { return g_err; }
int hfl_version(void) { return 100; }
int64_t hfl_launch_count(void) { return (int64_t)g_launches.load(); }

size_t hfl_octree_build_workspace_bytes(int64_t n_points, int32_t batch, int32_t depth) {
  if (n_points < 1) n_points = 1;
  return carve(nullptr, n_points, batch, depth).bytes;
}

int hfl_octree_build(const float* points, const int32_t* pt_offsets, const hfl_octree* o,
                     void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(o && points && pt_offsets && workspace, "null argument");
  const int D = o->depth, F = o->full_depth, B = o->batch;
  const int64_t n = o->n_points;
  HFL_CHECK_ARG(D >= 1 && D <= HFL_MAX_DEPTH && F >= 1 && F < D, "need 1 <= full_depth < depth <= 15");
  HFL_CHECK_ARG(B >= 1 && B < 32768, "batch must be in [1, 32767]");
  HFL_CHECK_ARG(n >= B && n < (1ll << 31), "need at least one point per submap and < 2^31 points");
  int bbits = 0;
  while ((1 << bbits) < B) ++bbits;
  const int nbits = 3 * D + bbits;
  HFL_CHECK_ARG(nbits <= 63, "key too wide");
  for (int d = 0; d <= D; ++d) {
    const int64_t full = (3 * d < 40) ? ((int64_t)B << (3 * d)) : (int64_t)1 << 62;
    const int64_t need = (d <= F) ? full : (full < n ? full : n);
    HFL_CHECK_ARG(o->cap[d] >= need, "node capacity too small");
    HFL_CHECK_ARG(o->nkey[d] && o->children[d] && o->nidx[d], "null node array");
  }
  HFL_CHECK_ARG(o->leaf_points && o->counts, "null output");
  BuildWs w = carve((char*)workspace, n, B, D);
  if (w.bytes > workspace_bytes) return fail(HFL_ERR_WORKSPACE, "workspace too small%s (need %lld)", "", (long long)w.bytes);
  const int stride = B + 2;
  int32_t* counts = o->counts;

  // 1. keys
  HFL_LAUNCH((k_quantize<<<grid_for(n, 256), 256, 0, st>>>(points, pt_offsets, n, B, D, w.keysA, w.valsA)));
  // 2. radix sort
  const int nblk = (int)ceil_div(n, RS_TILE);
  uint64_t *kin = w.keysA, *kout = w.keysB;
  uint32_t *vin = w.valsA, *vout = w.valsB;
  for (int shift = 0; shift < nbits; shift += 8) {
    HFL_LAUNCH((k_rs_hist<<<nblk, RS_THREADS, 0, st>>>(kin, n, shift, w.hist, nblk)));
    HFL_LAUNCH((k_scan_u32<<<1, 1024, 0, st>>>(w.hist, (int64_t)256 * nblk)));
    HFL_LAUNCH((k_rs_scatter<<<nblk, RS_THREADS, 0, st>>>(kin, vin, n, shift, w.hist, nblk, kout, vout)));
    uint64_t* tk = kin; kin = kout; kout = tk;
    uint32_t* tv = vin; vin = vout; vout = tv;
  }
  // 3. leaves
  const int nsc = (int)ceil_div(n, SC_TILE);
  int32_t* nD = counts + (size_t)D * stride + B;
  HFL_LAUNCH((k_uniq_count<<<nsc, SC_THREADS, 0, st>>>(kin, nullptr, n, 0, w.bsum)));
  HFL_LAUNCH((k_uniq_scan<<<1, 1024, 0, st>>>(w.bsum, nullptr, n, nD)));
  HFL_LAUNCH((k_uniq_leaf<<<nsc, SC_THREADS, 0, st>>>(kin, vin, n, w.bsum, o->nkey[D], w.leaf_start, o->point_leaf)));
  HFL_LAUNCH((k_leaf_mean<<<grid_for(o->cap[D], 128), 128, 0, st>>>(points, vin, w.leaf_start, nD, n, D, o->leaf_points)));
  // 4. inner levels D..F+1
  for (int d = D; d > F; --d) {
    int32_t* nd = counts + (size_t)d * stride + B;
    int32_t* np = counts + (size_t)(d - 1) * stride + B;
    const int g = (int)ceil_div(o->cap[d], SC_TILE);
    HFL_LAUNCH((k_uniq_count<<<g, SC_THREADS, 0, st>>>(o->nkey[d], nd, 0, 3, w.bsum)));
    HFL_LAUNCH((k_uniq_scan<<<1, 1024, 0, st>>>(w.bsum, nd, 0, np)));
    HFL_LAUNCH((k_fill_children<<<grid_for(8 * o->cap[d - 1], 256), 256, 0, st>>>(o->children[d], np, 8)));
    HFL_LAUNCH((k_uniq_parent<<<g, SC_THREADS, 0, st>>>(o->nkey[d], nd, w.bsum, o->nkey[d - 1], o->nidx[d], o->children[d])));
  }
  // 5. full-depth level and the complete grids below it
  {
    const int64_t cells = (int64_t)B << (3 * F);
    HFL_CUDA(cudaMemsetAsync(o->children[F], 0xFF, cells * sizeof(int32_t), st));
    HFL_LAUNCH((k_full_level<<<grid_for(cells, 256), 256, 0, st>>>(o->nkey[F], counts + (size_t)F * stride + B, o->nidx[F], o->children[F])));
    for (int d = 0; d < F; ++d) {
      const int64_t c = (int64_t)B << (3 * d);
      HFL_LAUNCH((k_grid_level<<<grid_for(c, 256), 256, 0, st>>>(c, o->nkey[d], o->nidx[d], o->children[d])));
    }
  }
  // 6. counts table
  {
    CountArgs ca;
    for (int d = 0; d <= HFL_MAX_DEPTH; ++d) ca.nkey[d] = d <= D ? o->nkey[d] : nullptr;
    const int t = (D + 1) * B;
    HFL_LAUNCH((k_counts<<<(int)ceil_div(t, 256), 256, 0, st>>>(ca, D, F, B, counts)));
  }
  return HFL_OK;
}

size_t hfl_octree_import_workspace_bytes(const hfl_ocnn_octree* in) {
  int64_t n = 1;
  if (in && in->depth >= 0 && in->depth <= HFL_MAX_DEPTH)
    for (int d = 0; d <= in->depth; ++d) n = in->nnum[d] > n ? in->nnum[d] : n;
  return align_up(4 * (ceil_div(n, SC_TILE) + 1)) + align_up(4);
}

int hfl_octree_import_check(const hfl_ocnn_octree* in) {
  HFL_CHECK_ARG(in, "null argument");
  const int D = in->depth, F = in->full_depth, B = in->batch;
  HFL_CHECK_ARG(D >= 1 && D <= HFL_MAX_DEPTH && F >= 1 && F < D, "need 1 <= full_depth < depth <= 15");
  HFL_CHECK_ARG(B >= 1 && B < 32768, "batch must be in [1, 32767]");
  for (int d = 0; d <= D; ++d) {
    const int64_t nn = in->nnum[d], ne = in->nnum_nempty[d];
    HFL_CHECK_ARG(nn < (1ll << 31) && ne >= 0 && ne <= nn, "need 0 <= nnum_nempty[d] <= nnum[d] < 2^31");
    if (d <= F) HFL_CHECK_ARG(nn == ((int64_t)B << (3 * d)), "need nnum[d] == batch * 8^d for d <= full_depth");
    if (d < F) HFL_CHECK_ARG(ne == nn, "need nnum_nempty[d] == nnum[d] for d < full_depth");
    if (d > F) HFL_CHECK_ARG(nn == 8 * in->nnum_nempty[d - 1], "need nnum[d] == 8 * nnum_nempty[d-1] for d > full_depth");
  }
  return HFL_OK;
}

int hfl_octree_import(const hfl_ocnn_octree* in, const hfl_octree* o, int32_t* status,
                      void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(in && o && status && workspace, "null argument");
  const int rc = hfl_octree_import_check(in);
  if (rc != HFL_OK) return rc;
  const int D = in->depth, F = in->full_depth, B = in->batch;
  HFL_CHECK_ARG(o->depth == D && o->full_depth == F && o->batch == B, "output octree shape differs");
  for (int d = 0; d <= D; ++d) {
    HFL_CHECK_ARG(in->nnum[d] == 0 || (in->keys[d] && in->children[d]), "null input array");
    HFL_CHECK_ARG(o->cap[d] >= in->nnum_nempty[d], "node capacity too small");
    HFL_CHECK_ARG(o->nkey[d] && o->children[d] && o->nidx[d], "null node array");
  }
  HFL_CHECK_ARG(in->nnum_nempty[D] == 0 || in->points, "null points");
  HFL_CHECK_ARG(o->leaf_points && o->counts, "null output");
  const size_t ws = hfl_octree_import_workspace_bytes(in);
  if (ws > workspace_bytes) return fail(HFL_ERR_WORKSPACE, "workspace too small%s (need %lld)", "", (long long)ws);
  uint32_t* bsum = (uint32_t*)workspace;
  int32_t* total = (int32_t*)((char*)workspace + ws - align_up(4));
  const int stride = B + 2;

  HFL_CUDA(cudaMemsetAsync(status, 0, 2 * sizeof(int32_t), st));
  for (int d = 0; d <= D; ++d) {        // top down: depth d reads the compact keys of depth d-1
    const int64_t n = in->nnum[d];
    const int g = (int)(ceil_div(n, SC_TILE) > 0 ? ceil_div(n, SC_TILE) : 1);
    HFL_LAUNCH((k_import_count<<<g, SC_THREADS, 0, st>>>(in->children[d], n, bsum)));
    HFL_LAUNCH((k_uniq_scan<<<1, 1024, 0, st>>>(bsum, nullptr, n, total)));
    HFL_LAUNCH((k_import_level<<<g, SC_THREADS, 0, st>>>(
        in->children[d], in->keys[d], n, in->nnum_nempty[d], d, F, d > F ? o->nkey[d - 1] : nullptr,
        bsum, total, o->nkey[d], o->nidx[d], o->children[d], o->counts + (size_t)d * stride + B, status)));
  }
  HFL_CUDA(cudaMemcpyAsync(o->leaf_points, in->points, 12 * in->nnum_nempty[D], cudaMemcpyDeviceToDevice, st));
  CountArgs ca;
  for (int d = 0; d <= HFL_MAX_DEPTH; ++d) ca.nkey[d] = d <= D ? o->nkey[d] : nullptr;
  HFL_LAUNCH((k_counts<<<(int)ceil_div((D + 1) * B, 256), 256, 0, st>>>(ca, D, F, B, o->counts)));
  return HFL_OK;
}

int hfl_octree_neigh(const hfl_octree* o, int32_t d, const int32_t* na_parent, int32_t* grid,
                     int32_t* na_out, int32_t* ne_out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(o && na_out, "null argument");
  HFL_CHECK_ARG(d >= 1 && d <= o->depth, "depth out of range");
  const int B = o->batch, stride = B + 2;
  const int32_t* nd = o->counts + (size_t)d * stride + B;
  if (d <= o->full_depth) {
    HFL_CHECK_ARG(grid, "grid table required at or below full depth");
    const int64_t total = ((int64_t)B << (3 * d)) * 27;
    HFL_LAUNCH((k_neigh_grid<<<grid_for(total, 256), 256, 0, st>>>(d, B, grid)));
    HFL_LAUNCH((k_neigh_from_grid<<<grid_for(o->cap[d] * 27, 256), 256, 0, st>>>(grid, o->nidx[d], o->children[d], nd, na_out, ne_out)));
  } else {
    HFL_CHECK_ARG(na_parent, "parent table required above full depth");
    HFL_LAUNCH((k_neigh_child<<<grid_for(o->cap[d] * 27, 256), 256, 0, st>>>(na_parent, o->children[d - 1], o->children[d], o->nidx[d], nd, 1, na_out, ne_out)));
  }
  return HFL_OK;
}

int hfl_octree_neigh_full(const hfl_octree* o, int32_t d, const int32_t* na_parent,
                          int32_t* full_out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(o && full_out, "null argument");
  HFL_CHECK_ARG(d >= 1 && d <= o->depth, "depth out of range");
  const int B = o->batch, stride = B + 2;
  if (d <= o->full_depth) {
    const int64_t total = ((int64_t)B << (3 * d)) * 27;
    HFL_LAUNCH((k_neigh_grid<<<grid_for(total, 256), 256, 0, st>>>(d, B, full_out)));
  } else {
    HFL_CHECK_ARG(na_parent, "parent table required above full depth");
    const int32_t* np = o->counts + (size_t)(d - 1) * stride + B;
    HFL_LAUNCH((k_neigh_child<<<grid_for(o->cap[d - 1] * 8 * 27, 256), 256, 0, st>>>(na_parent, o->children[d - 1], nullptr, nullptr, np, 8, full_out, nullptr)));
  }
  return HFL_OK;
}

int hfl_octree_full_keys(const hfl_octree* o, int32_t d, int64_t* keys_out, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(o && keys_out, "null argument");
  HFL_CHECK_ARG(d >= 0 && d <= o->depth, "depth out of range");
  const int B = o->batch, stride = B + 2, F = o->full_depth;
  const int64_t cap = d <= F ? ((int64_t)B << (3 * d)) : 8 * o->cap[d - 1];
  const uint64_t* pk = d > F ? o->nkey[d - 1] : nullptr;
  const int32_t* np = d > F ? o->counts + (size_t)(d - 1) * stride + B : nullptr;
  HFL_LAUNCH((k_full_keys<<<grid_for(cap, 256), 256, 0, st>>>(pk, d, F, B, np, keys_out)));
  return HFL_OK;
}

int hfl_octree_tokens(const hfl_octree* o, int32_t d, int64_t n_pad, int16_t* xyzb_out,
                      void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  HFL_CHECK_ARG(o && xyzb_out, "null argument");
  HFL_CHECK_ARG(d >= 0 && d <= o->depth && n_pad >= 0, "bad depth / padding");
  const int B = o->batch, stride = B + 2;
  HFL_LAUNCH((k_tokens<<<grid_for(n_pad, 256), 256, 0, st>>>(o->nkey[d], o->counts + (size_t)d * stride + B, d, B, n_pad, (short4*)xyzb_out)));
  return HFL_OK;
}

}  // extern "C"
