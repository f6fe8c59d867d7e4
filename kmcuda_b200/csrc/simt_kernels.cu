// simt_kernels.cu -- exact (reference-arithmetic) CUDA-core kernels.
//
// Everything here consumes the caller's row-major [N][D] layout directly (the reference first
// transposes to feature-major through a managed staging copy, transpose.cu:83-117; that component
// does not exist here).  Sample tiles are staged through padded shared memory so that the
// sequential Kahan chains of exact.cuh read conflict-free, and centroid features are warp-uniform
// broadcast loads.
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>

#include "exact.cuh"
#include "kernels.h"

namespace kmb {

static inline unsigned cdiv(size_t a, size_t b) { return static_cast<unsigned>((a + b - 1) / b); }

// row lists up to this length are handled one CTA per row (exact_rows_few_kernel)
constexpr uint32_t kFewRows = 8192;

// ------------------------------------------------------------------------------------------------
// ||c||^2 table (reference computes it per CTA per chunk, kmeans.cu:322-323)
// ------------------------------------------------------------------------------------------------
// One warp per 32 centroids: 32 features x 32 rows at a time are staged through shared memory with coalesced loads
// (lane = feature), then lane r walks row r in feature order -- the reference's sequential Kahan sum (round 2's first
// version let every thread walk its own row in global memory: a chain of dependent 4-byte loads, 21 us per pass, which
// is a visible part of the 0.58 ms step of a 1 M-row shard).
template <int METRIC>
__global__ void __launch_bounds__(32)
csqr_kernel(const float* __restrict__ C, uint32_t K, int D, float* __restrict__ csq) {
  __shared__ float tile[32 * 33];
  const int lane = threadIdx.x;
  const uint32_t c0 = blockIdx.x * 32u;
  if (METRIC == 1) {
    if (c0 + lane < K) csq[c0 + lane] = 1.f;
    return;
  }
  Kahan k;
  for (int f0 = 0; f0 < D; f0 += 32) {
    const int fl = min(32, D - f0);
    float v[32];
#pragma unroll
    for (int r = 0; r < 32; r++) {   // all 32 row segments in flight at once
      const uint32_t c = min(c0 + r, K - 1);
      v[r] = lane < fl ? C[static_cast<size_t>(c) * D + f0 + lane] : 0.f;
    }
#pragma unroll
    for (int r = 0; r < 32; r++) tile[r * 33 + lane] = v[r];
    __syncwarp();
    for (int f = 0; f < fl; f++) {
      const float v = tile[lane * 33 + f];
      k.mac(v, v);
    }
    __syncwarp();
  }
  if (c0 + lane < K) csq[c0 + lane] = k.sum;
}

cudaError_t launch_csqr(int metric, const float* C, uint32_t K, int D, float* csq, cudaStream_t st) {
  if (metric == 1) csqr_kernel<1><<<cdiv(K, 32), 32, 0, st>>>(C, K, D, csq);
  else csqr_kernel<0><<<cdiv(K, 32), 32, 0, st>>>(C, K, D, csq);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Exact pass over ALL K centroids.  MODE 0: Lloyd argmin (reference kmeans.cu:293-364).
// MODE 1: Yinyang bounds refresh (reference kmeans.cu:431-485).
// A CTA owns RB sample rows (staged once in padded shared memory) and TPR threads per row; thread
// part t of a row scans the centroid quads {t, t+TPR, ...} in ascending order with 4 independent Kahan
// chains in flight, so a row's K*D dependent operations are spread over TPR threads and the SM holds
// up to 32 warps.  Parts are merged towards the lowest index on equal scores == the reference's
// ascending strict-'<' scan.  Warps are (same part, 32 consecutive rows): centroid loads are
// warp-uniform broadcasts, sample reads are conflict-free.
// ------------------------------------------------------------------------------------------------
template <int METRIC, int MODE>
__global__ void __launch_bounds__(1024)
exact_pass_kernel(const float* __restrict__ X, const float* __restrict__ C,
                  const float* __restrict__ csq, uint32_t n, int D, uint32_t K,
                  const uint32_t* __restrict__ rows, const uint32_t* __restrict__ d_nrows,
                  uint32_t* __restrict__ result, int use_smem, int RB,
                  // MODE 1 only
                  uint32_t G, const uint32_t* __restrict__ assign,
                  const uint32_t* __restrict__ groups, float* __restrict__ bounds) {
  extern __shared__ float sX[];
  const int TPR = blockDim.x / RB;
  const int r = threadIdx.x % RB, t = threadIdx.x / RB;
  float* s_best = sX + (use_smem ? static_cast<size_t>(RB + 1) * D : 0);   // [TPR][RB]
  uint32_t* s_arg = reinterpret_cast<uint32_t*>(s_best + static_cast<size_t>(TPR) * RB);
  const uint32_t nrows = d_nrows ? *d_nrows : n;
  if (MODE == 0 && d_nrows && nrows <= kFewRows) return;  // exact_rows_few_kernel handles short lists
  for (uint32_t tile0 = blockIdx.x * RB; tile0 < nrows; tile0 += gridDim.x * RB) {
    const uint32_t slot = tile0 + r;
    const bool active = slot < nrows;
    const uint32_t row = active ? (rows ? rows[slot] : slot) : 0;
    const float* xs;
    int xstride;
    __syncthreads();
    if (use_smem) {
      const int cnt = min(static_cast<uint32_t>(RB), nrows - tile0);
      for (int e = threadIdx.x; e < cnt * D; e += blockDim.x) {
        int s = e / D, f = e - s * D;
        uint32_t rr = rows ? rows[tile0 + s] : tile0 + s;
        sX[f * (RB + 1) + s] = X[static_cast<size_t>(rr) * D + f];
      }
      xs = sX + r;
      xstride = RB + 1;
    } else {
      xs = X + static_cast<size_t>(row) * D;
      xstride = 1;
    }
    uint32_t mine = 0;
    if (MODE == 1 && active) {
      mine = assign[row];
      if (t == 0)
        for (uint32_t g = 0; g <= G; g++) bounds[static_cast<size_t>(row) * (G + 1) + g] = FLT_MAX;
    }
    __syncthreads();
    float best = FLT_MAX;
    uint32_t arg = UINT32_MAX;
    const bool insane = MODE == 0 && active && (xs[0] != xs[0]);  // first feature NaN (kmeans.cu:312,355)
    if (active && !insane) {
      for (uint32_t c0 = 4u * t; c0 < K; c0 += 4u * TPR) {
        const float* cp[4];
#pragma unroll
        for (int j = 0; j < 4; j++) cp[j] = C + static_cast<size_t>(min(c0 + j, K - 1)) * D;
        Kahan k[4];
        for (int f = 0; f < D; f++) {
          float x = xs[f * xstride];
#pragma unroll
          for (int j = 0; j < 4; j++) {
            float cv = __ldg(cp[j] + f);
            if (MODE == 1 && METRIC == 0) k[j].sqdiff(x, cv);
            else k[j].mac(x, cv);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
          uint32_t c = c0 + j;
          if (c >= K) break;
          if (MODE == 0) {
            float score = lloyd_score<METRIC>(k[j].sum, csq[c]);
            if (score < best) {
              best = score;
              arg = c;
            }
          } else {
            uint32_t g = groups[c];
            if (g >= G) continue;  // NaN centroid (kmeans.cu:464-468)
            float dist = finalize_distance<METRIC>(k[j].sum);
            if (c != mine) {
              // distances are >= +0: their bit patterns order like unsigned integers; NaN never lowers a bound
              atomicMin(reinterpret_cast<uint32_t*>(bounds + static_cast<size_t>(row) * (G + 1) + 1 + g),
                        __float_as_uint(dist));
            } else {
              bounds[static_cast<size_t>(row) * (G + 1)] = dist;
            }
          }
        }
      }
    }
    if (MODE == 0) {
      s_best[t * RB + r] = best;
      s_arg[t * RB + r] = arg;
      __syncthreads();
      if (t == 0 && active) {
        if (insane) {
          result[row] = K;
        } else {
          for (int tt = 1; tt < TPR; tt++) {
            float b2 = s_best[tt * RB + r];
            uint32_t a2 = s_arg[tt * RB + r];
            if (a2 != UINT32_MAX && (arg == UINT32_MAX || b2 < best || (b2 == best && a2 < arg))) {
              best = b2;
              arg = a2;
            }
          }
          result[row] = (arg == UINT32_MAX) ? kUntouched : arg;
        }
      }
    }
  }
}

// Row-list variant for FEW rows (the tensor-core filter's overflow list is normally a handful of rows
// out of millions): one CTA per row, the K centroids spread over the 512 threads, so a single row does
// not serialise K*D dependent operations on one thread.  Each thread scans its centroids in ascending
// order with strict '<'; the block reduction breaks equal scores towards the lowest index, which is
// exactly the reference's ascending strict-'<' scan (kmeans.cu:343-346).

template <int METRIC>
__global__ void __launch_bounds__(512)
exact_rows_few_kernel(const float* __restrict__ X, const float* __restrict__ C,
                      const float* __restrict__ csq, int D, uint32_t K,
                      const uint32_t* __restrict__ rows, const uint32_t* __restrict__ d_nrows,
                      uint32_t* __restrict__ result) {
  extern __shared__ float sx[];
  __shared__ float s_best[512];
  __shared__ uint32_t s_arg[512];
  const uint32_t nrows = *d_nrows;
  if (nrows > kFewRows) return;  // the tiled kernel takes over
  for (uint32_t e = blockIdx.x; e < nrows; e += gridDim.x) {
    const uint32_t row = rows[e];
    __syncthreads();
    for (int f = threadIdx.x; f < D; f += 512) sx[f] = X[static_cast<size_t>(row) * D + f];
    __syncthreads();
    if (sx[0] != sx[0]) {
      if (threadIdx.x == 0) result[row] = K;
      continue;
    }
    float best = FLT_MAX;
    uint32_t arg = UINT32_MAX;
    for (uint32_t c = threadIdx.x; c < K; c += 512) {
      const float* cp = C + static_cast<size_t>(c) * D;
      Kahan k;
      for (int f = 0; f < D; f++) k.mac(sx[f], __ldg(cp + f));
      float score = lloyd_score<METRIC>(k.sum, csq[c]);
      if (score < best) {
        best = score;
        arg = c;
      }
    }
    s_best[threadIdx.x] = best;
    s_arg[threadIdx.x] = arg;
    __syncthreads();
    for (int o = 256; o > 0; o >>= 1) {
      if (threadIdx.x < o) {
        float b2 = s_best[threadIdx.x + o];
        uint32_t a2 = s_arg[threadIdx.x + o];
        if (a2 != UINT32_MAX && (s_arg[threadIdx.x] == UINT32_MAX || b2 < s_best[threadIdx.x] ||
                                 (b2 == s_best[threadIdx.x] && a2 < s_arg[threadIdx.x]))) {
          s_best[threadIdx.x] = b2;
          s_arg[threadIdx.x] = a2;
        }
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) result[row] = (s_arg[0] == UINT32_MAX) ? kUntouched : s_arg[0];
  }
}

struct ExactCfg {
  int rb, tpr, use_smem;
  size_t smem;
};
static ExactCfg exact_cfg(int D) {
  const size_t limit = 200 * 1024;
  for (int rb : {128, 64, 32}) {
    int tpr = 1024 / rb > 8 ? 8 : 1024 / rb;
    size_t need = static_cast<size_t>(rb + 1) * D * sizeof(float) + static_cast<size_t>(tpr) * rb * 8;
    if (need <= limit) return {rb, tpr, 1, need};
  }
  return {128, 8, 0, static_cast<size_t>(8) * 128 * 8};
}

template <int METRIC, int MODE>
static cudaError_t launch_exact_pass(const float* X, const float* C, const float* csq, uint32_t n,
                                     int D, uint32_t K, const uint32_t* rows,
                                     const uint32_t* d_nrows, uint32_t* result, uint32_t G,
                                     const uint32_t* assign, const uint32_t* groups, float* bounds,
                                     cudaStream_t st) {
  ExactCfg cfg = exact_cfg(D);
  auto kern = exact_pass_kernel<METRIC, MODE>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(cfg.smem));
  if (e != cudaSuccess) return e;
  unsigned grid = d_nrows ? 148 * 2 : cdiv(n, cfg.rb);
  if (grid == 0) return cudaSuccess;
  kern<<<grid, cfg.rb * cfg.tpr, cfg.smem, st>>>(X, C, csq, n, D, K, rows, d_nrows, result, cfg.use_smem, cfg.rb, G,
                                                 assign, groups, bounds);
  return cudaGetLastError();
}

cudaError_t launch_assign_exact(int metric, const float* X, const float* C, const float* csq,
                                uint32_t n, int D, uint32_t K, const uint32_t* rows,
                                const uint32_t* d_nrows, uint32_t* result, cudaStream_t st) {
  if (d_nrows) {  // list mode: short lists go to the one-CTA-per-row kernel (decided on the device)
    const size_t smem = sizeof(float) * D;
    if (metric == 1) exact_rows_few_kernel<1><<<148 * 4, 512, smem, st>>>(X, C, csq, D, K, rows, d_nrows, result);
    else exact_rows_few_kernel<0><<<148 * 4, 512, smem, st>>>(X, C, csq, D, K, rows, d_nrows, result);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  if (metric == 1)
    return launch_exact_pass<1, 0>(X, C, csq, n, D, K, rows, d_nrows, result, 0, nullptr, nullptr,
                                   nullptr, st);
  return launch_exact_pass<0, 0>(X, C, csq, n, D, K, rows, d_nrows, result, 0, nullptr, nullptr,
                                 nullptr, st);
}

cudaError_t launch_yy_init(int metric, const float* X, const float* C, uint32_t n, int D, uint32_t K,
                           uint32_t G, const uint32_t* assign, const uint32_t* groups, float* bounds,
                           cudaStream_t st) {
  if (metric == 1)
    return launch_exact_pass<1, 1>(X, C, nullptr, n, D, K, nullptr, nullptr, nullptr, G, assign,
                                   groups, bounds, st);
  return launch_exact_pass<0, 1>(X, C, nullptr, n, D, K, nullptr, nullptr, nullptr, G, assign, groups,
                                 bounds, st);
}

cudaError_t launch_yy_init_rows(int metric, const float* X, const float* C, uint32_t n, int D, uint32_t K,
                                uint32_t G, const uint32_t* assign, const uint32_t* groups, float* bounds,
                                const uint32_t* rows, const uint32_t* d_nrows, cudaStream_t st) {
  if (metric == 1)
    return launch_exact_pass<1, 1>(X, C, nullptr, n, D, K, rows, d_nrows, nullptr, G, assign, groups, bounds, st);
  return launch_exact_pass<0, 1>(X, C, nullptr, n, D, K, rows, d_nrows, nullptr, G, assign, groups, bounds, st);
}

// ------------------------------------------------------------------------------------------------
// prev/assign bookkeeping + reassignment counter (reference kmeans.cu:358-363)
// ------------------------------------------------------------------------------------------------
__global__ void finalize_assign_kernel(uint32_t n, const uint32_t* __restrict__ result,
                                       uint32_t* __restrict__ assign, uint32_t* __restrict__ prev,
                                       uint32_t* __restrict__ d_changed) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  int changed = 0;
  if (i < n) {
    uint32_t r = result[i];
    if (r != kUntouched) {
      uint32_t a = assign[i];
      prev[i] = a;
      if (a != r) {
        assign[i] = r;
        changed = 1;
      }
    }
  }
  unsigned mask = __ballot_sync(0xffffffffu, changed);
  if ((threadIdx.x & 31) == 0 && mask) atomicAdd(d_changed, __popc(mask));
}

cudaError_t launch_finalize_assign(uint32_t n, const uint32_t* result, uint32_t* assign,
                                   uint32_t* prev, uint32_t* d_changed, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  finalize_assign_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, result, assign, prev, d_changed);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Centroid update.  The reference updates incrementally with one thread per centroid scanning all
// N assignments (kmeans.cu:366-429); here: stable radix sort by cluster, per-cluster compensated
// sums in sample-index order (deterministic), all-reduce across shards by the caller, normalise.
// ------------------------------------------------------------------------------------------------
__global__ void iota_kernel(uint32_t* p, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}

// first position of the sorted keys[0..n) whose key is >= c, by one warp: 32 probes per step (a 33-ary search, 4 steps +
// a final window at n = 8M; one thread per cluster doing a binary search was a chain of 23 dependent DRAM reads, 27 us)
__device__ __forceinline__ uint32_t warp_lower_bound(const uint32_t* __restrict__ keys, uint32_t n, uint32_t c, int lane) {
  uint32_t lo = 0, hi = n;     // every position < lo has key < c; position hi has key >= c (or hi == n)
  while (hi - lo > 32) {
    const uint64_t s = hi - lo;
    const uint32_t q = lo + static_cast<uint32_t>((static_cast<uint64_t>(lane + 1) * s) / 33);   // lo < q < hi, increasing in lane
    const unsigned m = __ballot_sync(0xffffffffu, keys[q] >= c);
    const int t = m ? __ffs(m) - 1 : 32;
    const uint32_t q_prev = __shfl_sync(0xffffffffu, q, t > 0 ? t - 1 : 0);
    const uint32_t q_t = __shfl_sync(0xffffffffu, q, t < 32 ? t : 31);
    if (t < 32) hi = q_t;
    if (t > 0) lo = q_prev + 1;
  }
  const uint32_t p = lo + lane;
  const unsigned m = __ballot_sync(0xffffffffu, p < hi && keys[p] >= c);
  return m ? lo + (__ffs(m) - 1) : hi;
}

__global__ void segment_offsets_kernel(const uint32_t* __restrict__ keys, uint32_t n, uint32_t K,
                                       uint32_t* __restrict__ offsets, uint32_t* __restrict__ counts) {
  const uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // one warp per cluster (and one for the end marker K)
  const int lane = threadIdx.x & 31;
  if (c > K) return;
  const uint32_t lo = warp_lower_bound(keys, n, c, lane);
  if (lane == 0) offsets[c] = lo;
  if (c < K) {
    const uint32_t lo2 = warp_lower_bound(keys, n, c + 1, lane);
    if (lane == 0) counts[c] = lo2 - lo;
  }
}

// (the only way this kernel is launched: its grid is one WARP per cluster plus one for the end marker)
static void launch_segment_offsets(const uint32_t* keys, uint32_t n, uint32_t K, uint32_t* offsets, uint32_t* counts,
                                   cudaStream_t st) {
  segment_offsets_kernel<<<cdiv((static_cast<size_t>(K) + 1) * 32, 128), 128, 0, st>>>(keys, n, K, offsets, counts);
}

constexpr int kUpdateUnroll = 8;

// Member sums, balanced: CTA b owns the sorted positions [b * kSumChunk, (b + 1) * kSumChunk) whatever clusters they
// belong to, and writes one partial row per (chunk, cluster) run it meets, into slot b + c (unique: along the sorted
// array b and c never decrease and one of them grows from run to run).  The previous layout -- a fixed number of CTAs
// per cluster -- made the pass as slow as the largest cluster (4.9 ms instead of 2.1 ms at 8M x 256 @ 1024 when the
// centroids are random rows and the cell sizes differ by an order of magnitude).  Within a run the additions are
// compensated and in sample order, kUpdateUnroll member rows in flight per thread (with 4 the gather ran at
// ~4.7 TB/s, short of the bytes in flight the HBM latency asks for).  The sample rows are read once, so they are loaded
// with ld.global.cs (evict-first).
// (VEC = 4: D % 4 == 0 and 16-byte aligned rows -- a thread owns four adjacent features and reads them with one
// 16-byte load, so a CTA is D / 4 threads and every thread keeps 8 x 16 bytes in flight: the gather is latency-bound,
// 2.26 ms at 8M x 256 with 4-byte loads and 8 rows in flight, 1.89 ms with 16 rows in flight)
// (the minimum-blocks bound is there for the register budget: without it ptxas aims at 32 registers = full occupancy
// and sinks the row loads between the additions, one or two in flight instead of kUpdateUnroll)
template <int VEC>
__global__ void __launch_bounds__(256, VEC == 4 ? 3 : 5)
cluster_sums_kernel(const float* __restrict__ X, int D, const uint32_t* __restrict__ keys,
                    const uint32_t* __restrict__ idx, const uint32_t* __restrict__ offsets, uint32_t K,
                    float* __restrict__ partial) {
  const uint32_t b = blockIdx.x;
  const uint32_t total = offsets[K];                     // positions past it carry the "unassigned" key
  uint32_t lo = b * kSumChunk;
  const uint32_t hi = min(total, lo + kSumChunk);
  const int nf = D / VEC;
  while (lo < hi) {
    const uint32_t c = keys[lo];
    const uint32_t e = min(hi, offsets[c + 1]);
    for (int f = threadIdx.x; f < nf; f += blockDim.x) {
      float sum[VEC], comp[VEC];
#pragma unroll
      for (int q = 0; q < VEC; q++) sum[q] = comp[q] = 0.f;
      uint32_t j = lo;
      uint32_t id[kUpdateUnroll];   // member indices of the NEXT group: their loads overlap this group's row reads
#pragma unroll
      for (int u = 0; u < kUpdateUnroll; u++) id[u] = idx[min(j + u, e - 1)];
      for (; j + kUpdateUnroll <= e; j += kUpdateUnroll) {
        float v[kUpdateUnroll][VEC];
#pragma unroll
        for (int u = 0; u < kUpdateUnroll; u++) {
          const float* src = X + static_cast<size_t>(id[u]) * D + f * VEC;
          if (VEC == 4) {
            const float4 t4 = __ldcs(reinterpret_cast<const float4*>(src));
            v[u][0] = t4.x; v[u][VEC > 1 ? 1 : 0] = t4.y; v[u][VEC > 2 ? 2 : 0] = t4.z; v[u][VEC > 3 ? 3 : 0] = t4.w;
          } else {
            v[u][0] = __ldcs(src);
          }
        }
#pragma unroll
        for (int u = 0; u < kUpdateUnroll; u++) id[u] = idx[min(j + kUpdateUnroll + u, e - 1)];
#pragma unroll
        for (int u = 0; u < kUpdateUnroll; u++)
#pragma unroll
          for (int q = 0; q < VEC; q++) {
            const float y = v[u][q] - comp[q], t = sum[q] + y;
            comp[q] = (t - sum[q]) - y;
            sum[q] = t;
          }
      }
      for (; j < e; j++) {
        const float* src = X + static_cast<size_t>(idx[j]) * D + f * VEC;
#pragma unroll
        for (int q = 0; q < VEC; q++) {
          const float y = __ldcs(src + q) - comp[q], t = sum[q] + y;
          comp[q] = (t - sum[q]) - y;
          sum[q] = t;
        }
      }
#pragma unroll
      for (int q = 0; q < VEC; q++) partial[(static_cast<size_t>(b) + c) * D + f * VEC + q] = sum[q];
    }
    lo = e;
  }
}

// sums[c] = compensated sum of the cluster's runs in chunk order
__global__ void combine_partials_kernel(const float* __restrict__ partial, const uint32_t* __restrict__ offsets,
                                        uint32_t K, int D, float* __restrict__ sums) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<size_t>(K) * D) return;
  const uint32_t c = i / D;
  const int f = i - static_cast<size_t>(c) * D;
  const uint32_t beg = offsets[c], end = offsets[c + 1];
  float sum = 0.f, comp = 0.f;
  if (end > beg) {
    const uint32_t b0 = beg / kSumChunk, b1 = (end - 1) / kSumChunk;
    for (uint32_t b = b0; b <= b1; b++) {
      const float v = partial[(static_cast<size_t>(b) + c) * D + f];
      const float y = v - comp, t = sum + y;
      comp = (t - sum) - y;
      sum = t;
    }
  }
  sums[i] = sum;
}

size_t update_partial_rows(uint32_t n, uint32_t K) { return static_cast<size_t>(cdiv(n, kSumChunk)) + K; }

size_t update_cub_bytes(uint32_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n, 0, 32);
  return bytes;
}

cudaError_t launch_partial_sums(const float* X, uint32_t n, int D, uint32_t K, const uint32_t* assign,
                                UpdateWorkspace& ws, float* sums, uint32_t* counts, cudaStream_t st) {
  if (n == 0) {
    cudaMemsetAsync(sums, 0, sizeof(float) * static_cast<size_t>(K) * D, st);
    cudaMemsetAsync(counts, 0, sizeof(uint32_t) * K, st);
    return cudaGetLastError();
  }
  if (ws.iota_n < n) {   // the identity permutation is an input the sort never modifies: written once per workspace
    iota_kernel<<<cdiv(n, 256), 256, 0, st>>>(ws.vals_in, n);
    ws.iota_n = n;
  }
  int bits = 1;
  while ((1ull << bits) <= K) bits++;  // keys are in [0, K] (K = "insane")
  size_t bytes = ws.cub_tmp_bytes;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(ws.cub_tmp, bytes, assign, ws.keys_out, ws.vals_in,
                                                  ws.vals_out, (int)n, 0, bits, st);
  if (e != cudaSuccess) return e;
  launch_segment_offsets(ws.keys_out, n, K, ws.offsets, counts, st);
  if (D % 4 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0) {
    const int threads = std::min(256, (D / 4 + 31) / 32 * 32);
    cluster_sums_kernel<4><<<cdiv(n, kSumChunk), threads, 0, st>>>(X, D, ws.keys_out, ws.vals_out, ws.offsets, K, ws.partial);
  } else {
    cluster_sums_kernel<1><<<cdiv(n, kSumChunk), 256, 0, st>>>(X, D, ws.keys_out, ws.vals_out, ws.offsets, K, ws.partial);
  }
  combine_partials_kernel<<<cdiv(static_cast<size_t>(K) * D, 256), 256, 0, st>>>(ws.partial, ws.offsets, K, D, sums);
  return cudaGetLastError();
}

cudaError_t launch_knn_inverse(const uint32_t* assign, uint32_t n, uint32_t K, uint32_t* iota,
                               uint32_t* keys_out, uint32_t* inv, uint32_t* off, uint32_t* counts,
                               UpdateWorkspace& ws, cudaStream_t st) {
  iota_kernel<<<cdiv(n, 256), 256, 0, st>>>(iota, n);
  int bits = 1;
  while ((1ull << bits) <= K) bits++;
  size_t bytes = ws.cub_tmp_bytes;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(ws.cub_tmp, bytes, assign, keys_out, iota, inv, (int)n, 0,
                                                  bits, st);
  if (e != cudaSuccess) return e;
  launch_segment_offsets(keys_out, n, K, off, counts, st);
  return cudaGetLastError();
}

// reference kmeans_adjust (kmeans.cu:366-429) + METRIC::normalize (metric_abstraction.h:138-144 L2: multiply by
// __frcp_rn(count); :255-272 cosine).  The reference updates incrementally: centroid * old count, plus the samples
// that joined, minus the samples that left, then normalise.  For L2 that is the mean of the current members (what
// the segmented sums give directly).  For the cosine metric the stored centroid is the UNIT vector, so
// "centroid * old count" is not the old member sum and the recurrence is its own algorithm:
//     raw_new = count_old * c_old + (S_cur - S_prev),   c_new = raw_new / ||raw_new||
// with S_* the member sums of the current / previous assignment (prev_sums caches S_prev between iterations).
template <int METRIC>
__global__ void normalize_kernel(const float* __restrict__ sums, const uint32_t* __restrict__ counts,
                                 uint32_t K, int D, float* __restrict__ C,
                                 uint32_t* __restrict__ ccounts, float* __restrict__ prev_sums) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= K) return;
  const float* s = sums + static_cast<size_t>(c) * D;
  float* o = C + static_cast<size_t>(c) * D;
  uint32_t cnt = counts[c];
  if (METRIC == 1) {
    float* ps = prev_sums + static_cast<size_t>(c) * D;
    const float old_cnt = static_cast<float>(ccounts[c]);
    Kahan k;
    for (int f = 0; f < D; f++) {
      const float cur = s[f];
      const float raw = o[f] * old_cnt + (cur - ps[f]);
      ps[f] = cur;
      o[f] = raw;
      k.mac(raw, raw);
    }
    const float scale = __frcp_rn(__fsqrt_rn(k.sum));
    for (int f = 0; f < D; f++) o[f] = o[f] * scale;
  } else {
    const float scale = __frcp_rn(static_cast<float>(cnt));
    for (int f = 0; f < D; f++) o[f] = s[f] * scale;
  }
  ccounts[c] = cnt;
}

// ------------------------------------------------------------------------------------------------
// Reference-ORDER centroid update (strict parity mode, KMCUDA_B200_STRICT_UPDATE=1; single GPU).
// The reference's kmeans_adjust (kmeans.cu:366-429) is a running sum: centroid * old count, then every sample that
// joined / left the cluster is added / subtracted in SAMPLE ORDER, feature by feature, with ONE compensation term
// that is carried across features and samples, then the normalisation.  Its result depends on that order in the
// last ulps, which is what makes whole runs of two implementations drift apart on structureless data.  This path
// reproduces the order: the (cluster, sample, sign) events of the pass are sorted by cluster (stable: sample order
// survives) and one thread per centroid replays its events.  The default update (sorted compensated sums, parallel
// over clusters, features and splits) is ~1e-7 relative away from it and much faster; this one is for bit-identical
// trajectories (tests, bisecting) and costs O(changed samples per cluster x D) sequential steps per thread.
// ------------------------------------------------------------------------------------------------
__global__ void strict_events_kernel(uint32_t n, uint32_t K, const uint32_t* __restrict__ prev,
                                     const uint32_t* __restrict__ cur, uint32_t* __restrict__ keys,
                                     uint32_t* __restrict__ vals) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t p = prev[i], c = cur[i];
  const bool moved = p != c;
  keys[2 * i] = (moved && p < K) ? p : K;           // key K = "no event" (sorted to the end, never replayed)
  vals[2 * i] = 2 * i;                              // bit 0: 0 = left the cluster, 1 = joined it
  keys[2 * i + 1] = (moved && c < K) ? c : K;
  vals[2 * i + 1] = 2 * i + 1;
}

template <int METRIC>
__global__ void __launch_bounds__(32)
strict_adjust_kernel(const float* __restrict__ X, int D, uint32_t K, const uint32_t* __restrict__ offsets,
                     const uint32_t* __restrict__ events, float* __restrict__ C, uint32_t* __restrict__ ccounts) {
  extern __shared__ float srow[];                    // [D][32]: feature-major, one column per thread (no bank conflicts)
  const uint32_t c = blockIdx.x * 32 + threadIdx.x;
  if (c >= K) return;
  float* row = C + static_cast<size_t>(c) * D;
  float* mine = srow + threadIdx.x;
  uint32_t cnt = ccounts[c];
  const float fc = static_cast<float>(cnt);
  for (int f = 0; f < D; f++) mine[f * 32] = row[f] * fc;
  float corr = 0.f;
  const uint32_t beg = offsets[c], end = offsets[c + 1];
  for (uint32_t e = beg; e < end; e++) {
    const uint32_t v = events[e];
    const float fs = (v & 1u) ? 1.f : -1.f;
    cnt += (v & 1u) ? 1u : 0xFFFFFFFFu;
    const float* xs = X + static_cast<size_t>(v >> 1) * D;
    for (int f = 0; f < D; f++) {
      const float cv = mine[f * 32];
      const float y = __fmaf_rd(xs[f], fs, corr);
      const float t = cv + y;
      corr = y - (t - cv);
      mine[f * 32] = t;
    }
  }
  if (METRIC == 1) {
    Kahan k;
    for (int f = 0; f < D; f++) {
      const float v = mine[f * 32];
      k.mac(v, v);
    }
    const float scale = __frcp_rn(__fsqrt_rn(k.sum));
    for (int f = 0; f < D; f++) row[f] = mine[f * 32] * scale;
  } else {
    const float scale = __frcp_rn(static_cast<float>(cnt));   // count 0 -> inf -> NaN centroid (kmeans.cu:425-427)
    for (int f = 0; f < D; f++) row[f] = mine[f * 32] * scale;
  }
  ccounts[c] = cnt;
}

size_t strict_update_cub_bytes(uint32_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)(2 * static_cast<size_t>(n)), 0, 32);
  return bytes;
}

// keys_in / vals_in / keys_out / vals_out: [2n] each, offsets [K + 2], cub_tmp from strict_update_cub_bytes(n)
cudaError_t launch_strict_update(int metric, const float* X, uint32_t n, int D, uint32_t K, const uint32_t* prev,
                                 const uint32_t* cur, float* C, uint32_t* ccounts, uint32_t* keys_in,
                                 uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out, uint32_t* offsets,
                                 void* cub_tmp, size_t cub_bytes, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  if (static_cast<size_t>(D) * 32 * sizeof(float) > 200 * 1024) return cudaErrorInvalidValue;
  strict_events_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, K, prev, cur, keys_in, vals_in);
  int bits = 1;
  while ((1ull << bits) <= K) bits++;  // keys are in [0, K]
  cudaError_t e = cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, keys_in, keys_out, vals_in, vals_out,
                                                  (int)(2 * static_cast<size_t>(n)), 0, bits, st);
  if (e != cudaSuccess) return e;
  // offsets[c] = first event of cluster c (binary search in the sorted keys); counts are not needed
  launch_segment_offsets(keys_out, 2 * n, K, offsets, keys_in /* scratch */, st);
  const size_t smem = static_cast<size_t>(D) * 32 * sizeof(float);
  if (metric == 1) {
    if ((e = cudaFuncSetAttribute(strict_adjust_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(smem))) != cudaSuccess) return e;
    strict_adjust_kernel<1><<<cdiv(K, 32), 32, smem, st>>>(X, D, K, offsets, vals_out, C, ccounts);
  } else {
    if ((e = cudaFuncSetAttribute(strict_adjust_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(smem))) != cudaSuccess) return e;
    strict_adjust_kernel<0><<<cdiv(K, 32), 32, smem, st>>>(X, D, K, offsets, vals_out, C, ccounts);
  }
  return cudaGetLastError();
}

// all-reduce of the update's partial sums over peer memory: every GPU gathers and adds all shards' sums itself (K*D*4
// bytes per peer over NVLink; 16-byte loads, each peer's buffer read exactly once, coalesced)
__global__ void __launch_bounds__(256)
peer_reduce_kernel(const PeerBuffers pb, size_t nvec4, size_t nsums, uint32_t K, float* __restrict__ out_sums,
                   uint32_t* __restrict__ out_counts) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec4; i += stride) {
    float4 acc = reinterpret_cast<const float4*>(pb.sums[0])[i];
    for (int d = 1; d < pb.n; d++) {
      const float4 v = reinterpret_cast<const float4*>(pb.sums[d])[i];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    reinterpret_cast<float4*>(out_sums)[i] = acc;
  }
  for (size_t i = nvec4 * 4 + static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < nsums; i += stride) {
    float acc = pb.sums[0][i];
    for (int d = 1; d < pb.n; d++) acc += pb.sums[d][i];
    out_sums[i] = acc;
  }
  for (size_t c = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < K; c += stride) {
    uint32_t acc = 0;
    for (int d = 0; d < pb.n; d++) acc += pb.counts[d][c];   // exact integer sum (counts never go through fp32)
    out_counts[c] = acc;
  }
}

__global__ void peer_min_u32_kernel(const PeerU32 pb, size_t count, uint32_t* __restrict__ out) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += stride) {
    uint32_t v = pb.p[0][i];
    for (int d = 1; d < pb.n; d++) v = min(v, pb.p[d][i]);
    out[i] = v;
  }
}
cudaError_t launch_peer_min_u32(const PeerU32& pb, size_t count, uint32_t* out, cudaStream_t st) {
  const unsigned grid = static_cast<unsigned>(std::min<size_t>(148 * 8, (count + 255) / 256 + 1));
  peer_min_u32_kernel<<<grid, 256, 0, st>>>(pb, count, out);
  return cudaGetLastError();
}

cudaError_t launch_peer_reduce(const PeerBuffers& pb, uint32_t K, int D, float* out_sums, uint32_t* out_counts,
                               cudaStream_t st) {
  const size_t nsums = static_cast<size_t>(K) * D;
  const size_t nvec4 = nsums / 4;
  const unsigned grid = static_cast<unsigned>(std::min<size_t>(148 * 4, (nvec4 + 255) / 256 + 1));
  peer_reduce_kernel<<<grid, 256, 0, st>>>(pb, nvec4, nsums, K, out_sums, out_counts);
  return cudaGetLastError();
}

// L2: element-wise (the same two operations per element as normalize_kernel<0>, one thread per element instead of one
// thread walking a whole centroid with strided accesses: 24 us -> a few us at 1024 x 256)
__global__ void normalize_l2_kernel(const float* __restrict__ sums, const uint32_t* __restrict__ counts, uint32_t K, int D,
                                    float* __restrict__ C, uint32_t* __restrict__ ccounts) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<size_t>(K) * D) return;
  const uint32_t c = i / D;
  const uint32_t cnt = counts[c];
  C[i] = sums[i] * __frcp_rn(static_cast<float>(cnt));
  if (i - static_cast<size_t>(c) * D == 0) ccounts[c] = cnt;
}

cudaError_t launch_normalize(int metric, const float* sums, const uint32_t* counts, uint32_t K, int D,
                             float* C, uint32_t* ccounts, float* prev_sums, cudaStream_t st) {
  if (metric == 1) normalize_kernel<1><<<cdiv(K, 64), 64, 0, st>>>(sums, counts, K, D, C, ccounts, prev_sums);
  else normalize_l2_kernel<<<cdiv(static_cast<size_t>(K) * D, 256), 256, 0, st>>>(sums, counts, K, D, C, ccounts);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Yinyang bound maintenance (reference kmeans.cu:487-672), exact arithmetic, row-major samples.
// ------------------------------------------------------------------------------------------------
template <int METRIC>
__global__ void yy_drifts_kernel(const float* __restrict__ Cnew, const float* __restrict__ Cold,
                                 uint32_t K, int D, float* __restrict__ drift) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= K) return;
  drift[c] = distance_exact<METRIC>(Cnew + static_cast<size_t>(c) * D, Cold + static_cast<size_t>(c) * D, D);
}

__global__ void yy_group_max_kernel(const float* __restrict__ drift, const uint32_t* __restrict__ groups,
                                    uint32_t K, uint32_t G, float* __restrict__ maxdrift) {
  uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  float m = -FLT_MAX;
  for (uint32_t c = 0; c < K; c++)
    if (groups[c] == g) {
      float d = drift[c];
      if (m < d) m = d;
    }
  maxdrift[g] = m;
}

cudaError_t launch_yy_drifts(int metric, const float* Cnew, const float* Cold, uint32_t K, int D,
                             uint32_t G, const uint32_t* groups, float* drift, float* maxdrift,
                             cudaStream_t st) {
  if (metric == 1) yy_drifts_kernel<1><<<cdiv(K, 64), 64, 0, st>>>(Cnew, Cold, K, D, drift);
  else yy_drifts_kernel<0><<<cdiv(K, 64), 64, 0, st>>>(Cnew, Cold, K, D, drift);
  yy_group_max_kernel<<<cdiv(G, 64), 64, 0, st>>>(drift, groups, K, G, maxdrift);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// average distance (kmeans.cu:674-691) and the k-means++ distance step (kmeans.cu:42-67)
// ------------------------------------------------------------------------------------------------
template <int METRIC>
__global__ void average_distance_kernel(const float* __restrict__ X, const float* __restrict__ C,
                                        uint32_t n, int D, const uint32_t* __restrict__ assign,
                                        double* __restrict__ d_sum) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  float dist = 0.f;
  if (i < n)
    dist = distance_exact<METRIC>(X + static_cast<size_t>(i) * D, C + static_cast<size_t>(assign[i]) * D, D);
  for (int o = 16; o > 0; o >>= 1) dist += __shfl_down_sync(0xffffffffu, dist, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(d_sum, static_cast<double>(dist));
}

cudaError_t launch_average_distance(int metric, const float* X, const float* C, uint32_t n, int D,
                                    const uint32_t* assign, double* d_sum, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  if (metric == 1) average_distance_kernel<1><<<cdiv(n, 256), 256, 0, st>>>(X, C, n, D, assign, d_sum);
  else average_distance_kernel<0><<<cdiv(n, 256), 256, 0, st>>>(X, C, n, D, assign, d_sum);
  return cudaGetLastError();
}

template <int METRIC>
__global__ void plusplus_kernel(const float* __restrict__ X, uint32_t n, int D,
                                const float* __restrict__ centroid, int first,
                                float* __restrict__ dists, double* __restrict__ d_sum) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  float dist = 0.f;
  if (i < n) {
    const float* x = X + static_cast<size_t>(i) * D;
    if (x[0] == x[0]) dist = distance_exact<METRIC>(x, centroid, D);
    float prev;
    if (first || dist < (prev = dists[i])) dists[i] = dist;
    else dist = prev;
  }
  for (int o = 16; o > 0; o >>= 1) dist += __shfl_down_sync(0xffffffffu, dist, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(d_sum, static_cast<double>(dist));
}

cudaError_t launch_plusplus_step(int metric, const float* X, uint32_t n, int D, const float* centroid,
                                 int first, float* dists, double* d_sum, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  if (metric == 1) plusplus_kernel<1><<<cdiv(n, 256), 256, 0, st>>>(X, n, D, centroid, first, dists, d_sum);
  else plusplus_kernel<0><<<cdiv(n, 256), 256, 0, st>>>(X, n, D, centroid, first, dists, d_sum);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Device-resident k-means++ (reference kmcuda.cc:262-333 + kmeans.cu:42-67).  The reference runs K - 1 rounds of
// {distance kernel, D2H of all N distances, sequential CDF walk on the host, H2D of the chosen row}; here a round is
// two kernels and nothing crosses PCIe: pp_update_kernel refreshes the min-distances and leaves one partial sum per
// 256 samples, pp_pick_kernel (one CTA) scans the partial sums, resolves the draw to a sample with the reference's
// walk semantics (including its backward branch, kmcuda.cc:304-320) and copies that sample into the centroid table.
// The random draws are the reference's: rand() on the host, one per round, uploaded once.
// ------------------------------------------------------------------------------------------------
constexpr int kPpBlock = 256;

template <int METRIC>
__global__ void __launch_bounds__(kPpBlock)
pp_update_kernel(const float* __restrict__ X, uint32_t n, int D, const float* __restrict__ centroid, int first,
                 float* __restrict__ dists, double* __restrict__ bsum) {
  __shared__ double s_part[kPpBlock / 32];
  const uint32_t i = blockIdx.x * kPpBlock + threadIdx.x;
  float dist = 0.f;
  if (i < n) {
    const float* x = X + static_cast<size_t>(i) * D;
    if (x[0] == x[0]) dist = distance_exact<METRIC>(x, centroid, D);
    float prev;
    if (first || dist < (prev = dists[i])) dists[i] = dist;
    else dist = prev;
  }
  double v = (dist == dist) ? static_cast<double>(dist) : 0.0;
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kPpBlock / 32; w++) t += s_part[w];
    bsum[blockIdx.x] = t;            // deterministic (fixed order), unlike an atomic total
  }
}

// prefix P(t) = sum of the first t distances, from the scanned block sums + the tail of one block
__device__ double pp_prefix(const float* __restrict__ dists, const double* __restrict__ bpre, uint32_t t) {
  const uint32_t b = t / kPpBlock;
  double p = bpre[b];
  for (uint32_t u = b * kPpBlock; u < t; u++) {
    const float d = dists[u];
    if (d == d) p += static_cast<double>(d);
  }
  return p;
}

__global__ void __launch_bounds__(1024)
pp_pick_kernel(const float* __restrict__ X, uint32_t n, int D, const float* __restrict__ dists,
               const double* __restrict__ bsum, double* __restrict__ bpre, uint32_t nb, double choice,
               float* __restrict__ next_centroid, uint32_t* __restrict__ chosen_out) {
  __shared__ double s_chunk[1024];
  __shared__ double s_total;
  __shared__ uint32_t s_j;
  // exclusive scan of the block sums into bpre[0 .. nb] (bpre[nb] = total): each thread owns a contiguous chunk
  const uint32_t per = (nb + 1023) / 1024;
  const uint32_t lo = min(nb, threadIdx.x * per), hi = min(nb, lo + per);
  double acc = 0.0;
  for (uint32_t b = lo; b < hi; b++) acc += bsum[b];
  s_chunk[threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double run = 0.0;
    for (int t = 0; t < 1024; t++) {
      const double c = s_chunk[t];
      s_chunk[t] = run;
      run += c;
    }
    s_total = run;
  }
  __syncthreads();
  double run = s_chunk[threadIdx.x];
  for (uint32_t b = lo; b < hi; b++) {
    bpre[b] = run;
    run += bsum[b];
  }
  if (threadIdx.x == 0) bpre[nb] = s_total;
  __syncthreads();
  if (threadIdx.x == 0) {
    const double total = bpre[nb];
    const double cs = choice * total;
    uint32_t ca = static_cast<uint32_t>(choice * n);
    uint32_t j;
    // smallest j >= from with P(j) >= cs (n if none): binary search over the block prefixes, then inside the block
    auto first_reaching = [&](uint32_t from) -> uint32_t {
      if (pp_prefix(dists, bpre, from) >= cs) return from;
      uint32_t blo = from / kPpBlock, bhi = nb;          // invariant: prefix at block start blo < cs <= ... search block
      while (blo + 1 < bhi) {
        const uint32_t mid = blo + (bhi - blo) / 2;
        if (bpre[mid] >= cs) bhi = mid; else blo = mid;
      }
      double p = bpre[blo];
      uint32_t u = blo * kPpBlock;
      if (u < from) { p = pp_prefix(dists, bpre, from); u = from; }
      const uint32_t end = min(n, (blo + 1) * kPpBlock);
      for (; u < end; u++) {
        const float d = dists[u];
        if (d == d) p += static_cast<double>(d);
        if (p >= cs) return u + 1;
      }
      // rounding left the crossing in the next block (or nowhere): continue linearly
      for (; u < n; u++) {
        const float d = dists[u];
        if (d == d) p += static_cast<double>(d);
        if (p >= cs) return u + 1;
      }
      return n;
    };
    if (ca < 100) {
      j = first_reaching(0);                                              // kmcuda.cc:298-302
    } else {
      ca = min(ca, n - 1);
      const double s2 = pp_prefix(dists, bpre, ca);
      if (s2 < cs) {
        j = first_reaching(ca);                                           // kmcuda.cc:309-313
      } else {
        // backward walk (kmcuda.cc:314-320): it subtracts d[ca], d[ca-1], ... from P(ca) until the sum drops below the
        // draw or j reaches 1, i.e. it stops at the largest t <= ca with P(t) - d[ca] < cs, and picks sample t - 1
        const float dca = dists[ca];
        const double lim = cs + ((dca == dca) ? static_cast<double>(dca) : 0.0);
        // largest t <= ca with P(t) < lim: the block by binary search over the block prefixes (P at block starts),
        // then a scan inside that block
        uint32_t tlo = 0;
        if (0.0 < lim) {
          uint32_t blo = 0, bhi = ca / kPpBlock;                          // bpre[blo] < lim holds for blo = 0
          while (blo < bhi) {
            const uint32_t mid = blo + (bhi - blo + 1) / 2;
            if (bpre[mid] < lim) blo = mid; else bhi = mid - 1;
          }
          double pcur = bpre[blo];
          tlo = blo * kPpBlock;
          while (tlo < ca) {
            const float d = dists[tlo];
            const double pn = pcur + ((d == d) ? static_cast<double>(d) : 0.0);
            if (!(pn < lim)) break;
            pcur = pn;
            tlo++;
          }
        }
        const uint32_t t = max(tlo, 2u);
        j = t;                                                            // chosen sample t - 1  (j = j_end + 1 = t)
      }
    }
    if (j == 0 || j > n) j = min(max(j, 1u), n);                          // kmcuda.cc:322-327
    s_j = j - 1;
    *chosen_out = j - 1;
  }
  __syncthreads();
  const float* src = X + static_cast<size_t>(s_j) * D;
  for (int f = threadIdx.x; f < D; f += 1024) next_centroid[f] = src[f];
}

// one k-means++ round on the device: distances to C[i-1], pick sample for C[i]
cudaError_t launch_plusplus_round(int metric, const float* X, uint32_t n, int D, float* C, uint32_t i, double choice,
                                  float* dists, double* bsum, double* bpre, uint32_t* chosen, cudaStream_t st) {
  const uint32_t nb = cdiv(n, kPpBlock);
  const float* cprev = C + static_cast<size_t>(i - 1) * D;
  if (metric == 1) pp_update_kernel<1><<<nb, kPpBlock, 0, st>>>(X, n, D, cprev, i == 1, dists, bsum);
  else pp_update_kernel<0><<<nb, kPpBlock, 0, st>>>(X, n, D, cprev, i == 1, dists, bsum);
  pp_pick_kernel<<<1, 1024, 0, st>>>(X, n, D, dists, bsum, bpre, nb, choice, C + static_cast<size_t>(i) * D, chosen + i);
  return cudaGetLastError();
}

// AFK-MC2 (reference kmeans_afkmc2_min_dist, kmeans.cu:159-176): for every candidate sample the distance to the
// nearest of the first k centroids.  One thread per (candidate, centroid) pair (the reference walks the k
// centroids serially per candidate); the minimum is taken on the float bit patterns (distances are >= 0, NaN
// never lowers it).  rows[] are shard-local sample indices.
template <int METRIC>
__global__ void afkmc2_min_dist_kernel(const float* __restrict__ X, const float* __restrict__ C, int D, uint32_t k,
                                       const uint32_t* __restrict__ rows, uint32_t m,
                                       uint32_t* __restrict__ min_bits) {
  const uint64_t p = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= static_cast<uint64_t>(m) * k) return;
  const uint32_t cand = static_cast<uint32_t>(p / k), c = static_cast<uint32_t>(p % k);
  const float d = distance_exact<METRIC>(X + static_cast<size_t>(rows[cand]) * D, C + static_cast<size_t>(c) * D, D);
  if (d == d) atomicMin(min_bits + cand, __float_as_uint(fmaxf(d, 0.f)));
}

cudaError_t launch_afkmc2_min_dist(int metric, const float* X, const float* C, int D, uint32_t k,
                                   const uint32_t* rows, uint32_t m, float* min_dists, cudaStream_t st) {
  if (m == 0 || k == 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(min_dists, 0x7f, sizeof(float) * m, st);   // 0x7f7f7f7f = 3.39e38: "no centroid yet"
  if (e != cudaSuccess) return e;
  const uint64_t pairs = static_cast<uint64_t>(m) * k;
  const unsigned grid = static_cast<unsigned>((pairs + 127) / 128);
  if (metric == 1)
    afkmc2_min_dist_kernel<1><<<grid, 128, 0, st>>>(X, C, D, k, rows, m, reinterpret_cast<uint32_t*>(min_dists));
  else
    afkmc2_min_dist_kernel<0><<<grid, 128, 0, st>>>(X, C, D, k, rows, m, reinterpret_cast<uint32_t*>(min_dists));
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// fp16x2 ingest / egress (exact widening; centroids narrowed round-to-nearest on the way out)
// ------------------------------------------------------------------------------------------------
}  // namespace kmb
#include <cuda_fp16.h>
namespace kmb {

__global__ void half_to_float_kernel(const __half* __restrict__ src, float* __restrict__ dst, size_t n) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) dst[i] = __half2float(src[i]);
}
__global__ void float_to_half_kernel(const float* __restrict__ src, __half* __restrict__ dst, size_t n) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) dst[i] = __float2half_rn(src[i]);
}
__global__ void fill_u32_kernel(uint32_t* p, uint32_t v, size_t n) {
  size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

cudaError_t launch_half_to_float(const void* src, float* dst, size_t n, cudaStream_t st) {
  if (!n) return cudaSuccess;
  half_to_float_kernel<<<min(cdiv(n, 256), 148u * 32u), 256, 0, st>>>(static_cast<const __half*>(src), dst, n);
  return cudaGetLastError();
}
cudaError_t launch_float_to_half(const float* src, void* dst, size_t n, cudaStream_t st) {
  if (!n) return cudaSuccess;
  float_to_half_kernel<<<min(cdiv(n, 256), 148u * 32u), 256, 0, st>>>(src, static_cast<__half*>(dst), n);
  return cudaGetLastError();
}
cudaError_t launch_fill_u32(uint32_t* p, uint32_t v, size_t n, cudaStream_t st) {
  if (!n) return cudaSuccess;
  fill_u32_kernel<<<min(cdiv(n, 256), 148u * 32u), 256, 0, st>>>(p, v, n);
  return cudaGetLastError();
}

}  // namespace kmb
