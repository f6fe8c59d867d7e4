// assign_tc.cu -- the B200 hot path: samples x centroids L2 ranking as a dense fp16 contraction on
// tcgen05 tensor cores, fused with a per-sample candidate filter; the exact fp32 re-check
// (below + simt_kernels.cu) then makes the final, reference-identical decision.
//
// What the reference does here: kmeans_assign_lloyd (reference src/kmeans.cu:293-364) -- one CUDA
// thread per sample, N*K*D Kahan-compensated round-down FMAs on the FP32 pipe.
//
// What this file does instead, per persistent CTA (one per SM) and per tile of 128 samples:
//   X producer      : TMA (cp.async.bulk.tensor, 128B swizzle) streams the caller's fp32 rows, 32
//                     features x 128 rows per stage, through a 4-deep mbarrier ring
//   converter warps : one thread per sample row: LDS the fp32 stage -> *s (power of two) -> fp16 ->
//                     tcgen05.st into TMEM, where the A operand lives double-buffered (so the next
//                     tile is converted while the current one is multiplied); per row ||x~||,
//                     ||x - x~|| are accumulated for the error bound
//   B producer      : TMA streams the fp16 centroid table (128 centroids x 64 features per stage,
//                     128B swizzle) + the per-n-tile bias block through mbarrier rings
//   MMA thread      : tcgen05.mma kind::f16, A from TMEM, B from shared memory, M=128 N=128 K=16,
//                     fp32 accumulators double-buffered in TMEM (2 x 128 columns); one extra K=16
//                     step (A and B from shared memory) adds -||c||^2/2 as three fp16 terms against
//                     constant ones, so acc = x.c - ||c||^2/2.  The Lloyd pass on large inputs runs as
//                     clusters of two CTAs: one tcgen05.mma.cta_group::2 of M=256 per K step, issued by
//                     the leader CTA, every CTA staging half of each centroid tile (template parameter CG)
//   epilogue warps  : tcgen05.ld 32 columns at a time; running row maximum M; every column whose
//                     value is within `margin` of M is recorded (bit mask per 32-column chunk);
//                     margin is a rigorous bound on |approx - exact| derived from the actual
//                     rounding residuals (Cauchy-Schwarz), so the reference's fp32 winner is
//                     guaranteed to be among the recorded candidates.
//   rows with one candidate are final; rows with several go to the exact re-check queue; rows with
//   non-finite data or too many candidates go to the exact full pass.  Assignments are therefore
//   bit-identical to the reference kernel's, ties included.
//
// TMEM map (512 columns): [0,128) accumulator 0, [128,256) accumulator 1, [256,384) A buffer 0,
// [384,512) A buffer 1 (128 rows x 256 fp16 = 128 lanes x 128 32-bit columns); for D > 256 one A buffer of up to
// 256 columns.
//
// The same kernel template serves two more callers (MODE template parameter, see tc::Params):
//   MODE 1  Yinyang local step (reference kmeans.cu:584-672): the samples are a compacted row list read straight
//           from global memory by the converter warps; candidates = every centroid within the margin of the
//           row's SECOND best; all of them get their exact true distance (yinyang.cu finishes the step).
//   MODE 2  k-NN (reference knn.cu:177-347): queries and candidates are the samples in a cluster-aligned table;
//           a tile is multiplied with one segment per candidate cluster, both operands centred on that
//           cluster's centroid; the epilogue keeps the k+1 largest 4-column-group maxima per half-row as its
//           threshold and records candidate masks in global lists (namespace knn below has the passes around it).
#include <cuda.h>
#include <cuda_fp16.h>

#include <cstdio>
#include <algorithm>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include <cub/cub.cuh>

#include "exact.cuh"
#include "kernels.h"
#include "sm100_ptx.cuh"

namespace kmb {

namespace tc {
constexpr int TM = 128;                 // samples per tile (UMMA M)
constexpr int TN = 128;                 // centroids per n-tile (UMMA N)
constexpr int KB = 64;                  // fp16 elements per K-block = one 128-byte swizzle row of B
constexpr int MAX_NKB = 8;              // D <= 512: A needs 32 TMEM columns per K-block; double-buffered up to 4 K-blocks
constexpr int X_STAGES = 4;             // fp32 sample stages: 32 features x 128 rows = 16 KiB
constexpr int B_STAGES = 5;             // fp16 centroid stages of ONE K-block (64 features x 128 rows = 16 KiB): a stage is
                                        // refilled as soon as its 4 MMAs retire; 4 stages x 256 MMA cycles in flight cover
                                        // the L2 round trip (round 1: 2 stages of 32 KiB left the MMA warp waiting)
constexpr int B_STAGES_PAIR = 8;        // CTA-pair mode (cta_group::2): every CTA stages HALF a centroid tile per K-block, 8 KiB
constexpr int B_STAGES_MAX = B_STAGES > B_STAGES_PAIR ? B_STAGES : B_STAGES_PAIR;
constexpr int X_STAGE_BYTES = TM * 128;
constexpr int B_KB_BYTES = TN * 128;     // one K-block of the centroid tile: 16 KiB
constexpr int B_STAGE_BYTES = B_KB_BYTES;
constexpr int AUG_A_BYTES = TM * 32;    // 4 KiB  (K=16 fp16, no swizzle)
constexpr int AUG_B_BYTES = TN * 32;    // 4 KiB
constexpr int LIST_LEN = 5;             // entries per epilogue thread: one per n-tile that held a candidate (max, 2 x 32-bit mask, n-tile)
// Warp roles.  The SM's issue arbiter prefers the highest warp id of a scheduler (B300_MICROARCH.md), so the warp
// whose stalls cost tensor-pipe time -- the MMA issuer -- gets the highest id and the warps with slack (emitters)
// the lowest.  Converter / epilogue warps keep warp % 4 = TMEM lane quarter.
// There is ONE MMA issuer: round 2 measured a second one taking alternate n-tiles, and with the lean single-thread issue
// loop it was slower (3.88 -> 4.29 ms), because with two n-tiles in flight the 5-stage B ring, 1.25 n-tiles deep,
// becomes the limit.
constexpr int FIRST_EMIT_WARP = 0;      // 4 emitter warps (merge + global emission)
constexpr int FIRST_CONV_WARP = 4;      // 4 converter warps, warp % 4 = TMEM lane quarter
constexpr int FIRST_EPI_WARP = 8;       // 8 epilogue warps
constexpr int WARP_B_PRODUCER = 16, WARP_X_PRODUCER = 17, WARP_MMA = 19;
constexpr int N_CONV_WARPS = 4;
constexpr int N_EPI_WARPS = 8;
constexpr int N_EMIT_WARPS = 4;
constexpr int N_THREADS = 20 * 32;      // 640
constexpr int MAX_CAND = 32;            // candidates per row before falling back to the full exact pass (one per lane of the finishing warp)
constexpr int KNN_CAP = 40;             // k-NN: (chunk, mask) entries per half-row in global memory
constexpr int KNN_MAX_KK = 16;          // k + 1 <= 16 on the tensor-core path
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t TMEM_ACC0 = 0, TMEM_A0 = 256;
constexpr float SENTINEL_GUARD = -65000.f;   // padded / dead centroids score exactly -65504: thresholds below this are not trusted

// counters[] slots
enum { CNT_PAIRS = 0, CNT_ROWQ = 1, CNT_OVF = 2, CNT_ERR = 3, CNT_N = 4 };

struct Stats {       // written by the centroid prep kernels, read by the main kernel
  float scale;       // s = 2^k applied to samples and centroids before fp16 rounding
  float cmax;        // max_c ||s*c||  (finite centroids)
  float dcmax;       // max_c ||s*c - fp16(s*c)||
  uint32_t csq_max_bits;
  uint32_t force_exact; // cosine only: a centroid with an infinite element / norm can still win -> no filtering
  float yabs;           // k-NN: max over samples of s * (|y| + |c(y)|): bounds the rounding of the centring y - c
  float mun;            // s * ||mu|| (upper bound): mu = centring vector of the assignment filter (0 when not centred)
  float knn_extra;      // k-NN, angular metric served through the L2 pass: s^2 * max |1 - ||y||^2| (see tc_knn_search)
};

constexpr uint32_t LIST_ARRAY = 2 * LIST_LEN * 256 * 4;   // bytes of one of the four list arrays (both tile parities)
struct SmemLayout {  // byte offsets from the 1024-aligned dynamic smem base
  uint32_t x, b, aug_a, aug_b, list, norms, fin, mu, bars, tmem_slot, total;
};

__host__ __device__ inline SmemLayout smem_layout() {
  SmemLayout L;
  uint32_t o = 0;
  L.x = o; o += X_STAGES * X_STAGE_BYTES;
  L.b = o; o += B_STAGES * B_STAGE_BYTES;
  L.aug_a = o; o += AUG_A_BYTES;
  L.aug_b = o; o += 2 * AUG_B_BYTES;
  // candidate lists: 4 arrays (entry maximum | mask of columns 0-31 | mask of columns 32-63 | n-tile) of
  // [tile parity][entry][epilogue thread] words, LIST_ARRAY bytes apart.  MODE 2 reuses [list, norms) as its top-kk /
  // bucket scratch: 48 rows x 256 x 4 bytes (static_assert below)
  L.list = o; o += 4 * LIST_ARRAY;
  L.fin = o; o += 2 * 5 * 256 * 4;    // [tile parity][M|cnt|flags|margin|M2][epilogue thread]
  L.norms = o; o += 4 * 4 * TM * 4;   // [tile % 4][x|d][row]  x~^2 | residual^2 | (k-NN) exact s^2|x-c|^2 | (k-NN) s^2(|x|+|c|)^2; 4 deep: the converters run up to 2 segments ahead
  L.mu = o; o += MAX_NKB * KB * 4;    // -mu * s per feature (zero padded): the converters' centring term
  L.bars = o; o += 64 * 8;
  L.tmem_slot = o; o += 16;
  L.total = o;
  return L;
}
static_assert(4 * LIST_ARRAY + 2 * 5 * 256 * 4 >= 48 * 256 * 4, "k-NN scratch overlaps the norms");

// barrier indices inside the bars[] array
enum {
  BAR_X_FULL = 0,                         // [X_STAGES]
  BAR_X_EMPTY = BAR_X_FULL + X_STAGES,    // [X_STAGES]
  BAR_B_FULL = BAR_X_EMPTY + X_STAGES,    // [B_STAGES_MAX]
  BAR_B_EMPTY = BAR_B_FULL + B_STAGES_MAX,    // [B_STAGES_MAX]
  BAR_AUG_FULL = BAR_B_EMPTY + B_STAGES_MAX,  // [2]
  BAR_AUG_EMPTY = BAR_AUG_FULL + 2,       // [2]
  BAR_A_FULL = BAR_AUG_EMPTY + 2,         // [2][MAX_NKB]
  BAR_A_FREE = BAR_A_FULL + 2 * MAX_NKB,  // [2]
  BAR_ACC_FULL = BAR_A_FREE + 2,          // [2]
  BAR_ACC_EMPTY = BAR_ACC_FULL + 2,       // [2]
  BAR_EMIT_FULL = BAR_ACC_EMPTY + 2,      // [2] epilogue -> emitter (per tile parity)
  BAR_EMIT_EMPTY = BAR_EMIT_FULL + 2,     // [2]
  BAR_COUNT = BAR_EMIT_EMPTY + 2
};
static_assert(BAR_COUNT <= 63, "barrier array too small");   // slot 63 is the CTA's "a wait has given up" flag

struct Params {
  uint32_t n;
  int D;
  uint32_t K;
  int nkb;                   // K-blocks of 64 features
  int nt;                    // n-tiles of 128 centroids
  uint32_t ntiles;           // sample tiles
  const __half* aug_blob;    // [nt][AUG_B_BYTES] in the shared-memory byte layout
  const Stats* stats;
  uint32_t* result;          // [n]
  uint32_t* pair_row;        // re-check queue: (row, candidate) pairs
  uint32_t* pair_cand;
  uint32_t max_pairs;
  uint32_t* rowq;            // [3*i]: row, first pair, pair count
  uint32_t* ovf_rows;        // rows for the full exact pass
  uint32_t* counters;        // CNT_*
  int metric;                // 0 = L2 (score x.c - ||c||^2/2), 1 = cosine (score x.c; larger dot = smaller angle)
  const float* neg_mu_s;     // [nkb*64] -mu*s (zero padded), nullptr = no centring: MODE 0/1 multiply (x - mu) with the
                             // table of (c - mu); scores shift by a per-row constant, so the ranking is unchanged while
                             // the fp16 rounding error (proportional to |x - mu| |c - mu|) shrinks
  // MODE 0 with assign != nullptr: the bookkeeping of the assignment pass is fused (reference kmeans.cu:356-363):
  // prev[row] = assign[row]; assign[row] = winner; *d_changed += (winner != old); rows that go to the re-check /
  // exact queues are finished by those kernels
  uint32_t* assign;
  uint32_t* prev;
  uint32_t* d_changed;
  // MODE 3 (Yinyang bounds refresh, reference kmeans_yy_init kmeans.cu:431-485): the table is the GROUP-SORTED
  // centroid list, every group padded to whole 4-column quads (yy_qgroup[(n-tile * 2 + half) * 16 + quad] = group of
  // that quad, UINT32_MAX past the end).  The epilogue folds the quad maxima into per-group maxima and turns each
  // into a LOWER bound of the distance to the nearest centroid of that group, d >= sqrt(|x^|^2 - 2 (max + E)) / s,
  // merged into bounds[row][1 + g] with an atomic minimum; the sample's own group and its upper bound are exact
  // (yy_own_group_kernel).  Valid bounds are all Yinyang needs: the assignments stay those of Lloyd's algorithm.
  const uint32_t* yy_qgroup;
  const uint32_t* yy_groups;     // [K] centroid -> group
  const uint32_t* yy_assign;     // [n]
  float* yy_bounds;              // [n][G + 1]
  uint32_t G;
  // MODE 1 (Yinyang local step): the samples are the rows listed in rows[0 .. *d_nrows), read straight from
  // global memory by the converter warps; every column within the margin of the row's SECOND best score is a
  // candidate and every candidate goes to the pair queue (the caller needs exact best and second-best distances)
  const float* X;
  const uint32_t* rows;
  const uint32_t* d_nrows;
  // MODE 2 (k-NN candidate pass): queries AND candidates are the samples in the cluster-aligned table order: cluster
  // c owns the blocks [blk_first[c], blk_first[c+1]) of 128 table rows (zero-padded), rows[] maps a table row to the
  // original sample (UINT32_MAX = padding), so query tile t IS block t.  A tile is multiplied with a list of
  // SEGMENTS knn_ranges[knn_roff[t] .. +knn_rcount[t]): each segment is the block range of ONE candidate cluster B,
  // and for it the queries are re-converted relative to B's centroid -- both operands are then small vectors
  // (x - c_B, y - c_B), which is what gives the fp16 product enough resolution inside tight clusters.  The per-row
  // constant s^2 |x - c_B|^2 / 2 is folded into the threshold, so everything the epilogue keeps (top-kk list, entry
  // maxima) lives in the translation-invariant score g = -s^2 d^2 / 2.  Every column within the margin of the row's
  // kk-th largest 4-column-group maximum (kk = k + 1, self included) is recorded as (max, mask, chunk id, margin).
  const uint32_t* d_ntiles;
  const uint32_t* tile_nrows;
  const uint32_t* blk_cluster;
  const float* C;                // centroids [K][D] (fp32)
  const uint2* knn_ranges;
  const uint32_t* knn_roff;
  const uint32_t* knn_rcount;
  const uint32_t* knn_nblk;      // blocks per tile (sum over its segments)
  int kk;
  int knn_first_pass;            // 1: the per-row state starts empty; the tile has TWO segments, both its own cluster:
                                 //    the first sweep only builds the top-kk threshold, the second one only records
  uint32_t knn_stride;           // = 2 * (table rows): stride of the [kk][stride] top-kk state
  float* knn_topk;               // [kk][stride] descending group maxima (g-space) of half-row (table row * 2 + h)
  uint32_t* knn_cnt;             // [stride] entries used
  uint32_t* knn_flags;           // [stride]
  float* knn_dub;                // [stride] upper bound of the exact distance to the kk-th nearest candidate seen so far
  uint4* knn_entries;            // [stride][KNN_CAP]: (group max bits (g-space), mask, chunk id, margin bits)
  uint32_t knn_part, knn_nparts; // query-tile shard of this device (0, 1 = everything)
};

// ---------------------------------------------------------------------------------------------------
// centroid preparation: scale, fp16 table (zero padded to [nt*256][nkb*64]), bias blobs, statistics
// ---------------------------------------------------------------------------------------------------
__global__ void tc_prep_stats_kernel(const float* __restrict__ csq, uint32_t K, Stats* __restrict__ st) {
  // max finite ||c||^2 (positive floats order like unsigned ints)
  uint32_t best = 0;
  for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < K; c += gridDim.x * blockDim.x) {
    float v = csq[c];
    if (v == v && v < 3.0e38f) best = max(best, __float_as_uint(fmaxf(v, 0.f)));
  }
  for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0) atomicMax(&st->csq_max_bits, best);
}

__global__ void tc_prep_scale_kernel(Stats* __restrict__ st) {   // one thread
  float cmax = __fsqrt_ru(__uint_as_float(st->csq_max_bits));
  float s = 1.f;
  if (cmax > 0.f && cmax < 3.0e38f) {
    int e;
    frexpf(cmax, &e);          // cmax = m * 2^e, m in [0.5, 1)
    s = ldexpf(1.f, 6 - e);    // s*cmax in [32, 64)
  }
  st->scale = s;
  st->cmax = cmax * s * 1.001f;
  st->dcmax = 0.f;
}

// one table row (a centroid, or a zero padding row up to nt*TN) by one warp; s = Stats::scale; csq / mu may have been
// written earlier in the SAME launch by other CTAs (fused preparation), hence no __restrict__ / read-only loads on them
__device__ __forceinline__ void prep_table_row(uint32_t row, int lane, float s, int metric, const float* __restrict__ C,
                                               const float* csq, uint32_t K, int D, int nkb, __half* __restrict__ table,
                                               __half* __restrict__ aug_blob, Stats* st,
                                               const uint32_t* __restrict__ gather, const float* mu, int by_source,
                                               int pair_blob) {
  // by_source (Yinyang refresh layout): table row r holds centroid gather[r] (UINT32_MAX = padding) and csq[] is
  // indexed by the centroid; otherwise csq[] is indexed by the table row and rows >= K are padding
  const int Dp = nkb * KB;
  uint32_t src = row;
  bool finite = row < K;
  if (by_source) {
    src = gather[row];
    finite = src != UINT32_MAX;
    if (!finite) src = 0;
  } else if (finite && gather) {
    src = gather[row];
  }
  const uint32_t qrow = by_source ? src : row;
  const float* Crow = C + static_cast<size_t>(src) * D;
  if (finite) {
    float q = __ldcg(csq + qrow);
    finite = (q == q) && q < 3.0e38f;
    for (int f = lane; f < D; f += 32) {
      float v = Crow[f];
      if (!(fabsf(v) < 3.0e38f)) finite = false;
    }
    finite = __all_sync(0xffffffffu, finite);
    if (metric == 1 && !finite) {
      // a NaN centroid never wins (acos(NaN) fails every '<'), but one with +-Inf elements or an
      // overflowing norm can: the filter has no bound for it, so the whole pass runs exact
      bool has_nan = false;
      for (int f = lane; f < D; f += 32) {
        float v = Crow[f];
        has_nan |= (v != v);
      }
      has_nan = __any_sync(0xffffffffu, has_nan);
      if (!has_nan && lane == 0) st->force_exact = 1u;
    }
  }
  float d2 = 0.f;
  for (int f = lane; f < Dp; f += 32) {
    float v = (finite && f < D) ? (mu ? Crow[f] - mu[f] : Crow[f]) * s : 0.f;
    __half h = __float2half_rn(v);
    float r = v - __half2float(h);
    d2 = fmaf(r, r, d2);
    table[static_cast<size_t>(row) * Dp + f] = h;
  }
  for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
  if (lane == 0) {
    if (finite) atomicMax(reinterpret_cast<uint32_t*>(&st->dcmax), __float_as_uint(__fsqrt_ru(d2) * 1.0001f));
    // bias: three fp16 terms of -(s^2 ||c - mu||^2 / 2); invalid / padded centroids get -65504
    __half b[3];
    if (finite) {
      float h = metric == 1 ? 0.f : -0.5f * ((s * __ldcg(csq + qrow)) * s);   // s = 2^k: exact; this order cannot overflow for tiny data
      b[0] = __float2half_rn(h);
      float r1 = h - __half2float(b[0]);
      b[1] = __float2half_rn(r1);
      float r2 = r1 - __half2float(b[1]);
      b[2] = __float2half_rn(r2);
    } else {
      b[0] = __float2half_rn(-65504.f);
      b[1] = b[2] = __float2half_rn(0.f);
    }
    // shared-memory layout of the K=16 no-swizzle block: core matrix = 8 rows x 16 bytes contiguous,
    // 8-row groups 128 bytes apart, second K half TN*16 bytes further
    const uint32_t t = row / TN, r = row % TN;
    __half* blob = aug_blob + static_cast<size_t>(t) * (AUG_B_BYTES / 2);
    for (int k = 0; k < 16; k++) {
      int j = k >> 3, e = k & 7;
      // CTA-pair mode: the block is two 2 KiB pieces (rows 0-63 for the leader CTA, 64-127 for its peer), each in the
      // layout of a 64-row operand (K halves 64 * 16 bytes apart)
      const uint32_t off = pair_blob ? (r >> 6) * 2048u + j * 1024u + ((r & 63u) >> 3) * 128u + (r & 7u) * 16u
                                     : j * (TN * 16) + (r >> 3) * 128 + (r & 7) * 16;
      blob[off / 2 + e] = k < 3 ? b[k] : __float2half_rn(0.f);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// The whole centroid preparation of one pass as ONE launch (Lloyd / Yinyang tables; the k-NN tables have their own
// kernels).  As a chain of small kernels it was ten stream operations (three memsets, ||c||^2, mean, mu, centred norms,
// maximum, scale, table) of 3-12 us each on a 1 MB centroid matrix: ~0.05 ms of dependent launches per pass, 1 % of the
// step of an 8M-row shard and 8 % of the step of a 1M-row shard (8 GPUs), as measured in round 2; that chain has since
// been removed.  Here the same arithmetic runs as four phases of one small grid separated by a sense-reversing grid
// barrier; every CTA is resident (grid <= number of SMs, 256 threads, 34 KB static shared memory),
// so the barrier cannot deadlock.  Values produced by other CTAs in an earlier phase are read with ld.global.cg.
// ---------------------------------------------------------------------------------------------------
struct PrepArgs {
  int metric, D, nkb, by_source, pair_blob;
  uint32_t K, rows_pad;
  const float* C;
  float* csq;            // reference-order ||c||^2 (L2) / 1 (cosine); written here when compute_csq
  int compute_csq;
  float* cnorm2;         // L2: ||c - mu||^2; cosine: upper bound of ||c||^2
  double* musum;         // [D] + valid-row count
  float* neg_mu_s;       // [nkb * KB]
  Stats* stats;
  uint32_t* counters;    // CNT_N words, zeroed here
  __half* table;
  __half* aug_blob;
  const uint32_t* gather;
  unsigned* barrier;     // {arrivals, generation}
};

__device__ __forceinline__ void prep_grid_barrier(unsigned* bar, unsigned nblocks) {
  __syncthreads();
  if (threadIdx.x == 0) {
    volatile unsigned* gen = bar + 1;
    const unsigned g = *gen;          // cannot advance before this CTA has arrived
    __threadfence();
    if (atomicAdd(bar, 1u) == nblocks - 1u) {
      atomicExch(bar, 0u);
      __threadfence();
      atomicAdd(bar + 1, 1u);
    } else {
      while (*gen == g) __nanosleep(32);
    }
    __threadfence();
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256)
tc_prep_fused_kernel(const PrepArgs a) {
  __shared__ float s_tile[8][32 * 33];   // ||c||^2: one 32 x 32 staging tile per warp
  __shared__ float s_mu[MAX_NKB * KB];
  __shared__ float s_scale;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t gw = blockIdx.x * 8u + warp, nw = gridDim.x * 8u;
  const uint32_t gt = blockIdx.x * 256u + tid, nthr = gridDim.x * 256u;
  const int D = a.D;
  const uint32_t K = a.K;

  // ---- phase 0: zero the pass counters / statistics / column sums; ||c||^2 in the reference's order
  if (gt < CNT_N) a.counters[gt] = 0u;
  if (gt < sizeof(Stats) / 4) reinterpret_cast<uint32_t*>(a.stats)[gt] = 0u;
  if (a.metric == 0)
    for (uint32_t i = gt; i < static_cast<uint32_t>(D) + 1u; i += nthr) a.musum[i] = 0.0;
  if (a.compute_csq) {
    float* tile = s_tile[warp];
    for (uint32_t c0 = gw * 32u; c0 < K; c0 += nw * 32u) {
      if (a.metric == 1) {
        if (c0 + lane < K) a.csq[c0 + lane] = 1.f;
        continue;
      }
      // lane r walks row c0 + r in feature order (the reference's sequential Kahan sum); 32 features x 32 rows are
      // staged through shared memory with coalesced loads (lane = feature), and the loads of the NEXT 32 features are
      // in flight during the walk -- this phase is the longest of the launch (a 256-step dependent chain per row)
      kmb::Kahan k;
      float v[32];
      auto load32 = [&](int f0) {
        const int fl = min(32, D - f0);
#pragma unroll
        for (int r = 0; r < 32; r++) {
          const uint32_t c = min(c0 + r, K - 1);
          v[r] = lane < fl ? a.C[static_cast<size_t>(c) * D + f0 + lane] : 0.f;
        }
      };
      load32(0);
      for (int f0 = 0; f0 < D; f0 += 32) {
        const int fl = min(32, D - f0);
#pragma unroll
        for (int r = 0; r < 32; r++) tile[r * 33 + lane] = v[r];
        __syncwarp();
        if (f0 + 32 < D) load32(f0 + 32);
        for (int f = 0; f < fl; f++) {
          const float x = tile[lane * 33 + f];
          k.mac(x, x);
        }
        __syncwarp();
      }
      if (c0 + lane < K) a.csq[c0 + lane] = k.sum;
    }
  }
  prep_grid_barrier(a.barrier, gridDim.x);

  const float* nsq = a.csq;
  if (a.metric == 1) {
    // ---- cosine: upper bound of ||c||^2 per centroid (one warp per row) + its maximum
    uint32_t best = 0;
    for (uint32_t row = gw; row < K; row += nw) {
      const float* src = a.C + static_cast<size_t>(row) * D;
      float acc = 0.f;
      for (int f = lane; f < D; f += 32) {
        float v = src[f];
        acc = fmaf(v, v, acc);
      }
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      const float v = acc * 1.0001f;
      if (lane == 0) a.cnorm2[row] = v;
      if (v == v && v < 3.0e38f) best = max(best, __float_as_uint(fmaxf(v, 0.f)));
    }
    if (lane == 0 && best) atomicMax(&a.stats->csq_max_bits, best);
    nsq = a.cnorm2;
    prep_grid_barrier(a.barrier, gridDim.x);
  } else {
    // ---- phase 1: column sums of the valid centroids (rows whose ||c||^2 is finite), 128 features per half CTA.  ANY
    // vector is a correct choice of mu (scores shift by a per-row constant); the mean minimises the operand norms.
    {
      const int fb = (D + 127) / 128;
      const uint32_t nvb = static_cast<uint32_t>(fb) * ((K + 15u) / 16u);   // 16 rows per half CTA: two load groups deep
      const int ht = tid & 127;
      for (uint32_t vb = blockIdx.x * 2u + (tid >> 7); vb < nvb; vb += gridDim.x * 2u) {
        const int f = static_cast<int>(vb % fb) * 128 + ht;
        const uint32_t r0 = (vb / fb) * 16u, r1 = min(K, r0 + 16u);
        double acc = 0.0;
        uint32_t nv = 0;
        for (uint32_t rb = r0; rb < r1; rb += 8) {
          float v[8], q[8];
#pragma unroll
          for (int j = 0; j < 8; j++) {
            const uint32_t r = min(rb + j, r1 - 1);
            q[j] = __ldcg(a.csq + r);
            v[j] = f < D ? a.C[static_cast<size_t>(r) * D + f] : 0.f;
          }
#pragma unroll
          for (int j = 0; j < 8; j++) {
            if (rb + j >= r1 || !(q[j] == q[j] && q[j] < 3.0e38f)) continue;
            nv++;
            acc += static_cast<double>(v[j]);
          }
        }
        if (f < D && nv) atomicAdd(&a.musum[f], acc);
        if (vb % fb == 0 && ht == 0 && nv) atomicAdd(reinterpret_cast<uint32_t*>(a.musum + D), nv);
      }
    }
    prep_grid_barrier(a.barrier, gridDim.x);
    // ---- phase 2: mu (every CTA keeps its own copy), ||c - mu||^2 per centroid, its maximum
    {
      const uint32_t nv = __ldcg(reinterpret_cast<const uint32_t*>(a.musum + D));
      for (int f = tid; f < D; f += 256) {
        const float m = nv ? static_cast<float>(__ldcg(a.musum + f) / nv) : 0.f;
        s_mu[f] = (fabsf(m) < 3.0e38f) ? m : 0.f;
      }
      __syncthreads();
      uint32_t best = 0;
      for (uint32_t row = gw; row < K; row += nw) {
        const float* src = a.C + static_cast<size_t>(row) * D;
        double acc = 0.0;
        for (int f = lane; f < D; f += 32) {
          const float v = src[f] - s_mu[f];
          acc += static_cast<double>(v) * v;
        }
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        const float q = __ldcg(a.csq + row);
        const float v = (q == q && q < 3.0e38f) ? static_cast<float>(acc) : q;   // dead centroids stay dead
        if (lane == 0) a.cnorm2[row] = v;
        if (v == v && v < 3.0e38f) best = max(best, __float_as_uint(fmaxf(v, 0.f)));
      }
      if (lane == 0 && best) atomicMax(&a.stats->csq_max_bits, best);
    }
    nsq = a.cnorm2;
    prep_grid_barrier(a.barrier, gridDim.x);
  }

  // ---- phase 3: scale (every CTA derives it; CTA 0 publishes Stats and -mu*s), then the fp16 table + bias blocks
  const bool have_mu = a.metric == 0;
  if (warp == 0) {
    float cmax = __fsqrt_ru(__uint_as_float(__ldcg(&a.stats->csq_max_bits)));
    float s = 1.f;
    if (cmax > 0.f && cmax < 3.0e38f) {
      int e;
      frexpf(cmax, &e);
      s = ldexpf(1.f, 6 - e);
    }
    if (lane == 0) s_scale = s;
    if (blockIdx.x == 0) {
      const int Dp = a.nkb * KB;
      float m2 = 0.f;
      for (int f = lane; f < Dp; f += 32) {
        const float m = (have_mu && f < D) ? s_mu[f] : 0.f;
        a.neg_mu_s[f] = -m * s;
        m2 = fmaf(m * s, m * s, m2);
      }
      for (int o = 16; o > 0; o >>= 1) m2 += __shfl_xor_sync(0xffffffffu, m2, o);
      if (lane == 0) {
        a.stats->scale = s;
        a.stats->cmax = cmax * s * 1.001f;
        a.stats->mun = __fsqrt_ru(m2) * 1.002f;
      }
    }
  }
  __syncthreads();
  const float s = s_scale;
  for (uint32_t row = gw; row < a.rows_pad; row += nw)
    prep_table_row(row, lane, s, a.metric, a.C, nsq, K, D, a.nkb, a.table, a.aug_blob, a.stats, a.gather,
                   have_mu ? s_mu : nullptr, a.by_source, a.pair_blob);
}

// ---------------------------------------------------------------------------------------------------
// the main kernel
// ---------------------------------------------------------------------------------------------------
// bars_u32 = shared-space address of bars[0] (computed once per thread)
#define TC_WAIT(bar, parity, site) \
  ptx::mbar_wait(bars_u32 + 8u * static_cast<uint32_t>(bar), (parity), p.counters + CNT_ERR, site, bars_u32 + 8u * 63u)

// the reference's bookkeeping for one decided row (kmeans.cu:356-363); returns 1 if the assignment changed
__device__ __forceinline__ uint32_t commit_assignment(uint32_t* __restrict__ assign, uint32_t* __restrict__ prev,
                                                      uint64_t row, uint32_t winner) {
  const uint32_t a = assign[row];
  prev[row] = a;
  if (a == winner) return 0u;
  assign[row] = winner;
  return 1u;
}

// in-place compaction of one epilogue thread's chunk list: entries whose chunk maximum fell below the
// current threshold can never hold a candidate (the threshold only rises)
__device__ __forceinline__ uint32_t compact_list(uint32_t* lst, uint32_t cnt, float thr) {
  // lst = this thread's column of the entry arrays (stride 256 words per entry, LIST_ARRAY bytes between arrays)
  constexpr uint32_t A = LIST_ARRAY / 4;
  uint32_t w = 0;
  for (uint32_t i = 0; i < cnt; i++) {
    const uint32_t cmb = lst[i * 256];
    if (__uint_as_float(cmb) >= thr) {
      if (w != i) {
        lst[w * 256] = cmb;
        lst[A + w * 256] = lst[A + i * 256];
        lst[2 * A + w * 256] = lst[2 * A + i * 256];
        lst[3 * A + w * 256] = lst[3 * A + i * 256];
      }
      w++;
    }
  }
  return w;
}

// enumerates the n-tiles (blocks of 128 table rows) one sample tile is multiplied with, segment by segment
// (MODE 0 / 1: one segment = the whole table; MODE 2: one segment per candidate cluster)
template <int MODE>
struct BlockIter {
  uint32_t cur, lo, hi, left;    // current block, bounds of the current segment, blocks left including cur
  const uint2* rg;
  __device__ __forceinline__ BlockIter(const Params& p, uint32_t tile) {
    if (MODE == 2) {
      left = p.knn_nblk[tile];
      rg = p.knn_ranges + p.knn_roff[tile];
      if (left) { lo = cur = rg->x; hi = rg->y; } else { lo = cur = hi = 0; }
    } else {
      left = static_cast<uint32_t>(p.nt);
      lo = cur = 0;
      hi = left - 1;
      rg = nullptr;
    }
  }
  __device__ __forceinline__ bool valid() const { return left != 0; }
  __device__ __forceinline__ bool seg_first() const { return cur == lo; }
  __device__ __forceinline__ bool seg_last() const { return cur == hi; }
  __device__ __forceinline__ void next() {
    left--;
    if (MODE != 2) { cur++; return; }   // (keeps the range-list load out of the Lloyd / Yinyang loops: measured 0.65 ms per pass)
    if (cur == hi && left) { rg++; lo = cur = rg->x; hi = rg->y; } else { cur++; }
  }
};

// k-NN epilogue helpers (rare paths, kept out of line): sorted insert into the half-row's descending top-kk column
// in shared memory; returns the new kk-th largest value
__device__ __noinline__ float knn_topk_insert(float* col, int kk, float v) {
  int j = kk - 1;
  while (j > 0 && col[(j - 1) * 256] < v) {
    col[j * 256] = col[(j - 1) * 256];
    j--;
  }
  col[j * 256] = v;
  return col[(kk - 1) * 256];
}
// threshold sweep of the k-NN pass: every half-row keeps 32 running maxima over disjoint column buckets (branch
// free); afterwards the kk largest of the row's 64 buckets (both halves) become the descending top-kk list
__device__ __noinline__ void knn_select_buckets(const float* mine, const float* partner, int kk, float goff,
                                                float* out) {
  unsigned long long taken = 0ull;
  for (int o = 0; o < kk; o++) {
    float best = -INFINITY;
    int bi = -1;
    for (int j = 0; j < 64; j++) {
      const float v = j < 32 ? mine[j * 256] : partner[(j - 32) * 256];
      if (!((taken >> j) & 1ull) && v > best) { best = v; bi = j; }
    }
    if (bi >= 0) taken |= 1ull << bi;
    out[o] = best - goff;
  }
}
// append to the half-row's global entry list; when full, drop the entries that fell below the current kk-th
// best minus their own margin (g-space)
__device__ __noinline__ uint32_t knn_append(uint4* ent, uint32_t cnt, float kth, float cm, uint32_t mask, uint32_t cid,
                                            float margin, uint32_t* flags) {
  if (cnt == KNN_CAP) {
    uint32_t w = 0;
    for (uint32_t i = 0; i < cnt; i++) {
      const uint4 e = ent[i];
      if (__uint_as_float(e.x) >= kth - __uint_as_float(e.w)) ent[w++] = e;
    }
    cnt = w;
    if (cnt == KNN_CAP) { *flags |= 2u; return cnt; }
  }
  ent[cnt] = make_uint4(__float_as_uint(cm), mask, cid, __float_as_uint(margin));
  return cnt + 1;
}

// NKB: K-blocks of 64 features (compile-time: the MMA issue loop must be branch- and address-arithmetic-free); MODE 0 =
// Lloyd assignment, 1 = Yinyang local step, 2 = k-NN, 3 = Yinyang bounds refresh (see Params).
// CG = 2 (MODE 0 only): the kernel runs as clusters of two CTAs (the two SMs of a TPC) and the MMAs are
// tcgen05.mma.cta_group::2 with M = 256: every CTA converts, keeps and post-processes its own 128 sample rows exactly
// as with CG = 1, but stages only HALF of every centroid tile (64 of the 128 rows) in its shared memory; the leader CTA
// (cluster rank 0) issues the MMAs for both and its commits arrive on the barriers of both CTAs.  What it buys: the
// centroid table is streamed L2 -> shared memory once per PAIR of sample tiles (36 GB -> 18 GB per pass at 8M x 256 @
// 1024) and the tensor cores' shared-memory reads per SM halve -- the kernel runs against the board's power limit, and
// that traffic is energy.
template <int NKB, int MODE, int CG = 1>
__global__ void __launch_bounds__(N_THREADS, 1)
tc_assign_kernel(const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_x,
                 const __grid_constant__ CUtensorMap tmap_aug, const Params p) {
  static_assert(CG == 1 || MODE == 0, "CTA pairs are built for the Lloyd assignment pass only");
  constexpr bool PAIR = CG == 2;
  constexpr int BST = PAIR ? B_STAGES_PAIR : B_STAGES;                 // B ring depth
  constexpr uint32_t BSTAGE = PAIR ? B_KB_BYTES / 2 : B_STAGE_BYTES;   // bytes per B stage in this CTA
  const uint32_t cta_rank = PAIR ? ptx::cluster_ctarank() : 0u;
  // 1024-byte alignment (128B-swizzle atoms) by an OFFSET into the shared array: the pointer keeps its shared address
  // space, so every access below is LDS / STS.  (Round 1 aligned through uintptr_t; the compiler then treated
  // `smem` as a generic pointer: all shared traffic went through generic LD / ST and the aligned base was
  // re-derived -- S2R SR_SWINHI, IADD3, LOP3, IMAD.X -- in front of every barrier operation.)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  const SmemLayout L = smem_layout();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  const uint32_t bars_u32 = ptx::smem_u32(bars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L.tmem_slot);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int nkb = NKB;
  constexpr int NBUF = NKB <= 4 ? 2 : 1;   // A operand buffers in TMEM (256 columns are available for A)
  // The error bound needs |x~| (the fp16-rounded operand row) and the rounding residual |a - x~|; the converters MEASURE
  // both.  Round 2 measured bounding them analytically from |a|^2 instead, at 8M x 256 @ 1024: the kernel time did not
  // change (the converters are not on the critical path) while the margin widened and 8.1 % instead of 5.0 % of the
  // rows needed the exact re-check.
  const uint32_t n_eff = MODE == 1 ? min(*p.d_nrows, p.n) : p.n;
  const uint32_t ntiles = MODE == 1 ? (n_eff + TM - 1) / TM : (MODE == 2 ? *p.d_ntiles : p.ntiles);
  // MODE 2 on several GPUs: this device serves the query tiles of part knn_part of knn_nparts (every GPU holds the
  // whole candidate table; tiles are independent)
  uint32_t tile_lo = 0, tile_end = ntiles;
  if (MODE == 2 && p.knn_nparts > 1) {
    tile_lo = static_cast<uint32_t>(static_cast<uint64_t>(ntiles) * p.knn_part / p.knn_nparts);
    tile_end = static_cast<uint32_t>(static_cast<uint64_t>(ntiles) * (p.knn_part + 1) / p.knn_nparts);
  }
  // CTA pairs: consecutive tiles go to the two CTAs of a cluster (gridDim.x is even, cluster rank = blockIdx.x & 1); both
  // CTAs must make the same number of trips, so an odd tile count is rounded up (the phantom tile's rows are out of
  // range: TMA fills zeros, nothing is emitted)
  if (PAIR) tile_end = (tile_end + 1u) & ~1u;
  const uint32_t tile_begin = tile_lo + blockIdx.x;

  if (warp == WARP_B_PRODUCER && lane == 0) {
    bars[63] = 0ull;   // "a wait has given up" flag (mbar_wait_slow)
    ptx::prefetch_tmap(&tmap_b);
    ptx::prefetch_tmap(&tmap_x);
    for (int s = 0; s < X_STAGES; s++) {
      ptx::mbar_init(&bars[BAR_X_FULL + s], 1);
      ptx::mbar_init(&bars[BAR_X_EMPTY + s], N_CONV_WARPS);
    }
    for (int s = 0; s < BST; s++) {
      ptx::mbar_init(&bars[BAR_B_FULL + s], 1);
      ptx::mbar_init(&bars[BAR_B_EMPTY + s], 1);
    }
    for (int s = 0; s < 2; s++) {
      ptx::mbar_init(&bars[BAR_AUG_FULL + s], 1);
      ptx::mbar_init(&bars[BAR_AUG_EMPTY + s], 1);
      ptx::mbar_init(&bars[BAR_ACC_FULL + s], 1);
      ptx::mbar_init(&bars[BAR_ACC_EMPTY + s], N_EPI_WARPS * CG);   // pair: the leader's barrier counts both CTAs' warps
      ptx::mbar_init(&bars[BAR_A_FREE + s], 1);
      ptx::mbar_init(&bars[BAR_EMIT_FULL + s], N_EPI_WARPS);
      ptx::mbar_init(&bars[BAR_EMIT_EMPTY + s], N_EMIT_WARPS);
      for (int kb = 0; kb < MAX_NKB; kb++) ptx::mbar_init(&bars[BAR_A_FULL + s * MAX_NKB + kb], N_CONV_WARPS * CG);
    }
    ptx::fence_mbar_init();
  }
  if (warp == WARP_MMA) {
    if (PAIR) ptx::tmem_alloc_pair(tmem_slot, TMEM_COLS);   // the same warp of both CTAs
    else ptx::tmem_alloc(tmem_slot, TMEM_COLS);
  }
  // constant A-side bias block: ones in the first three K positions of every row
  for (int i = threadIdx.x; i < TM * 16; i += N_THREADS) {
    int r = i >> 4, k = i & 15;
    int j = k >> 3, e = k & 7;
    reinterpret_cast<__half*>(smem + L.aug_a)[(j * (TM * 16) + (r >> 3) * 128 + (r & 7) * 16) / 2 + e] =
        __float2half_rn(k < 3 ? 1.f : 0.f);
  }
  for (int i = threadIdx.x; i < MAX_NKB * KB; i += N_THREADS)
    reinterpret_cast<float*>(smem + L.mu)[i] = (MODE != 2 && p.neg_mu_s && i < nkb * KB) ? p.neg_mu_s[i] : 0.f;
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  if (PAIR) ptx::cluster_sync_all();   // the peer's barriers are initialised before anything arrives on them
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // pair mode: arrivals that the LEADER's MMA thread waits for go to the leader's copy of the barrier
  auto leader_bar = [&](int bar) -> uint32_t { return ptx::mapa_u32(bars_u32 + 8u * static_cast<uint32_t>(bar), 0u); };

  if (warp == WARP_B_PRODUCER) {
    // ================================ TMA producer: centroid table + bias blocks ================================
    if (lane == 0) {
      uint32_t bs = 0, bph = 0, ac = 0;      // B ring stage / phase, bias blocks issued
      for (uint32_t tile = tile_begin; tile < tile_end; tile += gridDim.x) {
        for (BlockIter<MODE> it(p, tile); it.valid(); it.next()) {
          const int n = static_cast<int>(it.cur);
          // the bias block first: it is consumed last, and its buffer was released two n-tiles ago, so the copy is
          // in flight for a whole n-tile before the MMA warp asks for it (round 1 issued it after the B stages and
          // the MMA warp waited for it 17 % of its time)
          const int as = ac & 1;
          const uint32_t aph = (ac >> 1) & 1;
          TC_WAIT(BAR_AUG_EMPTY + as, aph ^ 1, 2);
          if (PAIR) {
            // this CTA's half of the bias block (2 KiB, rows rank*64 ..) ; the leader's barrier counts both halves
            if (cta_rank == 0) ptx::mbar_arrive_expect_tx(&bars[BAR_AUG_FULL + as], AUG_B_BYTES);
            ptx::tma_load_2d_pair(ptx::smem_u32(smem + L.aug_b + as * AUG_B_BYTES), &tmap_aug, 0,
                                  (n * 2 + static_cast<int>(cta_rank)) * 2, leader_bar(BAR_AUG_FULL + as));
          } else {
            ptx::mbar_arrive_expect_tx(&bars[BAR_AUG_FULL + as], AUG_B_BYTES);
            ptx::bulk_load(smem + L.aug_b + as * AUG_B_BYTES,
                           reinterpret_cast<const uint8_t*>(p.aug_blob) + static_cast<size_t>(n) * AUG_B_BYTES,
                           AUG_B_BYTES, &bars[BAR_AUG_FULL + as]);
          }
          ac++;
#pragma unroll
          for (int kb = 0; kb < NKB; kb++) {
            TC_WAIT(BAR_B_EMPTY + bs, bph ^ 1, 1);
            if (PAIR) {
              if (cta_rank == 0) ptx::mbar_arrive_expect_tx(&bars[BAR_B_FULL + bs], B_KB_BYTES);   // both halves
              ptx::tma_load_2d_pair(ptx::smem_u32(smem + L.b + bs * BSTAGE), &tmap_b, kb * KB,
                                    n * TN + static_cast<int>(cta_rank) * (TN / 2), leader_bar(BAR_B_FULL + bs));
            } else {
              ptx::mbar_arrive_expect_tx(&bars[BAR_B_FULL + bs], B_KB_BYTES);
              ptx::tma_load_2d(smem + L.b + bs * B_STAGE_BYTES, &tmap_b, kb * KB, n * TN, &bars[BAR_B_FULL + bs]);
            }
            if (++bs == BST) { bs = 0; bph ^= 1; }
          }
        }
      }
    }
  } else if (warp == WARP_X_PRODUCER) {
    // ================================ TMA producer: fp32 sample rows ================================
    if ((MODE == 0 || MODE == 3) && lane == 0) {
      uint32_t xc = 0;
      for (uint32_t tile = tile_begin; tile < tile_end; tile += gridDim.x) {
        for (int hs = 0; hs < 2 * nkb; hs++, xc++) {
          const int s = xc % X_STAGES;
          const uint32_t ph = (xc / X_STAGES) & 1;
          TC_WAIT(BAR_X_EMPTY + s, ph ^ 1, 9);
          ptx::mbar_arrive_expect_tx(&bars[BAR_X_FULL + s], X_STAGE_BYTES);
          ptx::tma_load_2d(smem + L.x + s * X_STAGE_BYTES, &tmap_x, hs * 32, static_cast<int>(tile * TM),
                           &bars[BAR_X_FULL + s]);
        }
      }
    }
  } else if (warp == WARP_MMA) {
    // ================================ MMA issuer ================================
    // ONE thread runs the whole role (tcgen05.mma / commit are single-thread instructions): no election, no
    // reconvergence points, no warp-wide barrier probes.  ncu of the previous version (whole warp + elect per K-block,
    // profiles/r02_tc_assign_v6_*): ~330 SASS instructions per n-tile at ~6 cycles each = ~2000 cycles to issue 1088
    // cycles of tensor work -- the issuer, not the tensor pipe, paced the kernel.  Descriptors are built once; a K-block
    // is one asm statement (4 MMAs + commit).
    // CTA pairs: only the leader issues (M = 256 covers both CTAs' rows); its commits are multicast to both CTAs.
    if ((!PAIR || cta_rank == 0) && ptx::elect_one()) {   // (elect.sync, not `lane == 0`: ptxas then keeps the operands in
                              // uniform registers instead of wrapping every tcgen05 instruction in a per-lane R2UR.BROADCAST loop)
      const uint32_t idesc = ptx::make_idesc_f16(TM * CG, TN);
      const uint64_t bdesc0 = ptx::make_smem_desc(ptx::smem_u32(smem + L.b), 16, 1024, 2);
      const uint64_t aug_ad = ptx::make_smem_desc(ptx::smem_u32(smem + L.aug_a), TM * 16, 128, 0);
      // B-side bias block: (TN / CG) rows x 16 K in this CTA; the second K half lies rows * 16 bytes further
      const uint64_t aug_bd0 = ptx::make_smem_desc(ptx::smem_u32(smem + L.aug_b), (TN / CG) * 16, 128, 0);
      auto commit = [&](int bar) {
        if (PAIR) ptx::umma_commit_pair(bars_u32 + 8u * static_cast<uint32_t>(bar));
        else ptx::umma_commit_u32(bars_u32 + 8u * static_cast<uint32_t>(bar));
      };
      uint32_t bs = 0, bph = 0, ac = 0, si = 0;             // B ring stage / phase; n-tiles; segments (= A conversions) so far
      uint32_t a_ready_si = 0xFFFFFFFFu;                    // segment whose A operand has already been waited for
      for (uint32_t tile = tile_begin; tile < tile_end; tile += gridDim.x) {
        if (MODE == 2 && p.knn_nblk[tile] == 0) continue;   // nothing to visit: every role skips the tile
        for (BlockIter<MODE> it(p, tile); it.valid(); it.next(), ac++) {
          const uint32_t abuf = si % NBUF;
          const uint32_t a_par = (si / NBUF) & 1;
          const uint32_t buf = ac & 1;
          const uint32_t aph = (ac >> 1) & 1;
          const bool need_a = a_ready_si != si;             // first n-tile of this segment
          a_ready_si = si;
          const uint32_t a_tmem = tmem_base + TMEM_A0 + abuf * 128;
          const uint32_t d_tmem = tmem_base + TMEM_ACC0 + buf * TN;
          TC_WAIT(BAR_ACC_EMPTY + buf, aph ^ 1, 3);
          uint32_t s_ = bs, ph_ = bph;
#pragma unroll
          for (int kb = 0; kb < NKB; kb++) {
            if (need_a) TC_WAIT(BAR_A_FULL + abuf * MAX_NKB + kb, a_par, 4);
            TC_WAIT(BAR_B_FULL + s_, ph_, 5);
            ptx::tc_fence_after();
            if (PAIR)
              ptx::umma_f16_ts_kblock_pair(d_tmem, a_tmem + kb * 32, bdesc0 + s_ * (BSTAGE >> 4), idesc, kb ? 1u : 0u,
                                           bars_u32 + 8u * (BAR_B_EMPTY + s_));
            else
              ptx::umma_f16_ts_kblock(d_tmem, a_tmem + kb * 32, bdesc0 + s_ * (BSTAGE >> 4), idesc, kb ? 1u : 0u,
                                      bars_u32 + 8u * (BAR_B_EMPTY + s_));
            if (++s_ == BST) { s_ = 0; ph_ ^= 1; }
          }
          // bias step: acc += ones(128x16) * bias(128x16)^T  (both operands no-swizzle K-major smem blocks)
          TC_WAIT(BAR_AUG_FULL + buf, aph, 6);
          ptx::tc_fence_after();
          if (PAIR) ptx::umma_f16_pair(d_tmem, aug_ad, aug_bd0 + buf * (AUG_B_BYTES >> 4), idesc, 1u);
          else ptx::umma_f16(d_tmem, aug_ad, aug_bd0 + buf * (AUG_B_BYTES >> 4), idesc, 1u);
          commit(BAR_AUG_EMPTY + buf);
          commit(BAR_ACC_FULL + buf);
          bs += NKB;
          while (bs >= static_cast<uint32_t>(BST)) { bs -= BST; bph ^= 1; }
          if (it.seg_last()) {
            commit(BAR_A_FREE + abuf);   // the A buffer of this segment is free once its MMAs have retired
            si++;
          }
        }
      }
    }
  } else if (warp >= FIRST_CONV_WARP && warp < FIRST_CONV_WARP + N_CONV_WARPS) {
    // ================================ converters: fp32 smem stage -> fp16 A operand in TMEM ================================
    const int q = warp & 3;                 // TMEM lane quarter
    const int row = q * 32 + lane;          // this thread's sample row within the tile
    const float s = p.stats->scale;
    uint32_t xc = 0, si = 0;
    for (uint32_t tile = tile_begin; tile < tile_end; tile += gridDim.x) {
      if (MODE == 2 && p.knn_nblk[tile] == 0) continue;
      const float* xrow = nullptr;
      if (MODE == 1) {
        const uint32_t li = min(tile * TM + row, n_eff - 1);   // ragged tail: repeat the last listed row
        xrow = p.X + static_cast<size_t>(p.rows[li]) * p.D;
      }
      if (MODE == 2)   // padding rows of the table repeat sample 0; they are never recorded
        xrow = p.X + static_cast<size_t>(min(p.rows[tile * TM + row], p.n - 1)) * p.D;
      const uint32_t nseg = MODE == 2 ? p.knn_rcount[tile] : 1u;
      for (uint32_t seg = 0; seg < nseg; seg++, si++) {
        const int abuf = si % NBUF;
        TC_WAIT(BAR_A_FREE + abuf, ((si / NBUF) & 1) ^ 1, 7);   // MMAs of the previous user of this buffer are done
        ptx::tc_fence_after();
        // ||x~||^2 and ||s(x - mu) - x~||^2 as packed even/odd partial sums (FFMA2: two fp32 FMAs per issue slot)
        uint64_t nx2 = 0ull, nd2 = 0ull;
        const uint64_t s2 = ptx::pack2(s, s);
        const float* mu = reinterpret_cast<const float*>(smem + L.mu);
        float a2 = 0.f, a2c = 0.f, nraw = 0.f;     // MODE 2: Kahan sum of the exact (x-c)^2 s^2, and s^2 (|x|+|c|)^2
        const float* crow = nullptr;
        if (MODE == 2) crow = p.C + static_cast<size_t>(p.blk_cluster[p.knn_ranges[p.knn_roff[tile] + seg].x]) * p.D;
        for (int kb = 0; kb < nkb; kb++) {
          uint32_t pk[32];
#pragma unroll
          for (int half = 0; half < 2; half++, xc++) {
            const int st = xc % X_STAGES;
            const uint32_t ph = (xc / X_STAGES) & 1;
            float4 gv[8];
            const int f0 = kb * KB + half * 32;
            if (MODE == 0 || MODE == 3) {
              TC_WAIT(BAR_X_FULL + st, ph, 10);
            } else {
#pragma unroll
              for (int c = 0; c < 8; c++)
                gv[c] = (f0 + c * 4 < p.D) ? ptx::ldg_nc_f4(xrow + f0 + c * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            const uint8_t* xs = smem + L.x + st * X_STAGE_BYTES + row * 128;
#pragma unroll
            for (int c = 0; c < 8; c++) {
              float4 v = (MODE == 0 || MODE == 3) ? *reinterpret_cast<const float4*>(xs + ((c ^ (row & 7)) << 4)) : gv[c];
              float4 m4 = make_float4(0.f, 0.f, 0.f, 0.f);
              if (MODE == 2) {
                const float4 cv = (f0 + c * 4 < p.D) ? ptx::ldg_nc_f4(crow + f0 + c * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                const float r0 = fabsf(v.x) + fabsf(cv.x), r1 = fabsf(v.y) + fabsf(cv.y);
                const float r2 = fabsf(v.z) + fabsf(cv.z), r3 = fabsf(v.w) + fabsf(cv.w);
                nraw = fmaf(r0, r0, nraw); nraw = fmaf(r1, r1, nraw); nraw = fmaf(r2, r2, nraw); nraw = fmaf(r3, r3, nraw);
                v.x -= cv.x; v.y -= cv.y; v.z -= cv.z; v.w -= cv.w;
              } else {
                m4 = *reinterpret_cast<const float4*>(mu + f0 + c * 4);   // same address in every lane: broadcast
              }
              // a = s*v - s*mu in ONE rounding (s is a power of two, so this is exactly s * fl(v - mu))
              const uint64_t a01 = ptx::ffma2(ptx::pack2(v.x, v.y), s2, ptx::pack2(m4.x, m4.y));
              const uint64_t a23 = ptx::ffma2(ptx::pack2(v.z, v.w), s2, ptx::pack2(m4.z, m4.w));
              float a0, a1, a2_, a3;
              ptx::unpack2(a01, a0, a1);
              ptx::unpack2(a23, a2_, a3);
              __half2 h0 = __floats2half2_rn(a0, a1), h1 = __floats2half2_rn(a2_, a3);
              const float2 b0 = __half22float2(h0), b1 = __half22float2(h1);
              const uint64_t b01 = ptx::pack2(b0.x, b0.y), b23 = ptx::pack2(b1.x, b1.y);
              nx2 = ptx::ffma2(b01, b01, nx2);
              nx2 = ptx::ffma2(b23, b23, nx2);
              const uint64_t d01 = ptx::fsub2(a01, b01), d23 = ptx::fsub2(a23, b23);
              nd2 = ptx::ffma2(d01, d01, nd2);
              nd2 = ptx::ffma2(d23, d23, nd2);
              if (MODE == 2) {   // compensated: this sum is subtracted from scores of the same magnitude
                const float q4 = fmaf(a0, a0, fmaf(a1, a1, fmaf(a2_, a2_, a3 * a3)));
                const float y = q4 - a2c, t = a2 + y;
                a2c = (t - a2) - y;
                a2 = t;
              }
              pk[half * 16 + c * 2] = *reinterpret_cast<uint32_t*>(&h0);
              pk[half * 16 + c * 2 + 1] = *reinterpret_cast<uint32_t*>(&h1);
            }
            if (MODE == 0 || MODE == 3) {
              __syncwarp();
              if (lane == 0) ptx::mbar_arrive(&bars[BAR_X_EMPTY + st]);
            }
          }
          ptx::tmem_st_32x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + TMEM_A0 + abuf * 128 + kb * 32, pk);
          ptx::tmem_st_wait();
          if (kb == nkb - 1) {
            float* norms = reinterpret_cast<float*>(smem + L.norms) + (si & 3) * 4 * TM;
            float nxl, nxh, ndl, ndh;
            ptx::unpack2(nx2, nxl, nxh);
            ptx::unpack2(nd2, ndl, ndh);
            norms[row] = nxl + nxh;
            norms[TM + row] = ndl + ndh;
            if (MODE == 2) {
              norms[2 * TM + row] = a2;
              norms[3 * TM + row] = nraw * s * s;
            }
          }
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (PAIR) ptx::mbar_arrive_cluster(leader_bar(BAR_A_FULL + abuf * MAX_NKB + kb));
            else ptx::mbar_arrive(&bars[BAR_A_FULL + abuf * MAX_NKB + kb]);
          }
        }
      }
    }
  } else if (warp >= FIRST_EPI_WARP && warp < FIRST_EPI_WARP + N_EPI_WARPS) {
    // ================================ epilogue ================================
    const int e = warp - FIRST_EPI_WARP;       // 0..7
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    const int h = e >> 2;                      // column half of every 128-column accumulator
    const int row = q * 32 + lane;
    const int slot = h * TM + row;             // 0..255
    const float cmax = p.stats->cmax, dcmax = p.stats->dcmax;
    const float mun = MODE == 2 ? 0.f : p.stats->mun;
    const float knn_extra = MODE == 2 ? p.stats->knn_extra : 0.f;
    // cosine: every dot >= 1 is clamped to angle 0 by the reference, so all of them tie -> the threshold
    // never rises above s^2 * 1 (the accumulator holds s^2 * dot)
    const float cap = p.metric == 1 ? p.stats->scale * p.stats->scale : INFINITY;
    uint32_t ac = 0, ti = 0, si = 0;
    for (uint32_t tile = tile_begin; tile < tile_end; tile += gridDim.x) {
      if (MODE == 2 && p.knn_nblk[tile] == 0) continue;
      const int par = ti & 1;
      uint32_t* lst = reinterpret_cast<uint32_t*>(smem + L.list) + par * LIST_LEN * 256 + slot;   // this thread's entries
      float* fin = reinterpret_cast<float*>(smem + L.fin) + par * 5 * 256;
      // the emitter warps must have consumed this parity's lists (tile ti-2)
      if (MODE < 2) TC_WAIT(BAR_EMIT_EMPTY + par, ((ti >> 1) & 1) ^ 1, 11);
      float M = -INFINITY, M2 = -INFINITY, margin = 0.f;   // M2: MODE 1, second largest chunk maximum
      uint32_t cnt = 0, flags = 0;
      // MODE 2: this half-row's persistent state (global) and its top-kk column (the list_cm region is free)
      float* topk = reinterpret_cast<float*>(smem + L.list) + slot;   // [kk][256], kk <= 16 rows of the scratch
      uint32_t kslot = 0;
      bool klive = false;
      uint4* kent = nullptr;
      float goff = 0.f, mmax = 0.f;     // MODE 2: s^2 |x - c_B|^2 / 2 of the current segment; largest margin so far
      // MODE 3: this row's record, own group (handled exactly elsewhere), lower bound of |s (x - mu)|^2
      float xa2lo = 0.f;
      uint32_t gown = UINT32_MAX;
      uint32_t* yb = nullptr;
      bool ylive = false;
      if (MODE == 3) {
        const uint64_t grow = static_cast<uint64_t>(tile) * TM + row;
        ylive = grow < p.n;
        if (ylive) {
          const uint32_t a = p.yy_assign[grow];
          if (a < p.K) gown = p.yy_groups[a];
          yb = reinterpret_cast<uint32_t*>(p.yy_bounds + grow * (p.G + 1) + 1);
        }
      }
      uint32_t seg = 0;
      if (MODE == 2) {
        klive = static_cast<uint32_t>(row) < p.tile_nrows[tile];
        kslot = (tile * TM + row) * 2u + h;
        kent = p.knn_entries + static_cast<size_t>(kslot) * KNN_CAP;
        if (p.knn_first_pass || !klive) {
          for (int j = 0; j < p.kk; j++) topk[j * 256] = -INFINITY;
          if (p.knn_first_pass)
            for (int j = 0; j < 32; j++) topk[(16 + j) * 256] = -INFINITY;   // bucket maxima: rows 16..47 of the region
        } else {
          // second pass: both halves saved the same merged list at the end of the first pass (no insertion happens
          // in the recording sweep); from here on each half adds its own, disjoint, columns
          for (int j = 0; j < p.kk; j++) topk[j * 256] = p.knn_topk[static_cast<size_t>(j) * p.knn_stride + kslot];
          cnt = p.knn_cnt[kslot];
          flags = p.knn_flags[kslot];
        }
        M = topk[(p.kk - 1) * 256];                 // MODE 2: M holds the kk-th largest group maximum (g-space)
      }
      for (BlockIter<MODE> it(p, tile); it.valid(); it.next(), ac++) {
        const int n = static_cast<int>(it.cur);
        const int buf = ac & 1;
        const uint32_t aph = (ac >> 1) & 1;
        TC_WAIT(BAR_ACC_FULL + buf, aph, 8);
        ptx::tc_fence_after();
        // both 32-column chunks of this warp are fetched up front so that their dependency chains interleave
        uint32_t r0[32], r1[32];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + TMEM_ACC0 + buf * TN + h * 64;
        ptx::tmem_ld_32x32(taddr, r0);
        ptx::tmem_ld_32x32(taddr + 32, r1);
        if (it.seg_first()) {
          const float* norms = reinterpret_cast<const float*>(smem + L.norms) + (si & 3) * 4 * TM;
          // rigorous bound on |acc - (s^2 x.c - s^2||c||^2/2)| (see header): Cauchy-Schwarz on the
          // actual rounding residuals + accumulation + the reference's own rounding slack
          const float nx = __fsqrt_ru(norms[row]) * 1.0001f;
          const float nd = __fsqrt_ru(norms[TM + row]) * 1.0001f;
          const float xn = nx + nd;
          float E = nx * dcmax + nd * cmax + nd * dcmax;
          E += static_cast<float>(p.nkb * KB + 16) * 2.4e-7f * nx * cmax;   // fp32 accumulation in the tensor core
          // reference Kahan/rd rounding + bias split + fp32 centring of both operands: the reference works on the
          // UNCENTRED vectors, whose norms are bounded by the centred ones + ||mu||
          const float xu = xn + mun, cu = cmax + mun;
          if (MODE == 0) {
            // the reference ranks with fma_rd(-2, Kahan dot, csq): |error| <= 1.2e-7 cu^2 + 2.4e-7 xu cu in score units
            // (2^-23 per directed rounding, Kahan sums to ~1 ulp); 2.5x - 5x of that is allowed for
            E += 6.0e-7f * (cu * cu + xu * cu);
          } else if (MODE == 2) {
            E += 2.0e-6f * (cu * cu + xu * cu) + 2.0e-6f * xu * xu;
          } else {
            // MODE 1 / 3 decide on TRUE distances sqrt(Kahan sum (x - c)^2): their rounding is relative to |x - c|^2 <=
            // (|x^| + |c^|)^2 (the subtraction cancels the common offset exactly), plus the fp32 centring of both operands
            E += 2.0e-6f * (xn + cmax) * (xn + cmax) + 2.4e-7f * (xn * cmax + cmax * cmax);
          }
          if (MODE == 3) {
            xa2lo = norms[row] * (1.f - 1.0e-4f);                          // lower bound of |s (x - mu)|^2 (fp32 summation error)
            // scores this low are not separable from the padding sentinel (-65504): such rows take the exact pass
            if (!(nx * cmax < 6.0e4f)) flags |= 1u;
          }
          if (MODE == 2) {
            goff = 0.5f * norms[2 * TM + row];
            // centring x - c_B and y - c_B rounds in fp32 (relative to |x|+|c|), and the row constant is subtracted
            // from scores of its own magnitude
            E += 1.2e-7f * (__fsqrt_ru(norms[3 * TM + row]) * cmax + p.stats->yabs * xn) + 4.8e-7f * (goff + xn * cmax);
          }
          margin = 2.f * E * 1.001f + 1e-30f;
          if (MODE == 2) margin += knn_extra;
          if (!(margin < 1.0e30f)) flags |= 1u;                            // NaN / Inf somewhere in the row
          if (MODE == 2) {
            mmax = fmaxf(mmax, margin);
            if (p.knn_first_pass && seg == 1) {
              // threshold sweep done: both column halves of the row adopt the merged top-kk (the partner warp
              // e ^ 4 sits on the same row quarter); named barrier per quarter, 64 threads
              float mg[KNN_MAX_KK];
              asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
              knn_select_buckets(topk + 16 * 256, reinterpret_cast<float*>(smem + L.list) + ((1 - h) * TM + row) + 16 * 256,
                                 p.kk, goff, mg);
              asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
              for (int j = 0; j < p.kk; j++) topk[j * 256] = mg[j];
              M = mg[p.kk - 1];
            }
          }
        }
        ptx::tmem_ld_wait();
        // the accumulator values are in registers: hand the TMEM buffer back to the MMA warp right away
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) ptx::mbar_arrive_cluster(leader_bar(BAR_ACC_EMPTY + buf));
          else ptx::mbar_arrive(&bars[BAR_ACC_EMPTY + buf]);
        }
        if (MODE == 3) {
          // quad maxima (2 instructions per 4 columns), folded into per-group maxima along the (warp-uniform) group ids
          // of this 64-column half; every finished group turns into a lower bound of the distance
          float qm[16];
#pragma unroll
          for (int i = 0; i < 8; i++) {
            qm[i] = fmaxf(ptx::fmax3(__uint_as_float(r0[4 * i]), __uint_as_float(r0[4 * i + 1]), __uint_as_float(r0[4 * i + 2])),
                          __uint_as_float(r0[4 * i + 3]));
            qm[8 + i] = fmaxf(ptx::fmax3(__uint_as_float(r1[4 * i]), __uint_as_float(r1[4 * i + 1]), __uint_as_float(r1[4 * i + 2])),
                              __uint_as_float(r1[4 * i + 3]));
          }
          uint32_t gq[16];
          {
            const uint4* src = reinterpret_cast<const uint4*>(p.yy_qgroup) + (static_cast<size_t>(n) * 2 + h) * 4;
#pragma unroll
            for (int i = 0; i < 4; i++) {
              const uint4 v = __ldg(src + i);
              gq[4 * i] = v.x; gq[4 * i + 1] = v.y; gq[4 * i + 2] = v.z; gq[4 * i + 3] = v.w;
            }
          }
          const float Eb = 0.5f * margin;                       // >= E
          const float sc = p.stats->scale;
          const float inv_s = 1.f / sc, inv_s2 = inv_s * inv_s;   // s is a power of two: exact
          const bool emit_ok = ylive && !(flags & 1u);
          float run = qm[0];
#pragma unroll
          for (int i = 1; i <= 16; i++) {
            if (i == 16 || gq[i] != gq[i - 1]) {                // warp-uniform: the table layout is the same for every row
              const uint32_t g = gq[i - 1];
              if (emit_ok && g < p.G && g != gown) {
                float v;
                if (p.metric == 1) {
                  // angular: every dot of the group <= (run + E) / s^2; acos is decreasing; libdevice acosf is good to 2 ulp
                  const float dot = fminf(1.f, fmaxf(-1.f, (run + Eb) * inv_s2));
                  v = fmaxf(0.f, acosf(dot) - 4.0e-6f);
                } else {
                  // L2: s^2 d^2 = |x^|^2 - 2 score  >=  |x^|^2 - 2 (run + E)
                  const float t = xa2lo - 2.f * (run + Eb);
                  v = t > 0.f ? __fsqrt_rd(t) * inv_s * (1.f - 4.0e-6f) : 0.f;
                }
                atomicMin(yb + g, __float_as_uint(v));        // bounds are >= +0: ordered like unsigned integers
              }
              if (i < 16) run = qm[i];
            } else {
              run = fmaxf(run, qm[i]);
            }
          }
          if (it.seg_last()) si++;
          continue;
        }
        // chunk maxima with three-input maxima (FMNMX3): 16 instructions per 32 columns
        float t0[8], t1[8];      // MODE 2 only: maxima of the 4-column groups
        float cm0, cm1;
        if (MODE == 2) {
#pragma unroll
          for (int i = 0; i < 8; i++) {
            t0[i] = fmaxf(fmaxf(__uint_as_float(r0[4 * i]), __uint_as_float(r0[4 * i + 1])),
                          fmaxf(__uint_as_float(r0[4 * i + 2]), __uint_as_float(r0[4 * i + 3])));
            t1[i] = fmaxf(fmaxf(__uint_as_float(r1[4 * i]), __uint_as_float(r1[4 * i + 1])),
                          fmaxf(__uint_as_float(r1[4 * i + 2]), __uint_as_float(r1[4 * i + 3])));
          }
          cm0 = fmaxf(fmaxf(fmaxf(t0[0], t0[1]), fmaxf(t0[2], t0[3])), fmaxf(fmaxf(t0[4], t0[5]), fmaxf(t0[6], t0[7])));
          cm1 = fmaxf(fmaxf(fmaxf(t1[0], t1[1]), fmaxf(t1[2], t1[3])), fmaxf(fmaxf(t1[4], t1[5]), fmaxf(t1[6], t1[7])));
        } else {
          float u0[10], u1[10];
#pragma unroll
          for (int i = 0; i < 10; i++) {
            u0[i] = ptx::fmax3(__uint_as_float(r0[3 * i]), __uint_as_float(r0[3 * i + 1]), __uint_as_float(r0[3 * i + 2]));
            u1[i] = ptx::fmax3(__uint_as_float(r1[3 * i]), __uint_as_float(r1[3 * i + 1]), __uint_as_float(r1[3 * i + 2]));
          }
          const float w00 = ptx::fmax3(u0[0], u0[1], u0[2]), w01 = ptx::fmax3(u0[3], u0[4], u0[5]);
          const float w02 = ptx::fmax3(u0[6], u0[7], u0[8]), w03 = ptx::fmax3(u0[9], __uint_as_float(r0[30]), __uint_as_float(r0[31]));
          const float w10 = ptx::fmax3(u1[0], u1[1], u1[2]), w11 = ptx::fmax3(u1[3], u1[4], u1[5]);
          const float w12 = ptx::fmax3(u1[6], u1[7], u1[8]), w13 = ptx::fmax3(u1[9], __uint_as_float(r1[30]), __uint_as_float(r1[31]));
          cm0 = fmaxf(ptx::fmax3(w00, w01, w02), w03);
          cm1 = fmaxf(ptx::fmax3(w10, w11, w12), w13);
        }
        float thr;
        if (MODE == 0) {
          M = fmaxf(M, fmaxf(cm0, cm1));
          thr = fminf(M, cap) - margin;
        } else if (MODE == 1) {
          // two distinct columns reach min(two largest chunk maxima): a lower bound of the second best score
          M2 = fmaxf(M2, fminf(M, cm0));
          M = fmaxf(M, cm0);
          M2 = fmaxf(M2, fminf(M, cm1));
          M = fmaxf(M, cm1);
          thr = fminf(M2, cap) - margin;
        } else {
          // kk distinct columns reach the kk-th largest 4-column-group maximum (first level of the max tree): a
          // lower bound of the kk-th best score; finer than whole chunks because near neighbours sit close together
          // in the table.  M and the list live in g-space (score - goff).
          if (p.knn_first_pass && seg == 0) {
            // threshold sweep: bucket (block parity, 4-column group) <- max; raw scores, the row constant is
            // subtracted once at the end of the sweep
            float* bk = topk + (16 + 16 * (n & 1)) * 256;
#pragma unroll
            for (int i = 0; i < 8; i++) {
              bk[i * 256] = fmaxf(bk[i * 256], t0[i]);
              bk[(8 + i) * 256] = fmaxf(bk[(8 + i) * 256], t1[i]);
            }
          } else if (!p.knn_first_pass) {
            const float lim = M + goff;
            if (cm0 > lim) {
#pragma unroll
              for (int i = 0; i < 8; i++)
                if (t0[i] - goff > M) M = knn_topk_insert(topk, p.kk, t0[i] - goff);
            }
            if (cm1 > lim) {
#pragma unroll
              for (int i = 0; i < 8; i++)
                if (t1[i] - goff > M) M = knn_topk_insert(topk, p.kk, t1[i] - goff);
            }
          }
          thr = (M - margin) + goff;
        }
        // candidate masks: d_j = v_j - thr as packed pairs (FADD2), then the sign bits are shifted into a mask with
        // one funnel shift per column: 1.5 issue slots per accumulator element (round 1: 2.4 -- two FFMAs per
        // element plus conversions).  NaN scores only occur in rows whose margin is not finite (flag 1).
        uint32_t nc0, nc1;
        {
          const uint64_t nthr2 = ptx::pack2(-thr, -thr);
          uint32_t c00 = 0, c01 = 0, c10 = 0, c11 = 0;   // two 16-column chains per chunk (shorter dependency chains)
#pragma unroll
          for (int jj = 0; jj < 32; jj += 2) {
            float x0, y0, x1, y1;
            ptx::unpack2(ptx::fadd2(ptx::pack2(__uint_as_float(r0[jj]), __uint_as_float(r0[jj + 1])), nthr2), x0, y0);
            ptx::unpack2(ptx::fadd2(ptx::pack2(__uint_as_float(r1[jj]), __uint_as_float(r1[jj + 1])), nthr2), x1, y1);
            if (jj < 16) {
              c00 = __funnelshift_l(__float_as_uint(x0), c00, 1);
              c00 = __funnelshift_l(__float_as_uint(y0), c00, 1);
              c10 = __funnelshift_l(__float_as_uint(x1), c10, 1);
              c10 = __funnelshift_l(__float_as_uint(y1), c10, 1);
            } else {
              c01 = __funnelshift_l(__float_as_uint(x0), c01, 1);
              c01 = __funnelshift_l(__float_as_uint(y0), c01, 1);
              c11 = __funnelshift_l(__float_as_uint(x1), c11, 1);
              c11 = __funnelshift_l(__float_as_uint(y1), c11, 1);
            }
          }
          // bit (31 - j) of (c?0 << 16 | c?1) = sign of d_j = "column j is below the threshold"
          nc0 = (c00 << 16) | c01;
          nc1 = (c10 << 16) | c11;
        }
        const uint32_t mask0 = __brev(~nc0), mask1 = __brev(~nc1);
        if (MODE == 2) {
          if (klive && !(p.knn_first_pass && seg == 0)) {
            if (mask0)
              cnt = knn_append(kent, cnt, M, cm0 - goff, mask0, static_cast<uint32_t>(n) * 4 + h * 2, margin, &flags);
            if (mask1)
              cnt = knn_append(kent, cnt, M, cm1 - goff, mask1, static_cast<uint32_t>(n) * 4 + h * 2 + 1, margin, &flags);
          }
          if (it.seg_last()) { si++; seg++; }
          continue;
        }
        if (it.seg_last()) si++;
        // one entry per n-tile that holds a candidate in this thread's 64 columns (round 2 v7: one per 32-column chunk,
        // two divergent append blocks per n-tile)
        if (mask0 | mask1) {
          constexpr uint32_t A = LIST_ARRAY / 4;
          if (cnt >= LIST_LEN - 1) cnt = compact_list(lst, cnt, thr);   // rare: drop entries below the risen threshold
          if (cnt < LIST_LEN) {
            lst[cnt * 256] = __float_as_uint(fmaxf(cm0, cm1));
            lst[A + cnt * 256] = mask0;
            lst[2 * A + cnt * 256] = mask1;
            lst[3 * A + cnt * 256] = static_cast<uint32_t>(n);
            cnt++;
          } else {
            flags |= 2u;
          }
        }
      }
      if (MODE == 2) {
        if (klive) {
          for (int j = 0; j < p.kk; j++) p.knn_topk[static_cast<size_t>(j) * p.knn_stride + kslot] = topk[j * 256];
          p.knn_cnt[kslot] = cnt;
          p.knn_flags[kslot] = flags;
          // exact distance to the kk-th nearest candidate seen so far, upper bound in the caller's units:
          // every recorded score is within its margin of g = -s^2 d^2 / 2
          const float sc = p.stats->scale;
          const float d2 = fmaxf(0.f, -2.f * (M - mmax));
          p.knn_dub[kslot] = (M > -INFINITY && !flags) ? __fsqrt_ru(d2) / sc * 1.0001f : INFINITY;
        }
        ti++;
        continue;
      }
      if (MODE == 3) {
        // rows the filter cannot bound (non-finite data, scores beyond the sentinel range): exact refresh of the row
        if (ylive && (flags & 1u) && h == 0)
          p.ovf_rows[atomicAdd(&p.counters[CNT_OVF], 1u)] = static_cast<uint32_t>(tile * TM + row);
        ti++;
        continue;
      }
      // publish this half-row's state; the emitter warps merge the halves and write the results
      fin[slot] = M;
      reinterpret_cast<uint32_t*>(fin)[256 + slot] = cnt;
      reinterpret_cast<uint32_t*>(fin)[512 + slot] = flags;
      fin[768 + slot] = margin;
      if (MODE == 1) fin[1024 + slot] = M2;
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars[BAR_EMIT_FULL + par]);
      ti++;
    }
  } else if (warp >= FIRST_EMIT_WARP && warp < FIRST_EMIT_WARP + N_EMIT_WARPS && MODE < 2) {
    // ================================ emitters: merge column halves, write results / queues ================================
    const int row = (warp - FIRST_EMIT_WARP) * 32 + lane;
    const float cap = p.metric == 1 ? p.stats->scale * p.stats->scale : INFINITY;
    const uint32_t force = p.stats->force_exact ? 16u : 0u;
    uint32_t ti = 0, nchanged = 0;
    for (uint32_t tile = tile_begin; tile < tile_end; tile += gridDim.x, ti++) {
      const int par = ti & 1;
      const uint32_t* lst = reinterpret_cast<const uint32_t*>(smem + L.list) + par * LIST_LEN * 256;
      const float* fin = reinterpret_cast<const float*>(smem + L.fin) + par * 5 * 256;
      const uint32_t* finu = reinterpret_cast<const uint32_t*>(fin);
      TC_WAIT(BAR_EMIT_FULL + par, (ti >> 1) & 1, 12);
      uint64_t grow = static_cast<uint64_t>(tile) * TM + row;
      uint32_t cand[MAX_CAND];
      uint32_t total = 0, fl = 0;
      const bool live = grow < n_eff;
      if (MODE == 1 && live) grow = p.rows[grow];
      if (live) {
        float Mf = fmaxf(fin[row], fin[TM + row]);
        if (MODE == 1)   // second largest of the two halves' (largest, second largest) pairs
          Mf = fmaxf(fminf(fin[row], fin[TM + row]), fmaxf(fin[1024 + row], fin[1024 + TM + row]));
        const float thr = fminf(Mf, cap) - fin[768 + row];
        fl = finu[512 + row] | finu[512 + TM + row] | force;
        // cosine: if every dot may be <= -1 they all clamp to pi and the lowest index wins -> exact pass
        if (p.metric == 1 && !(Mf >= fin[768 + row] - cap)) fl |= 8u;
        // padded table rows and dead (non-finite) centroids score exactly -65504 (zero row + sentinel bias): a
        // threshold that low cannot tell them from real candidates (an outlier far from every centroid) -> exact pass
        if (!(thr > SENTINEL_GUARD)) fl |= 8u;
        for (int hh = 0; hh < 2; hh++) {
          const int sl = hh * TM + row;
          const uint32_t c2 = finu[256 + sl];
          for (uint32_t i = 0; i < c2; i++) {
            constexpr uint32_t A = LIST_ARRAY / 4;
            if (!(__uint_as_float(lst[i * 256 + sl]) >= thr)) continue;
            const uint32_t base = lst[3 * A + i * 256 + sl] * TN + hh * 64;
#pragma unroll
            for (int c = 0; c < 2; c++) {
              uint32_t m = lst[(1 + c) * A + i * 256 + sl];
              while (m) {
                const int b = __ffs(m) - 1;
                m &= m - 1;
                const uint32_t col = base + c * 32 + b;
                if (col < p.K) {
                  if (total < MAX_CAND) cand[total] = col;
                  total++;
                }
              }
            }
          }
        }
      }
      // the lists of this parity are consumed: the epilogue may start tile ti+2
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars[BAR_EMIT_EMPTY + par]);
      const bool overflow = live && (fl || total > MAX_CAND || (MODE == 1 && total == 0));
      const bool multi = live && !overflow && total >= (MODE == 1 ? 1u : 2u);
      // warp-aggregated queue reservation: one atomic per warp for the pairs, one for the row queue
      uint32_t want = multi ? total : 0, pre = want;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t v = __shfl_up_sync(0xffffffffu, pre, o);
        if (lane >= o) pre += v;
      }
      const uint32_t warp_total = __shfl_sync(0xffffffffu, pre, 31);
      const unsigned mmask = __ballot_sync(0xffffffffu, multi);
      uint32_t base = 0, rqbase = 0;
      if (lane == 0 && warp_total) {
        base = atomicAdd(&p.counters[CNT_PAIRS], warp_total);
        rqbase = atomicAdd(&p.counters[CNT_ROWQ], static_cast<uint32_t>(__popc(mmask)));
      }
      base = __shfl_sync(0xffffffffu, base, 0) + (pre - want);
      rqbase = __shfl_sync(0xffffffffu, rqbase, 0) + __popc(mmask & ((1u << lane) - 1));
      if (live) {
        if (overflow) {
          p.ovf_rows[atomicAdd(&p.counters[CNT_OVF], 1u)] = static_cast<uint32_t>(grow);
        } else if (MODE == 0 && total == 1) {
          if (p.assign) nchanged += commit_assignment(p.assign, p.prev, grow, cand[0]);
          else p.result[grow] = cand[0];
        } else if (MODE == 0 && total == 0) {
          // every score NaN: nothing wins, the assignment stays (reference kmeans.cu:349-353)
          if (!p.assign) p.result[grow] = kUntouched;
        } else if (base + total <= p.max_pairs) {
          for (uint32_t i = 0; i < total; i++) {
            p.pair_row[base + i] = static_cast<uint32_t>(grow);
            p.pair_cand[base + i] = cand[i];
          }
          p.rowq[3 * rqbase] = static_cast<uint32_t>(grow);
          p.rowq[3 * rqbase + 1] = base;
          p.rowq[3 * rqbase + 2] = total;
        } else {
          // queue full: the row goes to the full exact pass; its reserved row-queue slot is neutralised
          p.rowq[3 * rqbase] = static_cast<uint32_t>(grow);
          p.rowq[3 * rqbase + 1] = 0;
          p.rowq[3 * rqbase + 2] = 0;
          p.ovf_rows[atomicAdd(&p.counters[CNT_OVF], 1u)] = static_cast<uint32_t>(grow);
        }
      }
    }
    if (MODE == 0 && p.assign) {
      nchanged = __reduce_add_sync(0xffffffffu, nchanged);
      if (lane == 0 && nchanged) atomicAdd(p.d_changed, nchanged);
    }
  }
  // teardown
  ptx::tc_fence_before();
  __syncthreads();
  if (PAIR) ptx::cluster_sync_all();   // no CTA leaves while its peer may still arrive on its barriers / use the pair's TMEM
  if (warp == WARP_MMA) {
    ptx::tc_fence_after();
    if (PAIR) ptx::tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else ptx::tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace tc

// ---------------------------------------------------------------------------------------------------
// exact re-check of (row, candidate) pairs + per-row reduction
// ---------------------------------------------------------------------------------------------------
template <int METRIC, int MODE>   // MODE 0: Lloyd ranking score; MODE 1: true distance (Yinyang bounds)
__global__ void __launch_bounds__(128)
recheck_pairs_kernel(const float* __restrict__ X, const float* __restrict__ C,
                     const float* __restrict__ csq, int D, const uint32_t* __restrict__ pair_row,
                     const uint32_t* __restrict__ pair_cand, const uint32_t* __restrict__ d_npairs,
                     uint32_t max_pairs, uint32_t n, uint32_t K, float* __restrict__ pair_score) {
  // 128 (row, candidate) pairs per CTA; features stream through shared memory 32 at a time.
  // Staging: every thread issues 16 independent 16-byte loads per chunk (8 lanes cover one 128-byte row segment).  The
  // loads of chunk i+1 are issued BEFORE the sequential Kahan loop of chunk i (32 features x a 4-instruction dependent
  // chain per pair), so the global-memory latency of a chunk hides behind the previous chunk's arithmetic (round 2:
  // load -> store -> compute ran back to back, 233 us for 0.92 M pairs at the headline shape).
  __shared__ float sX[32 * 129];     // [feature][pair]   (+1 padding: conflict-free both ways)
  __shared__ float sC[128 * 33];     // [pair][feature]
  __shared__ uint32_t s_row[128], s_cand[128];
  const uint32_t np = min(*d_npairs, max_pairs);
  const int nchunks = (D + 31) / 32;
  for (uint32_t tile0 = blockIdx.x * 128; tile0 < np; tile0 += gridDim.x * 128) {
    const uint32_t pidx = tile0 + threadIdx.x;
    const bool active = pidx < np;
    __syncthreads();
    // (slots past the last complete row group may hold stale data: stay in bounds)
    s_row[threadIdx.x] = active ? min(pair_row[pidx], n - 1) : 0;
    s_cand[threadIdx.x] = active ? min(pair_cand[pidx], K - 1) : 0;
    __syncthreads();
    // the whole sample row of this thread's pair is requested from DRAM now, line after line (one open DRAM page per
    // row), so that the chunk loads below -- 128 bytes of the row per chunk, spread over the chunk loop -- hit L2
    // instead of making eight scattered DRAM accesses per row
    if (active) {
      const char* xr = reinterpret_cast<const char*>(X + static_cast<size_t>(s_row[threadIdx.x]) * D);
      for (int b = 128; b < D * 4; b += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(xr + b));
    }
    Kahan k;
    float4 v[16];
    auto load_chunk = [&](int f0) {
      const int fl = min(32, D - f0);
#pragma unroll
      for (int i = 0; i < 16; i++) {
        const int idx = i * 128 + threadIdx.x;  // [which(1)][pair(7)][quad(3)]
        const int q = idx & 7, e = (idx >> 3) & 127, which = idx >> 10;
        const float* src = which ? C + static_cast<size_t>(s_cand[e]) * D : X + static_cast<size_t>(s_row[e]) * D;
        v[i] = (q * 4 < fl) ? *reinterpret_cast<const float4*>(src + f0 + q * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    load_chunk(0);
    for (int ch = 0; ch < nchunks; ch++) {
      const int fl = min(32, D - ch * 32);
      __syncthreads();                      // the previous chunk has been consumed
#pragma unroll
      for (int i = 0; i < 16; i++) {
        const int idx = i * 128 + threadIdx.x;
        const int q = idx & 7, e = (idx >> 3) & 127, which = idx >> 10;
        if (which) {
          float* d = sC + e * 33 + q * 4;
          d[0] = v[i].x; d[1] = v[i].y; d[2] = v[i].z; d[3] = v[i].w;
        } else {
          float* d = sX + (q * 4) * 129 + e;
          d[0] = v[i].x; d[129] = v[i].y; d[258] = v[i].z; d[387] = v[i].w;
        }
      }
      __syncthreads();
      if (ch + 1 < nchunks) load_chunk((ch + 1) * 32);   // in flight during the loop below
      if (active)
        for (int f = 0; f < fl; f++) {
          if (MODE == 1 && METRIC == 0) k.sqdiff(sX[f * 129 + threadIdx.x], sC[threadIdx.x * 33 + f]);
          else k.mac(sX[f * 129 + threadIdx.x], sC[threadIdx.x * 33 + f]);
        }
    }
    if (active)
      pair_score[pidx] = MODE == 1 ? finalize_distance<METRIC>(k.sum)
                                   : lloyd_score<METRIC>(k.sum, csq[s_cand[threadIdx.x]]);
  }
}

__global__ void recheck_reduce_kernel(const uint32_t* __restrict__ rowq, const uint32_t* __restrict__ d_nrowq,
                                      const uint32_t* __restrict__ pair_cand,
                                      const float* __restrict__ pair_score, uint32_t* __restrict__ result,
                                      uint32_t* __restrict__ assign, uint32_t* __restrict__ prev,
                                      uint32_t* __restrict__ d_changed) {
  const uint32_t nq = *d_nrowq;
  uint32_t nchanged = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += gridDim.x * blockDim.x) {
    const uint32_t row = rowq[3 * i], base = rowq[3 * i + 1], cnt = rowq[3 * i + 2];
    if (cnt == 0) continue;  // neutralised slot (pair queue was full; the row is on the overflow list)
    float best = FLT_MAX;
    uint32_t arg = UINT32_MAX;
    for (uint32_t j = 0; j < cnt; j++) {
      const float sc = pair_score[base + j];
      const uint32_t c = pair_cand[base + j];
      // strict '<' in ascending centroid order == lowest index among equal scores
      if (sc < best || (sc == best && c < arg)) {
        best = sc;
        arg = c;
      }
    }
    if (assign) {
      if (arg != UINT32_MAX) nchanged += tc::commit_assignment(assign, prev, row, arg);
    } else {
      result[row] = (arg == UINT32_MAX) ? kUntouched : arg;
    }
  }
  if (assign) {
    nchanged = __reduce_add_sync(0xffffffffu, nchanged);
    if ((threadIdx.x & 31) == 0 && nchanged) atomicAdd(d_changed, nchanged);
  }
}

// bookkeeping for the rows that took the full exact pass (their winners are in result[])
__global__ void finalize_rows_kernel(const uint32_t* __restrict__ rows, const uint32_t* __restrict__ d_nrows,
                                     const uint32_t* __restrict__ result, uint32_t* __restrict__ assign,
                                     uint32_t* __restrict__ prev, uint32_t* __restrict__ d_changed) {
  const uint32_t nr = *d_nrows;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nr; i += gridDim.x * blockDim.x) {
    const uint32_t row = rows[i], r = result[row];
    if (r != kUntouched && tc::commit_assignment(assign, prev, row, r)) atomicAdd(d_changed, 1u);
  }
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
struct TcPlan {
  int metric, D, device, nkb, nt;
  uint32_t K, max_n, max_pairs;
  __half* table = nullptr;
  __half* aug_blob = nullptr;
  tc::Stats* stats = nullptr;
  float* cnorm2 = nullptr;         // cosine: ||c||^2 (the reference's 'csqr' is the constant 1 there); L2: ||c - mu||^2
  double* musum = nullptr;         // [D] column sums of the valid centroids, followed by the valid-row count
  float* neg_mu_s = nullptr;       // [nkb*64] L2: -mu*s with mu = mean of the valid centroids, see Params::neg_mu_s
  bool inject_error = false;       // test hook (KMCUDA_B200_INJECT_PIPELINE_ERROR=1): report a timed-out barrier
  // Yinyang bounds refresh (MODE 3): group-sorted table layout, built once per run by tc_yy_layout()
  int nt3 = 0;
  uint32_t G3 = 0;
  __half* table3 = nullptr;
  __half* aug_blob3 = nullptr;
  uint32_t* yy_perm = nullptr;     // [nt3*128] table row -> centroid (UINT32_MAX = padding)
  uint32_t* yy_qgroup = nullptr;   // [nt3*32] group of every 4-column quad
  uint32_t* yy_goff = nullptr;     // [G+1] CSR of the group members
  uint32_t* yy_gmem = nullptr;     // [K]
  uint32_t yy_max_gsize = 0;       // members of the largest group
  CUtensorMap tmap3;
  uint32_t *pair_row = nullptr, *pair_cand = nullptr, *rowq = nullptr, *ovf_rows = nullptr, *counters = nullptr;
  float* pair_score = nullptr;
  uint32_t* h_counters = nullptr;  // pinned
  unsigned* prep_barrier = nullptr;   // {arrivals, generation} of tc_prep_fused_kernel's grid barrier (zero between launches)
  CUtensorMap tmap;     // fp16 centroid table
  // CTA-pair mode of the Lloyd pass (cta_group::2, see tc_assign_kernel): half-tile boxes of the table, the bias blocks
  // as 2 KiB pieces per (n-tile, CTA rank), number of CTA pairs that can be resident at once
  bool pair = false;
  int pair_clusters = 0;
  CUtensorMap tmap_pair, tmap_aug;
  int num_sms = 148;
  size_t smem_bytes = 0;
  // CUDA-event pairs around the main kernel of the most recent passes (bench.py roofline)
  static constexpr int kEvRing = 64;
  cudaEvent_t ev0[kEvRing] = {}, ev1[kEvRing] = {};
  uint64_t passes = 0;
  bool capturing = false;          // the pass is being captured into a CUDA graph (Shard::assign): events are recorded as
  int graph_slot = -1;             // external event nodes into one fixed slot, which every replay of the graph refreshes
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

template <int MODE>
static void tc_launch_mode(int nkb, unsigned grid, size_t smem, cudaStream_t st, const CUtensorMap& tb,
                           const CUtensorMap& tx, const tc::Params& prm) {
  using namespace tc;
  switch (nkb) {   // (the third tensor map is only read in CTA-pair mode)
    case 1: tc_assign_kernel<1, MODE><<<grid, N_THREADS, smem, st>>>(tb, tx, tb, prm); break;
    case 2: tc_assign_kernel<2, MODE><<<grid, N_THREADS, smem, st>>>(tb, tx, tb, prm); break;
    case 3: tc_assign_kernel<3, MODE><<<grid, N_THREADS, smem, st>>>(tb, tx, tb, prm); break;
    case 4: tc_assign_kernel<4, MODE><<<grid, N_THREADS, smem, st>>>(tb, tx, tb, prm); break;
    case 5: tc_assign_kernel<5, MODE><<<grid, N_THREADS, smem, st>>>(tb, tx, tb, prm); break;
    case 6: tc_assign_kernel<6, MODE><<<grid, N_THREADS, smem, st>>>(tb, tx, tb, prm); break;
    case 7: tc_assign_kernel<7, MODE><<<grid, N_THREADS, smem, st>>>(tb, tx, tb, prm); break;
    default: tc_assign_kernel<8, MODE><<<grid, N_THREADS, smem, st>>>(tb, tx, tb, prm); break;
  }
}
static void tc_launch_main(int mode, int nkb, unsigned grid, size_t smem, cudaStream_t st, const CUtensorMap& tb,
                           const CUtensorMap& tx, const tc::Params& prm) {
  if (mode == 3) tc_launch_mode<3>(nkb, grid, smem, st, tb, tx, prm);
  else if (mode == 2) tc_launch_mode<2>(nkb, grid, smem, st, tb, tx, prm);
  else if (mode == 1) tc_launch_mode<1>(nkb, grid, smem, st, tb, tx, prm);
  else tc_launch_mode<0>(nkb, grid, smem, st, tb, tx, prm);
}
// CTA-pair launch of the Lloyd pass: clusters of 2 CTAs
template <int NKB>
static cudaError_t tc_launch_pair_one(unsigned grid, size_t smem, cudaStream_t st, const CUtensorMap& tb,
                                      const CUtensorMap& tx, const CUtensorMap& ta, const tc::Params& prm) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(tc::N_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, tc::tc_assign_kernel<NKB, 0, 2>, tb, tx, ta, prm);
}
static cudaError_t tc_launch_pair(int nkb, unsigned grid, size_t smem, cudaStream_t st, const CUtensorMap& tb,
                                  const CUtensorMap& tx, const CUtensorMap& ta, const tc::Params& prm) {
  switch (nkb) {
    case 1: return tc_launch_pair_one<1>(grid, smem, st, tb, tx, ta, prm);
    case 2: return tc_launch_pair_one<2>(grid, smem, st, tb, tx, ta, prm);
    case 3: return tc_launch_pair_one<3>(grid, smem, st, tb, tx, ta, prm);
    case 4: return tc_launch_pair_one<4>(grid, smem, st, tb, tx, ta, prm);
    case 5: return tc_launch_pair_one<5>(grid, smem, st, tb, tx, ta, prm);
    case 6: return tc_launch_pair_one<6>(grid, smem, st, tb, tx, ta, prm);
    case 7: return tc_launch_pair_one<7>(grid, smem, st, tb, tx, ta, prm);
    default: return tc_launch_pair_one<8>(grid, smem, st, tb, tx, ta, prm);
  }
}
template <int NKB>
static int tc_pair_clusters_one(int bytes) {
  // how many CTA pairs fit on the device at once (0: pair mode unavailable)
  if (cudaFuncSetAttribute(tc::tc_assign_kernel<NKB, 0, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2);
  cfg.blockDim = dim3(tc::N_THREADS);
  cfg.dynamicSmemBytes = bytes;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, tc::tc_assign_kernel<NKB, 0, 2>, &cfg) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}
static int tc_pair_clusters_query(int bytes, int nkb) {
  switch (nkb) {
    case 1: return tc_pair_clusters_one<1>(bytes);
    case 2: return tc_pair_clusters_one<2>(bytes);
    case 3: return tc_pair_clusters_one<3>(bytes);
    case 4: return tc_pair_clusters_one<4>(bytes);
    case 5: return tc_pair_clusters_one<5>(bytes);
    case 6: return tc_pair_clusters_one<6>(bytes);
    case 7: return tc_pair_clusters_one<7>(bytes);
    default: return tc_pair_clusters_one<8>(bytes);
  }
}
// (cudaOccupancyMaxActiveClusters and the pinned allocation below are milliseconds each: a plan is created by every
// kmeans_cuda call, so their results are kept per process)
static int tc_pair_clusters(int bytes, int nkb) {
  static std::mutex mu;
  static std::map<std::tuple<int, int, int>, int> cache;
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(mu);
  auto key = std::make_tuple(dev, bytes, nkb);
  auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  const int n = tc_pair_clusters_query(bytes, nkb);
  cache[key] = n;
  return n;
}
static std::mutex g_pinned_mu;
static std::vector<uint32_t*> g_pinned_free;   // CNT_N-word pinned blocks of destroyed plans
static uint32_t* pinned_counters_alloc() {
  {
    std::lock_guard<std::mutex> lk(g_pinned_mu);
    if (!g_pinned_free.empty()) {
      uint32_t* p = g_pinned_free.back();
      g_pinned_free.pop_back();
      return p;
    }
  }
  void* p = nullptr;
  if (cudaHostAlloc(&p, sizeof(uint32_t) * tc::CNT_N, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return static_cast<uint32_t*>(p);
}
static void pinned_counters_free(uint32_t* p) {
  if (!p) return;
  std::lock_guard<std::mutex> lk(g_pinned_mu);
  g_pinned_free.push_back(p);
}

template <int NKB>
static cudaError_t tc_set_smem_attr_one(int bytes) {
  cudaError_t e = cudaFuncSetAttribute(tc::tc_assign_kernel<NKB, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(tc::tc_assign_kernel<NKB, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(tc::tc_assign_kernel<NKB, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(tc::tc_assign_kernel<NKB, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
static cudaError_t tc_set_smem_attr(int bytes, int nkb) {   // only the instantiation this shape launches
  switch (nkb) {
    case 1: return tc_set_smem_attr_one<1>(bytes);
    case 2: return tc_set_smem_attr_one<2>(bytes);
    case 3: return tc_set_smem_attr_one<3>(bytes);
    case 4: return tc_set_smem_attr_one<4>(bytes);
    case 5: return tc_set_smem_attr_one<5>(bytes);
    case 6: return tc_set_smem_attr_one<6>(bytes);
    case 7: return tc_set_smem_attr_one<7>(bytes);
    default: return tc_set_smem_attr_one<8>(bytes);
  }
}

bool tc_supported(int metric, uint32_t n, int D, uint32_t K) {
  if (D < 4 || D % 4 != 0 || D > tc::MAX_NKB * tc::KB) return false;   // TMA row pitch must be 16-byte aligned
  if (K < 2 || K > 16383u * 128u) return false;        // chunk ids are 16 bit (4 per n-tile)
  if (n == 0) return false;
  return true;
}

void tc_plan_destroy(TcPlan* p) {
  if (!p) return;
  pool_free(p->table);
  pool_free(p->aug_blob);
  pool_free(p->stats);
  pool_free(p->cnorm2);
  pool_free(p->musum);
  pool_free(p->neg_mu_s);
  pool_free(p->table3);
  pool_free(p->aug_blob3);
  pool_free(p->yy_perm);
  pool_free(p->yy_qgroup);
  pool_free(p->yy_goff);
  pool_free(p->yy_gmem);
  pool_free(p->pair_row);
  pool_free(p->pair_cand);
  pool_free(p->pair_score);
  pool_free(p->rowq);
  pool_free(p->ovf_rows);
  pool_free(p->counters);
  pool_free(p->prep_barrier);
  pinned_counters_free(p->h_counters);
  for (int i = 0; i < TcPlan::kEvRing; i++) {
    if (p->ev0[i]) cudaEventDestroy(p->ev0[i]);
    if (p->ev1[i]) cudaEventDestroy(p->ev1[i]);
  }
  delete p;
}

cudaError_t tc_plan_create(TcPlan** out, int metric, uint32_t max_n, int D, uint32_t K, int device) {
  using namespace tc;
  TcPlan* p = new TcPlan;
  p->metric = metric;
  p->D = D;
  p->K = K;
  p->device = device;
  p->max_n = max_n;
  p->nkb = (D + KB - 1) / KB;
  p->nt = static_cast<int>((K + TN - 1) / TN);
  p->max_pairs = max_n < (1u << 28) ? 10 * max_n + 1024 : 0xFFFFFFF0u;   // Lloyd needs ~0.4 n, the Yinyang top-2 mode up to ~7 n
  cudaError_t e;
#define TC_TRY(x) do { e = (x); if (e != cudaSuccess) { tc_plan_destroy(p); return e; } } while (0)
  TC_TRY(cudaDeviceGetAttribute(&p->num_sms, cudaDevAttrMultiProcessorCount, device));
  const size_t rows_pad = static_cast<size_t>(p->nt) * TN;
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->table), rows_pad * p->nkb * KB * sizeof(__half)));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->aug_blob), static_cast<size_t>(p->nt) * AUG_B_BYTES));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->stats), sizeof(Stats)));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->cnorm2), sizeof(float) * K));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->musum), sizeof(double) * (D + 1)));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->neg_mu_s), sizeof(float) * MAX_NKB * KB));
  {
    const char* ie = getenv("KMCUDA_B200_INJECT_PIPELINE_ERROR");
    p->inject_error = ie && ie[0] == '1';
  }
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->pair_row), sizeof(uint32_t) * p->max_pairs));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->pair_cand), sizeof(uint32_t) * p->max_pairs));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->pair_score), sizeof(float) * p->max_pairs));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->rowq), sizeof(uint32_t) * 3 * static_cast<size_t>(max_n)));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->ovf_rows), sizeof(uint32_t) * static_cast<size_t>(max_n)));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->counters), sizeof(uint32_t) * CNT_N));
  TC_TRY(pool_alloc(reinterpret_cast<void**>(&p->prep_barrier), sizeof(unsigned) * 2));
  TC_TRY(cudaMemset(p->prep_barrier, 0, sizeof(unsigned) * 2));
  TC_TRY(cudaStreamSynchronize(nullptr));   // the passes run on non-blocking streams, which do not order against this memset
  p->h_counters = pinned_counters_alloc();
  if (!p->h_counters) { tc_plan_destroy(p); return cudaErrorMemoryAllocation; }
  memset(p->h_counters, 0, sizeof(uint32_t) * CNT_N);
  // tensor map over the fp16 centroid table [rows_pad][nkb*64], box 64 x 256, 128-byte swizzle
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { tc_plan_destroy(p); return cudaErrorNotSupported; }
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(p->nkb * KB), static_cast<cuuint64_t>(rows_pad)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(p->nkb * KB) * sizeof(__half)};
  cuuint32_t box[2] = {KB, TN};
  cuuint32_t estr[2] = {1, 1};
  CUresult cr = enc(&p->tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, p->table, gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) { tc_plan_destroy(p); return cudaErrorInvalidValue; }
  for (int i = 0; i < TcPlan::kEvRing; i++) {
    TC_TRY(cudaEventCreate(&p->ev0[i]));
    TC_TRY(cudaEventCreate(&p->ev1[i]));
  }
  p->smem_bytes = smem_layout().total + 1024;
  TC_TRY(tc_set_smem_attr(static_cast<int>(p->smem_bytes), p->nkb));
  {
    // CTA-pair mode (KMCUDA_B200_PAIR=0 switches it off): half-tile boxes of the table, the bias blocks as a
    // [nt * 4][256 words] matrix whose rows (t, rank, K half) are the 1 KiB halves of the 2 KiB pieces
    const char* pe = getenv("KMCUDA_B200_PAIR");
    bool want = !(pe && pe[0] == '0');
    if (want) {
      cuuint32_t boxp[2] = {KB, TN / 2};
      CUresult c1 = enc(&p->tmap_pair, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, p->table, gdim, gstride, boxp, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      cuuint64_t gdima[2] = {256, static_cast<cuuint64_t>(p->nt) * 4};
      cuuint64_t gstridea[1] = {1024};
      cuuint32_t boxa[2] = {256, 2};
      CUresult c2 = enc(&p->tmap_aug, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, p->aug_blob, gdima, gstridea, boxa, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (c1 == CUDA_SUCCESS && c2 == CUDA_SUCCESS) {
        p->pair_clusters = tc_pair_clusters(static_cast<int>(p->smem_bytes), p->nkb);
        // only worth it when (nearly) every SM finds a partner
        p->pair = p->pair_clusters * 2 >= p->num_sms - 4;
      }
    }
  }
#undef TC_TRY
  *out = p;
  return cudaSuccess;
}

// counters reset + centroid preparation (scale, fp16 table, bias blobs) + the parameter block shared by both modes
static cudaError_t tc_prepare(TcPlan* p, const float* C, const float* csq, uint32_t n, tc::Params* out,
                              cudaStream_t st, bool yy_layout = false, bool pair_blob = false, bool compute_csq = false) {
  using namespace tc;
  cudaError_t e;
  {
    PrepArgs a;
    a.metric = p->metric;
    a.D = p->D;
    a.nkb = p->nkb;
    a.by_source = yy_layout ? 1 : 0;
    a.pair_blob = pair_blob ? 1 : 0;
    a.K = p->K;
    a.rows_pad = static_cast<uint32_t>(yy_layout ? p->nt3 : p->nt) * TN;
    a.C = C;
    a.csq = const_cast<float*>(csq);
    a.compute_csq = compute_csq ? 1 : 0;
    a.cnorm2 = p->cnorm2;
    a.musum = p->musum;
    a.neg_mu_s = p->neg_mu_s;
    a.stats = p->stats;
    a.counters = p->counters;
    a.table = yy_layout ? p->table3 : p->table;
    a.aug_blob = yy_layout ? p->aug_blob3 : p->aug_blob;
    a.gather = yy_layout ? p->yy_perm : nullptr;
    a.barrier = p->prep_barrier;
    // one table row per warp up to the number of SMs (every CTA must be resident for the grid barrier)
    const unsigned grid = std::min<unsigned>(static_cast<unsigned>(p->num_sms), std::max(1u, (a.rows_pad + 7u) / 8u));
    tc_prep_fused_kernel<<<grid, 256, 0, st>>>(a);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  Params prm;
  prm.n = n;
  prm.D = p->D;
  prm.K = p->K;
  prm.nkb = p->nkb;
  prm.nt = p->nt;
  prm.ntiles = (n + TM - 1) / TM;
  prm.aug_blob = p->aug_blob;
  prm.stats = p->stats;
  prm.result = nullptr;
  prm.pair_row = p->pair_row;
  prm.pair_cand = p->pair_cand;
  prm.max_pairs = p->max_pairs;
  prm.rowq = p->rowq;
  prm.ovf_rows = p->ovf_rows;
  prm.counters = p->counters;
  prm.metric = p->metric;
  prm.neg_mu_s = p->neg_mu_s;
  prm.assign = prm.prev = prm.d_changed = nullptr;
  prm.yy_qgroup = prm.yy_groups = prm.yy_assign = nullptr;
  prm.yy_bounds = nullptr;
  prm.G = 0;
  if (yy_layout) {
    prm.nt = p->nt3;
    prm.aug_blob = p->aug_blob3;
  }
  prm.X = nullptr;
  prm.rows = nullptr;
  prm.d_nrows = nullptr;
  prm.d_ntiles = nullptr;
  prm.tile_nrows = prm.blk_cluster = prm.knn_roff = prm.knn_rcount = prm.knn_nblk = nullptr;
  prm.C = nullptr;
  prm.knn_ranges = nullptr;
  prm.kk = 0;
  prm.knn_first_pass = 0;
  prm.knn_stride = 0;
  prm.knn_topk = prm.knn_dub = nullptr;
  prm.knn_cnt = prm.knn_flags = nullptr;
  prm.knn_entries = nullptr;
  prm.knn_part = 0;
  prm.knn_nparts = 1;
  *out = prm;
  return cudaGetLastError();
}

cudaError_t tc_assign(TcPlan* p, const float* X, const float* C, const float* csq, uint32_t n,
                      uint32_t* result, uint32_t* assign, uint32_t* prev, uint32_t* d_changed, cudaStream_t st,
                      bool compute_csq) {
  using namespace tc;
  if (n > p->max_n) return cudaErrorInvalidValue;
  // TMA needs 16-byte aligned rows; the re-check kernels read both matrices with 16-byte vector loads
  if ((reinterpret_cast<uintptr_t>(X) & 15) || (reinterpret_cast<uintptr_t>(C) & 15)) return cudaErrorMisalignedAddress;
  cudaError_t e;
  // tensor map over the caller's fp32 samples [n][D]: box 32 features x 128 rows, 128-byte swizzle,
  // out-of-range rows / features read as zero (ragged last tile, D not a multiple of 32)
  CUtensorMap tmap_x;
  {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return cudaErrorNotSupported;
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(p->D), static_cast<cuuint64_t>(n)};
    cuuint64_t gstride[1] = {static_cast<cuuint64_t>(p->D) * sizeof(float)};
    cuuint32_t box[2] = {32, TM};
    cuuint32_t estr[2] = {1, 1};
    CUresult cr = enc(&tmap_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(X), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) return cudaErrorInvalidValue;
  }
  Params prm;
  // CTA pairs pay off once every pair has several tile pairs to stream the table for
  const bool pair = p->pair && (n + TM - 1) / TM >= 4u * static_cast<uint32_t>(p->num_sms);
  if ((e = tc_prepare(p, C, csq, n, &prm, st, false, pair, compute_csq)) != cudaSuccess) return e;
  prm.result = result;
  prm.assign = assign;      // non-null: the pass's bookkeeping (prev / assign / changed counter) is fused
  prm.prev = prev;
  prm.d_changed = d_changed;
  unsigned grid = min(static_cast<uint32_t>(p->num_sms), prm.ntiles);
  if (pair) grid = min(static_cast<uint32_t>(p->pair_clusters) * 2u, (prm.ntiles + 1u) & ~1u);
  const int slot = static_cast<int>(p->passes % TcPlan::kEvRing);
  if (p->capturing) {
    p->graph_slot = slot;
    cudaEventRecordWithFlags(p->ev0[slot], st, cudaEventRecordExternal);
  } else {
    p->graph_slot = -1;
    cudaEventRecord(p->ev0[slot], st);
  }
  if (pair) {
    if ((e = tc_launch_pair(p->nkb, grid, p->smem_bytes, st, p->tmap_pair, tmap_x, p->tmap_aug, prm)) != cudaSuccess) return e;
  } else {
    tc_launch_main(0, p->nkb, grid, p->smem_bytes, st, p->tmap, tmap_x, prm);
  }
  if (p->capturing) cudaEventRecordWithFlags(p->ev1[slot], st, cudaEventRecordExternal);
  else cudaEventRecord(p->ev1[slot], st);
  p->passes++;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  // exact re-check of the multi-candidate rows, then the rows that need the full exact pass
  const unsigned rgrid = p->num_sms * 4;
  if (p->metric == 1)
    recheck_pairs_kernel<1, 0><<<rgrid, 128, 0, st>>>(X, C, csq, p->D, p->pair_row, p->pair_cand,
                                                      p->counters + CNT_PAIRS, p->max_pairs, n, p->K, p->pair_score);
  else
    recheck_pairs_kernel<0, 0><<<rgrid, 128, 0, st>>>(X, C, csq, p->D, p->pair_row, p->pair_cand,
                                                      p->counters + CNT_PAIRS, p->max_pairs, n, p->K, p->pair_score);
  recheck_reduce_kernel<<<p->num_sms * 2, 256, 0, st>>>(p->rowq, p->counters + CNT_ROWQ, p->pair_cand,
                                                        p->pair_score, result, assign, prev, d_changed);
  if ((e = launch_assign_exact(p->metric, X, C, csq, n, p->D, p->K, p->ovf_rows, p->counters + CNT_OVF, result,
                               st)) != cudaSuccess)
    return e;
  if (assign)
    finalize_rows_kernel<<<p->num_sms, 256, 0, st>>>(p->ovf_rows, p->counters + CNT_OVF, result, assign, prev, d_changed);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (p->inject_error) cudaMemsetAsync(p->counters + CNT_ERR, 0x11, sizeof(uint32_t), st);
  return cudaMemcpyAsync(p->h_counters, p->counters, sizeof(uint32_t) * CNT_N, cudaMemcpyDeviceToHost, st);
}

// Yinyang local step, candidate generation: for the listed rows, every centroid whose approximate score is
// within the rigorous margin of the row's second best, with its exact TRUE distance (reference
// METRIC::distance, metric_abstraction.h:59-101,179-222).  Results stay in the plan's queues (tc_queues()).
// Rows the filter cannot bound (NaN/Inf, > MAX_CAND candidates, queue full) are put on the overflow list.
cudaError_t tc_yy_candidates(TcPlan* p, const float* X, const float* C, const float* csq, uint32_t n,
                             const uint32_t* rows, const uint32_t* d_nrows, cudaStream_t st) {
  using namespace tc;
  if (n > p->max_n) return cudaErrorInvalidValue;
  if ((reinterpret_cast<uintptr_t>(X) & 15) || (reinterpret_cast<uintptr_t>(C) & 15)) return cudaErrorMisalignedAddress;
  cudaError_t e;
  Params prm;
  if ((e = tc_prepare(p, C, csq, n, &prm, st)) != cudaSuccess) return e;
  prm.X = X;
  prm.rows = rows;
  prm.d_nrows = d_nrows;
  const unsigned grid = min(static_cast<uint32_t>(p->num_sms), prm.ntiles);
  tc_launch_main(1, p->nkb, grid, p->smem_bytes, st, p->tmap, p->tmap /* unused */, prm);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = tc_exact_distances(p, X, C, n, p->pair_row, p->pair_cand, p->counters + CNT_PAIRS, p->max_pairs,
                              p->pair_score, st)) != cudaSuccess)
    return e;
  return cudaMemcpyAsync(p->h_counters, p->counters, sizeof(uint32_t) * CNT_N, cudaMemcpyDeviceToHost, st);
}

// exact true distances of (row, centroid) pairs: 128 pairs per CTA, coalesced staging (see recheck_pairs_kernel)
cudaError_t tc_exact_distances(TcPlan* p, const float* X, const float* C, uint32_t n, const uint32_t* pair_row,
                               const uint32_t* pair_cand, const uint32_t* d_npairs, uint32_t max_pairs,
                               float* pair_score, cudaStream_t st) {
  const unsigned rgrid = p->num_sms * 4;
  if (p->metric == 1)
    recheck_pairs_kernel<1, 1><<<rgrid, 128, 0, st>>>(X, C, nullptr, p->D, pair_row, pair_cand, d_npairs, max_pairs,
                                                      n, p->K, pair_score);
  else
    recheck_pairs_kernel<0, 1><<<rgrid, 128, 0, st>>>(X, C, nullptr, p->D, pair_row, pair_cand, d_npairs, max_pairs,
                                                      n, p->K, pair_score);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// Yinyang bounds refresh on the tensor cores (reference kmeans_yy_init, kmeans.cu:431-485)
// ---------------------------------------------------------------------------------------------------
// exact part of the refresh: upper bound = distance to the own centroid, lower bound of the OWN group = nearest other
// member (both as the reference computes them).  Round 2's first version gave every sample a warp whose lanes each walked
// one member's row from global memory -- a chain of 256 dependent Kahan steps per lane with 10 of 32 lanes busy: 1.1 s
// at 8M x 256 @ 1024 (G = 102), more than the whole Lloyd run.  Now: (1) the (sample, group member) pairs of a chunk of
// rows are written to the plan's pair queue, (2) recheck_pairs_kernel computes their exact true distances (128 pairs
// per CTA, coalesced staging), (3) one thread per row folds its pairs into the two bounds.
__global__ void __launch_bounds__(256)
yy_own_pairs_kernel(uint32_t row0, uint32_t row1, uint32_t K, uint32_t G, const uint32_t* __restrict__ assign,
                    const uint32_t* __restrict__ groups, const uint32_t* __restrict__ goff,
                    const uint32_t* __restrict__ gmem, uint32_t* __restrict__ pair_row, uint32_t* __restrict__ pair_cand,
                    uint32_t max_pairs, uint32_t* __restrict__ rowq, uint32_t* __restrict__ counters) {
  const int lane = threadIdx.x & 31;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t base_row = row0 + blockIdx.x * blockDim.x; base_row < row1; base_row += stride) {
    const uint32_t row = base_row + threadIdx.x;
    uint32_t cnt = 0, beg = 0;
    if (row < row1) {
      const uint32_t a = assign[row];
      if (a < K) {                                   // "insane" samples keep FLT_MAX bounds
        const uint32_t g = groups[a];
        if (g < G) { beg = goff[g]; cnt = goff[g + 1] - beg; }
      }
    }
    uint32_t pre = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, pre, o);
      if (lane >= o) pre += v;
    }
    const uint32_t warp_total = __shfl_sync(0xffffffffu, pre, 31);
    const unsigned have = __ballot_sync(0xffffffffu, cnt != 0);
    uint32_t pbase = 0, qbase = 0;
    if (lane == 0 && warp_total) {
      pbase = atomicAdd(&counters[tc::CNT_PAIRS], warp_total);
      qbase = atomicAdd(&counters[tc::CNT_ROWQ], static_cast<uint32_t>(__popc(have)));
    }
    pbase = __shfl_sync(0xffffffffu, pbase, 0) + (pre - cnt);
    qbase = __shfl_sync(0xffffffffu, qbase, 0) + __popc(have & ((1u << lane) - 1));
    if (cnt && pbase + cnt <= max_pairs) {           // (the host sizes the chunks so that this always holds)
      for (uint32_t j = 0; j < cnt; j++) {
        pair_row[pbase + j] = row;
        pair_cand[pbase + j] = gmem[beg + j];
      }
      rowq[3 * qbase] = row;
      rowq[3 * qbase + 1] = pbase;
      rowq[3 * qbase + 2] = cnt;
    } else if (cnt) {
      rowq[3 * qbase] = row;
      rowq[3 * qbase + 1] = 0;
      rowq[3 * qbase + 2] = 0;
    }
  }
}

__global__ void yy_own_reduce_kernel(const uint32_t* __restrict__ rowq, const uint32_t* __restrict__ d_nrowq,
                                     const uint32_t* __restrict__ pair_cand, const float* __restrict__ pair_score,
                                     const uint32_t* __restrict__ assign, const uint32_t* __restrict__ groups, uint32_t G,
                                     float* __restrict__ bounds) {
  const uint32_t nq = *d_nrowq;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += gridDim.x * blockDim.x) {
    const uint32_t row = rowq[3 * i], base = rowq[3 * i + 1], cnt = rowq[3 * i + 2];
    if (cnt == 0) continue;
    const uint32_t a = assign[row];
    float lb = FLT_MAX, ub = FLT_MAX;
    for (uint32_t j = 0; j < cnt; j++) {
      const float d = pair_score[base + j];
      if (pair_cand[base + j] == a) ub = d;
      else if (d < lb) lb = d;                       // NaN never lowers a bound (as the reference's `dist < bound`)
    }
    float* b = bounds + static_cast<size_t>(row) * (G + 1);
    b[0] = ub;
    b[1 + groups[a]] = lb;
  }
}

// Builds the group-sorted table layout from the centroid -> group map of this run (host vector, G groups; ids >= G
// mark dead centroids, which get no table row).  Call again whenever the grouping changes.
void tc_yy_layout_host(const uint32_t* host_groups, uint32_t K, uint32_t G, std::vector<uint32_t>* perm_out,
                       std::vector<uint32_t>* qgroup_out, std::vector<uint32_t>* goff_out,
                       std::vector<uint32_t>* gmem_out, int* nt3_out) {
  using namespace tc;
  std::vector<uint32_t> gsz(G, 0);
  for (uint32_t c = 0; c < K; c++)
    if (host_groups[c] < G) gsz[host_groups[c]]++;
  std::vector<uint32_t> goff(G + 1, 0), gfill(G, 0), gmem(K ? K : 1, 0);
  for (uint32_t g = 0; g < G; g++) goff[g + 1] = goff[g] + gsz[g];
  for (uint32_t c = 0; c < K; c++)
    if (host_groups[c] < G) gmem[goff[host_groups[c]] + gfill[host_groups[c]]++] = c;
  size_t rows = 0;
  for (uint32_t g = 0; g < G; g++) rows += (gsz[g] + 3) / 4 * 4;
  const int nt3 = static_cast<int>(std::max<size_t>(1, (rows + TN - 1) / TN));
  const size_t rows_pad = static_cast<size_t>(nt3) * TN;
  std::vector<uint32_t> perm(rows_pad, UINT32_MAX), qgroup(rows_pad / 4, UINT32_MAX);
  size_t r = 0;
  for (uint32_t g = 0; g < G; g++) {
    if (gsz[g] == 0) continue;
    for (uint32_t j = 0; j < gsz[g]; j++) perm[r + j] = gmem[goff[g] + j];
    const size_t padded = (gsz[g] + 3) / 4 * 4;
    for (size_t qd = r / 4; qd < (r + padded) / 4; qd++) qgroup[qd] = g;
    r += padded;
  }
  *perm_out = std::move(perm);
  *qgroup_out = std::move(qgroup);
  *goff_out = std::move(goff);
  *gmem_out = std::move(gmem);
  *nt3_out = nt3;
}

cudaError_t tc_yy_layout(TcPlan* p, const uint32_t* host_groups, uint32_t G) {
  using namespace tc;
  std::vector<uint32_t> perm, qgroup, goff, gmem;
  int nt3 = 0;
  tc_yy_layout_host(host_groups, p->K, G, &perm, &qgroup, &goff, &gmem, &nt3);
  const size_t rows_pad = static_cast<size_t>(nt3) * TN;
  cudaError_t e;
  if (nt3 != p->nt3 || !p->table3) {
    pool_free(p->table3); pool_free(p->aug_blob3); pool_free(p->yy_perm); pool_free(p->yy_qgroup);
    p->table3 = nullptr; p->aug_blob3 = nullptr; p->yy_perm = nullptr; p->yy_qgroup = nullptr;
    if ((e = pool_alloc(reinterpret_cast<void**>(&p->table3), rows_pad * p->nkb * KB * sizeof(__half))) != cudaSuccess) return e;
    if ((e = pool_alloc(reinterpret_cast<void**>(&p->aug_blob3), static_cast<size_t>(nt3) * AUG_B_BYTES)) != cudaSuccess) return e;
    if ((e = pool_alloc(reinterpret_cast<void**>(&p->yy_perm), rows_pad * sizeof(uint32_t))) != cudaSuccess) return e;
    if ((e = pool_alloc(reinterpret_cast<void**>(&p->yy_qgroup), rows_pad / 4 * sizeof(uint32_t))) != cudaSuccess) return e;
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return cudaErrorNotSupported;
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(p->nkb * KB), static_cast<cuuint64_t>(rows_pad)};
    cuuint64_t gstride[1] = {static_cast<cuuint64_t>(p->nkb * KB) * sizeof(__half)};
    cuuint32_t box[2] = {KB, TN};
    cuuint32_t estr[2] = {1, 1};
    if (enc(&p->tmap3, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, p->table3, gdim, gstride, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return cudaErrorInvalidValue;
    p->nt3 = nt3;
  }
  if (G != p->G3 || !p->yy_goff) {
    pool_free(p->yy_goff); pool_free(p->yy_gmem);
    p->yy_goff = nullptr; p->yy_gmem = nullptr;
    if ((e = pool_alloc(reinterpret_cast<void**>(&p->yy_goff), (static_cast<size_t>(G) + 1) * sizeof(uint32_t))) != cudaSuccess) return e;
    if ((e = pool_alloc(reinterpret_cast<void**>(&p->yy_gmem), gmem.size() * sizeof(uint32_t))) != cudaSuccess) return e;
    p->G3 = G;
  }
  p->yy_max_gsize = 0;
  for (uint32_t g = 0; g < G; g++) p->yy_max_gsize = std::max(p->yy_max_gsize, goff[g + 1] - goff[g]);
  if ((e = cudaMemcpy(p->yy_perm, perm.data(), perm.size() * 4, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
  if ((e = cudaMemcpy(p->yy_qgroup, qgroup.data(), qgroup.size() * 4, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
  if ((e = cudaMemcpy(p->yy_goff, goff.data(), goff.size() * 4, cudaMemcpyHostToDevice)) != cudaSuccess) return e;
  return cudaMemcpy(p->yy_gmem, gmem.data(), gmem.size() * 4, cudaMemcpyHostToDevice);
}

bool tc_yy_layout_ready(TcPlan* p, uint32_t G) { return p && p->table3 && p->G3 == G; }

// One bounds refresh: bounds[row] = {ub exact, lb[g] valid lower bounds} (see Params, MODE 3).  Rows the filter
// cannot bound are left on the overflow list (tc_queues) for the caller's exact row refresh.
cudaError_t tc_yy_refresh(TcPlan* p, const float* X, const float* C, const float* csq, uint32_t n,
                          const uint32_t* assign, const uint32_t* groups, uint32_t G, float* bounds, cudaStream_t st) {
  using namespace tc;
  if (n > p->max_n || !tc_yy_layout_ready(p, G)) return cudaErrorInvalidValue;
  if ((reinterpret_cast<uintptr_t>(X) & 15) || (reinterpret_cast<uintptr_t>(C) & 15)) return cudaErrorMisalignedAddress;
  cudaError_t e;
  CUtensorMap tmap_x;
  {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return cudaErrorNotSupported;
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(p->D), static_cast<cuuint64_t>(n)};
    cuuint64_t gstride[1] = {static_cast<cuuint64_t>(p->D) * sizeof(float)};
    cuuint32_t box[2] = {32, TM};
    cuuint32_t estr[2] = {1, 1};
    if (enc(&tmap_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(X), gdim, gstride, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return cudaErrorInvalidValue;
  }
  if ((e = launch_fill_u32(reinterpret_cast<uint32_t*>(bounds), 0x7f7fffffu /* FLT_MAX */,
                           static_cast<size_t>(n) * (G + 1), st)) != cudaSuccess)
    return e;
  Params prm;
  if ((e = tc_prepare(p, C, csq, n, &prm, st, true)) != cudaSuccess) return e;
  prm.yy_qgroup = p->yy_qgroup;
  prm.yy_groups = groups;
  prm.yy_assign = assign;
  prm.yy_bounds = bounds;
  prm.G = G;
  const unsigned grid = min(static_cast<uint32_t>(p->num_sms), prm.ntiles);
  tc_launch_main(3, p->nkb, grid, p->smem_bytes, st, p->tmap3, tmap_x, prm);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  // own group + upper bound, exactly: chunks of rows whose pairs fit the queue (yy_max_gsize members per row at most)
  const uint32_t per_row = max(1u, p->yy_max_gsize);
  const uint32_t chunk = max(1u, p->max_pairs / per_row);
  for (uint32_t r0 = 0; r0 < n; r0 += chunk) {
    const uint32_t r1 = min(n, r0 + chunk);
    if ((e = cudaMemsetAsync(p->counters, 0, sizeof(uint32_t) * 2, st)) != cudaSuccess) return e;   // CNT_PAIRS, CNT_ROWQ
    yy_own_pairs_kernel<<<p->num_sms * 8, 256, 0, st>>>(r0, r1, p->K, G, assign, groups, p->yy_goff, p->yy_gmem, p->pair_row,
                                                       p->pair_cand, p->max_pairs, p->rowq, p->counters);
    if ((e = tc_exact_distances(p, X, C, n, p->pair_row, p->pair_cand, p->counters + CNT_PAIRS, p->max_pairs,
                                p->pair_score, st)) != cudaSuccess)
      return e;
    yy_own_reduce_kernel<<<p->num_sms * 4, 256, 0, st>>>(p->rowq, p->counters + CNT_ROWQ, p->pair_cand, p->pair_score, assign,
                                                        groups, G, bounds);
  }
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  return cudaMemcpyAsync(p->h_counters, p->counters, sizeof(uint32_t) * CNT_N, cudaMemcpyDeviceToHost, st);
}

void tc_queues(TcPlan* p, TcQueues* q) {
  q->rowq = p->rowq;
  q->d_nrowq = p->counters + tc::CNT_ROWQ;
  q->pair_cand = p->pair_cand;
  q->pair_score = p->pair_score;
  q->ovf_rows = p->ovf_rows;
  q->d_novf = p->counters + tc::CNT_OVF;
}

// valid after the stream has been synchronised
void tc_last_stats(TcPlan* p, uint32_t* n_recheck, uint32_t* n_overflow) {
  *n_recheck = p->h_counters[tc::CNT_ROWQ];
  *n_overflow = p->h_counters[tc::CNT_OVF];
}

uint32_t tc_last_error(TcPlan* p) { return p->h_counters[tc::CNT_ERR]; }
void tc_set_capture(TcPlan* p, bool on) { p->capturing = on; }
uint32_t tc_last_pairs(TcPlan* p) { return p->h_counters[tc::CNT_PAIRS]; }

// device time (ms) of the main kernel in the most recent passes, oldest first; call after a sync
int tc_kernel_times(TcPlan* p, float* ms_out, int max_out) {
  const uint64_t have = p->passes < static_cast<uint64_t>(TcPlan::kEvRing) ? p->passes : TcPlan::kEvRing;
  const int n = static_cast<int>(have < static_cast<uint64_t>(max_out) ? have : max_out);
  for (int i = 0; i < n; i++) {
    // graph replays refresh the one slot that was captured; otherwise the ring holds one pair per pass
    const int slot = p->graph_slot >= 0 ? p->graph_slot : static_cast<int>((p->passes - n + i) % TcPlan::kEvRing);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p->ev0[slot], p->ev1[slot]) != cudaSuccess) ms = -1.f;
    ms_out[i] = ms;
  }
  return n;
}
void tc_debug_stats(TcPlan* p, float* out4) {
  tc::Stats st;
  cudaMemcpy(&st, p->stats, sizeof(st), cudaMemcpyDeviceToHost);
  out4[0] = st.scale;
  out4[1] = st.cmax;
  out4[2] = st.dcmax;
  out4[3] = __builtin_bit_cast(float, st.csq_max_bits);
}

// ===================================================================================================
// k-NN on the tensor cores (reference knn.cu:177-347: cluster-pruned exact k nearest neighbours)
//
// Queries and candidates are the samples in cluster-sorted order (the inverse assignment).  Pass 1 multiplies
// every query tile (<= 128 queries of one cluster) with the blocks covering its own cluster; that yields, per
// query, an upper bound of the distance to its k-th neighbour.  The reference's skip test
// `Cd[B][A] - d(q, A) - R[B] > kth` (knn.cu:218-225) is then evaluated per tile (a cluster is visited if ANY
// query of the tile needs it) and pass 2 visits the surviving clusters' blocks.  The epilogue records every
// column whose fp16 score is within the rigorous margin of the row's (k+1)-th best (self included); those
// candidates get their exact distance (reference METRIC::distance) and the k smallest are written in
// ascending order.  Any superset of the reference's visited clusters gives the same exact top-k.
// ===================================================================================================
namespace knn {

__global__ void tile_count_kernel(const uint32_t* __restrict__ off, uint32_t K, uint32_t* __restrict__ ntile) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < K) ntile[c] = (off[c + 1] - off[c] + tc::TM - 1) / tc::TM;
}

// per cluster: its blocks (= query tiles), the two own-cluster segments of pass 1
__global__ void tile_fill_kernel(const uint32_t* __restrict__ off, uint32_t K, const uint32_t* __restrict__ blk_first,
                                 uint32_t* __restrict__ tile_nrows, uint32_t* __restrict__ blk_cluster,
                                 uint2* __restrict__ ranges1, uint32_t* __restrict__ roff1,
                                 uint32_t* __restrict__ rcount1, uint32_t* __restrict__ nblk1,
                                 uint32_t* __restrict__ d_ntiles, unsigned long long* __restrict__ d_pairs) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= K) return;
  const uint32_t m = off[c + 1] - off[c];
  const uint32_t t0 = blk_first[c], nt = (m + tc::TM - 1) / tc::TM;
  for (uint32_t i = 0; i < nt; i++) {
    const uint32_t t = t0 + i;
    tile_nrows[t] = min(static_cast<uint32_t>(tc::TM), m - i * tc::TM);
    blk_cluster[t] = c;
    ranges1[2 * t] = ranges1[2 * t + 1] = make_uint2(t0, t0 + nt - 1);   // threshold sweep + recording sweep
    roff1[t] = 2 * t;
    rcount1[t] = 2;
    nblk1[t] = 2 * nt;
  }
  if (c == K - 1) *d_ntiles = t0 + nt;
}

// table row of every valid sorted position (cluster-aligned, zero padded): tab2orig[row] = original sample index
__global__ void layout_kernel(const uint32_t* __restrict__ inv, const uint32_t* __restrict__ assign,
                              const uint32_t* __restrict__ off, const uint32_t* __restrict__ blk_first, uint32_t nv,
                              uint32_t* __restrict__ tab2orig) {
  uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= nv) return;
  const uint32_t s = inv[pos], c = assign[s];
  tab2orig[blk_first[c] * tc::TM + (pos - off[c])] = s;
}

// one warp per table row: ||y - c||^2 (fp32) and the largest s-free magnitude |y| + |c| (for the centring error)
__global__ void prep_norms_kernel(const float* __restrict__ X, const float* __restrict__ C, int D,
                                  const uint32_t* __restrict__ tab2orig, const uint32_t* __restrict__ blk_cluster,
                                  const uint32_t* __restrict__ d_ntiles, float* __restrict__ ysq,
                                  float* __restrict__ yabs_max, int angular) {
  const uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= *d_ntiles * tc::TM) return;
  const uint32_t sidx = tab2orig[row];
  if (sidx == UINT32_MAX) {
    if (lane == 0) ysq[row] = 0.f;
    return;
  }
  const float* x = X + static_cast<size_t>(sidx) * D;
  const float* c = C + static_cast<size_t>(blk_cluster[row / tc::TM]) * D;
  float a = 0.f, r = 0.f;
  for (int f = lane; f < D; f += 32) {
    const float xv = x[f], cv = c[f], d = xv - cv, m = fabsf(xv) + fabsf(cv);
    a = fmaf(d, d, a);
    r = fmaf(m, m, r);
  }
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    r += __shfl_xor_sync(0xffffffffu, r, o);
  }
  if (lane == 0) {
    ysq[row] = a;
    if (r == r && r < 3.0e38f) atomicMax(reinterpret_cast<uint32_t*>(yabs_max), __float_as_uint(__fsqrt_ru(r)));
  }
  if (angular) {   // deviation of the sample from unit length (yabs_max[1]); NaN / Inf rows count as "far off"
    float xx = 0.f;
    for (int f = lane; f < D; f += 32) xx = fmaf(x[f], x[f], xx);
    for (int o = 16; o > 0; o >>= 1) xx += __shfl_xor_sync(0xffffffffu, xx, o);
    const float dev = fabsf(xx - 1.f) + 4.0e-6f * (1.f + xx);    // + the fp32 rounding of the sum itself
    if (lane == 0) atomicMax(reinterpret_cast<uint32_t*>(yabs_max + 1), (dev == dev) ? __float_as_uint(dev) : 0x7f800000u);
  }
}

// one warp per table row: fp16(s (y - c)), rounding residual, bias -(s^2 |y - c|^2 / 2) in three fp16 terms;
// padding and non-finite rows: zero vector, bias -65504
__global__ void prep_table_kernel(const float* __restrict__ X, const float* __restrict__ C, int D, int nkb,
                                  const uint32_t* __restrict__ tab2orig, const uint32_t* __restrict__ blk_cluster,
                                  const uint32_t* __restrict__ d_ntiles, const float* __restrict__ ysq,
                                  __half* __restrict__ table, __half* __restrict__ aug_blob,
                                  tc::Stats* __restrict__ st, const float* __restrict__ yabs_max, int angular,
                                  uint32_t* __restrict__ d_error) {
  using namespace tc;
  const uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= *d_ntiles * TM) return;
  const int Dp = nkb * KB;
  const float s = st->scale;
  if (row == 0 && lane == 0) {
    st->yabs = *yabs_max * s * 1.0001f;
    st->knn_extra = 0.f;
    if (angular) {
      // angular neighbours through the L2 pass: for |1 - |y|^2| <= eps the true top-k by dot product lie within
      // s^2 * eps of the (k+1)-th best L2 score (x.y = (|x|^2 + |y|^2 - d^2) / 2), so the margin grows by that much;
      // samples far from unit length make the equivalence useless -> the caller runs the exact search instead
      const float eps = yabs_max[1];
      if (!(eps <= 1.0e-2f)) *d_error = 2u;
      st->knn_extra = (s * s) * eps * 1.01f;
    }
  }
  const uint32_t sidx = tab2orig[row];
  bool finite = sidx != UINT32_MAX;
  const float* x = X + static_cast<size_t>(finite ? sidx : 0) * D;
  const float* c = C + static_cast<size_t>(blk_cluster[row / TM]) * D;
  if (finite) {
    const float q = ysq[row];
    finite = (q == q) && q < 3.0e38f;
    finite = __all_sync(0xffffffffu, finite);
  }
  float d2 = 0.f;
  for (int f = lane; f < Dp; f += 32) {
    const float v = (finite && f < D) ? (x[f] - c[f]) * s : 0.f;
    const __half h = __float2half_rn(v);
    const float r = v - __half2float(h);
    d2 = fmaf(r, r, d2);
    table[static_cast<size_t>(row) * Dp + f] = h;
  }
  for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
  if (lane == 0) {
    if (finite) atomicMax(reinterpret_cast<uint32_t*>(&st->dcmax), __float_as_uint(__fsqrt_ru(d2) * 1.0001f));
    __half b[3];
    if (finite) {
      const float hh = -0.5f * ((s * ysq[row]) * s);
      b[0] = __float2half_rn(hh);
      const float r1 = hh - __half2float(b[0]);
      b[1] = __float2half_rn(r1);
      b[2] = __float2half_rn(r1 - __half2float(b[1]));
    } else {
      b[0] = __float2half_rn(-65504.f);
      b[1] = b[2] = __float2half_rn(0.f);
    }
    const uint32_t t = row / TN, r = row % TN;
    __half* blob = aug_blob + static_cast<size_t>(t) * (AUG_B_BYTES / 2);
    for (int k = 0; k < 16; k++) {
      const int j = k >> 3, e = k & 7;
      blob[(j * (TN * 16) + (r >> 3) * 128 + (r & 7) * 16) / 2 + e] = k < 3 ? b[k] : __float2half_rn(0.f);
    }
  }
}

// one warp per tile: the clusters pass 2 must visit, one segment (block range) per cluster
__global__ void __launch_bounds__(256)
range_build_kernel(const uint32_t* __restrict__ d_ntiles, const uint32_t* __restrict__ tile_nrows,
                   const uint32_t* __restrict__ blk_cluster, const uint32_t* __restrict__ blk_first,
                   const uint32_t* __restrict__ off, uint32_t K, const float* __restrict__ cd,
                   const float* __restrict__ radii, const float* __restrict__ ysq, const float* __restrict__ dub,
                   uint2* __restrict__ pool, uint32_t pool_cap, uint32_t* __restrict__ pool_used,
                   uint32_t* __restrict__ roff2, uint32_t* __restrict__ rcount2, uint32_t* __restrict__ nblk2,
                   uint32_t* __restrict__ d_error, unsigned long long* __restrict__ d_pairs, uint32_t part,
                   uint32_t nparts) {
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t T = *d_ntiles;
  const uint32_t t_lo = static_cast<uint32_t>(static_cast<uint64_t>(T) * part / nparts);
  const uint32_t t_hi = static_cast<uint32_t>(static_cast<uint64_t>(T) * (part + 1) / nparts);
  for (uint32_t t = t_lo + warp; t < t_hi; t += nwarps) {
    const uint32_t nr = tile_nrows[t], A = blk_cluster[t];
    // W = max over the tile's queries of d(q, A) + (upper bound of the distance to the k-th neighbour so far);
    // d(q, A) is bounded by the fp32 centred norm (the reference's Kahan value differs by rounding only)
    float W = 0.f;
    for (uint32_t r = lane; r < nr; r += 32) {
      const uint32_t row = t * tc::TM + r;
      const float w = __fsqrt_ru(ysq[row]) * 1.00001f + fminf(dub[2 * row], dub[2 * row + 1]);
      W = (w == w) ? fmaxf(W, w) : INFINITY;
    }
    for (int o = 16; o > 0; o >>= 1) W = fmaxf(W, __shfl_xor_sync(0xffffffffu, W, o));
    W = W * 1.000002f + 1e-30f;   // the reference rounds `cd - dA - R` twice: stay on the visiting side
    for (int pass = 0; pass < 2; pass++) {   // pass 0 counts, pass 1 writes
      uint32_t count = 0, blocks = 0, base = 0;
      unsigned long long pairs = 0;
      if (pass == 0 && lane == 0 && A < K) pairs = static_cast<unsigned long long>(nr) * (off[A + 1] - off[A]);   // own cluster
      if (pass == 1) {
        const uint32_t c0 = rcount2[t];
        if (lane == 0) base = atomicAdd(pool_used, c0);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base + c0 > pool_cap) {
          if (lane == 0) { *d_error = 1u; rcount2[t] = 0; nblk2[t] = 0; roff2[t] = 0; }
          break;
        }
        if (lane == 0) roff2[t] = base;
      }
      for (uint32_t B0 = 0; B0 < K; B0 += 32) {
        const uint32_t B = B0 + lane;
        bool visit = false;
        uint32_t lo = 0, hi = 0;
        if (B < K && B != A) {
          const uint32_t m = off[B + 1] - off[B];
          const float c = cd[static_cast<size_t>(B) * K + A];
          if (m && c == c && !(c - radii[B] > W)) {
            visit = true;
            lo = blk_first[B];
            hi = blk_first[B + 1] - 1;
            pairs += static_cast<unsigned long long>(m) * nr;
          }
        }
        const unsigned mk = __ballot_sync(0xffffffffu, visit);
        if (visit) {
          if (pass == 1) pool[base + count + __popc(mk & ((1u << lane) - 1))] = make_uint2(lo, hi);
        }
        uint32_t nb = visit ? hi - lo + 1 : 0;
        for (int o = 16; o > 0; o >>= 1) nb += __shfl_xor_sync(0xffffffffu, nb, o);
        blocks += nb;
        count += __popc(mk);
      }
      if (pass == 0) {
        if (lane == 0) { rcount2[t] = count; nblk2[t] = blocks; }
        for (int o = 16; o > 0; o >>= 1) pairs += __shfl_xor_sync(0xffffffffu, pairs, o);
        if (lane == 0 && pairs) atomicAdd(d_pairs, pairs);
        __syncwarp();
      }
    }
  }
}

// one warp per query (table row): final threshold, expansion of the recorded entries into candidate pairs
__global__ void __launch_bounds__(256)
expand_kernel(const uint32_t* __restrict__ d_ntiles, int kk, uint32_t stride, const float* __restrict__ topk,
              const uint32_t* __restrict__ cnts, const uint32_t* __restrict__ flags,
              const uint4* __restrict__ entries, const uint32_t* __restrict__ tab2orig, uint32_t max_pairs,
              uint32_t* __restrict__ pair_row, uint32_t* __restrict__ pair_cand, uint32_t* __restrict__ rowq,
              uint32_t* __restrict__ fb_rows, uint32_t* __restrict__ counters, uint32_t* __restrict__ dbg,
              uint32_t part, uint32_t nparts) {
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t T = *d_ntiles;
  const uint32_t row_lo = static_cast<uint32_t>(static_cast<uint64_t>(T) * part / nparts) * tc::TM;
  const uint32_t nrows = static_cast<uint32_t>(static_cast<uint64_t>(T) * (part + 1) / nparts) * tc::TM;
  for (uint32_t row = row_lo + warp; row < nrows; row += nwarps) {
    const uint32_t self = tab2orig[row];
    if (self == UINT32_MAX) continue;   // padding
    const uint32_t s0 = 2 * row, s1 = 2 * row + 1;
    const float k0 = topk[static_cast<size_t>(kk - 1) * stride + s0], k1 = topk[static_cast<size_t>(kk - 1) * stride + s1];
    const float kth = fmaxf(k0, k1);   // each half saw kk distinct columns at or above its own value
    const uint32_t fl = flags[s0] | flags[s1];
    const uint32_t c0 = cnts[s0], c1 = cnts[s1];
    bool fallback = fl != 0 || !(kth > -INFINITY);
    if (lane == 0 && dbg) {
      if (fl & 1) atomicAdd(dbg + 0, 1u);
      if (fl & 2) atomicAdd(dbg + 1, 1u);
      if (fl & 4) atomicAdd(dbg + 2, 1u);
      if (!(kth > -INFINITY)) atomicAdd(dbg + 3, 1u);
    }
    // each lane takes entries lane, lane+32, ... of the concatenated (half 0, half 1) lists; an entry survives if
    // its group maximum is within ITS margin of the final kk-th best
    uint32_t mine = 0;
    const uint32_t total_e = c0 + c1;
    for (uint32_t i = lane; i < total_e && !fallback; i += 32) {
      const uint4 e = i < c0 ? entries[static_cast<size_t>(s0) * tc::KNN_CAP + i]
                             : entries[static_cast<size_t>(s1) * tc::KNN_CAP + (i - c0)];
      if (__uint_as_float(e.x) >= kth - __uint_as_float(e.w)) {
        uint32_t m = e.y;
        const uint32_t p0 = (e.z >> 2) * 128u + ((e.z >> 1) & 1u) * 64u + (e.z & 1u) * 32u;
        while (m) {
          const uint32_t cp = p0 + __ffs(m) - 1;
          m &= m - 1;
          if (cp != row && tab2orig[cp] != UINT32_MAX) mine++;
        }
      }
    }
    uint32_t pre = mine;
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t v = __shfl_up_sync(0xffffffffu, pre, o);
      if (lane >= o) pre += v;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, pre, 31);
    if (lane == 0 && dbg && !fallback) {
      if (total > 64) atomicAdd(dbg + 4, 1u);
      if (total < static_cast<uint32_t>(kk - 1)) atomicAdd(dbg + 5, 1u);
      atomicAdd(dbg + 6, total);
    }
    if (total > 64 || total < static_cast<uint32_t>(kk - 1)) fallback = true;
    uint32_t base = 0;
    if (!fallback) {
      if (lane == 0) base = atomicAdd(&counters[tc::CNT_PAIRS], total);
      base = __shfl_sync(0xffffffffu, base, 0);
      if (base + total > max_pairs) fallback = true;
    }
    if (fallback) {
      if (lane == 0) fb_rows[atomicAdd(&counters[tc::CNT_OVF], 1u)] = self;
      continue;
    }
    uint32_t w = base + pre - mine;
    for (uint32_t i = lane; i < total_e; i += 32) {
      const uint4 e = i < c0 ? entries[static_cast<size_t>(s0) * tc::KNN_CAP + i]
                             : entries[static_cast<size_t>(s1) * tc::KNN_CAP + (i - c0)];
      if (__uint_as_float(e.x) >= kth - __uint_as_float(e.w)) {
        uint32_t m = e.y;
        const uint32_t p0 = (e.z >> 2) * 128u + ((e.z >> 1) & 1u) * 64u + (e.z & 1u) * 32u;
        while (m) {
          const uint32_t cp = p0 + __ffs(m) - 1;
          m &= m - 1;
          const uint32_t o = tab2orig[cp];
          if (cp != row && o != UINT32_MAX) {
            pair_row[w] = self;
            pair_cand[w] = o;
            w++;
          }
        }
      }
    }
    if (lane == 0) {
      const uint32_t q = atomicAdd(&counters[tc::CNT_ROWQ], 1u);
      rowq[3 * q] = self;
      rowq[3 * q + 1] = base;
      rowq[3 * q + 2] = total;
    }
  }
}

// one warp per query: the k smallest exact distances in ascending order (knn.cu:239-242)
__global__ void __launch_bounds__(256)
select_kernel(int k, const uint32_t* __restrict__ rowq, const uint32_t* __restrict__ counters,
              const uint32_t* __restrict__ pair_cand, const float* __restrict__ pair_score, uint32_t q_offset,
              uint32_t* __restrict__ neighbors) {
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t nq = counters[tc::CNT_ROWQ];
  for (uint32_t q = warp; q < nq; q += nwarps) {
    const uint32_t row = rowq[3 * q], base = rowq[3 * q + 1], cnt = rowq[3 * q + 2];
    float d[2];
    uint32_t id[2];
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const uint32_t i = lane + 32 * j;
      d[j] = INFINITY;
      id[j] = UINT32_MAX;
      if (i < cnt) {
        const float v = pair_score[base + i];
        if (v == v) { d[j] = v; id[j] = pair_cand[base + i]; }
      }
    }
    for (int r = 0; r < k; r++) {
      // lexicographic (distance, index) minimum over the 64 slots
      float bd = d[0];
      uint32_t bi = id[0];
      if (d[1] < bd || (d[1] == bd && id[1] < bi)) { bd = d[1]; bi = id[1]; }
      for (int o = 16; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(0xffffffffu, bd, o);
        const uint32_t oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (od < bd || (od == bd && oi < bi)) { bd = od; bi = oi; }
      }
      if (lane == 0) neighbors[static_cast<size_t>(row - q_offset) * k + r] = bi;
      if (id[0] == bi) { d[0] = INFINITY; id[0] = UINT32_MAX; }
      if (id[1] == bi) { d[1] = INFINITY; id[1] = UINT32_MAX; }
    }
  }
}

}  // namespace knn

bool tc_knn_supported(int metric, int k, uint32_t N, int D, uint32_t K) {
  // (the angular metric is served through the L2 pass when the samples have unit length, see tc_knn_search)
  if (k + 1 > tc::KNN_MAX_KK) return false;
  if (D < 4 || D % 4 != 0 || D > tc::MAX_NKB * tc::KB) return false;
  if (N < 4096 || N > (1u << 30)) return false;                    // tiny inputs: not worth the set-up
  if (static_cast<uint64_t>(K) * K > (1ull << 31)) return false;
  return true;
}

#define KNN_TRY(x) do { e = (x); if (e != cudaSuccess) goto done; } while (0)

// neighbors: device array [N][k] indexed by the original sample index (this build shards k-NN queries only on the
// SIMT path).  Rows the filter cannot serve are appended to fb_rows / d_nfb for the caller's exact search.
cudaError_t tc_knn_search(int metric, int k, const float* X, const float* C, uint32_t N, int D, uint32_t K,
                          const uint32_t* assign, const uint32_t* inv, const uint32_t* off, const float* cd,
                          const float* radii, uint32_t nv, uint32_t* neighbors, uint32_t* fb_rows, uint32_t* d_nfb,
                          unsigned long long* d_pairs, uint32_t* h_error, uint32_t part, uint32_t nparts,
                          cudaStream_t st) {
  using namespace tc;
  cudaError_t e = cudaSuccess;
  *h_error = 0;
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return cudaErrorNotSupported;
  int dev = 0, num_sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  const int nkb = (D + KB - 1) / KB, kk = k + 1;
  const uint32_t tmax = nv / TM + K + 1;                 // upper bound of the number of cluster-aligned blocks
  const uint32_t rows_max = tmax * TM;
  const uint32_t stride = 2 * rows_max;
  const uint64_t want_pool = static_cast<uint64_t>(tmax) * K;
  const uint32_t pool_cap = static_cast<uint32_t>(want_pool < (48u << 20) ? want_pool : (48u << 20));
  const uint32_t pair_cap = static_cast<uint32_t>(std::min<uint64_t>(40ull * nv + 4096, 0xFFFFFFF0ull));
  __half *table = nullptr, *blobs = nullptr;
  float *ysq = nullptr, *topk = nullptr, *dub = nullptr, *pair_score = nullptr, *yabs = nullptr;
  Stats* stats = nullptr;
  uint32_t *u32 = nullptr, *kcnt = nullptr, *kflags = nullptr, *pair_row = nullptr, *pair_cand = nullptr, *rowq = nullptr;
  uint32_t *counters = nullptr, *tab2orig = nullptr;
  uint2 *ranges1 = nullptr, *pool = nullptr;
  uint4* entries = nullptr;
  void* cub_tmp = nullptr;
  size_t cub_bytes = 0;
  uint32_t h_cnt[CNT_N + 2] = {0};
  uint32_t h_dbg[8] = {0};
  CUtensorMap tmap;
  Params prm;
  const unsigned grid = static_cast<unsigned>(num_sms);
  const size_t smem_bytes = smem_layout().total + 1024;
  uint32_t *ntile, *blk_first, *t_nrows, *blk_cluster, *roff1, *rcount1, *nblk1, *roff2, *rcount2, *nblk2, *d_ntiles,
      *pool_used, *d_err;
  {
    const size_t words = static_cast<size_t>(K) + (K + 1) + 8ull * tmax + 16;
    KNN_TRY(pool_alloc(reinterpret_cast<void**>(&u32), words * sizeof(uint32_t)));
    KNN_TRY(cudaMemsetAsync(u32, 0, words * sizeof(uint32_t), st));
    uint32_t* q = u32;
    ntile = q; q += K;
    blk_first = q; q += K + 1;
    t_nrows = q; q += tmax; blk_cluster = q; q += tmax;
    roff1 = q; q += tmax; rcount1 = q; q += tmax; nblk1 = q; q += tmax;
    roff2 = q; q += tmax; rcount2 = q; q += tmax; nblk2 = q; q += tmax;
    d_ntiles = q++; pool_used = q++; d_err = q++;   // pool_used + 2 .. + 9: debug counters of expand_kernel
  }
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&table), static_cast<size_t>(rows_max) * nkb * KB * sizeof(__half)));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&blobs), static_cast<size_t>(tmax) * AUG_B_BYTES));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&ysq), sizeof(float) * rows_max));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&yabs), 2 * sizeof(float)));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&stats), sizeof(Stats)));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&tab2orig), sizeof(uint32_t) * rows_max));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&topk), sizeof(float) * static_cast<size_t>(kk) * stride));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&dub), sizeof(float) * stride));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&kcnt), sizeof(uint32_t) * stride));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&kflags), sizeof(uint32_t) * stride));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&entries), sizeof(uint4) * static_cast<size_t>(stride) * KNN_CAP));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&ranges1), sizeof(uint2) * 2ull * tmax));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&pool), sizeof(uint2) * pool_cap));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&pair_row), sizeof(uint32_t) * pair_cap));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&pair_cand), sizeof(uint32_t) * pair_cap));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&pair_score), sizeof(float) * pair_cap));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&rowq), sizeof(uint32_t) * 3ull * nv));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&counters), sizeof(uint32_t) * CNT_N));
  KNN_TRY(cudaMemsetAsync(counters, 0, sizeof(uint32_t) * CNT_N, st));
  KNN_TRY(cudaMemsetAsync(stats, 0, sizeof(Stats), st));
  KNN_TRY(cudaMemsetAsync(yabs, 0, 2 * sizeof(float), st));
  KNN_TRY(cudaMemsetAsync(ysq, 0, sizeof(float) * rows_max, st));   // rows past the last block stay 0 for the max
  KNN_TRY(cudaMemsetAsync(kcnt, 0, sizeof(uint32_t) * stride, st));
  KNN_TRY(cudaMemsetAsync(kflags, 0, sizeof(uint32_t) * stride, st));
  KNN_TRY(cudaMemsetAsync(tab2orig, 0xff, sizeof(uint32_t) * rows_max, st));
  KNN_TRY(tc_set_smem_attr(static_cast<int>(smem_bytes), nkb));
  // cluster-aligned table layout: blocks per cluster, first block of every cluster, table row -> sample
  knn::tile_count_kernel<<<(K + 255) / 256, 256, 0, st>>>(off, K, ntile);
  KNN_TRY(cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, ntile, blk_first, static_cast<int>(K), st));
  KNN_TRY(pool_alloc(reinterpret_cast<void**>(&cub_tmp), cub_bytes ? cub_bytes : 16));
  KNN_TRY(cub::DeviceScan::ExclusiveSum(cub_tmp, cub_bytes, ntile, blk_first, static_cast<int>(K), st));
  knn::tile_fill_kernel<<<(K + 255) / 256, 256, 0, st>>>(off, K, blk_first, t_nrows, blk_cluster, ranges1, roff1, rcount1,
                                                         nblk1, d_ntiles, d_pairs);
  KNN_TRY(cudaMemcpyAsync(blk_first + K, d_ntiles, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
  knn::layout_kernel<<<(nv + 255) / 256, 256, 0, st>>>(inv, assign, off, blk_first, nv, tab2orig);
  // fp16 table of the centred samples + bias blobs + statistics
  knn::prep_norms_kernel<<<(rows_max / 8) + 1, 256, 0, st>>>(X, C, D, tab2orig, blk_cluster, d_ntiles, ysq, yabs, metric);
  tc_prep_stats_kernel<<<8, 256, 0, st>>>(ysq, rows_max, stats);
  tc_prep_scale_kernel<<<1, 1, 0, st>>>(stats);
  knn::prep_table_kernel<<<(rows_max / 8) + 1, 256, 0, st>>>(X, C, D, nkb, tab2orig, blk_cluster, d_ntiles, ysq, table,
                                                             blobs, stats, yabs, metric, d_err);
  KNN_TRY(cudaGetLastError());
  {
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(nkb * KB), static_cast<cuuint64_t>(rows_max)};
    cuuint64_t gstride[1] = {static_cast<cuuint64_t>(nkb * KB) * sizeof(__half)};
    cuuint32_t box[2] = {KB, TN};
    cuuint32_t estr[2] = {1, 1};
    CUresult cr = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, table, gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { e = cudaErrorInvalidValue; goto done; }
  }
  prm.n = N; prm.D = D; prm.K = K; prm.nkb = nkb; prm.nt = 0; prm.ntiles = 0;
  prm.aug_blob = blobs; prm.stats = stats; prm.result = nullptr; prm.pair_row = nullptr; prm.pair_cand = nullptr;
  prm.max_pairs = 0; prm.rowq = nullptr; prm.ovf_rows = nullptr; prm.counters = counters; prm.metric = 0;
  prm.X = X; prm.rows = tab2orig; prm.d_nrows = nullptr; prm.d_ntiles = d_ntiles; prm.tile_nrows = t_nrows;
  prm.blk_cluster = blk_cluster; prm.C = C;
  prm.knn_ranges = ranges1; prm.knn_roff = roff1; prm.knn_rcount = rcount1; prm.knn_nblk = nblk1;
  prm.kk = kk; prm.knn_first_pass = 1; prm.knn_stride = stride; prm.knn_topk = topk;
  prm.knn_cnt = kcnt; prm.knn_flags = kflags; prm.knn_dub = dub; prm.knn_entries = entries;
  prm.neg_mu_s = nullptr; prm.assign = prm.prev = prm.d_changed = nullptr;
  prm.yy_qgroup = prm.yy_groups = prm.yy_assign = nullptr; prm.yy_bounds = nullptr; prm.G = 0;
  prm.knn_part = part; prm.knn_nparts = nparts ? nparts : 1;
  tc_launch_main(2, nkb, grid, smem_bytes, st, tmap, tmap, prm);
  KNN_TRY(cudaGetLastError());
  knn::range_build_kernel<<<num_sms * 4, 256, 0, st>>>(d_ntiles, t_nrows, blk_cluster, blk_first, off, K, cd, radii, ysq,
                                                       dub, pool, pool_cap, pool_used, roff2, rcount2, nblk2, d_err,
                                                       d_pairs, part, prm.knn_nparts);
  KNN_TRY(cudaGetLastError());
  prm.knn_ranges = pool; prm.knn_roff = roff2; prm.knn_rcount = rcount2; prm.knn_nblk = nblk2; prm.knn_first_pass = 0;
  tc_launch_main(2, nkb, grid, smem_bytes, st, tmap, tmap, prm);
  KNN_TRY(cudaGetLastError());
  knn::expand_kernel<<<num_sms * 8, 256, 0, st>>>(d_ntiles, kk, stride, topk, kcnt, kflags, entries, tab2orig, pair_cap,
                                                  pair_row, pair_cand, rowq, fb_rows, counters, pool_used + 2, part,
                                                  prm.knn_nparts);
  KNN_TRY(cudaGetLastError());
  // the exact distance of every candidate pair in the CALLER's metric (angular: acos of the Kahan dot product)
  if (metric == 1)
    recheck_pairs_kernel<1, 1><<<num_sms * 4, 128, 0, st>>>(X, X, nullptr, D, pair_row, pair_cand, counters + CNT_PAIRS,
                                                            pair_cap, N, N, pair_score);
  else
    recheck_pairs_kernel<0, 1><<<num_sms * 4, 128, 0, st>>>(X, X, nullptr, D, pair_row, pair_cand, counters + CNT_PAIRS,
                                                            pair_cap, N, N, pair_score);
  knn::select_kernel<<<num_sms * 8, 256, 0, st>>>(k, rowq, counters, pair_cand, pair_score, 0u, neighbors);
  KNN_TRY(cudaGetLastError());
  KNN_TRY(cudaMemcpyAsync(h_cnt, counters, sizeof(uint32_t) * CNT_N, cudaMemcpyDeviceToHost, st));
  KNN_TRY(cudaMemcpyAsync(h_cnt + CNT_N, d_err, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  KNN_TRY(cudaMemcpyAsync(d_nfb, counters + CNT_OVF, sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
  KNN_TRY(cudaMemcpyAsync(h_dbg, pool_used + 2, sizeof(h_dbg), cudaMemcpyDeviceToHost, st));
  KNN_TRY(cudaStreamSynchronize(st));
  *h_error = h_cnt[CNT_ERR] | (h_cnt[CNT_N] ? 0x80000000u : 0u);
  if (getenv("KMCUDA_B200_TIMING"))
    fprintf(stderr, "[kmcuda_b200 timing]   knn tensor-core path: %u rows, %u candidate pairs, %u rows to the exact search, "
            "error word 0x%x; fallback reasons: nan/inf %u, list full %u, tiny diff %u, no threshold %u, >64 cand %u, "
            "<k cand %u; candidates seen %u\n", h_cnt[CNT_ROWQ], h_cnt[CNT_PAIRS], h_cnt[CNT_OVF], *h_error, h_dbg[0],
            h_dbg[1], h_dbg[2], h_dbg[3], h_dbg[4], h_dbg[5], h_dbg[6]);
done:
  pool_free(u32); pool_free(table); pool_free(blobs); pool_free(ysq); pool_free(yabs); pool_free(stats); pool_free(tab2orig);
  pool_free(topk); pool_free(dub); pool_free(kcnt); pool_free(kflags); pool_free(entries); pool_free(ranges1);
  pool_free(pool); pool_free(pair_row); pool_free(pair_cand); pool_free(pair_score); pool_free(rowq); pool_free(counters);
  pool_free(cub_tmp);
  return e;
}
#undef KNN_TRY

}  // namespace kmb
