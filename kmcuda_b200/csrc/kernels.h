// kernels.h -- host-callable launchers of the device code (one CUDA stream per device context).
//
// Two families:
//   * exact kernels (simt_kernels.cu, knn_kernels.cu): bit-for-bit the reference's fp32 arithmetic
//     (exact.cuh); they make every decision that leaves the library.
//   * the tensor-core filter (assign_tc.cu): tcgen05 fp16 distance GEMM that proposes, per sample,
//     the short list of centroids the exact re-check has to look at.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <vector>

namespace kmb {

// Device-memory cache (shard.cu).  kmeans_cuda / knn_cuda allocate their whole workspace at entry like the reference
// (wrappers.h:16-21); on a B200 the GB-sized cudaMalloc / cudaFree pairs of a call cost more than its kernels (round 1:
// 0.30 of 0.38 s of a 3 M-point knn_cuda), so freed blocks are kept per device and handed to the next call.  Blocks are
// only returned here after the owning stream has been synchronised.  KMCUDA_B200_CACHE_MB caps what is kept (default
// 24576; 0 disables the cache); kmcuda_b200_trim_cache() releases everything.
cudaError_t pool_alloc(void** p, size_t bytes);   // on the current device
void pool_free(void* p);
void pool_trim();

constexpr uint32_t kUntouched = 0xFFFFFFFEu;  // "no centroid won": leave the assignment alone

// ---- exact Lloyd assignment (all K centroids), optional row list -------------------------------
// result[i] = argmin (strict <, ascending index), K for "insane" rows, kUntouched if nothing wins.
// rows == nullptr: rows 0..n-1; else the n row ids in rows[] (device), results still indexed by row.
cudaError_t launch_csqr(int metric, const float* C, uint32_t K, int D, float* csq, cudaStream_t st);
cudaError_t launch_assign_exact(int metric, const float* X, const float* C, const float* csq,
                                uint32_t n, int D, uint32_t K, const uint32_t* rows,
                                const uint32_t* d_nrows, uint32_t* result, cudaStream_t st);

// prev[i]=assign[i]; assign[i]=result[i] unless kUntouched; *changed += #(assign changed)
cudaError_t launch_finalize_assign(uint32_t n, const uint32_t* result, uint32_t* assign,
                                   uint32_t* prev, uint32_t* d_changed, cudaStream_t st);

// ---- centroid update ----------------------------------------------------------------------------
// Deterministic: stable radix sort of (assignment, index), then per-cluster Kahan sums in index order.
struct UpdateWorkspace {
  uint32_t *keys_in = nullptr, *keys_out = nullptr, *vals_in = nullptr, *vals_out = nullptr;
  uint32_t* offsets = nullptr;   // [K+1]
  float* partial = nullptr;      // [update_partial_rows(max_n, K)][D]: one row per (chunk, cluster) run
  void* cub_tmp = nullptr;
  size_t cub_tmp_bytes = 0;
  uint32_t iota_n = 0;           // vals_in[0 .. iota_n) already holds the identity permutation
};
constexpr uint32_t kSumChunk = 512;   // sorted positions per CTA of the member-sum kernel
size_t update_partial_rows(uint32_t n, uint32_t K);
size_t update_cub_bytes(uint32_t n);
// sums[K][D] (fp32) and counts[K] (uint32) of this shard's samples
cudaError_t launch_partial_sums(const float* X, uint32_t n, int D, uint32_t K, const uint32_t* assign,
                                UpdateWorkspace& ws, float* sums, uint32_t* counts, cudaStream_t st);
// strict parity mode: the reference's running-sum update replayed in sample order (simt_kernels.cu)
size_t strict_update_cub_bytes(uint32_t n);
cudaError_t launch_strict_update(int metric, const float* X, uint32_t n, int D, uint32_t K, const uint32_t* prev,
                                 const uint32_t* cur, float* C, uint32_t* ccounts, uint32_t* keys_in,
                                 uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out, uint32_t* offsets,
                                 void* cub_tmp, size_t cub_bytes, cudaStream_t st);
// multi-GPU exchange through peer memory: out_sums = sums[0] + sums[1] + ... (device order, so every GPU computes
// the same bits), out_counts likewise; the pointers may live on other GPUs (peer access enabled by the caller)
constexpr int kMaxPeers = 32;
struct PeerBuffers {
  int n;
  const float* sums[kMaxPeers];
  const uint32_t* counts[kMaxPeers];
};
cudaError_t launch_peer_reduce(const PeerBuffers& pb, uint32_t K, int D, float* out_sums, uint32_t* out_counts,
                               cudaStream_t st);
// C = sums/count (L2, NaN for empty) or sums/||sums|| (cosine); ccounts = counts
cudaError_t launch_normalize(int metric, const float* sums, const uint32_t* counts, uint32_t K, int D,
                             float* C, uint32_t* ccounts, float* prev_sums, cudaStream_t st);

// ---- Yinyang -------------------------------------------------------------------------------------
// bounds layout [n][G+1] (one contiguous record per sample): [0] = upper bound, [1+g] = lower bound of group g
cudaError_t launch_yy_init(int metric, const float* X, const float* C, uint32_t n, int D, uint32_t K,
                           uint32_t G, const uint32_t* assign, const uint32_t* groups, float* bounds,
                           cudaStream_t st);
// exact refresh of the listed rows only (rows[0 .. *d_nrows))
cudaError_t launch_yy_init_rows(int metric, const float* X, const float* C, uint32_t n, int D, uint32_t K,
                                uint32_t G, const uint32_t* assign, const uint32_t* groups, float* bounds,
                                const uint32_t* rows, const uint32_t* d_nrows, cudaStream_t st);
cudaError_t launch_yy_drifts(int metric, const float* Cnew, const float* Cold, uint32_t K, int D,
                             uint32_t G, const uint32_t* groups, float* drift, float* maxdrift,
                             cudaStream_t st);
struct TcPlan;
// one Yinyang iteration after the centroid update (yinyang.cu): bound decay + group filter, exact tightening of
// the upper bound, tensor-core candidate pass over the surviving rows, bound / assignment update
struct YyWorkspace {
  float* minlb;            // [n]
  uint32_t* tight_rows;    // [n]
  uint32_t* tight_cand;    // [n]
  float* tight_score;      // [n]
  uint32_t* passed;        // [n]
  uint32_t* gsize;         // [G] members per group (NaN centroids excluded)
  uint32_t* counters;      // [4]: tight, passed, (spare)
};
cudaError_t launch_yy_group_sizes(const uint32_t* groups, uint32_t K, uint32_t G, uint32_t* gsize, cudaStream_t st);
cudaError_t launch_yy_step(int metric, TcPlan* plan, const float* X, const float* C, const float* csq, uint32_t n,
                           int D, uint32_t K, uint32_t G, const uint32_t* groups, const float* drift,
                           const float* maxdrift, uint32_t* assign, uint32_t* prev, float* bounds,
                           const YyWorkspace& ws, uint32_t* d_changed, bool reference_order_scan, cudaStream_t st);

// ---- misc ------------------------------------------------------------------------------------------
cudaError_t launch_average_distance(int metric, const float* X, const float* C, uint32_t n, int D,
                                    const uint32_t* assign, double* d_sum, cudaStream_t st);
cudaError_t launch_afkmc2_min_dist(int metric, const float* X, const float* C, int D, uint32_t k,
                                   const uint32_t* rows, uint32_t m, float* min_dists, cudaStream_t st);
cudaError_t launch_plusplus_step(int metric, const float* X, uint32_t n, int D, const float* centroid,
                                 int first, float* dists, double* d_sum, cudaStream_t st);
// device-resident k-means++ round (simt_kernels.cu): bsum / bpre hold ceil(n / 256) + 1 doubles, chosen [K]
cudaError_t launch_plusplus_round(int metric, const float* X, uint32_t n, int D, float* C, uint32_t i, double choice,
                                  float* dists, double* bsum, double* bpre, uint32_t* chosen, cudaStream_t st);
cudaError_t launch_half_to_float(const void* src, float* dst, size_t n, cudaStream_t st);
cudaError_t launch_float_to_half(const float* src, void* dst, size_t n, cudaStream_t st);
cudaError_t launch_fill_u32(uint32_t* p, uint32_t v, size_t n, cudaStream_t st);

// ---- k-NN ------------------------------------------------------------------------------------------
// inverse assignments: inv[] = sample ids sorted by (cluster, id), off[K+1] = CSR offsets
cudaError_t launch_knn_inverse(const uint32_t* assign, uint32_t n, uint32_t K, uint32_t* iota,
                               uint32_t* keys_out, uint32_t* inv, uint32_t* off, uint32_t* counts,
                               UpdateWorkspace& ws, cudaStream_t st);
cudaError_t launch_knn_radii(int metric, const float* X, const float* C, uint32_t n, int D, uint32_t K,
                             const uint32_t* assign, float* radii, cudaStream_t st);
cudaError_t launch_knn_centroid_distances(int metric, const float* C, uint32_t K, int D, float* cd,
                                          cudaStream_t st);
cudaError_t launch_knn_search(int metric, int k, const float* X, const float* C, uint32_t N, int D,
                              uint32_t K, uint32_t q_offset, uint32_t q_length, const uint32_t* assign,
                              const uint32_t* inv, const uint32_t* inv_off, const float* cd,
                              const float* radii, float* heap_scratch, uint32_t* neighbors,
                              unsigned long long* d_pairs, const uint32_t* rows, const uint32_t* d_nrows,
                              cudaStream_t st);
cudaError_t launch_knn_radii_fix(const uint32_t* inv_off, uint32_t K, float* radii, cudaStream_t st);
cudaError_t launch_knn_tail_rows(const uint32_t* inv, uint32_t nv, uint32_t n, uint32_t* rows, uint32_t* d_nrows,
                                 cudaStream_t st);

// ---- tensor-core filter (assign_tc.cu) -----------------------------------------------------------
struct TcPlan;  // opaque; owns the fp16 centroid table, tensor maps, queues
bool tc_supported(int metric, uint32_t n, int D, uint32_t K);
cudaError_t tc_plan_create(TcPlan** plan, int metric, uint32_t max_n, int D, uint32_t K, int device);
void tc_plan_destroy(TcPlan* plan);
// one full assignment pass.  assign == nullptr: result[i] as launch_assign_exact would produce it.  Otherwise the
// pass's bookkeeping (launch_finalize_assign) is fused: prev[i] = assign[i], assign[i] = winner, *d_changed +=
// changes; result[] is then scratch for the few rows that take the exact full pass.
// compute_csq: csq[] (the caller's buffer, K floats) is filled by the pass's own preparation launch (what launch_csqr
// would write) instead of being read as an input.
cudaError_t tc_assign(TcPlan* plan, const float* X, const float* C, const float* csq, uint32_t n,
                      uint32_t* result, uint32_t* assign, uint32_t* prev, uint32_t* d_changed, cudaStream_t st,
                      bool compute_csq = false);
// statistics of the last pass (for logging / bench): queue length and overflow rows
void tc_last_stats(TcPlan* plan, uint32_t* n_recheck, uint32_t* n_overflow);
// Yinyang local step (assign_tc.cu): candidate pairs with exact true distances for the listed rows
struct TcQueues {
  const uint32_t* rowq;       // [3*i]: row, first pair, pair count
  const uint32_t* d_nrowq;
  const uint32_t* pair_cand;
  const float* pair_score;    // exact distance of (row, pair_cand)
  const uint32_t* ovf_rows;   // rows the filter could not bound
  const uint32_t* d_novf;
};
cudaError_t tc_yy_candidates(TcPlan* plan, const float* X, const float* C, const float* csq, uint32_t n,
                             const uint32_t* rows, const uint32_t* d_nrows, cudaStream_t st);
cudaError_t tc_exact_distances(TcPlan* plan, const float* X, const float* C, uint32_t n, const uint32_t* pair_row,
                               const uint32_t* pair_cand, const uint32_t* d_npairs, uint32_t max_pairs,
                               float* pair_score, cudaStream_t st);
void tc_queues(TcPlan* plan, TcQueues* q);
// Yinyang bounds refresh on the tensor cores (assign_tc.cu, MODE 3): tc_yy_layout once per grouping (host map
// centroid -> group), then tc_yy_refresh per refresh; rows left on the overflow list need launch_yy_init_rows
cudaError_t tc_yy_layout(TcPlan* plan, const uint32_t* host_groups, uint32_t G);
// the host part of tc_yy_layout (pure function): table row -> centroid (UINT32_MAX = padding), group of every
// 4-row quad, CSR of the group members, number of 128-row n-tiles
void tc_yy_layout_host(const uint32_t* host_groups, uint32_t K, uint32_t G, std::vector<uint32_t>* perm,
                       std::vector<uint32_t>* qgroup, std::vector<uint32_t>* goff, std::vector<uint32_t>* gmem,
                       int* nt3);
bool tc_yy_layout_ready(TcPlan* plan, uint32_t G);
cudaError_t tc_yy_refresh(TcPlan* plan, const float* X, const float* C, const float* csq, uint32_t n,
                          const uint32_t* assign, const uint32_t* groups, uint32_t G, float* bounds, cudaStream_t st);
// k-NN candidate search on the tensor cores (assign_tc.cu); see the comment there
bool tc_knn_supported(int metric, int k, uint32_t N, int D, uint32_t K);
// metric 1 (angular): candidates come from the L2 pass (cd / radii must then be the L2 quantities), the margin is
// widened by the samples' deviation from unit length, exact distances and the selection use the angular metric; if the
// samples are not unit vectors (deviation > 1e-2) *h_error is set and the caller has to run the exact search
cudaError_t tc_knn_search(int metric, int k, const float* X, const float* C, uint32_t N, int D, uint32_t K,
                          const uint32_t* assign, const uint32_t* inv, const uint32_t* off, const float* cd,
                          const float* radii, uint32_t nv, uint32_t* neighbors, uint32_t* fb_rows, uint32_t* d_nfb,
                          unsigned long long* d_pairs, uint32_t* h_error, uint32_t part, uint32_t nparts,
                          cudaStream_t st);
// several GPUs: every device serves part `part` of `nparts` of the query tiles into its own full-size neighbour
// array (pre-filled with 0xFFFFFFFF); the arrays are merged with an element-wise minimum over peer memory
struct PeerU32 {
  int n;
  const uint32_t* p[kMaxPeers];
};
cudaError_t launch_peer_min_u32(const PeerU32& pb, size_t count, uint32_t* out, cudaStream_t st);
// 0 = clean; 0x1000+site = a pipeline wait timed out at `site` (results of that pass are invalid)
uint32_t tc_last_error(TcPlan* plan);
uint32_t tc_last_pairs(TcPlan* plan);
void tc_set_capture(TcPlan* plan, bool on);   // the next tc_assign is recorded into a CUDA graph (stream capture)
int tc_kernel_times(TcPlan* plan, float* ms_out, int max_out);
// diagnostics: prep statistics
void tc_debug_stats(TcPlan* plan, float* out4);

}  // namespace kmb
