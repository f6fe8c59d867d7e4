// shard.cu -- per-GPU hot-path steps + the shard-level C ABI (include/kmcuda_b200.h).
#include "shard.h"

#include <cstdlib>
#include <map>
#include <mutex>
#include <new>
#include <unordered_map>

#include "kmcuda_b200.h"

namespace kmb {

// ---------------------------------------------------------------------------------------------------
// device-memory cache (see shard.h)
// ---------------------------------------------------------------------------------------------------
namespace {
struct PoolState {
  std::mutex mu;
  std::map<int, std::multimap<size_t, void*>> free_blocks;          // per device: size -> block
  std::unordered_map<void*, std::pair<int, size_t>> live;           // block -> (device, size)
  std::map<int, size_t> cached_bytes;
  size_t cap = 0;
  bool cap_read = false;
};
PoolState& pool_state() {
  static PoolState st;
  return st;
}
size_t pool_round(size_t bytes) {
  if (bytes < 512) bytes = 512;
  const size_t q = bytes >= (1u << 20) ? (2u << 20) : 512;          // 2 MB granules for large blocks
  return (bytes + q - 1) / q * q;
}
}  // namespace

cudaError_t pool_alloc(void** p, size_t bytes) {
  PoolState& st = pool_state();
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const size_t want = pool_round(bytes);
  {
    std::lock_guard<std::mutex> lk(st.mu);
    if (!st.cap_read) {
      const char* c = getenv("KMCUDA_B200_CACHE_MB");
      st.cap = (c ? static_cast<size_t>(strtoull(c, nullptr, 10)) : 24576u) << 20;
      st.cap_read = true;
    }
    auto& fb = st.free_blocks[dev];
    auto it = fb.lower_bound(want);
    if (it != fb.end() && it->first <= want + want / 4) {           // close enough in size: reuse
      *p = it->second;
      st.live[*p] = {dev, it->first};
      st.cached_bytes[dev] -= it->first;
      fb.erase(it);
      return cudaSuccess;
    }
  }
  e = cudaMalloc(p, want);
  if (e != cudaSuccess) {                                            // out of memory: give the cache back and retry once
    cudaGetLastError();
    pool_trim();
    e = cudaMalloc(p, want);
    if (e != cudaSuccess) return e;
  }
  std::lock_guard<std::mutex> lk(st.mu);
  st.live[*p] = {dev, want};
  return cudaSuccess;
}

void pool_free(void* p) {
  if (!p) return;
  PoolState& st = pool_state();
  int dev = -1;
  size_t size = 0;
  bool keep = false;
  {
    std::lock_guard<std::mutex> lk(st.mu);
    auto it = st.live.find(p);
    if (it == st.live.end()) {       // not ours (should not happen): plain free
      cudaFree(p);
      return;
    }
    dev = it->second.first;
    size = it->second.second;
    st.live.erase(it);
    if (st.cap && st.cached_bytes[dev] + size <= st.cap) {
      st.free_blocks[dev].emplace(size, p);
      st.cached_bytes[dev] += size;
      keep = true;
    }
  }
  if (!keep) {
    int cur = 0;
    cudaGetDevice(&cur);
    if (cur != dev) cudaSetDevice(dev);
    cudaFree(p);
    if (cur != dev) cudaSetDevice(cur);
  }
}

void pool_trim() {
  PoolState& st = pool_state();
  std::lock_guard<std::mutex> lk(st.mu);
  int cur = 0;
  cudaGetDevice(&cur);
  for (auto& kv : st.free_blocks) {
    cudaSetDevice(kv.first);
    for (auto& b : kv.second) cudaFree(b.second);
    kv.second.clear();
    st.cached_bytes[kv.first] = 0;
  }
  cudaSetDevice(cur);
}

Shard::~Shard() {
  cudaSetDevice(device);
  if (assign_graph) cudaGraphExecDestroy(assign_graph);
  if (tc) tc_plan_destroy(tc);
}

KMCUDAResult Shard::create(bool with_update) {
  KMB_CU(cudaSetDevice(device), kmcudaNoSuchDevice);
  const char* fe = getenv("KMCUDA_B200_FORCE_EXACT");
  force_exact = fe && fe[0] == '1';
  const char* su = getenv("KMCUDA_B200_STRICT_UPDATE");
  strict_update = su && su[0] == '1';
  const char* ug = getenv("KMCUDA_B200_GRAPH");
  use_graph = ug && ug[0] == '1';
  KMB_CU(csq.alloc(K), kmcudaMemoryAllocationFailure);
  KMB_CU(result.alloc(max_n), kmcudaMemoryAllocationFailure);
  if (with_update) {
    KMB_CU(ws_keys_out.alloc(max_n), kmcudaMemoryAllocationFailure);
    KMB_CU(ws_vals_in.alloc(max_n), kmcudaMemoryAllocationFailure);
    KMB_CU(ws_vals_out.alloc(max_n), kmcudaMemoryAllocationFailure);
    KMB_CU(ws_offsets.alloc(static_cast<size_t>(K) + 1), kmcudaMemoryAllocationFailure);
    KMB_CU(ws_partial.alloc(update_partial_rows(max_n, K) * D), kmcudaMemoryAllocationFailure);
    ws.cub_tmp_bytes = update_cub_bytes(max_n);
    KMB_CU(ws_cub.alloc(ws.cub_tmp_bytes), kmcudaMemoryAllocationFailure);
    ws.keys_out = ws_keys_out;
    ws.vals_in = ws_vals_in;
    ws.vals_out = ws_vals_out;
    ws.offsets = ws_offsets;
    ws.partial = ws_partial;
    ws.cub_tmp = ws_cub.get();
    if (metric == 1) {
      KMB_CU(prev_sums.alloc(static_cast<size_t>(K) * D), kmcudaMemoryAllocationFailure);
      KMB_CU(cudaMemset(prev_sums.get(), 0, sizeof(float) * static_cast<size_t>(K) * D), kmcudaRuntimeError);
    }
  }
  if (!force_exact && tc_supported(metric, max_n, D, K)) {
    cudaError_t e = tc_plan_create(&tc, metric, max_n, D, K, device);
    if (e != cudaSuccess) {
      // No silent fallback: a shape the tensor-core path claims must get the tensor-core path.
      KMB_INFO("tensor-core plan creation failed: %s\n", cudaGetErrorString(e));
      tc = nullptr;
      return e == cudaErrorMemoryAllocation ? kmcudaMemoryAllocationFailure : kmcudaRuntimeError;
    }
  }
  return kmcudaSuccess;
}

KMCUDAResult Shard::enable_yinyang(uint32_t groups_size) {
  KMB_CU(cudaSetDevice(device), kmcudaNoSuchDevice);
  G = groups_size;
  KMB_CU(bounds.alloc(static_cast<size_t>(max_n) * (G + 1)), kmcudaMemoryAllocationFailure);
  KMB_CU(drift.alloc(K), kmcudaMemoryAllocationFailure);
  KMB_CU(maxdrift.alloc(G), kmcudaMemoryAllocationFailure);
  KMB_CU(oldC.alloc(static_cast<size_t>(K) * D), kmcudaMemoryAllocationFailure);
  KMB_CU(passed.alloc(max_n), kmcudaMemoryAllocationFailure);
  KMB_CU(groups.alloc(K), kmcudaMemoryAllocationFailure);
  KMB_CU(yy_counters.alloc(4), kmcudaMemoryAllocationFailure);
  KMB_CU(yy_minlb.alloc(max_n), kmcudaMemoryAllocationFailure);
  KMB_CU(yy_tight_rows.alloc(max_n), kmcudaMemoryAllocationFailure);
  KMB_CU(yy_tight_cand.alloc(max_n), kmcudaMemoryAllocationFailure);
  KMB_CU(yy_tight_score.alloc(max_n), kmcudaMemoryAllocationFailure);
  KMB_CU(yy_gsize.alloc(G), kmcudaMemoryAllocationFailure);
  return kmcudaSuccess;
}

// start of a run (the counts are reset to zero by the caller): forget the cached member sums (cosine update)
KMCUDAResult Shard::reset_update_state(cudaStream_t st) {
  if (prev_sums.get())
    KMB_CU(cudaMemsetAsync(prev_sums.get(), 0, sizeof(float) * static_cast<size_t>(K) * D, st), kmcudaRuntimeError);
  return kmcudaSuccess;
}

// after `groups` (device) has been filled; host_groups is the same map on the host
KMCUDAResult Shard::yy_prepare(const uint32_t* host_groups, cudaStream_t st) {
  KMB_CU(launch_yy_group_sizes(groups, K, G, yy_gsize, st), kmcudaRuntimeError);
  const char* er = getenv("KMCUDA_B200_YY_EXACT_REFRESH");   // A/B and parity tests: exact SIMT refresh
  if (tc && !force_exact && !(er && er[0] == '1'))
    KMB_CU(tc_yy_layout(tc, host_groups, G), kmcudaMemoryAllocationFailure);
  return kmcudaSuccess;
}

// Bounds refresh.  Tensor-core route (assign_tc.cu MODE 3): one distance GEMM against the group-sorted table gives
// valid lower bounds for every other group, the own centroid / own group are exact, rows the filter cannot bound
// are refreshed exactly.  Exact route: the reference's full pass (N * K exact distances).
KMCUDAResult Shard::yy_refresh(uint32_t n, const float* X, const float* C, const uint32_t* assignments,
                               cudaStream_t st) {
  if (n > max_n) return kmcudaInvalidArguments;
  if (n == 0) return kmcudaSuccess;
  if (tc && tc_yy_layout_ready(tc, G)) {
    KMB_CU(launch_csqr(metric, C, K, D, csq, st), kmcudaRuntimeError);
    KMB_CU(tc_yy_refresh(tc, X, C, csq, n, assignments, groups, G, bounds, st), kmcudaRuntimeError);
    TcQueues q;
    tc_queues(tc, &q);
    KMB_CU(launch_yy_init_rows(metric, X, C, n, D, K, G, assignments, groups, bounds, q.ovf_rows, q.d_novf, st),
           kmcudaRuntimeError);
    return kmcudaSuccess;
  }
  KMB_CU(launch_yy_init(metric, X, C, n, D, K, G, assignments, groups, bounds, st), kmcudaRuntimeError);
  return kmcudaSuccess;
}

// one Yinyang iteration after the centroid update: reference kmeans.cu:1180-1262 (drifts, global and local filter)
KMCUDAResult Shard::yy_step(uint32_t n, const float* X, const float* C, uint32_t* assignments, uint32_t* prev,
                            uint32_t* d_changed, cudaStream_t st) {
  if (n > max_n) return kmcudaInvalidArguments;
  KMB_CU(launch_yy_drifts(metric, C, oldC, K, D, G, groups, drift, maxdrift, st), kmcudaRuntimeError);
  if (tc) KMB_CU(launch_csqr(metric, C, K, D, csq, st), kmcudaRuntimeError);
  YyWorkspace ws{yy_minlb, yy_tight_rows, yy_tight_cand, yy_tight_score, passed, yy_gsize, yy_counters};
  KMB_CU(launch_yy_step(metric, tc, X, C, csq, n, D, K, G, groups, drift, maxdrift, assignments, prev, bounds, ws,
                        d_changed, force_exact, st), kmcudaRuntimeError);
  return kmcudaSuccess;
}

KMCUDAResult Shard::assign(uint32_t n, const float* X, const float* C, uint32_t* assignments,
                           uint32_t* prev, uint32_t* d_changed, cudaStream_t st) {
  if (n > max_n) return kmcudaInvalidArguments;
  // (the tensor-core pass computes ||c||^2 in its own preparation launch)
  if (!(tc && n > 0)) KMB_CU(launch_csqr(metric, C, K, D, csq, st), kmcudaRuntimeError);
  last_tc = false;
  if (tc && n > 0 && use_graph && st != nullptr) {   // (the legacy default stream cannot be captured)
    GraphKey key;
    key.X = X; key.C = C; key.a = assignments; key.prev = prev; key.ch = d_changed; key.n = n; key.st = st;
    if (!(assign_graph && key == graph_key)) {
      if (assign_graph) { cudaGraphExecDestroy(assign_graph); assign_graph = nullptr; }
      cudaGraph_t g = nullptr;
      KMB_CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal), kmcudaRuntimeError);
      tc_set_capture(tc, true);
      cudaError_t e2 = tc_assign(tc, X, C, csq, n, result, assignments, prev, d_changed, st, true);
      tc_set_capture(tc, false);
      cudaError_t e3 = cudaStreamEndCapture(st, &g);
      if (e2 != cudaSuccess || e3 != cudaSuccess || !g) {
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        KMB_INFO("CUDA graph capture of the assignment pass failed (%s / %s)\n", cudaGetErrorString(e2), cudaGetErrorString(e3));
        return kmcudaRuntimeError;
      }
      cudaError_t e4 = cudaGraphInstantiate(&assign_graph, g, 0);
      cudaGraphDestroy(g);
      KMB_CU(e4, kmcudaRuntimeError);
      graph_key = key;
    }
    KMB_CU(cudaGraphLaunch(assign_graph, st), kmcudaRuntimeError);
    last_tc = true;
    return kmcudaSuccess;
  }
  if (tc && n > 0) {
    KMB_CU(tc_assign(tc, X, C, csq, n, result, assignments, prev, d_changed, st, true), kmcudaRuntimeError);
    last_tc = true;
  } else {
    KMB_CU(launch_assign_exact(metric, X, C, csq, n, D, K, nullptr, nullptr, result, st),
           kmcudaRuntimeError);
    KMB_CU(launch_finalize_assign(n, result, assignments, prev, d_changed, st), kmcudaRuntimeError);
  }
  return kmcudaSuccess;
}

KMCUDAResult Shard::update_reference_order(uint32_t n, const float* X, const uint32_t* assignments,
                                           const uint32_t* prev, float* C, uint32_t* ccounts, cudaStream_t st) {
  if (n > max_n) return kmcudaInvalidArguments;
  if (!su_keys_in.get()) {   // first use: event buffers (2 entries per sample)
    const size_t m = 2 * static_cast<size_t>(max_n);
    KMB_CU(su_keys_in.alloc(m), kmcudaMemoryAllocationFailure);
    KMB_CU(su_vals_in.alloc(m), kmcudaMemoryAllocationFailure);
    KMB_CU(su_keys_out.alloc(m), kmcudaMemoryAllocationFailure);
    KMB_CU(su_vals_out.alloc(m), kmcudaMemoryAllocationFailure);
    KMB_CU(su_offsets.alloc(static_cast<size_t>(K) + 2), kmcudaMemoryAllocationFailure);
    su_cub_bytes = strict_update_cub_bytes(max_n);
    KMB_CU(su_cub.alloc(su_cub_bytes), kmcudaMemoryAllocationFailure);
  }
  KMB_CU(launch_strict_update(metric, X, n, D, K, prev, assignments, C, ccounts, su_keys_in, su_vals_in, su_keys_out,
                              su_vals_out, su_offsets, su_cub.get(), su_cub_bytes, st), kmcudaRuntimeError);
  return kmcudaSuccess;
}

KMCUDAResult Shard::check_pipeline() {
  if (!tc) return kmcudaSuccess;
  const uint32_t err = tc_last_error(tc);
  if (err == 0) return kmcudaSuccess;
  // never a silent success on garbage: the caller gets an error code (reference convention: RuntimeError)
  KMB_INFO("tensor-core pipeline error 0x%x on device %d: a barrier wait timed out, the pass is invalid\n", err, device);
  return kmcudaRuntimeError;
}

KMCUDAResult Shard::partial_sums(uint32_t n, const float* X, const uint32_t* assignments, float* sums,
                                 uint32_t* counts, cudaStream_t st) {
  if (n > max_n || ws.cub_tmp == nullptr) return kmcudaInvalidArguments;
  KMB_CU(launch_partial_sums(X, n, D, K, assignments, ws, sums, counts, st), kmcudaRuntimeError);
  return kmcudaSuccess;
}

KMCUDAResult Shard::finish_update(const float* sums, const uint32_t* counts, float* C,
                                  uint32_t* ccounts, cudaStream_t st) {
  KMB_CU(launch_normalize(metric, sums, counts, K, D, C, ccounts, prev_sums, st), kmcudaRuntimeError);
  return kmcudaSuccess;
}

}  // namespace kmb

// ---------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------
struct kmcuda_b200_shard {
  kmb::Shard* impl;
};

extern "C" {

KMCUDAResult kmcuda_b200_shard_create(kmcuda_b200_shard** shard, KMCUDADistanceMetric metric,
                                      uint32_t max_samples, uint16_t features_size,
                                      uint32_t clusters_size, int32_t verbosity) {
  if (!shard || features_size == 0 || clusters_size < 2 || clusters_size == UINT32_MAX)
    return kmcudaInvalidArguments;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return kmcudaNoSuchDevice;
  auto* impl = new (std::nothrow) kmb::Shard(metric == kmcudaDistanceMetricCosine ? 1 : 0, dev,
                                             max_samples, features_size, clusters_size, verbosity);
  if (!impl) return kmcudaMemoryAllocationFailure;
  KMCUDAResult r = impl->create(true);
  if (r != kmcudaSuccess) {
    delete impl;
    return r;
  }
  *shard = new kmcuda_b200_shard{impl};
  return kmcudaSuccess;
}

void kmcuda_b200_shard_destroy(kmcuda_b200_shard* shard) {
  if (!shard) return;
  delete shard->impl;
  delete shard;
}

KMCUDAResult kmcuda_b200_assign(kmcuda_b200_shard* shard, uint32_t samples_size, const float* samples,
                                const float* centroids, uint32_t* assignments,
                                uint32_t* assignments_prev, uint32_t* changed, void* stream) {
  if (!shard || !samples || !centroids || !assignments || !assignments_prev || !changed)
    return kmcudaInvalidArguments;
  return shard->impl->assign(samples_size, samples, centroids, assignments, assignments_prev, changed,
                             static_cast<cudaStream_t>(stream));
}

int32_t kmcuda_b200_last_pass_info(kmcuda_b200_shard* shard, uint32_t* rechecked, uint32_t* overflowed) {
  if (!shard) return 0;
  kmb::Shard* s = shard->impl;
  if (s->last_tc && s->tc) kmb::tc_last_stats(s->tc, &s->last_rechecked, &s->last_overflowed);
  else s->last_rechecked = s->last_overflowed = 0;
  if (rechecked) *rechecked = s->last_rechecked;
  if (overflowed) *overflowed = s->last_overflowed;
  return s->last_tc ? 1 : 0;
}

KMCUDAResult kmcuda_b200_partial_sums(kmcuda_b200_shard* shard, uint32_t samples_size,
                                      const float* samples, const uint32_t* assignments, float* sums,
                                      uint32_t* counts, void* stream) {
  if (!shard || !samples || !assignments || !sums || !counts) return kmcudaInvalidArguments;
  return shard->impl->partial_sums(samples_size, samples, assignments, sums, counts,
                                   static_cast<cudaStream_t>(stream));
}

KMCUDAResult kmcuda_b200_finish_update(kmcuda_b200_shard* shard, const float* sums,
                                       const uint32_t* counts, float* centroids, uint32_t* ccounts,
                                       void* stream) {
  if (!shard || !sums || !counts || !centroids || !ccounts) return kmcudaInvalidArguments;
  return shard->impl->finish_update(sums, counts, centroids, ccounts, static_cast<cudaStream_t>(stream));
}

KMCUDAResult kmcuda_b200_shard_reset(kmcuda_b200_shard* shard, void* stream) {
  if (!shard) return kmcudaInvalidArguments;
  return shard->impl->reset_update_state(static_cast<cudaStream_t>(stream));
}

uint32_t kmcuda_b200_last_error(kmcuda_b200_shard* shard) {
  if (!shard || !shard->impl->tc) return 0;
  return kmb::tc_last_error(shard->impl->tc);
}

// ---- diagnostics (used by tests; not part of the drop-in surface) ----
// returns the pipeline error word of the last tensor-core pass (0 = clean); call after a sync
uint32_t kmcuda_b200_debug_last_error(kmcuda_b200_shard* shard) {
  if (!shard || !shard->impl->tc) return 0;
  return kmb::tc_last_error(shard->impl->tc);
}
// device time (ms) of the tensor-core kernel in the most recent passes (CUDA events on the launching
// stream), oldest first; returns how many were written.  Call after synchronising the stream.
int32_t kmcuda_b200_kernel_times(kmcuda_b200_shard* shard, float* ms_out, int32_t max_out) {
  if (!shard || !shard->impl->tc || !ms_out) return 0;
  return kmb::tc_kernel_times(shard->impl->tc, ms_out, max_out);
}
// Yinyang bounds of one refresh (reference kmeans_yy_init) for the given assignments / grouping: use_tc = 1 takes the
// tensor-core route (valid lower bounds), 0 the exact pass.  bounds_out: device [n][G + 1].  Synchronous.
int32_t kmcuda_b200_debug_yy_bounds(kmcuda_b200_shard* shard, uint32_t n, const float* samples, const float* centroids,
                                    const uint32_t* assignments, const uint32_t* host_groups, uint32_t G,
                                    int32_t use_tc, float* bounds_out) {
  if (!shard || !samples || !centroids || !assignments || !host_groups || !bounds_out || G == 0) return -1;
  kmb::Shard* s = shard->impl;
  if (n > s->max_n) return -2;
  if (s->enable_yinyang(G) != kmcudaSuccess) return -3;
  if (cudaMemcpy(s->groups.get(), host_groups, sizeof(uint32_t) * s->K, cudaMemcpyHostToDevice) != cudaSuccess) return -4;
  cudaStream_t st = nullptr;
  if (use_tc) {
    if (!s->tc) return -5;
    if (kmb::tc_yy_layout(s->tc, host_groups, G) != cudaSuccess) return -6;
    if (s->yy_refresh(n, samples, centroids, assignments, st) != kmcudaSuccess) return -7;
  } else {
    if (kmb::launch_yy_init(s->metric, samples, centroids, n, s->D, s->K, G, assignments, s->groups, s->bounds, st) !=
        cudaSuccess)
      return -8;
  }
  if (cudaMemcpyAsync(bounds_out, s->bounds.get(), sizeof(float) * static_cast<size_t>(n) * (G + 1),
                      cudaMemcpyDeviceToDevice, st) != cudaSuccess)
    return -9;
  if (cudaStreamSynchronize(st) != cudaSuccess) return -10;
  return (use_tc && kmb::tc_last_error(s->tc)) ? -11 : 0;
}
int32_t kmcuda_b200_debug_stats(kmcuda_b200_shard* shard, float* out4) {
  if (!shard || !shard->impl->tc) return -1;
  kmb::tc_debug_stats(shard->impl->tc, out4);
  return 0;
}

// host layout of the Yinyang refresh table (assign_tc.cu::tc_yy_layout_host) for tests: perm_out [cap], qgroup_out
// [cap / 4]; returns the number of 128-row n-tiles, or -1 if cap is too small
int32_t kmcuda_b200_debug_yy_layout(uint32_t K, uint32_t G, const uint32_t* host_groups, uint32_t cap,
                                    uint32_t* perm_out, uint32_t* qgroup_out) {
  if (!host_groups || !perm_out || !qgroup_out) return -1;
  std::vector<uint32_t> perm, qgroup, goff, gmem;
  int nt3 = 0;
  kmb::tc_yy_layout_host(host_groups, K, G, &perm, &qgroup, &goff, &gmem, &nt3);
  if (perm.size() > cap) return -1;
  for (size_t i = 0; i < perm.size(); i++) perm_out[i] = perm[i];
  for (size_t i = 0; i < qgroup.size(); i++) qgroup_out[i] = qgroup[i];
  return nt3;
}

// the static (offset, length) split of `amount` rows over `ndev` devices that kmeans_cuda / knn_cuda use
// (api.cu::split_rows = the rule of the reference's distribute(), private.h:240-273); out: 2 * ndev values
int32_t kmcuda_b200_debug_split_rows(uint32_t amount, uint32_t row_bytes, uint32_t ndev, uint32_t* out) {
  if (!out || ndev == 0) return -1;
  auto plan = kmb::split_rows(amount, row_bytes, ndev);
  for (uint32_t i = 0; i < ndev; i++) {
    out[2 * i] = plan[i].first;
    out[2 * i + 1] = plan[i].second;
  }
  return 0;
}

// releases the device memory the library keeps cached between calls (see shard.h)
void kmcuda_b200_trim_cache(void) { kmb::pool_trim(); }

KMCUDAResult kmcuda_b200_device_malloc(int32_t device, uint64_t bytes, void** ptr) {
  if (!ptr) return kmcudaInvalidArguments;
  if (cudaSetDevice(device) != cudaSuccess) return kmcudaNoSuchDevice;
  return cudaMalloc(ptr, bytes ? bytes : 1) == cudaSuccess ? kmcudaSuccess : kmcudaMemoryAllocationFailure;
}

KMCUDAResult kmcuda_b200_device_free(int32_t device, void* ptr) {
  if (cudaSetDevice(device) != cudaSuccess) return kmcudaNoSuchDevice;
  return cudaFree(ptr) == cudaSuccess ? kmcudaSuccess : kmcudaRuntimeError;
}

KMCUDAResult kmcuda_b200_device_memcpy(int32_t device, void* dst, const void* src, uint64_t bytes,
                                       int32_t direction) {
  if (cudaSetDevice(device) != cudaSuccess) return kmcudaNoSuchDevice;
  cudaMemcpyKind kind = direction == 1 ? cudaMemcpyHostToDevice
                        : direction == 2 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  return cudaMemcpy(dst, src, bytes, kind) == cudaSuccess ? kmcudaSuccess : kmcudaMemoryCopyError;
}

KMCUDAResult kmcuda_b200_device_synchronize(int32_t device) {
  if (cudaSetDevice(device) != cudaSuccess) return kmcudaNoSuchDevice;
  return cudaDeviceSynchronize() == cudaSuccess ? kmcudaSuccess : kmcudaRuntimeError;
}

int32_t kmcuda_b200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

}  // extern "C"
