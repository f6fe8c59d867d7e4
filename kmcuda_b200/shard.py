"""Python mirror of the shard-level C ABI (include/kmcuda_b200.h) over torch device tensors.

torch is plumbing here: it owns device memory and streams (and, in bench.py / multi-process jobs,
the NCCL communicator).  Every computation goes through libKMCUDA.so.
"""
import ctypes

import numpy as np
import torch

from . import _lib, _raise_for

_lib.kmcuda_b200_shard_create.restype = ctypes.c_int
_lib.kmcuda_b200_shard_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_uint32,
                                          ctypes.c_uint16, ctypes.c_uint32, ctypes.c_int32]
_lib.kmcuda_b200_shard_destroy.restype = None
_lib.kmcuda_b200_shard_destroy.argtypes = [ctypes.c_void_p]
_lib.kmcuda_b200_assign.restype = ctypes.c_int
_lib.kmcuda_b200_assign.argtypes = [ctypes.c_void_p, ctypes.c_uint32] + [ctypes.c_void_p] * 6
_lib.kmcuda_b200_last_pass_info.restype = ctypes.c_int32
_lib.kmcuda_b200_last_pass_info.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint32),
                                            ctypes.POINTER(ctypes.c_uint32)]
_lib.kmcuda_b200_partial_sums.restype = ctypes.c_int
_lib.kmcuda_b200_partial_sums.argtypes = [ctypes.c_void_p, ctypes.c_uint32] + [ctypes.c_void_p] * 5
_lib.kmcuda_b200_finish_update.restype = ctypes.c_int
_lib.kmcuda_b200_finish_update.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 5
_lib.kmcuda_b200_shard_reset.restype = ctypes.c_int
_lib.kmcuda_b200_shard_reset.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
_lib.kmcuda_b200_last_error.restype = ctypes.c_uint32
_lib.kmcuda_b200_last_error.argtypes = [ctypes.c_void_p]
_lib.kmcuda_b200_kernel_times.restype = ctypes.c_int32
_lib.kmcuda_b200_kernel_times.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32]
_lib.kmcuda_b200_debug_last_error.restype = ctypes.c_uint32
_lib.kmcuda_b200_debug_last_error.argtypes = [ctypes.c_void_p]
_lib.kmcuda_b200_debug_yy_bounds.restype = ctypes.c_int32
_lib.kmcuda_b200_debug_yy_bounds.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p,
                                             ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int32,
                                             ctypes.c_void_p]
_lib.kmcuda_b200_debug_stats.restype = ctypes.c_int32
_lib.kmcuda_b200_debug_stats.argtypes = [ctypes.c_void_p, ctypes.c_void_p]


_lib.kmcuda_b200_exchange_handle_bytes.restype = ctypes.c_uint32
_lib.kmcuda_b200_exchange_handle_bytes.argtypes = []
_lib.kmcuda_b200_exchange_create.restype = ctypes.c_int
_lib.kmcuda_b200_exchange_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_uint32, ctypes.c_uint16,
                                             ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]
_lib.kmcuda_b200_exchange_connect.restype = ctypes.c_int
_lib.kmcuda_b200_exchange_connect.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
_lib.kmcuda_b200_exchange_buffers.restype = ctypes.c_int
_lib.kmcuda_b200_exchange_buffers.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p),
                                              ctypes.POINTER(ctypes.c_void_p)]
_lib.kmcuda_b200_exchange_reduce.restype = ctypes.c_int
_lib.kmcuda_b200_exchange_reduce.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
_lib.kmcuda_b200_exchange_error.restype = ctypes.c_uint32
_lib.kmcuda_b200_exchange_error.argtypes = [ctypes.c_void_p]
_lib.kmcuda_b200_exchange_destroy.restype = None
_lib.kmcuda_b200_exchange_destroy.argtypes = [ctypes.c_void_p]


def _stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t, dtype):
    assert t.is_cuda and t.is_contiguous() and t.dtype == dtype, (t.device, t.dtype, t.is_contiguous())
    return ctypes.c_void_p(t.data_ptr())


class Shard:
    """One GPU's share of a clustering job (the current torch CUDA device at construction)."""

    def __init__(self, max_samples, features, clusters, metric="L2", verbosity=0):
        self.device = torch.cuda.current_device()
        self.n, self.D, self.K = int(max_samples), int(features), int(clusters)
        self.metric = 1 if metric in ("cos", "cosine", "angular") else 0
        h = ctypes.c_void_p()
        _raise_for(_lib.kmcuda_b200_shard_create(ctypes.byref(h), self.metric, self.n, self.D, self.K,
                                                 int(verbosity)), "kmcuda_b200_shard_create")
        self._h = h

    def close(self):
        if self._h:
            _lib.kmcuda_b200_shard_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def assign(self, X, C, assignments, prev, changed):
        """One assignment pass, enqueued on the current torch stream (no host sync)."""
        _raise_for(_lib.kmcuda_b200_assign(self._h, X.shape[0], _ptr(X, torch.float32), _ptr(C, torch.float32),
                                           _ptr(assignments, torch.int32), _ptr(prev, torch.int32),
                                           _ptr(changed, torch.int32), _stream_ptr()), "kmcuda_b200_assign")

    def last_pass_info(self):
        """(used_tensor_cores, rows_rechecked, rows_overflowed) of the last pass; sync first."""
        a, b = ctypes.c_uint32(0), ctypes.c_uint32(0)
        tc = _lib.kmcuda_b200_last_pass_info(self._h, ctypes.byref(a), ctypes.byref(b))
        return bool(tc), a.value, b.value

    def kernel_times(self, max_out=64):
        """device ms of the tensor-core kernel in the most recent passes (sync first)"""
        buf = np.zeros(max_out, np.float32)
        n = _lib.kmcuda_b200_kernel_times(self._h, buf.ctypes.data, max_out)
        return buf[:n].tolist()

    def last_error(self):
        """pipeline status of the last tensor-core pass (0 = clean); sync first"""
        return int(_lib.kmcuda_b200_last_error(self._h))

    def reset(self):
        """start of a new run on this handle (angular metric: forget the cached member sums)"""
        _raise_for(_lib.kmcuda_b200_shard_reset(self._h, _stream_ptr()), "kmcuda_b200_shard_reset")

    def partial_sums(self, X, assignments, sums, counts):
        _raise_for(_lib.kmcuda_b200_partial_sums(self._h, X.shape[0], _ptr(X, torch.float32),
                                                 _ptr(assignments, torch.int32), _ptr(sums, torch.float32),
                                                 _ptr(counts, torch.int32), _stream_ptr()),
                   "kmcuda_b200_partial_sums")

    def partial_sums_into(self, X, assignments, sums_ptr, counts_ptr):
        """partial_sums() into raw device pointers (the buffers of a PeerExchange)"""
        _raise_for(_lib.kmcuda_b200_partial_sums(self._h, X.shape[0], _ptr(X, torch.float32),
                                                 _ptr(assignments, torch.int32), sums_ptr, counts_ptr, _stream_ptr()),
                   "kmcuda_b200_partial_sums")

    def finish_update(self, sums, counts, C, ccounts):
        _raise_for(_lib.kmcuda_b200_finish_update(self._h, _ptr(sums, torch.float32), _ptr(counts, torch.int32),
                                                  _ptr(C, torch.float32), _ptr(ccounts, torch.int32),
                                                  _stream_ptr()), "kmcuda_b200_finish_update")

    # diagnostics
    def debug_yy_bounds(self, X, C, assignments, groups, G, use_tc):
        """Yinyang bounds [n][G + 1] of one refresh (diagnostics / parity tests); groups: host uint32 [K]"""
        groups = np.ascontiguousarray(groups, dtype=np.uint32)
        out = torch.empty((X.shape[0], G + 1), dtype=torch.float32, device=X.device)
        rc = _lib.kmcuda_b200_debug_yy_bounds(self._h, X.shape[0], _ptr(X, torch.float32), _ptr(C, torch.float32),
                                              _ptr(assignments, torch.int32), groups.ctypes.data, int(G),
                                              1 if use_tc else 0, _ptr(out, torch.float32))
        if rc != 0:
            raise RuntimeError("kmcuda_b200_debug_yy_bounds failed (%d)" % rc)
        return out

    def debug_stats(self):
        out = np.zeros(4, np.float32)
        if _lib.kmcuda_b200_debug_stats(self._h, out.ctypes.data) != 0:
            return None
        return {"scale": float(out[0]), "cmax": float(out[1]), "dcmax": float(out[2])}


def assign_once(X, C, metric="L2", assignments=None):
    """Convenience: one pass over torch tensors; returns (assignments, prev, changed, info)."""
    n = X.shape[0]
    sh = Shard(n, X.shape[1], C.shape[0], metric)
    a = torch.full((n,), -1, dtype=torch.int32, device=X.device) if assignments is None else assignments
    prev = torch.full((n,), -1, dtype=torch.int32, device=X.device)
    changed = torch.zeros(1, dtype=torch.int32, device=X.device)
    sh.assign(X, C, a, prev, changed)
    torch.cuda.synchronize()
    info = sh.last_pass_info()
    err = sh.last_error()
    sh.close()
    if err:
        raise RuntimeError("tensor-core pipeline error 0x%x" % err)
    return a, prev, int(changed.item()), info


class PeerExchange:
    """Exchange step of the centroid update over peer memory (include/kmcuda_b200.h, csrc/exchange.cu) for one process
    per GPU on one node: replaces the all-reduce between `Shard.partial_sums` and `Shard.finish_update`.

        ex = PeerExchange(K, D)                      # collective: every rank of the default process group
        ex.update(shard, X, assignments, sums, counts)   # sums / counts = totals over all ranks, same bits everywhere
        shard.finish_update(sums, counts, C, ccounts)
        ex.close()                                   # collective

    Raises RuntimeError when the handles cannot be mapped (no peer access, different nodes): fall back to
    `torch.distributed.all_reduce` then."""

    def __init__(self, clusters, features, group=None):
        import torch.distributed as dist
        self._dist, self._group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.K, self.D = int(clusters), int(features)
        hb = int(_lib.kmcuda_b200_exchange_handle_bytes())
        mine = (ctypes.c_ubyte * hb)()
        h = ctypes.c_void_p()
        rc = _lib.kmcuda_b200_exchange_create(ctypes.byref(h), self.K, self.D, self.rank, self.world, mine)
        # every rank takes part in the gather, also one whose creation failed (no rank may be left waiting)
        mine_t = torch.tensor(list(bytes(mine)) + [rc], dtype=torch.uint8, device="cuda")
        allh = [torch.empty_like(mine_t) for _ in range(self.world)]
        dist.all_gather(allh, mine_t, group=group)
        blobs = [bytes(t.cpu().numpy().tobytes()) for t in allh]
        self._h = h if rc == 0 else None
        ok = all(b[hb] == 0 for b in blobs)
        if ok:
            flat = b"".join(b[:hb] for b in blobs)
            buf = (ctypes.c_ubyte * len(flat)).from_buffer_copy(flat)
            rc = _lib.kmcuda_b200_exchange_connect(self._h, buf)
            ok = rc == 0
        flag = torch.tensor([0 if ok else 1], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, group=group)
        if int(flag.item()) != 0:
            self.close(collective=False)
            raise RuntimeError("peer-memory exchange unavailable (CUDA IPC handles could not be created / mapped)")

    def update(self, shard, X, assignments, total_sums, total_counts):
        """this rank's partial sums -> totals over all ranks, enqueued on the current stream (no host sync)"""
        ps, pc = ctypes.c_void_p(), ctypes.c_void_p()
        _raise_for(_lib.kmcuda_b200_exchange_buffers(self._h, ctypes.byref(ps), ctypes.byref(pc)),
                   "kmcuda_b200_exchange_buffers")
        shard.partial_sums_into(X, assignments, ps, pc)
        self.reduce(total_sums, total_counts)

    def buffers(self):
        ps, pc = ctypes.c_void_p(), ctypes.c_void_p()
        _raise_for(_lib.kmcuda_b200_exchange_buffers(self._h, ctypes.byref(ps), ctypes.byref(pc)),
                   "kmcuda_b200_exchange_buffers")
        return ps, pc

    def reduce(self, total_sums, total_counts):
        _raise_for(_lib.kmcuda_b200_exchange_reduce(self._h, _ptr(total_sums, torch.float32),
                                                    _ptr(total_counts, torch.int32), _stream_ptr()),
                   "kmcuda_b200_exchange_reduce")

    def error(self):
        """0 = every exchange so far completed (synchronise the stream first)"""
        return int(_lib.kmcuda_b200_exchange_error(self._h))

    def close(self, collective=True):
        if getattr(self, "_h", None):
            if collective:
                torch.cuda.synchronize()
                self._dist.barrier(group=self._group)   # no peer may still be reading this rank's block
            _lib.kmcuda_b200_exchange_destroy(self._h)
            self._h = None
