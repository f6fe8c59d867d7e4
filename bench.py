#!/usr/bin/env python
"""bench.py -- headline benchmark: k-means assignment step, points/sec, 8M x 256 fp32 @ 1024 clusters.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--points P] [--dump-outputs DIR]

Workload (BASELINE.json configs[1] / configs[3]): P = 8 000 000 samples IN TOTAL (U[0,1), the reference's own
benchmark distribution), 256 features, 1024 centroids = rows of the samples.  With N GPUs (one process per GPU
under torchrun) the samples are range-partitioned, P/N rows per rank -> "scaling": "strong".

A "step" is ONE assignment pass of the hot path (the reference's kmeans_assign_lloyd, src/kmeans.cu:293-364;
here: tcgen05 distance filter + exact fp32 re-check + fused bookkeeping) over the rank's shard, resident in HBM:
`value` = P / max-over-ranks(device time per step) (SURVEY.md 8d: the metric is the assignment step).  The same
run also times the FULL Lloyd iteration -- assign + per-cluster partial sums + NCCL all-reduce of the K*D fp32
sums and K integer counts + normalise (BASELINE configs[3]) -- and reports it per phase under `iteration`.

Other keys: `e2e` (the same pass through the reference-facing C ABI kmeans_cuda() with pinned HOST buffers: H2D
of the samples and D2H of the assignments inside the timed region), `roofline` (the tcgen05 kernel, CUDA events
around its launches, against the measured bf16 tensor peak of MEASURED_PEAKS.json), `cpu_baseline` (scikit-learn
KMeans labelling on all host cores, the CPU reference north_star names; the C oracle port is nested), `clocks`.

`--dump-outputs DIR` writes what the last timed step returned -- the assignments, the previous assignments and the
changed count; with `--impl reference` the assignments of its last timed call -- as DIR/<name>.npy (float32 / float64,
one set per rank with a _rank<r> suffix when there are several), so that two builds can be compared output for output
on the same seeded inputs.  All ranks together write at most 2^21 rows (under 64 MB); a larger shard is represented
by a fixed sample of its rows, listed in sample_rows.npy.

`--impl reference` times the UNMODIFIED reference (oracle/_ref/libKMCUDA.so, src-d/kmcuda rebuilt for sm_100 --
the reference has no CPU implementation, it is a CUDA library) through the same C ABI on the same P points with
device mask (1 << N) - 1: `value` with device-resident inputs (device_ptrs = 0), `e2e` with pinned host buffers.
If that library cannot be loaded the CPU oracle port is timed instead.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line: everything else that writes to fd 1 (NCCL_DEBUG output, C-library progress
# messages) goes to stderr, the JSON line goes to the saved descriptor.  NCCL_DEBUG is left as the caller set it.
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj):
    _JSON_OUT.write(json.dumps(obj) + "\n")
    _JSON_OUT.flush()


METRIC = "kmeans_assign_points_per_sec"
UNIT = "points/s"
N_POINTS, D, K = 8000000, 256, 1024
WORKLOAD = ("k-means assignment step, %d x %d fp32 samples in total (U[0,1)) @ %d clusters (rows of the samples), "
            "range-partitioned over the GPUs (BASELINE configs[1] at 1 GPU, configs[3] at 2/4/8)")
IMPORT = 3
# kernels of this library per assignment pass (L2, tensor-core path): tc_prep_fused_kernel (||c||^2, mean, centred
# norms, scale, fp16 table in one launch), tc_assign_kernel, recheck_pairs, recheck_reduce, exact_rows_few, exact_pass
# (row list), finalize_rows (profiles/r02_launches_iteration.csv lists them, next to the update's kernels)
LAUNCHES_PER_ASSIGN = 7


def _rank_info():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


def shard_range(total, rank, world):
    return total * rank // world, total * (rank + 1) // world


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region (B200_PROFILING.md's clocks line).

    The timed region of the default run is ~0.1 s, shorter than nvidia-smi's start-up and coarser than its averaged
    readings, so NVML is polled in-process by a thread (~1 ms period) and only the samples between the two `mark()`
    calls are used.  Falls back to an `nvidia-smi -lms 20` child process when pynvml is unavailable."""

    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"),
               ("hw_power_brake", "nvmlClocksEventReasonHwPowerBrakeSlowdown"))

    def __init__(self, index):
        self.index = index
        self.marks = []
        self.samples = []        # (t, sm_mhz, power_w, reasons_bitmask)
        self.thread = None
        self.stop_flag = False
        self.nv = None
        self.handle = None
        self.max_mhz = None
        self.path = None
        self.proc = None

    def _poll(self):
        nv, h = self.nv, self.handle
        while not self.stop_flag:
            try:
                clk = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = None
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = 0
                self.samples.append((time.time(), clk, pw, rs))
            except Exception:
                pass
            time.sleep(0.001)

    def start(self):
        try:
            import pynvml as nv
            import threading
            nv.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            idx = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:
                    pass
            self.handle = nv.nvmlDeviceGetHandleByIndex(idx)
            self.nv = nv
            try:
                self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM)
            except Exception:
                self.max_mhz = None
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nv = None
        q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.path = tempfile.mktemp(prefix="clocks_", suffix=".csv")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def wait_ready(self, timeout=5.0):
        t = time.time()
        while time.time() - t < timeout:
            if self.nv is not None:
                if self.samples:
                    return True
            elif self.proc is not None:
                try:
                    if os.path.getsize(self.path) > 0:
                        return True
                except OSError:
                    pass
            else:
                return False
            time.sleep(0.01)
        return False

    def mark(self):
        self.marks.append(time.time())

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        lo, hi = (self.marks[0], self.marks[1]) if len(self.marks) >= 2 else (0.0, 1e18)
        if self.nv is not None:
            self.stop_flag = True
            if self.thread:
                self.thread.join(timeout=2)
            inside = [x for x in self.samples if lo <= x[0] <= hi]
            out["source"] = "NVML polled in-process (~1 ms period)"
            if inside:
                out["sm_mhz"] = statistics.median(x[1] for x in inside)
                out["sm_min_mhz"] = min(x[1] for x in inside)
                out["sm_max_mhz"] = self.max_mhz
                out["samples"] = len(inside)
                pw = [x[2] for x in inside if x[2] is not None]
                if pw:
                    out["power_w_max"] = max(pw)
                bits = 0
                for x in inside:
                    bits |= x[3]
                out["reasons"] = sorted(name for name, attr in self.REASONS if bits & getattr(self.nv, attr, 0))
            else:
                out["note"] = "no NVML sample fell inside the timed region (%d outside it)" % len(self.samples)
            return out
        import datetime
        if not self.proc:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons, all_sm = [], [], [], set(), []
        lo, hi = lo - 0.02, hi + 0.02
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    clk, cmax = float(f[1]), float(f[2])
                except ValueError:
                    continue
                all_sm.append(clk)
                if not (lo <= ts <= hi):
                    continue
                sm.append(clk)
                mx.append(cmax)
                try:
                    pw.append(float(f[3]))
                except ValueError:
                    pass
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"],
                                   f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        out["source"] = "nvidia-smi -lms 20"
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["sm_max_mhz"] = max(mx)
            out["reasons"] = sorted(reasons)
            out["samples"] = len(sm)
            if pw:
                out["power_w_max"] = max(pw)
        elif all_sm:
            out["note"] = "no sample fell inside the timed region (%d outside it)" % len(all_sm)
        return out


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def cpu_baseline():
    """north_star's named CPU baseline: scikit-learn KMeans labelling (Lloyd assignment) on all host cores, bounded
    sample of the same workload; nested: the single-source C oracle port (exact reference arithmetic, OpenMP)."""
    cores = os.cpu_count() or 1
    rng = np.random.default_rng(777)
    sample = 1000000
    X = rng.random((sample, D), dtype=np.float32)
    C = X[rng.choice(sample, K, replace=False)].copy()
    out = {"unit": UNIT, "cores": cores, "kind": "port"}
    try:
        from sklearn.cluster import KMeans
        from threadpoolctl import threadpool_limits
        km = KMeans(n_clusters=K, init=C, n_init=1, max_iter=1, algorithm="lloyd", tol=0).fit(X[:8192])
        km.cluster_centers_ = C.astype(km.cluster_centers_.dtype)
        with threadpool_limits(limits=cores):
            km.predict(X[:65536])
            best, spent, reps = 1e30, 0.0, 0
            while spent < 10.0 and reps < 8:
                t = time.perf_counter()
                km.predict(X)
                dt = time.perf_counter() - t
                best, spent, reps = min(best, dt), spent + dt, reps + 1
        out.update({"value": sample / best, "implementation": "sklearn.cluster.KMeans.predict (Lloyd labelling)",
                    "sample": "%d points of the same %d-feature x %d-cluster workload, best of %d passes, %.1f s of CPU "
                              "work on %d threads" % (sample, D, K, reps, spent, cores)})
    except Exception as e:  # pragma: no cover
        out["sklearn_unavailable"] = repr(e)[:120]
    try:
        from oracle import oracle as O
        ocores = O.set_threads(cores)   # torchrun exports OMP_NUM_THREADS=1
        small = 16384
        O.assign_lloyd(X[:1024], C)
        t = time.perf_counter()
        O.assign_lloyd(X[:small], C)
        dt = time.perf_counter() - t
        out["oracle_port"] = {"value": small / dt, "unit": UNIT, "cores": ocores,
                              "sample": "%d points, C restatement of the reference arithmetic (TwoSum round-down FMA), "
                                        "%.1f s" % (small, dt)}
        if "value" not in out:
            out.update({"value": small / dt, "cores": ocores, "sample": out["oracle_port"]["sample"]})
    except Exception as e:  # pragma: no cover
        out["oracle_unavailable"] = repr(e)[:120]
    return out


DUMP_ROWS = 1 << 21    # over all ranks: at most 2^21 rows x (4 + 4 + 8) bytes = 32 MiB


def dump_outputs(dirname, rank, world, per_row, changed=None):
    """--dump-outputs: the arrays the caller of the timed call receives (`per_row`: name -> one value per row of this
    rank's shard) and the changed count.  The ranks share DUMP_ROWS; a larger shard is sampled with a fixed seed.
    Labels and row numbers below 2^24 are exact in float32."""
    os.makedirs(dirname, exist_ok=True)
    budget = DUMP_ROWS // world
    n = next(iter(per_row.values())).numel()
    rows = None if n <= budget else np.sort(np.random.default_rng(0).choice(n, budget, replace=False))
    out = {}
    for name, t in per_row.items():
        v = t.cpu().numpy()
        out[name] = (v if rows is None else v[rows]).astype(np.float32)
    if changed is not None:
        out["changed"] = np.array([int(changed.item())], np.float64)
    if rows is not None:
        out["sample_rows"] = rows.astype(np.float32 if n <= 1 << 24 else np.float64)
    suffix = "_rank%d" % rank if world > 1 else ""
    for name, v in out.items():
        np.save(os.path.join(dirname, name + suffix + ".npy"), v)


def time_c_abi(lib, n, x_ptr, c_ptr, a_ptr, device_mask, device_ptrs, steps, warmup):
    """kmeans_cuda(init=import, tolerance=1.0, yinyang_t=0): exactly one assignment pass (reference src/test.py:
    512-519); wall clock per call"""
    m = ctypes.c_uint32(0)

    def call():
        rc = lib.kmeans_cuda(IMPORT, ctypes.byref(m), 1.0, 0.0, 0, n, D, K, 0, device_mask, device_ptrs, 0, 0,
                             x_ptr, c_ptr, a_ptr, None)
        if rc != 0:
            raise RuntimeError("kmeans_cuda returned %d" % rc)

    for _ in range(warmup):
        call()
    t = time.perf_counter()
    for _ in range(steps):
        call()
    return (time.perf_counter() - t) / steps


def run_reference(args):
    rank, local, world = _rank_info()
    if rank != 0:
        return
    from oracle import oracle as O
    import torch
    n = args.points
    mask = (1 << args.gpus) - 1
    line = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD % (n, D, K), "l2": "inputs larger than L2",
                       "parallelism": "single process, device mask 0x%x (the reference replicates the samples on "
                                      "every GPU and splits the kernel ranges)" % mask}}
    try:
        if not (O.reference_available() and torch.cuda.is_available()):
            raise RuntimeError("oracle/_ref/libKMCUDA.so or GPU missing")
        ref = O.reference_lib()
        torch.cuda.set_device(0)
        g = torch.Generator(device="cuda").manual_seed(777)
        X = torch.rand((n, D), generator=g, device="cuda", dtype=torch.float32)
        C = X[torch.randperm(n, generator=g, device="cuda")[:K]].contiguous()
        A = torch.zeros(n, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        # resident: device pointers on GPU 0 (the reference still allocates, copies and transposes internally: its
        # public API has no finer-grained entry point)
        steps = args.steps
        dt = time_c_abi(ref, n, X.data_ptr(), C.data_ptr(), A.data_ptr(), mask, 0, steps, args.warmup)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, 0, 1, {"assignments": A})
        # end to end: pinned host buffers, H2D + D2H inside the call
        Xh = torch.empty((n, D), dtype=torch.float32, pin_memory=True)
        Xh.copy_(X)
        Ch = C.cpu().numpy().copy()
        Ah = torch.empty(n, dtype=torch.int32, pin_memory=True)
        del X, A
        torch.cuda.empty_cache()
        e2e_steps = max(1, min(steps, 3))
        dte = time_c_abi(ref, n, Xh.data_ptr(), Ch.ctypes.data, Ah.data_ptr(), mask, -1, e2e_steps, 1)
        note = ("unmodified src-d/kmcuda rebuilt for sm_100 (oracle/_ref), device mask 0x%x, kmeans_cuda(import, "
                "tolerance=1, yinyang_t=0) = one assign pass on all %d points; `value`: device-resident inputs "
                "(device_ptrs=0), %d timed calls; `e2e`: pinned host buffers, %d calls" % (mask, n, steps, e2e_steps))
        v = n / dt
        line.update({"value": v, "ms_per_step": dt * 1e3, "steps_timed": steps,
                     "cpu_baseline": {"value": v, "unit": UNIT, "cores": 0, "kind": "reference", "sample": note},
                     "e2e": {"value": n / dte, "unit": UNIT, "h2d_bytes_per_step": n * D * 4 + K * D * 4,
                             "d2h_bytes_per_step": n * 4 + K * D * 4, "steps": e2e_steps}})
    except Exception as e:
        if args.dump_outputs:     # the CPU port below does not compute the reference's outputs
            raise
        sample = 16384
        rng = np.random.default_rng(777)
        X = rng.random((sample, D), dtype=np.float32)
        C = X[rng.choice(sample, K, replace=False)].copy()
        cores = O.set_threads(os.cpu_count() or 1)
        reps = args.steps
        t = time.perf_counter()
        for _ in range(reps):
            O.assign_lloyd(X, C)
        dt = (time.perf_counter() - t) / reps
        v = sample / dt
        note = "CPU oracle port (reference library unavailable: %s); %d points" % (repr(e)[:80], sample)
        line.update({"value": v, "ms_per_step": dt * 1e3,
                     "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": note},
                     "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    emit(line)


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank, local, world = _rank_info()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import kmcuda_b200
    from kmcuda_b200.shard import Shard

    total = args.points
    lo, hi = shard_range(total, rank, world)
    n = hi - lo
    g = torch.Generator(device="cuda").manual_seed(777 + rank)
    X = torch.rand((n, D), generator=g, device="cuda", dtype=torch.float32)
    # centroids = K rows of the samples (BASELINE configs[1]); rank 0 draws them from its shard for everybody
    C = X[torch.randperm(n, generator=g, device="cuda")[:K]].contiguous()
    if world > 1:
        dist.broadcast(C, src=0)
    C0 = C.clone()
    sh = Shard(n, D, K)
    a = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    prev = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    changed = torch.zeros(1, dtype=torch.int32, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        a.fill_(-1)
        sh.assign(X, C, a, prev, changed)
    barrier()
    if sh.last_error():
        raise RuntimeError("tensor-core pipeline error 0x%x" % sh.last_error())
    sampler.wait_ready()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark()
    e0.record()
    for _ in range(args.steps):
        sh.assign(X, C, a, prev, changed)
    e1.record()
    barrier()
    sampler.mark()
    clocks = sampler.stop()
    ms_per_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    tc_used, rechecked, overflowed = sh.last_pass_info()
    if not tc_used or sh.last_error():
        raise RuntimeError("the tensor-core path did not run cleanly (tc=%s err=0x%x)" % (tc_used, sh.last_error()))
    kt = sh.kernel_times(min(args.steps, 64))
    kernel_ms = max_over_ranks(sum(kt) / len(kt))
    a_ref = a.clone()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, world, {"assignments": a, "previous_assignments": prev}, changed)

    if args.skip_extras:
        if rank == 0:
            emit({"metric": METRIC, "value": total / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world,
                  "ms_per_step": ms_per_step, "kernel_ms": kernel_ms, "note": "profiling run, extras skipped"})
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- the full Lloyd iteration (BASELINE configs[3]): assign + partial sums + NCCL all-reduce + normalise
    sums = torch.zeros((K, D), dtype=torch.float32, device="cuda")
    counts = torch.zeros(K, dtype=torch.int32, device="cuda")
    ccounts = torch.zeros(K, dtype=torch.int32, device="cuda")
    iters = max(3, min(args.steps, 10))
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(iters)]

    # the exchange step two ways when there are peers: summed over peer memory in rank order by one kernel per GPU
    # (kmcuda_b200.shard.PeerExchange, csrc/exchange.cu: CUDA IPC mappings over NVLink / NVSwitch), and the
    # communicator's all-reduce (two NCCL collectives: fp32 sums, integer counts)
    ex, ex_note = None, "none (1 GPU)"
    if world > 1 and os.environ.get("KMCUDA_B200_EXCHANGE", "") != "nccl":
        try:
            from kmcuda_b200.shard import PeerExchange
            ex = PeerExchange(K, D)
        except Exception as e:  # no peer access / IPC refused: the communicator's all-reduce is the exchange
            ex, ex_note = None, "peer-memory exchange unavailable: %s" % str(e)[:120]

    def iteration(evs=None, peer=False):
        if evs: evs[0].record()
        sh.assign(X, C, a, prev, changed)
        if evs: evs[1].record()
        if peer:
            ps, pc = ex.buffers()
            sh.partial_sums_into(X, a, ps, pc)
            if evs: evs[2].record()
            ex.reduce(sums, counts)
        else:
            sh.partial_sums(X, a, sums, counts)
            if evs: evs[2].record()
            if world > 1:
                dist.all_reduce(sums, op=dist.ReduceOp.SUM)
                dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        if evs: evs[3].record()
        sh.finish_update(sums, counts, C, ccounts)
        if evs: evs[4].record()

    def time_iterations(peer):
        """(ms per iteration, phase ms, failed).  Every rank runs the same sequence of collectives whatever happens
        inside the loop (a timed-out peer exchange raises on some ranks only)."""
        failed = 0
        C.copy_(C0)
        sh.reset()
        try:
            for _ in range(2):
                iteration(None, peer)
        except Exception as e:
            sys.stderr.write("iteration leg failed on rank %d: %s\n" % (rank, str(e)[:200]))
            failed = 1
        barrier()
        if not failed:
            try:
                for i in range(iters):
                    iteration(ev[i], peer)
            except Exception as e:
                sys.stderr.write("iteration leg failed on rank %d: %s\n" % (rank, str(e)[:200]))
                failed = 1
        barrier()
        if peer and not failed and ex.error() != 0:
            failed = 1
        ph = {}
        for j, name in enumerate(["assign", "partial_sums", "exchange", "normalise"]):
            v = 0.0 if failed else sum(ev[i][j].elapsed_time(ev[i][j + 1]) for i in range(iters)) / iters
            ph[name] = max_over_ranks(v)
        ms = max_over_ranks(0.0 if failed else ev[0][0].elapsed_time(ev[iters - 1][4]) / iters)
        return ms, ph, failed

    it_ms, phases, nccl_failed = time_iterations(False)
    if nccl_failed:
        raise RuntimeError("the Lloyd iteration leg failed")
    it_collective = "torch.distributed NCCL all_reduce x2" if world > 1 else "none (1 GPU)"
    it_other = None
    if ex is not None:
        nccl_ms, nccl_phases = it_ms, phases
        peer_ms, peer_phases, failed = time_iterations(True)
        bad = torch.tensor([failed], dtype=torch.int32, device="cuda")
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)     # every rank takes the same branch
        if int(bad.item()) == 0:
            it_ms, phases = peer_ms, peer_phases
            it_collective = ("peer memory: every GPU reads its peers' partial sums over NVLink / NVSwitch (CUDA IPC) and "
                             "adds them in rank order, one kernel per iteration")
            it_other = {"collective": "torch.distributed NCCL all_reduce x2", "value": total / (nccl_ms * 1e-3),
                        "unit": UNIT, "ms": nccl_ms, "phase_ms": nccl_phases}
        else:
            it_collective += " (the peer-memory exchange timed out on some rank: not reported)"
        ex.close()
    elif world > 1:
        it_collective += " (%s)" % ex_note
    C.copy_(C0)

    # ---- end to end through the reference-facing C ABI with host buffers (pinned), rank-local shard
    e2e_steps = max(1, min(args.steps, 3))
    Xh = torch.empty((n, D), dtype=torch.float32, pin_memory=True)
    Xh.copy_(X)
    Ch = C0.cpu().numpy().copy()
    Ah = torch.empty(n, dtype=torch.int32, pin_memory=True)
    del X
    torch.cuda.empty_cache()
    barrier()
    dt = time_c_abi(kmcuda_b200._lib, n, Xh.data_ptr(), Ch.ctypes.data, Ah.data_ptr(), 1 << local, -1, e2e_steps, 1)
    e2e_dt = max_over_ranks(dt)
    same = bool((Ah.cuda() == a_ref).all().item())

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        peak_tf = float(peaks.get("bf16_tflops", 1590.0))
        flops = 2.0 * n * K * D
        achieved = flops / (kernel_ms * 1e-3) / 1e12
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json"))).get("dram_bytes_per_launch")
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": total / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None,
            "dtype": "f16 tensor-core filter (f32 accumulate) + f32 exact re-check", "data": "synthetic",
            "config": {"workload": WORKLOAD % (total, D, K),
                       "parallelism": "%d rows per GPU x %d GPUs (one process per GPU); the assignment step needs no "
                                      "collective, the centroid update one exchange of the partial sums (see `iteration`)" % (n, world),
                       "l2": "inputs (%.2f GB per GPU) larger than L2, no flush needed" % (n * D * 4 / 1e9),
                       "rows_rechecked_exactly": rechecked, "rows_full_exact_fallback": overflowed},
            "step_tflops": 2.0 * total * K * D / (ms_per_step * 1e-3) / 1e12 / world,
            "iteration": {"what": "full Lloyd iteration: assign + partial sums + exchange (sum over GPUs of K*D f32 + K i32) + normalise",
                          "value": total / (it_ms * 1e-3), "unit": UNIT, "ms": it_ms, "iterations": iters,
                          "phase_ms": phases, "allreduce_bytes": K * D * 4 + K * 4,
                          "collective": it_collective, "same_iteration_over_nccl": it_other},
            "e2e": {"value": total / e2e_dt, "unit": UNIT, "h2d_bytes_per_step": n * D * 4 + K * D * 4,
                    "d2h_bytes_per_step": n * 4 + K * D * 4, "steps": e2e_steps,
                    "call": "kmeans_cuda(init=import, tolerance=1.0, yinyang_t=0) with pinned host buffers, one call "
                            "per rank on its shard",
                    "equal_to_resident_result": same},
            "gpu_launches": args.steps * LAUNCHES_PER_ASSIGN,
            "roofline": {"bound": "tensor", "kernel": "tc_assign_kernel", "achieved": achieved, "peak": peak_tf,
                         "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic,
                         "peak_source": "%s bf16_tflops (burst) of MEASURED_PEAKS.json; fp16 and bf16 share the "
                                        "tcgen05 rate" % peak_kind,
                         "kernel_ms": kernel_ms, "algorithmic_flops_per_launch": flops,
                         "algorithmic_hbm_bytes_per_launch": n * (D * 4 + 4),
                         "whole_step_frac": 2.0 * n * K * D / (ms_per_step * 1e-3) / 1e12 / peak_tf},
            "clocks": clocks,
        }
        line["cpu_baseline"] = cpu_baseline()
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=N_POINTS, help="samples IN TOTAL (default: the headline 8M)")
    ap.add_argument("--skip-extras", action="store_true", help="profiling runs: no iteration / e2e / cpu_baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
