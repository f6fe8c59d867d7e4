"""CPU dry run of bench.run_ours' control flow: every CUDA-touching piece (torch.cuda, the shard, the peer exchange, the
collectives, the C-ABI call) is a stub, so what runs is bench.py's own Python -- the timed loop, the iteration leg both
ways, the fallback when the peer-memory exchange fails on a rank, the JSON line and its contract keys.  Launched in a
subprocess by tests/test_bench_flow_cpu.py (it monkeypatches torch).  DRY_WORLD = ranks to pretend, DRY_PEER_FAIL = 1:
the exchange raises after three calls."""
import sys, types, time, json, io, contextlib
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench

# ---- torch stubs
_RealGen0 = torch.Generator
_real = {k: getattr(torch, k) for k in ("rand", "randperm", "full", "zeros", "tensor", "empty")}
def _strip(fn):
    def w(*a, **kw):
        kw.pop("device", None); kw.pop("pin_memory", None)
        g = kw.get("generator")
        if g is not None and not isinstance(g, _RealGen0): kw["generator"] = None
        return fn(*a, **kw)
    return w
for k, f in _real.items(): setattr(torch, k, _strip(f))
_RealGen = torch.Generator
class FakeGen:
    def __init__(self, device=None): self.g = _RealGen()
    def manual_seed(self, s): self.g.manual_seed(s); return self.g
torch.Generator = lambda device=None: FakeGen()
torch.Tensor.cuda = lambda self, *a, **k: self
class Ev:
    def __init__(self, enable_timing=True): self.t = None
    def record(self): self.t = time.perf_counter()
    def elapsed_time(self, other): return (other.t - self.t) * 1e3
torch.cuda.set_device = lambda d: None
torch.cuda.synchronize = lambda *a: None
torch.cuda.Event = Ev
torch.cuda.empty_cache = lambda: None

# ---- library stubs
import kmcuda_b200, kmcuda_b200.shard as shard_mod
class FakeShard:
    def __init__(self, n, D, K, **kw): self.n = n
    def assign(self, X, C, a, prev, ch): time.sleep(0.001)
    def partial_sums(self, X, a, sums, counts): pass
    def partial_sums_into(self, X, a, ps, pc): pass
    def finish_update(self, s, c, C, cc): pass
    def reset(self): pass
    def last_error(self): return 0
    def last_pass_info(self): return True, 12, 0
    def kernel_times(self, m): return [0.9] * min(m, 5)
shard_mod.Shard = FakeShard
bench.time_c_abi = lambda *a, **k: 0.05
class FakeSampler:
    def __init__(self, i): pass
    def start(self): pass
    def wait_ready(self): pass
    def mark(self): pass
    def stop(self): return {"sm_mhz": 1965, "sm_max_mhz": 1965, "reasons": []}
bench.ClockSampler = FakeSampler
bench.cpu_baseline = lambda: {"value": 1.0, "unit": "points/s", "cores": 1, "kind": "port", "sample": "stub"}
# data_ptr on pinned tensors works on CPU tensors too
import os
import torch.distributed as dist
if os.environ.get("DRY_WORLD", "1") != "1":
    os.environ["WORLD_SIZE"] = os.environ["DRY_WORLD"]; os.environ["RANK"] = "0"; os.environ["LOCAL_RANK"] = "0"
    dist.init_process_group = lambda *a, **k: None
    dist.all_reduce = lambda t, op=None, group=None: None
    dist.barrier = lambda *a, **k: None
    dist.broadcast = lambda *a, **k: None
    dist.destroy_process_group = lambda *a, **k: None
    class FakePeer:
        def __init__(self, K, D, group=None): self.fail = os.environ.get("DRY_PEER_FAIL") == "1"; self.n = 0
        def buffers(self): return 1, 2
        def reduce(self, s, c):
            self.n += 1
            if self.fail and self.n > 3: raise RuntimeError("kmcuda_b200_exchange_reduce -> kmcudaRuntimeError")
        def error(self): return 0
        def close(self, collective=True): pass
    shard_mod.PeerExchange = FakePeer
calls = [0]
def _assign(self, X, C, a, prev, ch):   # the n-th call writes (row + n) % 11 and changed = n
    time.sleep(0.001)
    calls[0] += 1
    a.copy_((torch.arange(len(a)) + calls[0]) % 11)
    ch.fill_(calls[0])
FakeShard.assign = _assign
dump = os.environ.get("DRY_DUMP")   # a directory: dump the outputs, the ranks sharing 1000 rows
if dump:
    bench.DUMP_ROWS = 1000
args = types.SimpleNamespace(gpus=1, steps=4, warmup=3, impl="ours", points=3000, skip_extras=False, dump_outputs=dump)
lines = []
bench.emit = lambda obj: lines.append(json.dumps(obj))
bench.run_ours(args)
assert len(lines) == 1
if dump:
    import numpy as np
    world = int(os.environ.get("DRY_WORLD", "1"))
    sfx = "_rank0" if world > 1 else ""
    last_timed = args.warmup + args.steps
    rows = np.load(os.path.join(dump, "sample_rows%s.npy" % sfx))
    a = np.load(os.path.join(dump, "assignments%s.npy" % sfx))
    assert rows.dtype == np.float32 and len(rows) == 1000 // world and (np.diff(rows) > 0).all()
    assert rows.max() < 3000 // world
    assert a.dtype == np.float32 and np.array_equal(a, (rows + last_timed) % 11)
    assert np.load(os.path.join(dump, "changed%s.npy" % sfx)).tolist() == [float(last_timed)]
    assert calls[0] > last_timed        # the iteration leg ran after the dump
    print("DUMP OK")
d = json.loads(lines[0])
for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
          "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks", "cpu_baseline", "iteration"):
    assert k in d, k
print("DRYRUN OK", {k: d[k] for k in ("value", "ms_per_step", "gpu_launches")}, d["iteration"]["collective"], d["iteration"]["phase_ms"])
