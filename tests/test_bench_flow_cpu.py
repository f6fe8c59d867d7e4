"""bench.py's control flow on CPU (tests/_bench_dryrun.py stubs everything that touches CUDA): one JSON line with the
contract's keys at 1 rank, the peer-memory iteration leg reported at 2 ranks, and the NCCL numbers kept -- with every rank
taking the same branch -- when the exchange fails on a rank."""
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("world,fail,expect", [(1, 0, "none (1 GPU)"), (2, 0, "peer memory"), (2, 1, "not reported")])
def test_bench_control_flow(world, fail, expect):
    env = dict(os.environ, DRY_WORLD=str(world), DRY_PEER_FAIL=str(fail))
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(HERE, "_bench_dryrun.py")], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=300)
    assert "DRYRUN OK" in r.stdout and expect in r.stdout, r.stdout[-1500:]


@pytest.mark.parametrize("world,suffix", [(1, ""), (2, "_rank0")])
def test_bench_dump_outputs(tmp_path, world, suffix):
    """--dump-outputs: the last timed step's outputs (not a warmup's, not the iteration leg's) on a fixed sorted row
    sample, float32, and the changed count; per-rank file names when there are several ranks"""
    env = dict(os.environ, DRY_WORLD=str(world), DRY_PEER_FAIL="0", DRY_DUMP=str(tmp_path))
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(HERE, "_bench_dryrun.py")], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=300)
    assert "DRYRUN OK" in r.stdout and "DUMP OK" in r.stdout, r.stdout[-1500:]
    assert sorted(os.listdir(tmp_path)) == [f + suffix + ".npy" for f in ("assignments", "changed",
                                                                         "previous_assignments", "sample_rows")]


def test_bench_dump_stays_under_64_mb_over_all_ranks(tmp_path):
    """the dumps of 3 ranks x 8M rows each (the largest shards at the default size) add up to less than 64 MB"""
    code = r'''
import sys, torch
sys.path.insert(0, %r)
import bench
n = 8000000
for rank in range(3):
    a = torch.arange(n, dtype=torch.int32) %% 1024
    bench.dump_outputs(%r, rank, 3, {"assignments": a, "previous_assignments": a}, torch.tensor([n]))
''' % (os.path.dirname(HERE), str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stdout[-1500:]
    files = os.listdir(tmp_path)
    assert len(files) == 12 and all("_rank" in f for f in files)
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in files) < 64e6
