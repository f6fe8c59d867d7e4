"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Everything goes through the C ABI of
kmcuda_b200/libKMCUDA.so; the oracle (oracle/) and the stored outputs of the unmodified reference library
(tests/golden/reference.npz, made by tests/golden/make_reference_golden.py) are checkers only.

Bars: bit-exact for assignments / neighbour indices (the tensor-core filter + exact re-check is
designed to be bit-identical to the reference kernel, ties included; cosine and k-NN distance ties are
exempt as in the reference's own suite); centroids within 1e-5 relative (fp32)."""
import ctypes
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))

import cases  # noqa: E402
from oracle import oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu

IMPORT = 3
GOLDEN = np.load(os.path.join(HERE, "golden", "golden.npz"))
REF = np.load(os.path.join(HERE, "golden", "reference.npz"))


@pytest.fixture(scope="module")
def km():
    import torch
    assert torch.cuda.is_available()
    import kmcuda_b200
    return kmcuda_b200


@pytest.fixture(scope="module")
def ours(km):
    return O.load_c_api(km.LIB_PATH)


def c_kmeans(lib, X, C0, tol, yy, metric=0, verbosity=0, init=IMPORT, seed=3):
    X = np.ascontiguousarray(X)
    N, D = X.shape
    K = C0.shape[0] if hasattr(C0, "shape") else int(C0)
    C = np.array(C0, copy=True, order="C") if hasattr(C0, "shape") else np.zeros((K, D), np.float32)
    A = np.zeros(N, np.uint32)
    m = ctypes.c_uint32(0)
    rc = lib.kmeans_cuda(init, ctypes.byref(m), tol, yy, metric, N, D, K, seed, 1, -1, 0, verbosity,
                         X.ctypes.data, C.ctypes.data, A.ctypes.data, None)
    assert rc == 0, rc
    return C, A


def one_pass(lib, X, C0, metric=0):
    return c_kmeans(lib, X, C0, 1.0, 0.0, metric)[1]


def reference_run(ours, key, X, C0, tol, yy, metric=0):
    """the reference library's whole run from C0: (centroids, assignments), replayed and checked by digest"""
    return cases.strict_replay(lambda: c_kmeans(ours, X, C0, tol, yy, metric), REF, key)


def test_oracle_matches_reference():
    """pins the CPU oracle (and the golden assignments made with it) against the UNMODIFIED reference kernels"""
    for name in cases.ORACLE_PIN_CASES:
        X, C = cases.make_assign_case(*cases.ASSIGN_CASES[name])
        exp = str(REF["oracle_pin/" + name])
        assert cases.digest(O.assign_lloyd(X, C)[0]) == exp and cases.digest(GOLDEN["assign/" + name]) == exp, name


@pytest.mark.parametrize("name", sorted(cases.ASSIGN_CASES))
@pytest.mark.parametrize("force_exact", ["0", "1"])
def test_assign_matches_golden(ours, name, force_exact, monkeypatch):
    """one assignment pass (tolerance=1 trick, reference src/test.py:512-519) == golden, bit for bit;
    force_exact=0 takes the tcgen05 filter + re-check wherever the shape allows it"""
    monkeypatch.setenv("KMCUDA_B200_FORCE_EXACT", force_exact)
    X, C = cases.make_assign_case(*cases.ASSIGN_CASES[name])
    got = one_pass(ours, X, C)
    exp = GOLDEN["assign/" + name]
    assert np.array_equal(got, exp), "%s: %d mismatches" % (name, int((got != exp).sum()))


def _shard_pass(X, C, assign=None, metric="L2", force_exact=False):
    import torch
    from kmcuda_b200.shard import assign_once
    old = os.environ.get("KMCUDA_B200_FORCE_EXACT")
    os.environ["KMCUDA_B200_FORCE_EXACT"] = "1" if force_exact else "0"   # read when the shard is created
    try:
        a, prev, changed, info = assign_once(torch.from_numpy(X).cuda(), torch.from_numpy(C).cuda(), metric=metric,
                                             assignments=None if assign is None else torch.from_numpy(
                                                 assign.astype(np.int32)).cuda())
    finally:
        if old is None:
            os.environ.pop("KMCUDA_B200_FORCE_EXACT", None)
        else:
            os.environ["KMCUDA_B200_FORCE_EXACT"] = old
    return a.cpu().numpy().astype(np.uint32), prev.cpu().numpy().astype(np.uint32), changed, info


def test_tensor_core_path_runs_and_matches_reference_100k():
    """C1-sized pass: the tcgen05 path must be the one that runs, and equal the reference kernel"""
    X, C = cases.uniform_rows(100000, 256, 1024, 777)
    a, prev, changed, info = _shard_pass(X, C)
    assert info[0], "tensor-core path not taken"
    assert cases.digest(a) == str(REF["tc_100k"])
    assert changed == len(X) and (prev == 0xFFFFFFFF).all()
    # idempotence: a second pass from the result changes nothing
    a2, prev2, changed2, _ = _shard_pass(X, C, assign=a)
    assert changed2 == 0 and np.array_equal(a2, a) and np.array_equal(prev2, a)


def _unit(a):
    return (a / np.linalg.norm(a, axis=1, keepdims=True)).astype(np.float32)


@pytest.mark.parametrize("n,d,k,metric", cases.WIDE_SHAPES)
def test_tensor_core_wide_shapes_match_reference(n, d, k, metric):
    """cosine, D up to 512 (single A buffer in TMEM) and K >> 1024 (chunk-list compaction) through the
    tcgen05 filter: bit-identical to the reference kernel"""
    X, C = cases.wide_shape(n, d, k, metric)
    a, prev, changed, info = _shard_pass(X, C, metric=metric)
    assert info[0], "tensor-core path not taken"
    assert info[2] < n // 20, "too many rows fell back to the exact pass: %d" % info[2]
    assert cases.digest(a) == str(REF["wide/%d_%d_%d_%s" % (n, d, k, metric)])


def test_tensor_core_cosine_unnormalised_clamps():
    """dots beyond +-1 are clamped by the reference (metric_abstraction.h:171-177): all such centroids tie
    and the lowest index wins -- the filter must not prune them"""
    rng = np.random.default_rng(5)
    X = _unit(rng.standard_normal((4096, 64)))
    C = _unit(X[rng.choice(4096, 300, replace=False)] + 0.05 * rng.standard_normal((300, 64)))
    Xs = X.copy()
    Xs[:1000] *= 3.0            # many dots > 1
    Xs[1000:1500] *= 1.0001     # borderline
    for Xc, Cc in ((Xs, C), (Xs, -np.abs(C)), (np.abs(Xs), -np.abs(C) * 4), (Xs, C * 2.5)):
        Xc, Cc = np.ascontiguousarray(Xc, np.float32), np.ascontiguousarray(Cc, np.float32)
        a, _, _, info = _shard_pass(Xc, Cc, metric="cos")
        assert info[0]
        # checker: this library's exact kernel (device acosf, as the reference; glibc's acosf in the CPU
        # oracle rounds differently in the last ulp, so the oracle only bounds the angle here)
        exp, _, _, info_e = _shard_pass(Xc, Cc, metric="cos", force_exact=True)
        assert not info_e[0]
        assert np.array_equal(a, exp), int((a != exp).sum())
        ang = O.assign_lloyd(Xc, Cc, metric=1, with_scores=True)[3]
        got_dot = np.clip(np.einsum("ij,ij->i", Xc.astype(np.float64), Cc[a].astype(np.float64)), -1, 1)
        assert np.abs(np.arccos(got_dot) - ang).max() < 2e-3   # acos is ill-conditioned next to the clamp
    Ci = C.copy()
    Ci[7, 63] = np.inf          # an infinite LAST feature survives the Kahan loop: dot=+inf clamps to angle 0 and wins
    Ci[9, 1] = np.nan
    a, _, _, info = _shard_pass(Xs, Ci, metric="cos")
    exp = _shard_pass(Xs, Ci, metric="cos", force_exact=True)[0]
    assert np.array_equal(a, exp), int((a != exp).sum())
    assert (a[Xs[:, 63] > 0] <= 7).all() and (a[Xs[:, 63] > 0] == 7).mean() > 0.9


def test_edge_cases_nan_ragged_ties(ours):
    X, C = cases.edge_cases()    # NaN rows / centroids, a 1e30 row, a duplicate centroid
    got = one_pass(ours, X, C)
    exp = REF["edge_cases"]
    keep = np.ones(len(X), bool)
    keep[77] = False            # left untouched by both (contents of the output buffer are unspecified)
    assert np.array_equal(got[keep], exp[keep])
    assert got[5] == 37 and got[300] == 4 and not (got[keep] == 3).any() and not (got[keep] == 10).any()


def test_headline_size_properties(km):
    """8M x 256 @ 1024 (BASELINE config 2): size-independent properties + exact spot check"""
    import torch
    from kmcuda_b200.shard import Shard
    n, d, k = 8000000, 256, 1024
    g = torch.Generator(device="cuda").manual_seed(777)
    X = torch.rand((n, d), generator=g, device="cuda", dtype=torch.float32)
    C = X[torch.randperm(n, generator=g, device="cuda")[:k]].contiguous()
    sh = Shard(n, d, k)
    a = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    prev = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    ch = torch.zeros(1, dtype=torch.int32, device="cuda")
    sh.assign(X, C, a, prev, ch)
    torch.cuda.synchronize()
    assert sh.last_error() == 0 and sh.last_pass_info()[0]
    assert int(ch.item()) == n and int(a.min()) >= 0 and int(a.max()) < k
    # the chosen centroid is at least as close (fp64) as any other, up to fp32 rounding, on a sample
    idx = torch.randperm(n, generator=g, device="cuda")[:20000]
    xs = X[idx].double()
    d2 = (C.double() ** 2).sum(1)[None, :] - 2 * xs @ C.double().T
    best = d2.min(1).values
    mine = d2.gather(1, a[idx].long()[:, None])[:, 0]
    assert float((mine - best).max()) <= 1e-4
    # rows whose source IS a centroid must map to it
    ch.zero_()
    sh.assign(X, C, a, prev, ch)
    torch.cuda.synchronize()
    assert int(ch.item()) == 0          # idempotent
    # bit-exact against the exact SIMT kernel of this library on the sample
    os.environ["KMCUDA_B200_FORCE_EXACT"] = "1"
    try:
        she = Shard(20000, d, k)
        ae = torch.full((20000,), -1, dtype=torch.int32, device="cuda")
        pe = torch.full((20000,), -1, dtype=torch.int32, device="cuda")
        she.assign(X[idx].contiguous(), C, ae, pe, ch)
        torch.cuda.synchronize()
        assert not she.last_pass_info()[0]
        assert bool((ae == a[idx]).all().item())
    finally:
        os.environ.pop("KMCUDA_B200_FORCE_EXACT", None)


def test_update_matches_oracle():
    import torch
    from kmcuda_b200.shard import Shard
    rng = np.random.default_rng(5)
    X = rng.random((20000, 64), dtype=np.float32)
    C0 = X[:100].copy()
    a, prev, _ = O.assign_lloyd(X, C0)
    Cexp, cnt = O.adjust(X, C0, prev, a, np.zeros(100, np.uint32))
    sh = Shard(len(X), 64, 100)
    Xt, at = torch.from_numpy(X).cuda(), torch.from_numpy(a.astype(np.int32)).cuda()
    sums = torch.zeros((100, 64), device="cuda")
    counts = torch.zeros(100, dtype=torch.int32, device="cuda")
    Ct = torch.zeros((100, 64), device="cuda")
    cc = torch.zeros(100, dtype=torch.int32, device="cuda")
    sh.partial_sums(Xt, at, sums, counts)
    sh.finish_update(sums, counts, Ct, cc)
    torch.cuda.synchronize()
    assert np.array_equal(cc.cpu().numpy().astype(np.uint32), cnt)
    np.testing.assert_allclose(Ct.cpu().numpy(), Cexp, rtol=1e-5)   # tolerance of north_star: 1e-5 relative


def _validate(X, centroids, assignments, tolerance):
    """reference src/test.py:176-183: one more sklearn Lloyd step changes < tolerance of the labels"""
    d = ((X[:, None, :].astype(np.float64) - centroids[None].astype(np.float64)) ** 2).sum(-1)
    assert (d.argmin(1) != assignments).mean() < tolerance


@pytest.mark.parametrize("init,yy", [("random", 0.0), ("k-means++", 0.0), ("k-means++", 0.1), ("afkmc2", 0.0),
                                     (("afkmc2", 100), 0.1)])
def test_kmeans_python_surface_validates(km, init, yy, capfd):
    """reference src/test.py:207-233,248-281 (random Lloyd / kmeans++ Lloyd / kmeans++ Yinyang / AFK-MC2)"""
    X = cases.blobs()
    cent, asg = km.kmeans_cuda(X, 50, init=init, device=1, verbosity=2, seed=3, tolerance=0.01, yinyang_t=yy)
    out = capfd.readouterr().out
    iters = sum(1 for line in out.split("\n") if line.startswith("iteration"))
    assert iters >= 2
    assert cent.shape == (50, 2) and asg.shape == (13000,) and asg.dtype == np.uint32
    assert not np.isnan(cent).any()
    _validate(X, cent, asg, 0.01)
    if "afkmc2" in str(init):   # the seeding must spread over the six blobs, like k-means++ does
        assert "afkmc2: calculating q" in out
        quadrant = (np.sign(np.round(cent[:, 0] / 2)) * 3 + np.sign(np.round(cent[:, 1] / 2))).astype(int)
        assert len(set(quadrant.tolist())) >= 5


def test_kmeans_runs_match_reference_trajectory(ours):
    """same imported centroids -> same assignments as the reference library after a whole run"""
    X, C0 = cases.blobs_start()
    for yy in (0.0, 0.1):
        C1, A1 = c_kmeans(ours, X, C0, 0.01, yy)
        C2, A2 = reference_run(ours, "trajectory/%.1f" % yy, X, C0, 0.01, yy)
        assert (A1 == A2).mean() > 0.99
        ok = ~np.isnan(C2).any(1)
        np.testing.assert_allclose(C1[ok], C2[ok], rtol=0, atol=2e-2)


@pytest.mark.parametrize("n,d,k,metric", cases.YY_LOCAL_SHAPES)
def test_yinyang_tensor_core_local_step_equals_reference_order_scan(ours, n, d, k, metric, monkeypatch):
    """Yinyang iterations: the tcgen05 candidate pass + exact finish (yinyang.cu) must give the same run as the
    reference-order per-row scan (KMCUDA_B200_FORCE_EXACT=1), and both the same as the reference library"""
    X, C0 = cases.yy_local(n, d, k, metric)            # structureless data: dozens of slow Yinyang iterations
    runs = {}
    for fe in ("0", "1"):
        monkeypatch.setenv("KMCUDA_B200_FORCE_EXACT", fe)
        runs[fe] = c_kmeans(ours, X, C0, 0.0005, 0.1, metric=metric)
    monkeypatch.setenv("KMCUDA_B200_FORCE_EXACT", "0")
    assert np.array_equal(runs["0"][1], runs["1"][1]), int((runs["0"][1] != runs["1"][1]).sum())
    np.testing.assert_array_equal(runs["0"][0], runs["1"][0])
    # Trajectory-independent check of the Yinyang result: the library returns the centroids of the LAST assignment
    # step (kmeans.cu:991-997), and a correct bound filter leaves every sample at the argmin over those centroids
    # (README.md:74-75) -- up to fp32 near-ties between the true-distance and the Lloyd ranking formulas.
    C_last, A_last = runs["0"]
    assert (one_pass(ours, X, C_last, metric=metric) == A_last).mean() > 0.9995
    # the reference library on the same input: same property, and the same run while the runs are short (over
    # dozens of iterations on structureless data 1e-7 centroid differences flip near-tie samples and any two
    # implementations drift apart)
    Co, Ao = c_kmeans(ours, X, C0, 0.04, 0.1, metric=metric)
    Cr, Ar = reference_run(ours, "yy_local/%d_%d_%d_%d" % (n, d, k, metric), X, C0, 0.04, 0.1, metric)
    assert (one_pass(ours, X, Cr, metric=metric) == Ar).mean() > 0.9995
    assert (Ao == Ar).mean() > 0.99, (Ao != Ar).mean()


def test_yinyang_log_lines_match_reference(ours, capfd):
    """the per-iteration reassignment counts (stdout contract, kmeans.cu:706) of a Yinyang run"""
    X, C0 = cases.mixture(50000, 16, 200, 9, sigma=0.12)
    capfd.readouterr()
    c_kmeans(ours, X, C0, 0.0002, 0.1, verbosity=1)
    out = capfd.readouterr().out
    outs = [[ln for ln in out.splitlines() if ln.startswith("iteration") or "refreshing" in ln],
            REF["yy_log_lines"].tolist()]
    print(outs[0])
    assert len(outs[0]) > 5 and any("refreshing" in ln for ln in outs[0])
    assert outs[0][:8] == outs[1][:8]


def test_fp16_and_average_distance(km):
    X = cases.blobs()
    c32, a32, avg = km.kmeans_cuda(X, 50, init="k-means++", device=1, seed=3, tolerance=0.01, yinyang_t=0,
                                   average_distance=True)
    dists = np.linalg.norm(X - c32[a32], axis=1)
    assert abs(avg - dists.mean()) < 1e-5
    c16, a16 = km.kmeans_cuda(X.astype(np.float16), 50, init="k-means++", device=1, seed=3, tolerance=0.01,
                              yinyang_t=0)
    assert c16.dtype == np.float16 and c16.shape == (50, 2)
    _validate(X.astype(np.float16).astype(np.float32), c16.astype(np.float32), a16, 0.02)


def test_cosine_lloyd(km):
    rng = np.random.default_rng(3)
    X = rng.standard_normal((5000, 32)).astype(np.float32)
    X /= np.linalg.norm(X, axis=1, keepdims=True)
    cent, asg = km.kmeans_cuda(X, 20, init="random", metric="cos", device=1, seed=3, yinyang_t=0, tolerance=0.01)
    norms = np.linalg.norm(cent, axis=1)
    assert ((norms > 0.9999) & (norms < 1.0001)).all()          # reference src/test.py:437-440
    assert ((X @ cent.T).argmax(1) != asg).mean() < 0.02
    with pytest.raises(ValueError):                               # un-normalised samples are rejected
        km.kmeans_cuda(X * 2, 20, metric="cos", device=1)


def test_cosine_runs_follow_reference_update_rule(ours):
    """angular metric, whole runs: the reference's incremental update (centroid * old count + joined - left, then
    L2-normalise, kmeans.cu:366-429) is NOT the spherical mean once the centroid has been normalised; the runs only
    agree if that recurrence is reproduced"""
    X, C0 = cases.cosine_runs()
    for tol, yy in cases.COSINE_RUNS:
        Co, Ao = c_kmeans(ours, X, C0, tol, yy, metric=1)
        Cr, Ar = reference_run(ours, "cosine_runs/%.2f_%.1f" % (tol, yy), X, C0, tol, yy, 1)
        assert (Ao == Ar).mean() > 0.999, (tol, yy, (Ao != Ar).mean())
        assert (np.abs(Co - Cr).max(1) < 1e-4).mean() > 0.9


def test_knn_matches_sklearn_exactly(km):
    """reference src/test.py:598-606: k=10 on the blobs must equal sklearn's neighbours"""
    X = cases.blobs()
    cent, asg = km.kmeans_cuda(X, 50, init="k-means++", device=1, seed=777, yinyang_t=0)
    nb = km.knn_cuda(10, X, cent, asg, device=1, verbosity=1)
    exp = GOLDEN["knn/blobs_k10"]
    assert nb.shape == exp.shape
    diff = nb != exp
    if diff.any():   # only exact distance ties may differ
        rows = np.unique(np.argwhere(diff)[:, 0])
        for r in rows:
            dg = np.linalg.norm(X[nb[r]].astype(np.float64) - X[r], axis=1)
            de = np.linalg.norm(X[exp[r]].astype(np.float64) - X[r], axis=1)
            assert np.allclose(dg, de, atol=1e-7)
    assert diff.mean() < 1e-3


def test_knn_matches_reference(ours):
    """the reference's neighbour lists on its own clustering, compared on the stored query sample"""
    X, C0 = cases.uniform_rows(20000, 48, 200, 9)
    C, A = reference_run(ours, "knn_20k", X, C0, 0.05, 0.0)
    k = 10
    out = np.zeros((len(X), k), np.uint32)
    rc = ours.knn_cuda(k, 0, len(X), 48, 200, 1, -1, 0, 0, X.ctypes.data, C.ctypes.data, A.ctypes.data,
                       out.ctypes.data)
    assert rc == 0
    assert (out[cases.sample_rows(len(X))] != REF["knn_20k/nb_sample"]).mean() < 1e-4


def _knn(lib, k, X, C, A, metric=0):
    out = np.zeros((len(X), k), np.uint32)
    rc = lib.knn_cuda(k, metric, X.shape[0], X.shape[1], C.shape[0], 1, -1, 0, 0, X.ctypes.data, C.ctypes.data,
                      A.ctypes.data, out.ctypes.data)
    assert rc == 0, rc
    return out


@pytest.mark.parametrize("kind,n,d,kc,k", cases.KNN_TC_SHAPES)
def test_knn_tensor_core_path_matches_reference(ours, capfd, monkeypatch, kind, n, d, kc, k):
    """knn_cuda through the tcgen05 candidate pass (cluster-sorted tiles, two passes, exact re-check + selection) on the
    reference's clustering: same neighbours as the reference library (stored query sample), and as a float64 brute
    force on a sample of the queries"""
    X, C0, rng = cases.knn_tc(kind, n, d, kc)
    key = "knn_tc/%s_%d_%d_%d_%d" % (kind, n, d, kc, k)
    C, A = reference_run(ours, key, X, C0, 0.05, 0.0)
    monkeypatch.setenv("KMCUDA_B200_TIMING", "1")
    capfd.readouterr()
    got = _knn(ours, k, X, C, A)
    err = capfd.readouterr().err
    monkeypatch.delenv("KMCUDA_B200_TIMING")
    line = [ln for ln in err.splitlines() if "knn tensor-core path" in ln]
    assert line, "tensor-core k-NN path not taken: " + err[-300:]
    served = int(line[0].split("path:")[1].split("rows")[0])
    assert served > 0.98 * n, line[0]
    exp = REF[key + "/nb_sample"]
    assert (got[cases.sample_rows(n)] != exp).mean() < 1e-4, (got[cases.sample_rows(n)] != exp).mean()
    # independent check: float64 brute force for 300 queries (ties at the k-th place aside)
    qs = rng.choice(n, 300, replace=False)
    Xd = X.astype(np.float64)
    bad = 0
    for q in qs:
        dist = ((Xd - Xd[q]) ** 2).sum(1)
        dist[q] = np.inf
        order = np.argsort(dist, kind="stable")[:k + 1]
        if abs(dist[order[k]] - dist[order[k - 1]]) < 1e-9 * max(1.0, dist[order[k]]):
            continue
        bad += set(got[q].tolist()) != set(order[:k].tolist())
    assert bad == 0, bad


def test_device_pointer_api(km):
    """reference src/test.py:348-372: raw device pointers in, raw device pointers out; samples untouched"""
    import torch
    X = cases.blobs()
    Xt = torch.from_numpy(X).cuda()
    before = Xt.clone()
    cptr, aptr = km.kmeans_cuda((Xt.data_ptr(), 0, X.shape), 50, init="k-means++", device=1, seed=3,
                                tolerance=0.01, yinyang_t=0)
    assert isinstance(cptr, int) and isinstance(aptr, int)
    cent = np.empty((50, 2), np.float32)
    asg = np.empty(13000, np.uint32)
    km._cuda_memcpy_d2h(0, cent.ctypes.data, cptr, cent.nbytes)
    km._cuda_memcpy_d2h(0, asg.ctypes.data, aptr, asg.nbytes)
    km._cuda_free(0, cptr)
    km._cuda_free(0, aptr)
    assert torch.equal(Xt, before)
    _validate(X, cent, asg, 0.01)
