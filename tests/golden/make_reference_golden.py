"""Records what the unmodified reference library computes on the inputs of the GPU tests that compare with it, so
that those tests run without it.  Needs a GPU and the reference built into oracle/_ref (oracle/build_ref.sh):

    python tests/golden/make_reference_golden.py RAW.npz         # run the reference, keep every output in RAW.npz
    python tests/golden/make_reference_golden.py RAW.npz --pack  # (no GPU needed) RAW.npz -> tests/golden/reference.npz

Inputs are regenerated from seeds by tests/golden/cases.py.  reference.npz keeps an output in full where it is small,
as a SHA-256 digest where the test asks for bit equality of a large output, and as a fixed row sample where the test
bounds a mismatch rate.  The centroids and assignments of whole runs are
kept as digests: the tests rebuild them with this library's strict-update mode (KMCUDA_B200_STRICT_UPDATE=1, which
replays the reference's centroid update) and check the digests.
"""
import ctypes
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

from oracle import oracle as O  # noqa: E402
import cases  # noqa: E402

IMPORT = 3
OUT = os.path.join(HERE, "reference.npz")


def c_kmeans(lib, X, C0, tol, yy, metric=0, verbosity=0):
    X = np.ascontiguousarray(X)
    N, D = X.shape
    C = np.array(C0, copy=True, order="C")
    A = np.zeros(N, np.uint32)
    m = ctypes.c_uint32(0)
    rc = lib.kmeans_cuda(IMPORT, ctypes.byref(m), tol, yy, metric, N, D, C.shape[0], 3, 1, -1, 0, verbosity,
                         X.ctypes.data, C.ctypes.data, A.ctypes.data, None)
    assert rc == 0, rc
    return C, A


def knn(lib, k, X, C, A, metric=0):
    out = np.zeros((len(X), k), np.uint32)
    rc = lib.knn_cuda(k, metric, X.shape[0], X.shape[1], C.shape[0], 1, -1, 0, 0, X.ctypes.data, C.ctypes.data,
                      A.ctypes.data, out.ctypes.data)
    assert rc == 0, rc
    return out


def logged_run(lib, X, C0, tol, yy, metric=0):
    """c_kmeans with verbosity 1; returns (C, A, the "iteration" / "refreshing" lines the library printed)"""
    libc = ctypes.CDLL(None)
    sys.stdout.flush()
    saved = os.dup(1)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 1)
        try:
            C, A = c_kmeans(lib, X, C0, tol, yy, metric, verbosity=1)
            libc.fflush(None)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
        f.seek(0)
        lines = [ln for ln in f.read().splitlines() if ln.startswith("iteration") or "refreshing" in ln]
    return C, A, lines


def run(raw_path):
    import torch
    assert torch.cuda.is_available() and O.reference_available()
    ref = O.reference_lib()
    raw = {}

    def one_pass(X, C, metric=0):
        return c_kmeans(ref, X, C, 1.0, 0.0, metric)[1]

    for name in cases.ORACLE_PIN_CASES:
        raw["oracle_pin/" + name] = one_pass(*cases.make_assign_case(*cases.ASSIGN_CASES[name]))
    raw["tc_100k"] = one_pass(*cases.uniform_rows(100000, 256, 1024, 777))
    for n, d, k, metric in cases.WIDE_SHAPES:
        raw["wide/%d_%d_%d_%s" % (n, d, k, metric)] = one_pass(*cases.wide_shape(n, d, k, metric),
                                                               metric=int(metric == "cos"))
    raw["edge_cases"] = one_pass(*cases.edge_cases())
    X, C0 = cases.blobs_start()
    for yy in (0.0, 0.1):
        raw["trajectory/%.1f/C" % yy], raw["trajectory/%.1f/A" % yy] = c_kmeans(ref, X, C0, 0.01, yy)
    for n, d, k, metric in cases.YY_LOCAL_SHAPES:
        key = "yy_local/%d_%d_%d_%d/" % (n, d, k, metric)
        raw[key + "C"], raw[key + "A"] = c_kmeans(ref, *cases.yy_local(n, d, k, metric), 0.04, 0.1, metric)
    raw["yy_log_lines"] = np.array(logged_run(ref, *cases.mixture(50000, 16, 200, 9, sigma=0.12), 0.0002, 0.1)[2])
    X, C0 = cases.cosine_runs()
    for tol, yy in cases.COSINE_RUNS:
        key = "cosine_runs/%.2f_%.1f/" % (tol, yy)
        raw[key + "C"], raw[key + "A"] = c_kmeans(ref, X, C0, tol, yy, 1)
    X, C0 = cases.uniform_rows(20000, 48, 200, 9)
    C, A = c_kmeans(ref, X, C0, 0.05, 0.0)
    raw["knn_20k/C"], raw["knn_20k/A"], raw["knn_20k/nb"] = C, A, knn(ref, 10, X, C, A)
    for kind, n, d, kc, k in cases.KNN_TC_SHAPES:
        X, C0, _ = cases.knn_tc(kind, n, d, kc)
        C, A = c_kmeans(ref, X, C0, 0.05, 0.0)
        key = "knn_tc/%s_%d_%d_%d_%d/" % (kind, n, d, kc, k)
        raw[key + "C"], raw[key + "A"], raw[key + "nb"] = C, A, knn(ref, k, X, C, A)
    for n, d, k, metric in cases.UPDATE_SHAPES:
        key = "update/%d_%d_%d_%d/" % (n, d, k, metric)
        raw[key + "C"], raw[key + "A"] = c_kmeans(ref, *cases.update_case(n, d, k, metric, n + d), 0.99, 0.0, metric)
    raw["adjust_pin/C"], raw["adjust_pin/A"] = c_kmeans(ref, *cases.adjust_pin(), 0.99, 0.0)
    X, C0 = cases.uniform_rows(100000, 256, 1024, 777)
    C, A, lines = logged_run(ref, X, C0, 0.002, 0.0)
    raw["c1_run/C"], raw["c1_run/A"], raw["c1_run/lines"] = C, A, np.array(lines)
    raw["headline_8m/sha256"] = np.array(cases.digest(one_pass(*cases.headline_8m())))
    raw["far_outliers"] = one_pass(*cases.far_outliers())
    X, C0, _ = cases.knn_angular()
    C, A = c_kmeans(ref, X, C0, 0.05, 0.0, 1)
    raw["knn_angular/C"], raw["knn_angular/A"], raw["knn_angular/nb"] = C, A, knn(ref, 10, X, C, A, 1)
    X, centers, _ = cases.knn_c5()
    C, A = c_kmeans(ref, X, centers, 0.01, 0.0)
    raw["knn_c5/C"], raw["knn_c5/A"], raw["knn_c5/nb"] = C, A, knn(ref, 10, X, C, A)
    for n, d, k, metric, tol, yy in cases.STRICT_RUNS:
        key = "strict/%d_%d_%d_%d_%g_%g/" % (n, d, k, metric, tol, yy)
        C, A, lines = logged_run(ref, *cases.update_case(n, d, k, metric, n + k), tol, yy, metric)
        raw[key + "C"], raw[key + "A"], raw[key + "lines"] = C, A, np.array(lines)
    for n in cases.CTA_PAIR_ROWS:
        raw["cta_pair/%d" % n] = one_pass(*cases.uniform_rows(n, 256, 1000, 4242))
    np.savez(raw_path, **raw)
    print("wrote", raw_path)


def pack(raw_path):
    raw = np.load(raw_path)
    out = {}
    for key in raw.files:
        v = raw[key]
        if key.endswith("/nb"):               # k-NN lists: the rows of the fixed query sample
            v = v[cases.sample_rows(len(v))]
            out[key + "_sample"] = v.astype(np.uint16) if v.max() < 1 << 16 else v
        elif v.dtype.kind == "U" or key in ("edge_cases", "far_outliers"):
            out[key] = v                      # log lines, digests, small outputs in full
        else:
            out[key] = np.array(cases.digest(v))
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    if "--pack" in sys.argv:
        pack(sys.argv[1])
    else:
        run(sys.argv[1])
        pack(sys.argv[1])
