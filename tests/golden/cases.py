"""Seeded input generators shared by make_golden.py, make_reference_golden.py and the tests (inputs are never
stored)."""
import hashlib
import os

import numpy as np

# name -> (n, d, k, seed, kind)
ASSIGN_CASES = {
    "uniform_3000x256_k1024": (3000, 256, 1024, 777, "uniform"),
    "uniform_5000x64_k100": (5000, 64, 100, 1, "uniform"),
    "normal_4000x128_k300": (4000, 128, 300, 2, "normal"),
    "ragged_1000x7_k3": (1000, 7, 3, 3, "uniform"),
    "ragged_4097x100_k33": (4097, 100, 33, 4, "uniform"),
    "blobs_13000x2_k50": (13000, 2, 50, 5, "blobs"),
    "wide_range_2000x32_k16": (2000, 32, 16, 6, "wide"),
    "dupes_1024x64_k64": (1024, 64, 64, 7, "dupes"),
}


def blobs():
    """reference src/test.py:158-169"""
    rng = np.random.RandomState(0)
    arr = np.empty((13000, 2), dtype=np.float32)
    arr[:2000] = rng.rand(2000, 2) + [0, 2]
    arr[2000:4000] = rng.rand(2000, 2) - [0, 2]
    arr[4000:6000] = rng.rand(2000, 2) + [2, 0]
    arr[6000:8000] = rng.rand(2000, 2) - [2, 0]
    arr[8000:10000] = rng.rand(2000, 2) - [2, 2]
    arr[10000:] = rng.rand(3000, 2) + [2, 2]
    return arr


def make_assign_case(n, d, k, seed, kind):
    rng = np.random.default_rng(seed)
    if kind == "blobs":
        X = blobs()
    elif kind == "normal":
        X = rng.standard_normal((n, d)).astype(np.float32)
    elif kind == "wide":      # features spanning 12 orders of magnitude
        X = (rng.standard_normal((n, d)) * (10.0 ** rng.integers(-6, 6, size=d))).astype(np.float32)
    else:
        X = rng.random((n, d), dtype=np.float32)
    C = X[rng.choice(len(X), k, replace=False)].copy()
    if kind == "dupes":       # exact duplicate centroids: ties must resolve to the lowest index
        C[k // 2:] = C[:k - k // 2]
    else:
        C += (rng.standard_normal(C.shape) * 0.01 * np.abs(C).mean()).astype(np.float32)
    return np.ascontiguousarray(X), np.ascontiguousarray(C)


# ---------------------------------------------------------------------------------------------------------------------
# Inputs of the tests that compare with the reference library (make_reference_golden.py stores its outputs on them).
# Functions that draw from a generator the test keeps drawing from afterwards return it.
# ---------------------------------------------------------------------------------------------------------------------
ORACLE_PIN_CASES = ["uniform_3000x256_k1024", "ragged_4097x100_k33", "blobs_13000x2_k50", "wide_range_2000x32_k16",
                    "dupes_1024x64_k64"]
WIDE_SHAPES = [(20000, 256, 500, "cos"), (20000, 480, 2000, "L2"), (20000, 480, 2000, "cos"), (30000, 64, 20000, "L2"),
               (9000, 324, 700, "L2")]
YY_LOCAL_SHAPES = [(60000, 64, 256, 0), (40000, 100, 120, 0), (30000, 32, 64, 1)]
COSINE_RUNS = [(0.12, 0.0), (0.04, 0.0), (0.04, 0.1)]
KNN_TC_SHAPES = [("uniform", 30000, 48, 200, 10), ("mixture", 60000, 64, 300, 10), ("mixture", 50000, 256, 100, 3),
                 ("uniform", 20000, 100, 50, 15)]
UPDATE_SHAPES = [(100000, 256, 1024, 0), (60000, 128, 300, 1), (30011, 100, 77, 0)]
STRICT_RUNS = [(100000, 256, 1024, 0, 0.002, 0.0), (30000, 32, 64, 1, 0.001, 0.0), (60000, 64, 256, 0, 0.001, 0.1)]
CTA_PAIR_ROWS = [75776 + 2 * 128 + 17, 75776 + 4 * 128]   # 595 tiles (odd: phantom tile in the last pair) and 596


def digest(a):
    """SHA-256 of an array's bytes (every NaN counted as the same NaN): stands for a large output that a test compares
    bit for bit"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.array(np.nan, a.dtype), a)
    return hashlib.sha256(a.tobytes()).hexdigest()


def strict_replay(run, ref, key):
    """A whole run of the reference library, replayed: `run()` calls this library with KMCUDA_B200_STRICT_UPDATE=1
    (the reference's running-sum centroid update in sample order), and the centroids and assignments its result ends
    with must match the digests of the reference's ("<key>/C", "<key>/A" in `ref`).  On the B200 the replay is bit for
    bit for Lloyd, Yinyang and cosine runs alike."""
    old = os.environ.get("KMCUDA_B200_STRICT_UPDATE")
    os.environ["KMCUDA_B200_STRICT_UPDATE"] = "1"    # read when the shard is created
    try:
        out = run()
    finally:
        if old is None:
            os.environ.pop("KMCUDA_B200_STRICT_UPDATE", None)
        else:
            os.environ["KMCUDA_B200_STRICT_UPDATE"] = old
    C, A = out[-2:]
    assert digest(C) == str(ref[key + "/C"]) and digest(A) == str(ref[key + "/A"]), \
        "%s: the strict-update run is not the reference's" % key
    return out


def sample_rows(n, m=1000):
    """the fixed rows of a large output whose values are stored"""
    return np.sort(np.random.default_rng(2024).choice(n, min(n, m), replace=False))


def unit(a):
    return (a / np.linalg.norm(a, axis=1, keepdims=True)).astype(np.float32)


def mixture(n, d, k, seed, sigma=0.25):
    """overlapping Gaussian blobs, initial centroids next to the true centres (no cluster runs empty: the
    reference library aborts in its Yinyang grouping when a centroid is NaN)"""
    rng = np.random.default_rng(seed)
    centers = rng.random((k, d), dtype=np.float32)
    X = centers[rng.integers(0, k, n)] + sigma * rng.standard_normal((n, d), dtype=np.float32)
    C0 = centers + 0.1 * rng.standard_normal((k, d), dtype=np.float32)
    return np.ascontiguousarray(X), np.ascontiguousarray(C0)


def uniform_rows(n, d, k, seed):
    """U[0,1) samples, centroids = k distinct rows of them"""
    rng = np.random.default_rng(seed)
    X = rng.random((n, d), dtype=np.float32)
    return X, X[rng.choice(n, k, replace=False)].copy()


def wide_shape(n, d, k, metric):
    rng = np.random.default_rng(n + d + k)
    X = rng.standard_normal((n, d)).astype(np.float32)
    if metric == "cos":
        X = unit(X)
    C = X[rng.choice(n, k, replace=False)].copy()
    C += (rng.standard_normal(C.shape) * 0.05 * np.abs(C).mean()).astype(np.float32)
    if metric == "cos":
        C = unit(C)
    return X, C


def edge_cases():
    rng = np.random.default_rng(11)
    X = rng.random((1000, 64), dtype=np.float32)
    C = X[rng.choice(1000, 37, replace=False)].copy()
    X[5, 0] = np.nan            # "insane" row -> K
    X[77, 13] = np.nan          # NaN elsewhere -> nothing wins
    X[200] = 1e30               # overflows the fp16 filter -> exact fallback
    C[3] = np.nan               # NaN centroid never wins
    C[10] = C[4]                # duplicate centroid -> lowest index
    X[300] = C[4]
    return X, C


def blobs_start():
    X = blobs()
    rng = np.random.default_rng(1)
    return X, X[rng.choice(len(X), 50, replace=False)].copy()


def yy_local(n, d, k, metric):
    rng = np.random.default_rng(42 + d)
    X = rng.random((n, d), dtype=np.float32) if metric == 0 else rng.standard_normal((n, d)).astype(np.float32)
    C0 = X[rng.choice(n, k, replace=False)].copy()     # structureless data: dozens of slow Yinyang iterations
    if metric == 1:
        X, C0 = unit(X), unit(C0)
    return X, C0


def cosine_runs():
    rng = np.random.default_rng(74)
    X = unit(rng.standard_normal((30000, 32)))
    return X, X[rng.choice(30000, 64, replace=False)].copy()


def knn_tc(kind, n, d, kc):
    rng = np.random.default_rng(n + d)
    if kind == "uniform":
        X = rng.random((n, d), dtype=np.float32)
        C0 = X[rng.choice(n, kc, replace=False)].copy()
    else:
        X, C0 = mixture(n, d, kc, 5, sigma=0.15)
    return X, C0, rng


def update_case(n, d, k, metric, seed):
    rng = np.random.default_rng(seed)
    X = rng.random((n, d), dtype=np.float32) if metric == 0 else unit(rng.standard_normal((n, d)))
    return X, X[rng.choice(n, k, replace=False)].copy()


def headline_8m():
    n, d, k = 8000000, 256, 1024
    rng = np.random.default_rng(777)
    X = np.empty((n, d), np.float32)
    for i in range(0, n, 1000000):               # chunked generation keeps the host RSS at the matrix itself
        X[i:i + 1000000] = rng.random((1000000, d), dtype=np.float32)
    return X, X[rng.choice(n, k, replace=False)].copy()


def far_outliers():
    rng = np.random.default_rng(3)
    n, d, k = 5000, 64, 200                      # 200 % 128 != 0: 56 padded columns
    X = (1.0 + 0.05 * rng.standard_normal((n, d))).astype(np.float32)
    C = (1.0 + 0.05 * rng.standard_normal((k, d))).astype(np.float32)
    C[17] = np.nan
    X[3] = -40.0
    X[77] = -900.0
    X[1234] = 3000.0
    X[99, :] = 0.0
    return X, C


def knn_angular():
    rng = np.random.default_rng(31)
    n, d, kc = 20000, 48, 100
    X = unit(rng.standard_normal((n, d)) + 2.0 * rng.standard_normal((1, d)))
    return X, X[rng.choice(n, kc, replace=False)].copy(), rng


def knn_c5():
    rng = np.random.default_rng(55)
    n, d, kc = 300000, 256, 100
    centers = rng.random((kc, d), dtype=np.float32)
    X = (centers[rng.integers(0, kc, n)] + 0.05 * rng.standard_normal((n, d), dtype=np.float32)).astype(np.float32)
    return X, centers, rng


def adjust_pin():
    rng = np.random.default_rng(12)
    X = rng.random((20000, 64), dtype=np.float32)
    return X, X[:100].copy()
