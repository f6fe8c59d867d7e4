"""In-tree build of libKMCUDA.so for sm_100a (nvcc cross-compiles without a GPU).

    python kmcuda_b200/build.py            # incremental (run by path: importing the package needs the built library)
    python kmcuda_b200/build.py --force

The product library is `kmcuda_b200/libKMCUDA.so`: it exports the reference's C ABI
(kmeans_cuda, knn_cuda -- include/kmcuda.h), the shard-level extension (include/kmcuda_b200.h) and,
when the CPython/NumPy headers are available, PyInit_libKMCUDA (the drop-in Python module).
"""
import concurrent.futures
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libKMCUDA.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

CU_SOURCES = ["simt_kernels.cu", "knn_kernels.cu", "assign_tc.cu", "yinyang.cu", "shard.cu", "exchange.cu", "api.cu"]
CC_SOURCES = ["py_module.cc"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-strict-aliasing", "-I" + os.path.join(ROOT, "include"),
              "-I" + CSRC]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hs += [os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))]
    return hs


def _run(cmd):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("build failed: %s\n%s" % (" ".join(cmd), r.stdout))
    return r.stdout


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = _headers()
    jobs = []
    objs = []
    for src in CU_SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src + ".o")
        objs.append(o)
        if force or _newer(o, [s] + headers):
            jobs.append([NVCC] + NVCC_FLAGS + ["-c", s, "-o", o])
    for src in CC_SOURCES:
        s = os.path.join(CSRC, src)
        if not os.path.exists(s):
            continue
        o = os.path.join(OBJ, src + ".o")
        objs.append(o)
        if force or _newer(o, [s] + headers):
            import numpy
            jobs.append(["g++", "-std=c++17", "-O2", "-fPIC", "-I" + os.path.join(ROOT, "include"),
                         "-I/usr/local/cuda/include", "-I" + sysconfig.get_paths()["include"],
                         "-I" + numpy.get_include(), "-c", s, "-o", o])
    if jobs:
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for out in ex.map(_run, jobs):
                if verbose and out.strip():
                    print(out)
    if force or jobs or _newer(LIB, objs):
        _run([NVCC, "-shared", "-o", LIB] + objs + ["-ldl"])  # NCCL is bound at run time (api.cu)
    return LIB


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    a = ap.parse_args()
    print(build(force=a.force, verbose=True))
