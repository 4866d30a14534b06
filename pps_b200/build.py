"""Build recipe for libpps_b200.so (hand-written sm_100a CUDA behind a C ABI).

The library is built in-tree (``pps_b200/_C/libpps_b200.so``) so that it travels with a
snapshot of the repository; nothing is JIT-compiled at run time.
"""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB_PATH = os.path.join(OUT_DIR, "libpps_b200.so")
SOURCES = ["pps_pool.cu", "split_prep.cu", "dist_gemm.cu", "pairs.cu", "rank.cu", "triplet.cu", "rerank.cu", "c_api.cu", "pass.cu", "index.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "ctx.cuh"), os.path.join(CSRC, "dist_tiles.cuh"), os.path.join(os.path.dirname(HERE), "include", "pps_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
]
OBJ_DIR = os.path.join(OUT_DIR, "obj")


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _compile_one(nvcc, src, obj, verbose):
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
    proc = subprocess.run(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return src, proc.returncode, proc.stdout


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a (one object per source, in parallel; objects newer than their source and
    the shared headers are reused) and link them into one shared library; returns its path."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = nvcc_path()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libpps_b200.so (set NVCC or install the CUDA toolkit)")
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdr_t = max(os.path.getmtime(h) for h in HEADERS if os.path.exists(h))
    jobs, objs = [], []
    for src in SOURCES:
        obj = os.path.join(OBJ_DIR, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        src_t = max(os.path.getmtime(os.path.join(CSRC, src)), hdr_t)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < src_t:
            jobs.append((src, obj))
    log = []
    if jobs:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as pool:
            for src, rc, out in pool.map(lambda j: _compile_one(nvcc, j[0], j[1], verbose), jobs):
                log.append("== %s ==\n%s" % (src, out))
                if rc != 0:
                    raise RuntimeError("nvcc failed on %s (%d):\n%s" % (src, rc, out))
    tmp = LIB_PATH + ".tmp.%d" % os.getpid()
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", tmp] + objs
    proc = subprocess.run(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise RuntimeError("nvcc link failed (%d):\n%s" % (proc.returncode, proc.stdout))
    os.replace(tmp, LIB_PATH)
    if verbose:
        print("\n".join(log))
    return LIB_PATH


TEST_HOOKS_PATH = os.path.join(OUT_DIR, "libpps_b200_testhooks.so")


def build_test_hooks(force: bool = False) -> str:
    """TEST-ONLY library (csrc/test_hooks.cu: the host replay of the distance kernels' tile schedule); never loaded by the
    product.  Returns its path."""
    src = os.path.join(CSRC, "test_hooks.cu")
    deps = [src] + [h for h in HEADERS if os.path.exists(h)]
    if (not force and os.path.exists(TEST_HOOKS_PATH)
            and all(os.path.getmtime(d) <= os.path.getmtime(TEST_HOOKS_PATH) for d in deps)):
        return TEST_HOOKS_PATH
    nvcc = nvcc_path()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build the test hooks")
    os.makedirs(OUT_DIR, exist_ok=True)
    tmp = TEST_HOOKS_PATH + ".tmp.%d" % os.getpid()
    proc = subprocess.run([nvcc] + NVCC_FLAGS + ["-shared", "-o", tmp, "test_hooks.cu"], cwd=CSRC, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed on test_hooks.cu:\n%s" % proc.stdout)
    os.replace(tmp, TEST_HOOKS_PATH)
    return TEST_HOOKS_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
