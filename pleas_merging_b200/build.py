"""Builds the sm_100a shared library in-tree (nvcc cross-compiles without a GPU).

    python -m pleas_merging_b200.build

The .so is git-ignored: a fresh checkout builds it with this module or ``__graft_entry__.build()``.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libpleas_b200.so")
SOURCES = ["api.cu", "gemm.cu", "gram_direct.cu", "gram_tma.cu", "pack.cu", "finalize.cu", "lap.cu", "blocks.cu", "chol.cu", "conv.cu"]


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(os.path.dirname(HERE), "include", "pleas_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_one(nvcc, src, obj, verbose):
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xcompiler", "-fPIC", "-c", src, "-o", obj]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)


def build(force=False, verbose=False):
    """One object per source (compiled in parallel, rebuilt only when the source or a header is newer), then
    one link: editing a single kernel costs one nvcc run."""
    if not force and not _stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor

    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + [
        os.path.join(os.path.dirname(HERE), "include", "pleas_b200.h")]
    newest_header = max(os.path.getmtime(h) for h in headers)
    jobs, objs = [], []
    for s in SOURCES:
        src, obj = os.path.join(CSRC, s), os.path.join(obj_dir, s[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), newest_header):
            jobs.append((src, obj))
    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as pool:
        for f in [pool.submit(_compile_one, nvcc, src, obj, verbose) for src, obj in jobs]:
            f.result()
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static",
                    *objs, "-o", LIB_PATH], check=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
