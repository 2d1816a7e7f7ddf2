"""Build libtwowl_b200.so (the C-ABI library of include/twowl.h) in-tree with nvcc for sm_100a.

    python link-prediction-gnn_b200/build.py [--force]

nvcc cross-compiles without a GPU. The .so lands next to the Python loader
(link-prediction-gnn_b200/twowl_b200/libtwowl_b200.so), is git-ignored, and travels to the GPU
box with the gpurun snapshot.
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "twowl_b200")
LIB = os.path.join(OUT_DIR, "libtwowl_b200.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["prims.cu", "index_ops.cu", "agg.cu", "norm.cu", "pair_ops.cu", "linear.cu", "pair_conv.cu", "dw_tc.cu", "metrics.cu", "sampler.cu", "nodefeat.cu", "train_ops.cu", "heuristics.cu", "walks.cu", "node2vec.cu", "seal.cu", "sketch.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"] + os.environ.get("TWOWL_NVCC_DEFS", "").split()   # e.g. -DTWOWL_DW_FLUSH=2 (tuning builds)


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _stale(target, deps) -> bool:
    if not os.path.isfile(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, "common.cuh"), os.path.join(HERE, "..", "include", "twowl.h"),
               os.path.abspath(__file__)]
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for log in ex.map(run, jobs):
            if verbose and log:
                print(log)
    objs = [os.path.join(OBJ_DIR, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        run([nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
