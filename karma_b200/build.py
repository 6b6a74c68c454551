"""Build libkarma_b200.so in-tree with nvcc for sm_100a (no torch extension machinery).

    python -m karma_b200.build [--force]

The shared library is a plain C-ABI (include/karma_b200.h); it links the CUDA
runtime statically and resolves cuTensorMapEncodeTiled from the driver at run
time, so it loads (and exports every symbol) on a machine without a GPU.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libkarma_b200.so")
SOURCES = ["kb_api.cu", "kb_count.cu", "kb_profile.cu", "kb_exotic.cu", "kb_knn.cu", "kb_knn_tc.cu", "kb_xchg.cu", "kb_fasta.cu", "kb_readgraph.cu", "kb_links.cu", "kb_umapgraph.cu", "kb_umaplayout.cu", "kb_hdbscan.cu", "kb_spectral.cu", "kb_mcl.cu"]
HEADERS = ["kb_common.cuh", "kb_knn.cuh", os.path.join("..", "..", "include", "karma_b200.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + hdrs):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (s, r.stdout, r.stderr))
        if verbose:
            print("compiled", os.path.basename(s))
        return o

    with ThreadPoolExecutor(max_workers=min(6, max(1, len(jobs)))) as ex:
        list(ex.map(compile_one, jobs))
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
               "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
        if verbose:
            print("linked", LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
