"""UMAP's spectral initialisation (K10) on the device against umap 0.3.9's formulation on the CPU.

Inputs: the K7 graph of the exact device kNN lists of S1 50 k (-k 5p6) at n_neighbors 2 (karma's default), 5 and 15,
and of S2 200 k (-k 5+6) at 15, pruned at max / 200 (umap's n_epochs above 10 000 rows); dim 10.  Per input:
  components_ms, eigensolve_ms, meta_ms   device time of the three stages (the library's CUDA-event stage timers),
                                          after one warm-up build, median of --repeats
  lanczos_steps, restarts                 over every solved component; meta_steps, meta_restarts for the meta points
  host_to_host_ms                         umap_spectral.spectral_layout (the 0.3.9 drop-in) on the pruned host graph
                                          and float32 data -> numpy layout, median of --repeats
  cpu_arm_ms                              oracle/umap_spectral_oracle.spectral_layout_reference (scipy eigsh with
                                          umap's arguments, scikit-learn's SpectralEmbedding) on the same graph and
                                          data, one run in a single-threaded child process stopped after --cpu-cap
                                          seconds (null, with the reason in ``cpu_arm``, when it does not finish)
    python scripts/bench_umap_spectral.py [--repeats 3] [--cpu-cap 600] [--inputs S1:50000:2,...]
Prints one JSON line, with the card's name and power limit read by nvidia-smi in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import warnings

import numpy as np
import scipy.sparse
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from karma_b200.engine import Engine  # noqa: E402
from karma_b200.umap_spectral import SOLVED, spectral_build, spectral_layout  # noqa: E402
from oracle import umap_spectral_oracle as so  # noqa: E402

DIM = 10
N_EPOCHS = 200
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def k7_graph(eng, kind, n, k):
    from karma_b200 import synth
    from karma_b200.engine import device_pass
    from karma_b200.umap_graph import build_graph
    asm = synth.make(kind, n)
    d_bases, d_offsets, d_key_len = eng.upload(asm.bases, asm.offsets, asm.key_len)
    r = device_pass(eng, d_bases, d_offsets, d_key_len, n, "5p6" if kind == "S1" else "5+6", n_neighbors=k,
                    want_profile=True)
    return build_graph(eng, r["idx"].contiguous(), r["dist"].contiguous()), r["profile"].contiguous()


_CPU_CHILD = """
import sys, time, warnings, numpy as np, scipy.sparse
sys.path.insert(0, sys.argv[2])
from oracle import umap_spectral_oracle as so
z = np.load(sys.argv[1])
g = scipy.sparse.csr_matrix((z["data"], z["indices"], z["indptr"]))
t0 = time.perf_counter()
with warnings.catch_warnings():
    warnings.simplefilter("ignore")
    so.spectral_layout_reference(z["x"], g, int(z["dim"]), np.random.RandomState(42))
print((time.perf_counter() - t0) * 1e3)
"""


def cpu_arm(path, cap_s):
    env = dict(os.environ, OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1")
    try:
        r = subprocess.run([sys.executable, "-c", _CPU_CHILD, path, ROOT], capture_output=True, text=True, timeout=cap_s,
                           env=env)
    except subprocess.TimeoutExpired:
        return None, "not run: did not end within %d s" % cap_s
    out = r.stdout.strip().splitlines()
    if r.returncode != 0 or not out:
        err = (r.stderr.strip().splitlines() or ["no output"])[-1]
        return None, "not run: failed (exit %d: %s)" % (r.returncode, err[:200])
    return float(out[-1]), "run"


def measure(eng, g, prof, repeats):
    stages = ("spectral_components", "spectral_eigensolve", "spectral_meta")
    spectral_build(eng, g, DIM, N_EPOCHS, data=prof)                   # warm-up
    eng.enable_timing(True)
    times = {s: [] for s in stages}
    res = None
    for _ in range(repeats):
        for s in stages:
            eng.stage_ms(s)                                           # reset
        res = spectral_build(eng, g, DIM, N_EPOCHS, data=prof)
        torch.cuda.synchronize()
        for s in stages:
            ms, cnt = eng.stage_ms(s)
            times[s].append(ms * cnt)
    eng.enable_timing(False)
    med = statistics.median
    st = res["stats"]
    return res, {"n_comp": res["n_comp"], "solved": int((res["status"] == SOLVED).sum()),
                 "largest": int(res["size"].max()), "components_ms": med(times["spectral_components"]),
                 "eigensolve_ms": med(times["spectral_eigensolve"]), "meta_ms": med(times["spectral_meta"]),
                 "lanczos_steps": int(st[0]), "restarts": int(st[1]), "meta_steps": int(st[2]),
                 "meta_restarts": int(st[3]), "component_rounds": int(st[4])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--inputs", default="S1:50000:2,S1:50000:5,S1:50000:15,S2:200000:15")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--cpu-cap", type=int, default=600)
    ap.add_argument("--no-cpu", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark measures the device: it needs a GPU"
    eng = Engine(0)
    rows = []
    with tempfile.TemporaryDirectory() as tmp:
        for spec in args.inputs.split(","):
            kind, n, k = spec.split(":")
            n, k = int(n), int(k)
            g, prof = k7_graph(eng, kind, n, k)
            _, row = measure(eng, g, prof, args.repeats)
            row.update(input="%s %d" % (kind, n), n_neighbors=k, dim=DIM, n_epochs=N_EPOCHS)
            csr = so.prune(scipy.sparse.csr_matrix(
                (g["data"].cpu().numpy(), g["indices"].cpu().numpy(), g["indptr"].cpu().numpy())), N_EPOCHS)
            x32 = prof.cpu().numpy().astype(np.float32)
            hh = []
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                for _ in range(args.repeats):
                    t0 = time.perf_counter()
                    spectral_layout(x32, csr, DIM, np.random.RandomState(42), engine=eng)
                    hh.append((time.perf_counter() - t0) * 1e3)
            row["host_to_host_ms"] = statistics.median(hh)
            if args.no_cpu:
                row["cpu_arm_ms"], row["cpu_arm"] = None, "not run: --no-cpu"
            else:
                path = os.path.join(tmp, "in.npz")
                np.savez(path, data=csr.data, indices=csr.indices, indptr=csr.indptr, x=x32, dim=DIM)
                row["cpu_arm_ms"], row["cpu_arm"] = cpu_arm(path, args.cpu_cap)
            print(json.dumps(row), file=sys.stderr, flush=True)
            rows.append(row)
    print(json.dumps({"bench": "umap_spectral", "card": gpu_card(), "repeats": args.repeats, "results": rows}))


if __name__ == "__main__":
    main()
