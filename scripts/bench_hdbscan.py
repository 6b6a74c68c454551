"""HDBSCAN (K9): the device MST and the host tree stage against scikit-learn's HDBSCAN on the CPU.

Inputs (10 dims, float32): the K8 embedding of a 50 k S1 pass (device_pass -> K7 -> K8, 200 epochs, random init,
seed 42) and synthetic blobs of 200 k and 1 M points (oracle/umap_layout_oracle.blobs, 30 blobs).  Each input runs at
min_cluster_size m = 2 (karma's default) and 15, hdbscan's min_samples defaulting to m, so core_k = m + 1.  Per
input and m:
  core_ms, mst_ms, sort_ms   device time of the three stages (the library's CUDA-event stage timers), after one
                             warm-up call at the start, median of --repeats; mst_ms sums the Boruvka rounds,
                             ``rounds`` is their number
  tree_ms                    host time of kb_hdbscan_labels (single linkage .. probabilities), median of --repeats
  host_to_host_ms            HDBSCAN(min_cluster_size=m).fit(numpy float32) -> labels_, probabilities_; median of
                             --repeats below 1 M points, one run at 1 M and above (each run is a full MST)
  pair_evals                 N^2 x (1 + rounds): the core sweep and every round visit all ordered pairs (i, j)
  pair_evals_per_s           pair_evals / (core_ms + mst_ms)
  cpu_arm_ms                 sklearn.cluster.HDBSCAN(min_cluster_size=m, min_samples=m + 1, algorithm="kd_tree").fit
                             on the same points, one run, in a child process stopped after --cpu-cap seconds
                             (null and ``cpu_arm`` = "not run: ..." when it does not end in time, fails or is not
                             attempted).  The child is single-threaded and runs on its own core, in a thread of its
                             own, while the device arm is measured; the two arms share no work.
    python scripts/bench_hdbscan.py [--sizes 200000,1000000] [--real 50000] [--repeats 3] [--cpu-sizes 50000,200000]
Prints one JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from karma_b200.engine import Engine  # noqa: E402
from karma_b200.hdbscan_ import HDBSCAN, mutual_reachability_mst, tree_labels  # noqa: E402
from oracle import umap_layout_oracle as lo  # noqa: E402

DIM = 10


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def s1_embedding(eng, n):
    from karma_b200 import synth
    from karma_b200.engine import device_pass
    from karma_b200.umap_graph import build_graph
    from karma_b200.umap_layout import find_ab_params, layout_graph
    asm = synth.make("S1", n)
    d_bases, d_offsets, d_key_len = eng.upload(asm.bases, asm.offsets, asm.key_len)
    r = device_pass(eng, d_bases, d_offsets, d_key_len, n, "5p6", n_neighbors=15, want_profile=False)
    g = build_graph(eng, r["idx"].contiguous(), r["dist"].contiguous())
    a, b = find_ab_params(1.0, 0.1)
    init = torch.rand(n, DIM, device=eng.device, generator=torch.Generator(eng.device).manual_seed(42)) * 20 - 10
    return layout_graph(eng, g, init, 200, a, b, 42).cpu().numpy()


_CPU_CHILD = """
import sys, time, numpy as np
from sklearn.cluster import HDBSCAN
x = np.load(sys.argv[1]); m = int(sys.argv[2])
t0 = time.perf_counter()
HDBSCAN(min_cluster_size=m, min_samples=m + 1, algorithm="kd_tree").fit(x.astype(np.float64))
print((time.perf_counter() - t0) * 1e3)
"""


def cpu_arm(path, m, cap_s):
    try:
        r = subprocess.run([sys.executable, "-c", _CPU_CHILD, path, str(m)], capture_output=True, text=True, timeout=cap_s)
    except subprocess.TimeoutExpired:
        return None, "not run: did not end within %d s" % cap_s
    out = r.stdout.strip().splitlines()
    if r.returncode != 0 or not out:
        err = (r.stderr.strip().splitlines() or ["no output"])[-1]
        return None, "not run: failed (exit %d: %s)" % (r.returncode, err[:200])
    return float(out[-1]), "run"


def cpu_arms(jobs, cap_s, results):
    """Run the CPU arm's jobs (key, points file, m) one after another; results[key] = (ms or None, status)."""
    for key, path, m in jobs:
        results[key] = cpu_arm(path, m, cap_s)


def stage_total(eng, stage):
    ms, n = eng.stage_ms(stage)
    return ms * n, n


def measure(eng, x, m, repeats):
    n = x.shape[0]
    core_k = m + 1
    dx = torch.from_numpy(x).to(eng.device)
    eng.enable_timing(True)
    core, mst, srt, tree, rounds = [], [], [], [], 0
    for _ in range(repeats):
        for s in ("hdbscan_core", "hdbscan_mst", "hdbscan_sort"):
            eng.stage_ms(s)                                           # reset
        r = mutual_reachability_mst(eng, dx, core_k)
        torch.cuda.synchronize()
        core.append(stage_total(eng, "hdbscan_core")[0])
        ms, rounds = stage_total(eng, "hdbscan_mst")
        mst.append(ms)
        srt.append(stage_total(eng, "hdbscan_sort")[0])
        edges, weights = r["edges"].cpu().numpy(), r["weights"].cpu().numpy()
        t0 = time.perf_counter()
        labels, probs, n_clusters = tree_labels(edges, weights, m)
        tree.append((time.perf_counter() - t0) * 1e3)
    eng.enable_timing(False)
    hh = []
    for _ in range(repeats if n < 1000000 else 1):
        t0 = time.perf_counter()
        c = HDBSCAN(min_cluster_size=m, engine=eng).fit(x)
        hh.append((time.perf_counter() - t0) * 1e3)
    assert np.array_equal(c.labels_, labels)
    pairs = float(n) * float(n) * (1 + rounds)
    med = statistics.median
    return {"rows": n, "min_cluster_size": m, "core_k": core_k, "core_ms": med(core), "mst_ms": med(mst), "rounds": rounds,
            "sort_ms": med(srt), "tree_ms": med(tree), "host_to_host_ms": med(hh), "pair_evals": pairs,
            "pair_evals_per_s": pairs / ((med(core) + med(mst)) * 1e-3), "n_clusters": int(n_clusters),
            "noise": int((labels == -1).sum()), "mean_probability": float(np.mean(probs))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="200000,1000000")
    ap.add_argument("--real", type=int, default=50000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--cpu-sizes", default="50000,200000")
    ap.add_argument("--cpu-cap", type=int, default=300)
    args = ap.parse_args()
    import tempfile
    eng = Engine(0)
    card = gpu_card()
    cpu_sizes = {int(s) for s in args.cpu_sizes.split(",") if s}
    inputs = []
    if args.real:
        inputs.append(("K8 embedding of S1 %d contigs (-k 5p6, k = 15, 200 epochs, seed 42)" % args.real,
                       s1_embedding(eng, args.real)))
    for n in [int(s) for s in args.sizes.split(",") if s]:
        inputs.append(("blobs %d x %d (30 blobs, seed 5)" % (n, DIM), lo.blobs(n, 30, DIM, seed=5)[0].astype(np.float32)))
    results = []
    with tempfile.TemporaryDirectory() as tmp:
        jobs = []
        for k, (name, x) in enumerate(inputs):
            if x.shape[0] in cpu_sizes:
                path = os.path.join(tmp, "points%d.npy" % k)
                np.save(path, x)
                jobs += [((k, m), path, m) for m in (2, 15)]
        cpu = {}
        worker = threading.Thread(target=cpu_arms, args=(jobs, args.cpu_cap, cpu))
        worker.start()
        mutual_reachability_mst(eng, torch.from_numpy(inputs[0][1][:4096]).to(eng.device), 3)       # warm-up
        torch.cuda.synchronize()
        for k, (name, x) in enumerate(inputs):
            for m in (2, 15):
                r = measure(eng, x, m, args.repeats)
                r["input"] = name
                results.append(((k, m), r))
                print(json.dumps(r), file=sys.stderr)
        worker.join()
    for key, r in results:
        r["cpu_arm_ms"], r["cpu_arm"] = cpu.get(key, (None, "not run: above the sizes attempted"))
    results = [r for _, r in results]
    print(json.dumps({"metric": "HDBSCAN (K9): mutual-reachability MST on the device, tree on the host, dim %d" % DIM,
                      "gpu": card, "cpu_count": os.cpu_count(), "cpu_arm_threads": 1, "cpu_cap_s": args.cpu_cap,
                      "results": results}))


if __name__ == "__main__":
    main()
