"""K11, MCL of many groups in one call: the read graph of 200 k synthetic contigs (the bench_readgraph.py input), grouped
like the device route's k-mer clusters (runs of 2-10 contigs) plus one unlabeled-sized group of 12 000 contigs.

    python scripts/bench_mcl.py [--contigs 200000] [--classes 4000000] [--unlabeled 12000] [--repeats 3]
Prints one JSON line: device ms of the set-up and of the iterations (stage timers), ms per iteration, iterations per
group, host-to-host ms of the array-level call, the overlap count, and the numba twin of the oracle on one CPU thread
over the same groups.  A real mcl binary is timed only when one is on PATH.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from karma_b200 import mcl as km  # noqa: E402
from karma_b200 import read_graph as rg  # noqa: E402
from karma_b200.engine import Engine  # noqa: E402
from oracle import mcl_oracle as mo  # noqa: E402
from oracle import readgraph_oracle as ro  # noqa: E402


def groups_of(n, unlabeled, seed):
    rng = np.random.default_rng(seed)
    group = np.full(n, -1, np.int32)
    group[:unlabeled] = 0
    g, i = 1, unlabeled
    while i < n:
        k = int(rng.integers(2, 11))
        group[i:i + k] = g
        g += 1
        i += k
    return group, g


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        return out
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs", type=int, default=200000)
    ap.add_argument("--classes", type=int, default=4000000)
    ap.add_argument("--unlabeled", type=int, default=12000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    a = ap.parse_args()
    names, classes = ro.synth_eq_classes(a.contigs, a.classes, seed=11, family=6, max_size=8)
    path = os.path.join(tempfile.mkdtemp(), "eq_classes.txt")
    ro.write_eq_file(path, names, classes)
    eng = Engine(0)
    _, ea, eb, w = rg.build_edges(eng, rg.parse(path))
    group, n_groups = groups_of(a.contigs, a.unlabeled, 5)
    dev = eng.device
    d = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (ea.astype(np.int32), eb.astype(np.int32), w, group)]
    eng.enable_timing(True)
    res = km.mcl_arrays(eng, a.contigs, *d, n_groups)                       # warm-up
    eng.stage_ms("mcl_setup"), eng.stage_ms("mcl_iteration")
    wall, setup, iteration = [], [], []
    for _ in range(a.repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = km.mcl_arrays(eng, a.contigs, *d, n_groups)
        wall.append((time.perf_counter() - t0) * 1e3)
        ms, n = eng.stage_ms("mcl_setup")
        setup.append(ms * n)
        ms, n_it = eng.stage_ms("mcl_iteration")
        iteration.append(ms * n_it)
    it = res["iterations"]
    out = {"metric": "MCL of every group of a read graph in one device call (K11)", "card": card(),
           "contigs": a.contigs, "classes": a.classes, "edges": int(len(ea)), "groups": int(n_groups),
           "stream_nodes": int((res["local"] >= 0).sum()), "unlabeled_group_nodes": int((res["local"][:a.unlabeled] >= 0).sum()),
           "clusters": int(res["n_clusters"].sum()), "overlap_nodes": int(res["overlap"].sum()),
           "groups_with_overlap": int((res["overlap"] > 0).sum()),
           "iterations_max": int(it.max()), "iterations_median": float(np.median(it[it > 0])),
           "iterations_unlabeled_group": int(it[0]),
           "device_ms_setup": float(np.median(setup)), "device_ms_iterations": float(np.median(iteration)),
           "device_ms_per_iteration": float(np.median(iteration)) / int(it.max()),
           "host_to_host_ms": float(np.median(wall)), "host_to_host_ms_min": float(np.min(wall)),
           "repeats": a.repeats}
    if not a.no_cpu:
        seg = mo.segment(a.contigs, ea, eb, w, group, n_groups)
        mo.mcl_union(mo.segment(2, [0], [1], [1.0], np.zeros(2, np.int32), 1), None, None, None, None)   # compile
        csc = mo.union_csc(seg, ea, eb, w, group)
        t0 = time.perf_counter()
        twin = mo._NB["union"](*csc, seg["col_group"], seg["off"], n_groups, 2.0, mo.MAX_ITER)
        out["cpu_numba_twin_ms_one_thread"] = (time.perf_counter() - t0) * 1e3
        out["cpu_twin_iterations_equal"] = bool(np.array_equal(twin[3], it))
    out["mcl_binary"] = "not measured (no mcl on PATH)" if shutil.which("mcl") is None else shutil.which("mcl")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
