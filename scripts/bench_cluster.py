"""KmerClustering.run on the device route, host to host: the GPU pass, then UMAP and HDBSCAN from the pass's own lists.

Inputs: synthetic assemblies as the OrderedDict karma hands to KmerClustering (S1 50 k and S2 200 k by default), at
karma's defaults (-k 5p6, n_neighbors 2, 10 components, min_dist 0, random_state 42, min_cluster_size 2).  Per input,
after one warm-up run, --repeats runs each into a fresh output directory:
  wall_ms                       KmerClustering(..., cluster_on="device").run(...), host to host (median, min, max)
  stage_ms                      medians of the per-stage host clocks of run(), each ended by a device synchronise:
                                pass (profile + kNN + k-list copy), graph (K7), spectral (K10), layout (K8),
                                hdbscan_mst (K9 device tree + edge copy), hdbscan_tree (K9 host labelling), files
  spectral                      K10's components and Lanczos statistics
  profile_bytes_not_downloaded  N * D' * 8: the float64 profile the host route copies back for umap and this route
                                does not
  cpu_arm                       not measured: umap-learn and hdbscan are not installed where this runs
A refusal (e.g. more components than K10's meta-embedding serves) is reported in ``refused`` instead of the times.
    python scripts/bench_cluster.py [--inputs S1:50000,S2:200000] [--repeats 3] [--out FILE]
Prints one JSON line per input, with the card's name and power limit read by nvidia-smi in the same run; --out
appends the lines to FILE too.
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

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from karma_b200 import _lib, synth  # noqa: E402
from karma_b200.engine import Engine  # noqa: E402
from karma_b200.kmer import KmerClustering  # noqa: E402

DEFAULTS = dict(neighbors=2, components=10, dist=0, r_state=42, min_cluster_size=2)


def gpu_card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def one_run(eng, seqs, tmp, i):
    out_dir = os.path.join(tmp, "run%d" % i)
    os.makedirs(out_dir)
    k = KmerClustering(seqs, out_dir, "5p6", 1, cluster_on="device")
    k._engine = eng
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")              # umap's meta-embedding notice
        k.run(**DEFAULTS)
    return (time.perf_counter() - t0) * 1e3, k


def measure(eng, kind, n, repeats):
    seqs = synth.make(kind, n).as_dict()
    row = {"input": "%s %d" % (kind, n), "kmer_size": "5p6", **DEFAULTS, "repeats": repeats,
           "cpu_arm": "not measured: umap-learn and hdbscan are not installed"}
    with tempfile.TemporaryDirectory() as tmp:
        try:
            one_run(eng, seqs, tmp, 0)                                   # warm-up
        except _lib.KarmaB200Error as e:
            row["refused"] = str(e)
            return row
        walls, stages, k = [], {}, None
        for i in range(repeats):
            ms, k = one_run(eng, seqs, tmp, i + 1)
            walls.append(ms)
            for s, v in k.stage_ms.items():
                stages.setdefault(s, []).append(v)
    med = statistics.median
    row.update(wall_ms=med(walls), wall_min_ms=min(walls), wall_max_ms=max(walls),
               stage_ms={s: med(v) for s, v in stages.items()},
               stage_max_ms={s: max(v) for s, v in stages.items()},
               spectral=k.spectral_stats, n_clusters=len(k.clusters), noise=len(k.unlabeled_cluster[0]),
               columns=len(k.kmers), profile_bytes_not_downloaded=n * len(k.kmers) * 8)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--inputs", default="S1:50000,S2:200000")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark measures the device: it needs a GPU"
    eng = Engine(0)
    card = gpu_card()
    for spec in args.inputs.split(","):
        kind, n = spec.split(":")
        row = measure(eng, kind, int(n), args.repeats)
        row = {"bench": "cluster", "card": card, **row}
        line = json.dumps(row)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
