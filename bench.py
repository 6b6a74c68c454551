#!/usr/bin/env python
"""Benchmark of the karma k-mer front end (profile matrix + exact kNN graph).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Metric (BASELINE.json): contigs/s for (profile + kNN).  Workload at every N is
BASELINE.json configs[1]: a 50 000-contig synthetic Trinity-like assembly (S1 gene
families, log-normal lengths), kmer.py's default -k 5p6 (1088 columns),
n_neighbors=2.  N>1 is strong scaling: the same 50k contigs, rows sharded for
counting, query rows sharded for the kNN, key shards exchanged over NVLink peer memory.

A step = one pass of the hot path over the whole assembly.
  value : T0 -- inputs already resident in HBM, one enqueue per step (the pre-planned pass of
          karma_b200.engine.PassPlan, a CUDA graph), CUDA-event time, max over ranks.  Step i is
          validated on the host while step i+1 runs.
  e2e   : T1 -- host (pinned) buffers in, host results out through the public API
          (karma_b200.engine.PassPlan.bind_host / run_host): chunked H2D, kernels, exchange, D2H of the float64
          profile rows, the kNN lists and the validation words of this rank, waited for and validated every
          step, all inside the timed region (wall clock between barriers, max over ranks).  e2e.single_shot
          (N=1) is the unplanned call karma_b200.engine.profile_and_knn that KmerClustering makes once per run.
  t2    : T2 -- from the Python dict karma.py builds (marshalling included), N=1 only
Per-kernel times (stage_ms, roofline) come from a separate eager pass with the library's event pairs on,
after the timed region.  Supplementary blocks (outside every timed region): the k=15 kernel rate, the
counting kernel on the 5120-column shape, a parity sample against the fp64 oracle at N>1, and at N=8 the
500k (BASELINE configs[2]) and 1M-contig (north_star target) runs.
One JSON line is printed by rank 0.

--dump-outputs DIR writes what the T0 pass left on the device after its last timed step (dump_outputs below):
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "contigs/sec (profile+kNN)"
UNIT = "contigs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--contigs", type=int, default=50000)
    ap.add_argument("--synth", default="S1")
    ap.add_argument("--kmer", default="5p6")
    ap.add_argument("--neighbors", type=int, default=2)
    ap.add_argument("--knn-impl", default="tc", choices=["tc", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the supplementary blocks")
    ap.add_argument("--no-graph", action="store_true", help="enqueue the pass eagerly instead of replaying a CUDA graph")
    ap.add_argument("--shard-gen", action="store_true", help="each rank synthesises only its own row shard")
    ap.add_argument("--big", default=None, help="comma list of contig counts for the sharded 5+6 / k=15 runs (default at N=8: 500000,1000000; 0: none)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (a seeded row sample, at most 64 MB)")
    return ap.parse_args()


def kmer_arg(s):
    return int(s) if s.isdigit() else s


def workload_name(a):
    return "%d-contig synthetic Trinity-like assembly (%s), -k %s, n_neighbors=%d" % (
        a.contigs, a.synth, a.kmer, a.neighbors)


def ncu_traffic(kernel_regex):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the newest
    committed `ncu --set full` summary of this bench command at N=1 (profiles/): None if absent."""
    import glob
    import re
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*", "ncu_k4_*summary.csv"))):
        rd = wr = None
        for line in open(path):
            parts = line.rstrip("\n").split(",")
            if parts[0] == "dram__bytes_read.sum":
                rd = (float(parts[-1]), parts[-2])
            if parts[0] == "dram__bytes_write.sum":
                wr = (float(parts[-1]), parts[-2])
        if rd and wr:
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            best = {"bytes": rd[0] * scale.get(rd[1], 1.0) + wr[0] * scale.get(wr[1], 1.0), "source": os.path.relpath(path, ROOT)}
    return best


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d["bf16_tflops"], "tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for nme, v in zip(names, r[4:8]):
                if v.strip().lower() == "active":
                    reasons.add(nme)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------ CPU arm (oracle port)
def _port_chunk(args):
    """Worker: kmer.py's counting loops (oracle port) on a chunk of the sample."""
    from oracle import kmer_oracle
    keys, seqs, kmer_size = args
    counters = [kmer_oracle._contig_counter(s, kmer_size) for s in seqs]
    return counters


def cpu_profile_rate(asm, kmer_size, n_sample, procs):
    """contigs/s of the kmer.py algorithm (oracle port) on the first n_sample contigs,
    counting loops spread over `procs` processes (more than kmer.py itself does:
    its counting is single-threaded, kmer.py:56-92)."""
    from multiprocessing import get_context
    sub = asm.slice(0, n_sample)
    d = sub.as_dict()
    keys, seqs = list(d.keys()), list(d.values())
    t0 = time.perf_counter()
    if procs > 1:
        step = -(-len(seqs) // procs)
        chunks = [(keys[i:i + step], seqs[i:i + step], kmer_size) for i in range(0, len(seqs), step)]
        with get_context("fork").Pool(procs) as pool:
            parts = pool.map(_port_chunk, chunks)
        counters = [c for p in parts for c in p]
    else:
        counters = _port_chunk((keys, seqs, kmer_size))
    kset = set()
    for c in counters:
        kset.update(c.keys())
    cols = sorted(kset)
    col = {k: i for i, k in enumerate(cols)}
    out = np.zeros((len(seqs), len(cols)), dtype=np.float64)
    for r, (key, c) in enumerate(zip(keys, counters)):
        ln = len(key)
        for kmer, cnt in c.items():
            out[r, col[kmer]] = cnt / ln
    dt = time.perf_counter() - t0
    return n_sample / dt, dt


def cpu_knn_rate(profile32, k, n_query):
    """queries/s of an exact CPU neighbour search (what UMAP does below 4096 points:
    full pairwise distances + partial sort), fp32 as UMAP casts, BLAS on all threads,
    for the first n_query rows against ALL keys."""
    t0 = time.perf_counter()
    q = profile32[:n_query]
    sq = np.einsum("ij,ij->i", profile32, profile32)
    d2 = sq[:n_query, None] + sq[None, :] - 2.0 * (q @ profile32.T)
    idx = np.argpartition(d2, k, axis=1)[:, :k]
    dd = np.take_along_axis(d2, idx, 1)
    order = np.argsort(dd, axis=1)
    idx = np.take_along_axis(idx, order, 1)
    dt = time.perf_counter() - t0
    return n_query / dt, dt, idx


def blas_threads(n):
    """Pin the BLAS/OpenMP pools to n threads at run time: torchrun exports OMP_NUM_THREADS=1 to its workers,
    which would silently run the reference arm's neighbour search on one core."""
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=n)
        got = [p.get("num_threads") for p in threadpool_info() if p.get("user_api") in ("blas", "openmp")]
        return max(got) if got else 1
    except Exception:
        return int(os.environ.get("OMP_NUM_THREADS", "1") or 1)


def cpu_arm(a, asm, steps, warmup):
    """contigs/s of the CPU path, extrapolated from a bounded sample of the same
    workload: profile is linear in contigs, exact kNN linear in query rows."""
    from oracle import kmer_oracle
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    threads = blas_threads(cores)
    kmer_size = kmer_arg(a.kmer)
    n_sample = min(asm.n, 1500)
    n_query = min(asm.n, 1024)
    # keys for the neighbour search: the full profile from the vectorised oracle (untimed)
    counts, _ = kmer_oracle.counts_mode(asm.bases, asm.offsets, kmer_size)
    prof32 = (counts / asm.key_len[:, None].astype(np.float64)).astype(np.float32)
    del counts
    vals, times = [], []
    for it in range(warmup + steps):
        rp, tp = cpu_profile_rate(asm, kmer_size, n_sample, cores)
        rk, tk, _ = cpu_knn_rate(prof32, a.neighbors, n_query)
        v = 1.0 / (1.0 / rp + 1.0 / rk)
        if it >= warmup:
            vals.append(v); times.append(tp + tk)
    value = statistics.mean(vals)
    sample = ("per step: oracle port of kmer.py (pure-Python counting loops over %d processes) on %d contigs + exact "
              "fp32 brute-force kNN (numpy/BLAS, %d threads) of %d query rows vs all %d keys; contigs/s = "
              "1/(1/profile_rate + 1/knn_rate); umap-learn/NN-descent not installed" %
              (cores, n_sample, threads, n_query, asm.n))
    return value, cores, sample, statistics.mean(times) * 1e3


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from karma_b200 import synth
    asm = synth.make(a.synth, a.contigs)
    steps = max(1, min(a.steps, 3))
    warm = min(a.warmup, 1)
    value, cores, sample, ms = cpu_arm(a, asm, steps, warm)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "python int / f64 (profile), f32 (kNN)", "data": "synthetic",
            "config": {"workload": workload_name(a)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------ parity sample (oracle as the checker)
def truth_from_counts(c_rows, l_rows, sq_rows, counts_all, l_all):
    """fp64 squared distances of sampled rows to all rows from INTEGER counts: the Gram entries and squared norms
    are integers below 2^53 (exact in fp64), so the only roundings are the final products and the division."""
    c_rows = np.asarray(c_rows, dtype=np.float64)
    n = counts_all.shape[0]
    sq = np.empty(n)
    gram = np.empty((c_rows.shape[0], n))
    for lo in range(0, n, 16384):
        blk = np.asarray(counts_all[lo:lo + 16384], dtype=np.float64)
        sq[lo:lo + 16384] = np.einsum("ij,ij->i", blk, blk)
        gram[:, lo:lo + 16384] = c_rows @ blk.T
    l_all = np.asarray(l_all, dtype=np.float64)
    l_rows = np.asarray(l_rows, dtype=np.float64)
    num = np.asarray(sq_rows)[:, None] * (l_all[None, :] ** 2) + sq[None, :] * (l_rows[:, None] ** 2) - 2.0 * gram * np.outer(l_rows, l_all)
    return num / np.outer(l_rows, l_all) ** 2


def parity_sample_small(asm, kmer_size, idx_all, dist_all, n_rows=256):
    """Rows of the gathered k-lists against the fp64 oracle (stated-ties rule, SURVEY 8c)."""
    from oracle import kmer_oracle, knn_oracle
    counts, _ = kmer_oracle.counts_mode(asm.bases, asm.offsets, kmer_size)
    rows = np.unique(np.linspace(0, asm.n - 1, n_rows).astype(np.int64))
    c = counts[rows].astype(np.float64)
    truth = truth_from_counts(c, asm.key_len[rows], np.einsum("ij,ij->i", c, c), counts, asm.key_len)
    rep = knn_oracle.check_knn(idx_all[rows], dist_all[rows], truth, rows=rows)
    rep["ok"] = bool(knn_oracle.parity_ok(rep))
    rep["checked_against"] = "fp64 distances from the oracle's integer counts (oracle/kmer_oracle.py), tie rule 1e-5"
    return rep


# ------------------------------------------------------------------ GPU arm
def timed_plan_loop(torch, dist, plan, steps, world):
    """K passes of a plan, each validated on the host while the next one runs.  Returns (ms total, checks)."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    checks = []
    ev0.record()
    prev = None
    for _ in range(steps):
        tok = plan.run()
        if prev is not None:
            checks.append(plan.check(prev))
        prev = tok
    ev1.record()
    checks.append(plan.check(prev))
    barrier()
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), checks


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, torch, dist, plan, n_total, lo, rank, world):
    """Write what a caller of PassPlan.run receives after the last pass: profile.npy (float64 profile rows),
    knn_idx.npy (neighbour indices, int32 held exactly in float64) and knn_dist.npy (float32 distances).  When all
    rows exceed DUMP_BYTES, a row sample drawn with a fixed seed is written; rows.npy holds the row numbers.  At N>1
    every rank contributes its profile rows; rank 0 writes."""
    per_row = plan.cols * 8 + plan.k * (8 + 4) + 8
    m = min(n_total, (DUMP_BYTES - 4096) // per_row)          # 4096: room for the four .npy headers
    rows = np.arange(n_total) if m == n_total else np.sort(np.random.default_rng(0).choice(n_total, m, replace=False))
    mine = rows[(rows >= lo) & (rows < lo + plan.n)] - lo
    prof = plan.profile[torch.from_numpy(mine).to(plan.profile.device)].cpu().numpy()
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, prof)
        prof = np.concatenate(parts)
    if rank != 0:
        return
    sel = torch.from_numpy(rows).to(plan.all_idx.device)       # gathered lists: row r of the assembly is row r here
    arrays = {"rows": rows.astype(np.float64), "profile": prof,
              "knn_idx": plan.all_idx[sel].cpu().numpy().astype(np.float64), "knn_dist": plan.all_dist[sel].cpu().numpy()}
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def big_run(torch, dist, eng, a, n_total, rank, world, local, pk):
    """One sharded run of the north-star shape (5120 dense columns, n_neighbors = 15): every rank synthesises its
    own row shard.  Device-resident steps, one host-to-host step, and a parity sample of rank 0's rows against
    distances computed on the CPU from the gathered integer counts."""
    from karma_b200 import _lib, synth
    from karma_b200.engine import PassPlan, shard_bounds
    lo, hi, per = shard_bounds(n_total, world, rank)
    t0 = time.perf_counter()
    kind = "S2" if n_total >= 2000000 else "S1"            # BASELINE configs[3] is the redundant multi-assembler merge
    shard = synth.make(kind, hi - lo, seed=4321 + rank)
    gen_s = time.perf_counter() - t0
    k, kmer = 15, "5+6"
    h_bases = torch.from_numpy(shard.bases.copy()).pin_memory()
    h_off = torch.from_numpy(shard.offsets.copy()).pin_memory()
    h_len = torch.from_numpy(shard.key_len.copy()).pin_memory()
    plan = PassPlan(eng, shard.n, int(shard.offsets[-1]), kmer, n_neighbors=k, impl=_lib.KB_KNN_TC, want_profile=True,
                    group=dist.group.WORLD if world > 1 else None, rank=rank, world=world, n_total=n_total, graph=False)
    def note(msg):
        if rank == 0:
            print("[bench big %d] %s" % (n_total, msg), file=sys.stderr, flush=True)
    try:
        note("plan ready (synth %.1f s)" % gen_s)
        plan.load(h_bases, h_off, h_len)
        eng.enable_timing(True)
        tok = plan.run()                                        # warm-up (uploads the piece table)
        first = plan.check(tok)
        note("first pass done: %r" % (first,))
        for st in ("count", "normalise", "knn_gemm", "rerank"):
            eng.stage_ms(st)
        ms, checks = timed_plan_loop(torch, dist, plan, 2, world)
        gemm_ms, _ = eng.stage_ms("knn_gemm")
        count_ms, _ = eng.stage_ms("count")
        norm_ms, _ = eng.stage_ms("normalise")
        rerank_ms, _ = eng.stage_ms("rerank")
        eng.enable_timing(False)
        note("timed passes done: %.1f ms per pass" % (ms / 2))
        if any(not c["ok"] for c in checks + [first]):
            raise RuntimeError("optimistic validation failed on the synthetic shard: %r" % (checks,))
        # rows K5 could not certify are redone exactly (all ranks take part: the count is the sum over ranks)
        unc = checks[-1]["uncertified"]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fixed = plan.fixup() if unc else 0
        torch.cuda.synchronize()
        fix_s = time.perf_counter() - t0
        # host to host: pinned inputs up, profile shard + this rank's lists down, uncertified rows redone
        h_prof = torch.empty(tuple(plan.profile.shape), dtype=torch.float64).pin_memory()
        h_idx = torch.empty(tuple(plan.idx.shape), dtype=torch.int32).pin_memory()
        h_dst = torch.empty(tuple(plan.dist.shape), dtype=torch.float32).pin_memory()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        plan.load(h_bases, h_off, h_len)
        tok = plan.run()
        h_prof.copy_(plan.profile, non_blocking=True)
        last = plan.check(tok)
        if last["uncertified"]:
            plan.fixup()
        h_idx.copy_(plan.idx, non_blocking=True)
        h_dst.copy_(plan.dist, non_blocking=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e2e_s = time.perf_counter() - t0
        tt = torch.tensor([e2e_s, fix_s], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s, fix_s = float(tt[0].item()), float(tt[1].item())
        note("host-to-host pass done: %.1f ms (exact redo %.1f ms)" % (e2e_s * 1e3, fix_s * 1e3))
        if not last["ok"]:
            raise RuntimeError("optimistic validation failed on the synthetic shard: %r" % (last,))
        rec = None
        if rank == 0:
            # parity sample: rows of rank 0 against ALL keys, truth from the gathered integer counts
            blas_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
            rows = np.unique(np.linspace(0, shard.n - 1, 128).astype(np.int64))
            meta = plan.rowmeta_all.cpu().numpy()
            real = (meta[:, 3] & 8) == 0
            l_all = meta[:, 2].astype(np.float64)
            sqn = meta[:, 0:2].copy().view(np.float64)[:, 0]
            op_rows = plan.operand_all[torch.from_numpy(rows).to(plan.operand_all.device)].cpu().numpy().astype(np.float64)
            n_keys = meta.shape[0]
            gram = np.empty((len(rows), n_keys))
            for b0 in range(0, n_keys, 32768):
                blk = plan.operand_all[b0:b0 + 32768].cpu().numpy().astype(np.float64)
                gram[:, b0:b0 + 32768] = op_rows @ blk.T
            lr = l_all[rows]
            num = sqn[rows][:, None] * (l_all[None, :] ** 2) + sqn[None, :] * (lr[:, None] ** 2) - 2.0 * gram * np.outer(lr, l_all)
            truth = num / np.outer(lr, l_all) ** 2
            truth[:, ~real] = np.inf
            from oracle import knn_oracle
            rep = knn_oracle.check_knn(plan.idx.cpu().numpy()[rows], plan.dist.cpu().numpy()[rows], truth, rows=rows)
            rep["ok"] = bool(knn_oracle.parity_ok(rep))
            rep["checked_against"] = "fp64 distances computed on the CPU from the gathered fp16 count rows (exact integers), tie rule 1e-5"
            flops = 2.0 * shard.n * float(n_total) * plan.cols
            tf = flops / (gemm_ms / 1e3) / 1e12
            rec = {"workload": "%d-contig %s assembly, -k 5+6 (5120 dense columns), n_neighbors=15, %d GPUs, shards synthesised per rank" % (n_total, kind, world),
                   "ms_per_step": ms / 2 + fix_s * 1e3, "contigs_per_s": n_total / (ms / 2e3 + fix_s), "steps": 2,
                   "pass_ms": ms / 2, "exact_redo_ms": fix_s * 1e3,
                   "e2e_ms_per_step": e2e_s * 1e3, "e2e_contigs_per_s": n_total / e2e_s,
                   "e2e_bytes": {"h2d": int(h_bases.numel() + h_off.numel() * 8 + h_len.numel() * 4),
                                 "d2h": int(h_prof.numel() * 8 + h_idx.numel() * 8)},
                   "stage_ms": {"count": count_ms, "normalise": norm_ms, "knn_gemm": gemm_ms, "rerank": rerank_ms},
                   "k4_tflops_per_gpu": tf, "k4_frac_of_sustained_peak": tf / pk["tflops_sustained"],
                   "uncertified_rows": int(unc), "rows_redone_exactly": int(fixed), "parity_sample": rep, "synth_s": gen_s}
        return rec
    finally:
        plan.close()
        del plan
        torch.cuda.empty_cache()


def run_ours(a):
    import torch
    import torch.distributed as dist
    from karma_b200 import _lib, synth
    from karma_b200.engine import Engine, PassPlan, mode_of, profile_and_knn, shard_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun (the driver launches torchrun itself)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(a.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000)] + sys.argv
        return subprocess.call(cmd)
    torch.cuda.set_device(local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        group = dist.group.WORLD
    eng = Engine(local)
    kmer_size = kmer_arg(a.kmer)
    mode = mode_of(kmer_size)
    impl = _lib.KB_KNN_TC if a.knn_impl == "tc" else _lib.KB_KNN_SIMT
    k = a.neighbors
    pk = peaks()

    n_total = a.contigs
    lo, hi, per = shard_bounds(n_total, world, rank)
    if world > 1 and (a.shard_gen or n_total >= 400000):
        # large assemblies: every rank synthesises only its own rows (seeded per rank)
        shard = synth.make(a.synth, hi - lo, seed=4321 + rank)
        asm = None
        tb = torch.tensor([int(shard.offsets[-1])], dtype=torch.int64, device="cuda")
        dist.all_reduce(tb)
        total_bases_all = int(tb.item())
    else:
        asm = synth.make(a.synth, a.contigs)
        shard = asm.slice(lo, hi) if world > 1 else asm
        total_bases_all = int(asm.offsets[-1])
    n = shard.n
    h_bases = torch.from_numpy(shard.bases.copy()).pin_memory()
    h_offsets = torch.from_numpy(shard.offsets.copy()).pin_memory()
    h_keylen = torch.from_numpy(shard.key_len.copy()).pin_memory()
    cols_full = eng.lib.kb_mode_columns(mode)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- T0: the pre-planned pass on device-resident inputs
    plan = PassPlan(eng, n, int(shard.offsets[-1]), kmer_size, n_neighbors=k, impl=impl, want_profile=True,
                    group=group, rank=rank, world=world, n_total=n_total, graph=not a.no_graph)
    plan.load(h_bases, h_offsets, h_keylen)
    launches0 = eng.launches()
    plan.capture(warmup=2)                                   # 2 eager passes (+1 captured)
    launches_per_step = (eng.launches() - launches0) // (3 if plan.graph is not None else 2)
    for _ in range(a.warmup):
        tok = plan.run()
    warm = plan.check(tok) if a.warmup else {"ok": True, "uncertified": 0}
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, checks = timed_plan_loop(torch, dist, plan, a.steps, world)
    if not all(c["ok"] for c in checks + [warm]):
        raise RuntimeError("optimistic validation failed on the synthetic assembly: %r" % (checks[-1],))
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, torch, dist, plan, n_total, lo, rank, world)
    uncertified = checks[-1]["uncertified"]
    value = n_total * a.steps / (total_ms / 1e3)
    d_cols = plan.cols

    # ---- per-kernel times: a separate eager pass with the library's event pairs on
    eng.enable_timing(True)
    n_stage = max(3, min(a.steps, 10))
    for _ in range(2):
        plan.enqueue()
    torch.cuda.synchronize()
    for st in ("count", "count_long", "normalise", "knn_gemm", "rerank"):
        eng.stage_ms(st)
    barrier()
    for _ in range(n_stage):
        plan.enqueue()
    barrier()
    gemm_ms, gemm_n = eng.stage_ms("knn_gemm")
    count_ms, _ = eng.stage_ms("count")
    long_ms, _ = eng.stage_ms("count_long")
    rerank_ms, _ = eng.stage_ms("rerank")
    norm_ms, _ = eng.stage_ms("normalise")
    eng.enable_timing(False)
    all_idx = plan.all_idx.cpu().numpy() if rank == 0 else None
    all_dist = plan.all_dist.cpu().numpy() if rank == 0 else None

    # ---- e2e: host buffers in, host results out
    e2e = None
    if not a.no_e2e:
        # the planned host-to-host pass: pinned host inputs -> (graph: chunked H2D || K1+K3 || profile D2H || exchange ||
        # K4 -> K5 -> lists D2H) -> float64 profile rows + k-lists of this rank's contigs in pinned host memory
        plan.bind_host(h_bases, h_offsets, h_keylen)
        for _ in range(max(2, min(a.warmup, 3))):
            res = plan.run_host()
        barrier()
        t0 = time.perf_counter()
        oks = []
        for _ in range(a.steps):
            res = plan.run_host()
            oks.append(res["ok"])
        barrier()
        dt = time.perf_counter() - t0
        if not all(oks):
            raise RuntimeError("host-to-host pass: optimistic validation failed: %r" % ({k_: v for k_, v in res.items() if not hasattr(v, "shape")},))
        tt = torch.tensor([dt], dtype=torch.float64, device=eng.device)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        h2d = int(shard.offsets[-1]) + h_offsets.numel() * 8 + h_keylen.numel() * 4
        d2h = res["profile"].nbytes + res["knn_idx"].nbytes + res["knn_dist"].nbytes + plan.host["h_rec"].numel() * 4
        e2e = {"value": n_total * a.steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": dt / a.steps * 1e3,
               "api": "PassPlan.bind_host + run_host (one graph replay per pass, results waited for and validated on the host)"}
        # the same e2e pass must return what the device-resident pass left on the GPU
        same = bool((torch.from_numpy(res["knn_idx"]).to(eng.device) == plan.idx).all().item()) and \
            bool((torch.from_numpy(res["profile"][:: max(1, n // 64)]).to(eng.device) == plan.profile[:: max(1, n // 64)]).all().item())
        e2e["equals_device_pass"] = same
        if world == 1:
            # the single-shot public call (what KmerClustering makes): eager, no plan, fresh device buffers
            for _ in range(2):
                r1 = profile_and_knn(eng, h_bases, h_offsets, h_keylen, kmer_size, n_neighbors=k, impl=impl, reuse_host=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ns = max(3, min(a.steps, 10))
            for _ in range(ns):
                r1 = profile_and_knn(eng, h_bases, h_offsets, h_keylen, kmer_size, n_neighbors=k, impl=impl, reuse_host=True)
            torch.cuda.synchronize()
            e2e["single_shot"] = {"ms_per_step": (time.perf_counter() - t0) / ns * 1e3, "api": "engine.profile_and_knn (eager, unplanned)"}
            del r1
    clocks = sampler.stop() if rank == 0 else None

    # ---- supplementary blocks (outside every timed region)
    extras = {}
    if not a.no_extras:
        try:
            if world == 1:
                # T2: from the Python dict karma.py builds (kmer.py's own input type), marshalling included
                from karma_b200.kmer import KmerClustering
                seqs = asm.as_dict()
                kc = KmerClustering(seqs, tempfile.gettempdir(), kmer_size, 1)
                kc._engine = eng
                t2 = []
                for it in range(3):
                    t0 = time.perf_counter()
                    kc._KmerClustering__calc_kmer_profile(n_neighbors=k)
                    t2.append(time.perf_counter() - t0)
                extras["t2"] = {"ms_per_step": min(t2[1:]) * 1e3, "value": n_total / min(t2[1:]), "unit": UNIT,
                                "what": "KmerClustering.__calc_kmer_profile(n_neighbors) from the Python dict: join/encode marshalling + T1"}
                # the same kernels with UMAP's default n_neighbors = 15
                p15 = PassPlan(eng, n, int(shard.offsets[-1]), kmer_size, n_neighbors=15, impl=impl, want_profile=False, graph=False)
                p15.load(h_bases, h_offsets, h_keylen)
                eng.enable_timing(True)
                for _ in range(2):
                    p15.enqueue()
                torch.cuda.synchronize(); eng.stage_ms("knn_gemm"); eng.stage_ms("rerank")
                for _ in range(5):
                    p15.enqueue()
                torch.cuda.synchronize()
                g15, _ = eng.stage_ms("knn_gemm"); r15, _ = eng.stage_ms("rerank")
                eng.enable_timing(False)
                tf15 = 2.0 * n * n * d_cols / (g15 / 1e3) / 1e12
                extras["neighbors15"] = {"knn_gemm_ms": g15, "rerank_ms": r15, "tflops": tf15, "frac_of_burst_peak": tf15 / pk["tflops"],
                                         "columns": d_cols, "ok": p15.check(p15.run())["ok"]}
                del p15
                # the counting kernel on north_star's dense 5120-column shape
                if mode != _lib.KB_MODE_DENSE_5_6:
                    eng.enable_timing(True)
                    eng.stage_ms("count")
                    cnt5120 = torch.empty((n, 5120), dtype=torch.int32, device=eng.device)
                    for _ in range(5):
                        eng.count(plan.d_bases, plan.d_offsets, n, _lib.KB_MODE_DENSE_5_6, counts=cnt5120, columns=False)
                    torch.cuda.synchronize()
                    dms, dn = eng.stage_ms("count")
                    eng.enable_timing(False)
                    del cnt5120
                    dbytes = float(shard.offsets[-1]) + 4.0 * n * 5120
                    extras["roofline_count_dense5120"] = {
                        "bound": "hbm", "kernel": "k1_count (5120 dense columns)", "achieved": dbytes / (dms / 1e3) / 1e9,
                        "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": dbytes / (dms / 1e3) / 1e9 / pk["hbm_gbs"],
                        "bytes_per_launch": dbytes, "launches": dn}
            elif rank == 0 and asm is not None:
                extras["parity_sample"] = parity_sample_small(asm, kmer_size, all_idx[:n_total], all_dist[:n_total])
            big = [int(x) for x in a.big.split(",") if int(x) > 0] if a.big else ([500000, 1000000] if world == 8 else [])
            for nb in big:
                rec = big_run(torch, dist, eng, a, nb, rank, world, local, pk)
                if rank == 0:
                    extras["north_star_1M" if nb == 1000000 else ("config3" if nb == 500000 else "sharded_%d" % nb)] = rec
        except Exception as ex:                               # supplementary: never lose the headline line
            import traceback
            extras["error"] = "%s: %s" % (type(ex).__name__, ex)
            extras["traceback"] = traceback.format_exc()[-1500:]

    if rank != 0:
        plan.close()
        if world > 1:
            dist.destroy_process_group()
        return 0

    flops = 2.0 * n * n_total * d_cols                     # this rank's query rows x all keys
    ach_tf = flops / (gemm_ms / 1e3) / 1e12
    # the fused counting kernel (K1+K3, kb_count_profile): bases read once; profile row (f64), operand row (f16) and the
    # 32-byte row record written once; the u32 count rows never reach HBM
    count_bytes = float(shard.offsets[-1]) + n * (8.0 * cols_full + 2.0 * plan.dp + 32.0)
    ach_gbs = count_bytes / (count_ms / 1e3) / 1e9
    traffic = ncu_traffic("k4_tc") if world == 1 else None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 counts, f16 x f16 -> f32 Gram (tcgen05), f64 profile + rerank", "data": "synthetic",
        "config": {"workload": workload_name(a), "columns": d_cols, "total_bases": total_bases_all,
                   "knn_impl": a.knn_impl,
                   "pass": ("one CUDA graph per step" if plan.graph is not None else "eager enqueue") +
                           ("; key shards and k-lists exchanged over NVLink peer memory (no NCCL call on the path)" if world > 1 else ""),
                   "l2": "no explicit flush: one step streams %.2f GB of inputs+intermediates (> 126 MB L2)" %
                         ((total_bases_all + n_total * d_cols * (4 + 8 + 2)) / 1e9)},
        "clocks": clocks, "gpu_launches": int(launches_per_step * a.steps),
        "gpu_launches_per_step": int(launches_per_step),
        "uncertified_rows": int(uncertified),
        "stage_ms": {"count": count_ms, "count_long": long_ms, "normalise": norm_ms, "knn_gemm": gemm_ms, "rerank": rerank_ms,
                     "how": "mean of %d eager passes after the timed region (event pairs around every launch)" % n_stage},
        "roofline": {"bound": "tensor", "kernel": "k4_tc2 (distance GEMM, 2-CTA tcgen05 MMA + fused top-k)" if a.knn_impl == "tc" else "k4_simt",
                     "achieved": ach_tf, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach_tf / pk["tflops"],
                     "traffic": (traffic or {}).get("bytes"), "traffic_source": (traffic or {}).get("source"),
                     "peak_source": pk["source"] + ", bf16 burst; sustained %s" % pk["tflops_sustained"],
                     "flops_per_launch": flops, "launches_timed": gemm_n},
        "roofline_count": {"bound": "hbm", "kernel": "k1_count_warp<fused> (K1+K3 in one kernel: bases -> f64 profile + f16 operand + row records)", "achieved": ach_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                           "frac": ach_gbs / pk["hbm_gbs"], "bytes_per_launch": count_bytes},
    }
    line.update(extras)
    if e2e:
        line["e2e"] = e2e
    if world == 1 and not a.no_cpu_baseline and asm is not None:
        v, cores, sample, _ = cpu_arm(a, asm, 1, 0)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
    print(json.dumps(line))
    plan.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    args = parse()
    sys.exit(run_reference(args) if args.impl == "reference" else run_ours(args))
