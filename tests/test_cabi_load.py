"""The C-ABI library loads without a GPU and exports every symbol include/*.h declares."""
import ctypes
import glob
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    names = set()
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        src = open(h).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names |= set(re.findall(r"KB_API\s+[\w\s\*]+?\b(kb_\w+)\s*\(", src))
    return names


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    from karma_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        __graft_entry__.build()
    return _lib.load()


def test_exports_every_declared_symbol(lib):
    from karma_b200 import _lib
    declared = _declared()
    assert len(declared) >= 18
    assert declared == set(_lib.SIGNATURES), "ctypes binding and header disagree"
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name


def test_ctypes_signatures_match_header_arity():
    """Every prototype in include/karma_b200.h must have as many parameters as its ctypes binding."""
    from karma_b200 import _lib
    src = open(os.path.join(ROOT, "include", "karma_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = re.findall(r"KB_API\s+[\w\s\*]+?\b(kb_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S)
    assert len(protos) == len(_lib.SIGNATURES)
    for name, params in protos:
        params = params.strip()
        n = 0 if params in ("", "void") else len([p for p in params.split(",") if p.strip()])
        assert n == len(_lib.SIGNATURES[name][1]), "%s: header has %d parameters, ctypes binding %d" % (
            name, n, len(_lib.SIGNATURES[name][1]))


def test_pure_host_entry_points(lib):
    from karma_b200 import _lib
    assert lib.kb_version() >= 100
    assert lib.kb_mode_columns(_lib.KB_MODE_5P6) == 1088
    assert lib.kb_mode_columns(_lib.KB_MODE_DENSE_5_6) == 5120
    assert lib.kb_mode_columns(_lib.KB_MODE_DENSE_4_5) == 1280
    assert [lib.kb_mode_columns(_lib.KB_MODE_K(k)) for k in range(1, 8)] == [4 ** k for k in range(1, 8)]
    assert lib.kb_mode_columns(999) < 0 and b"unknown column mode" in lib.kb_last_error()
    assert lib.kb_knn_workspace_bytes(None, 1000, 1000, 0, 1088, 2, 0, 0) > 0
    assert lib.kb_knn_workspace_bytes(None, 1000, 1000, 0, 1088, 200, 0, 0) > 0   # any n_neighbors <= keys (cmd_parser.py:101-107): exact pass
    assert lib.kb_knn_workspace_bytes(None, 10, 5, 0, 1088, 8, 0, 0) < 0          # k > nk


def test_no_cpu_fallback(lib):
    """Without a GPU the product path must fail loudly."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from karma_b200 import _lib
    h = ctypes.c_void_p()
    assert lib.kb_create(ctypes.byref(h), 0) == _lib.KB_ENOGPU
    assert b"no CPU fallback" in lib.kb_last_error()
    from karma_b200.engine import Engine
    with pytest.raises(_lib.KarmaB200Error):
        Engine()
    from karma_b200.kmer import KmerClustering
    k = KmerClustering({">a": "ACGTACGT"}, "/tmp", "5p6", 1)
    with pytest.raises(_lib.KarmaB200Error):
        k._KmerClustering__calc_kmer_profile()


def test_product_never_imports_oracle():
    for path in glob.glob(os.path.join(ROOT, "karma_b200", "**", "*.py"), recursive=True):
        src = open(path).read()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), path


def test_header_is_plain_c_and_a_c_host_links(lib, tmp_path):
    """include/karma_b200.h is consumed by a C99 compiler (no C++, no torch types) and a plain-C host
    program links against the library; without a GPU it stops at kb_create with the no-fallback error."""
    import shutil
    import subprocess
    from karma_b200 import _lib
    gcc = shutil.which("gcc")
    cuda_inc = "/usr/local/cuda/include"
    if not gcc or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime_api.h")):
        pytest.skip("gcc or the CUDA headers are not available")
    exe = str(tmp_path / "c_abi_demo")
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = [gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-I", cuda_inc,
           os.path.join(ROOT, "examples", "c_abi_demo.c"), "-L", libdir, "-lkarma_b200", "-L", "/usr/local/cuda/lib64", "-lcudart",
           "-Wl,-rpath," + libdir, "-o", exe]
    built = subprocess.run(cmd, capture_output=True, text=True)
    assert built.returncode == 0, built.stderr
    run = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    import torch
    if torch.cuda.is_available():
        assert run.returncode == 0 and "c_abi_demo OK" in run.stdout, run.stdout + run.stderr
    else:
        assert run.returncode != 0 and "no CPU fallback" in run.stderr, run.stdout + run.stderr


def test_knn_plan_workspace_bounds(lib):
    """kb_knn_workspace_bytes (host only) over the shapes of BASELINE.json and the shard shapes of 2-8 GPUs:
    the plan never asks for more candidate slots than K5 can merge (512 per row)."""
    from karma_b200 import _lib
    shapes = [(1000, 1000, 0), (50000, 50000, 0), (6250, 50000, 18750), (62500, 500000, 62500), (125000, 1000000, 0),
              (250000, 2000000, 1750000), (130, 130, 0), (513, 513, 0)]
    for nq, nk, q0 in shapes:
        for dp in (1088, 5120):
            for k in (2, 10, 15, 24, 40, 60):
                kp = 8 if k <= 2 else 16 if k <= 10 else 24 if k <= 18 else 32 if k <= 26 else 48 if k <= 42 else 64
                for impl in (_lib.KB_KNN_SIMT, _lib.KB_KNN_TC):
                    b = lib.kb_knn_workspace_bytes(None, nq, nk, q0, dp, k, impl, 0)
                    lo = nq * kp * 8 + nq * 4 + nq * 4                       # one list of candidates + row bounds + uncertified rows
                    hi = nq * 512 * 8 + nq * 8 + 8 * 256                     # at most 512 candidates per row
                    assert lo <= b <= hi, (nq, nk, k, impl, b, lo, hi)
                    assert lib.kb_knn_workspace_bytes(None, nq, nk, q0, dp, k, impl, 7) > b    # flagged rows add the fp64 side lists


def _plan(lib, nq, nk, q0, dp, k, sm=148):
    import numpy as np
    out = (ctypes.c_int64 * 8)()
    assert lib.kb_knn_plan_info(sm, 2, nq, nk, q0, dp, k, out) == 0, lib.kb_last_error()
    info = dict(zip(("kp", "slots", "bands", "kind", "workers", "pieces", "makespan", "ideal"), list(out)))
    pieces = np.zeros((info["pieces"], 8), dtype=np.int32)
    start = np.zeros(info["workers"] + 1, dtype=np.int32)
    m_blocks = -(-nq // 128)
    groups = -(-m_blocks // 2)                                            # CTA pairs, also for a lone query block
    slots = np.zeros(groups, dtype=np.int32)
    vp = ctypes.c_void_p
    assert lib.kb_knn_plan_table(sm, 2, nq, nk, q0, dp, k, pieces.ctypes.data_as(vp), start.ctypes.data_as(vp),
                                 slots.ctypes.data_as(vp)) == 0
    return info, pieces, start, slots, groups


@pytest.mark.parametrize("nq,nk,q0,dp,k", [(50000, 50000, 0, 1088, 2), (6250, 50000, 18750, 1088, 2), (6250, 50000, 43750, 1088, 15),
                                           (12500, 50000, 12500, 1088, 2), (25000, 50000, 25000, 1088, 2), (50000, 50000, 0, 5120, 15),
                                           (62500, 500000, 62500, 5120, 15), (700, 700, 0, 1088, 60), (130, 130, 0, 1088, 24),
                                           (257, 700, 300, 1088, 5), (1, 600, 599, 64, 1)])
def test_knn_piece_table_covers_every_tile_once(lib, nq, nk, q0, dp, k):
    """The host-built schedule of the tensor kernel (kb_knn.cuh: KbPiece): every (query group, key tile) pair is
    visited exactly once, every piece has a candidate slot of its own, and the busiest CTA pair carries at most
    a few tile visits more than the mean (SURVEY 8e: small shards must keep all 74 CTA pairs busy)."""
    import numpy as np
    info, pieces, start, slots, groups = _plan(lib, nq, nk, q0, dp, k)
    n_tiles = -(-nk // 256)
    cover = np.zeros((groups, n_tiles), dtype=np.int32)
    seen = set()
    for g, slot, t_lo, cnt, shift, i_lo, i_cnt, _ in pieces:
        assert (g, slot) not in seen and 0 <= slot < slots[g] <= info["slots"]
        seen.add((g, slot))
        assert 0 <= i_lo and i_lo + i_cnt <= cnt and i_cnt >= 1 and 0 <= shift < cnt and 0 <= t_lo < n_tiles
        i = np.arange(i_lo, i_lo + i_cnt) + shift
        cover[g, (np.where(i >= cnt, i - cnt, i) + t_lo) % n_tiles] += 1
    assert (cover == 1).all()
    assert info["slots"] * info["kp"] <= 512
    assert start[0] == 0 and start[-1] == len(pieces) and (np.diff(start) >= 0).all()
    loads = np.array([pieces[start[w]:start[w + 1], 6].sum() for w in range(info["workers"])])
    mean = groups * n_tiles / info["workers"]
    assert loads.max() <= mean * 1.04 + 2 * info["bands"], (loads.max(), mean, info)
    if nk * dp * 2 > 120e6 and n_tiles >= 2:
        # a key set beyond the L2 is swept in whole bands, dealt round-robin, so that concurrent clusters share key tiles
        assert info["kind"] == 0 and info["bands"] >= 2 and (pieces[:, 5] == 0).all() and (pieces[:, 6] == pieces[:, 3]).all()


@pytest.mark.parametrize("nq,nk,q0,dp,k", [(25000, 50000, 25000, 1088, 2), (12500, 50000, 12500, 1088, 2), (6250, 50000, 43750, 1088, 15),
                                           (6250, 50000, 0, 1088, 2), (62500, 500000, 187500, 5120, 15), (257, 700, 300, 1088, 5)])
def test_shard_sweeps_follow_the_arrival_order(lib, nq, nk, q0, dp, k):
    """A query shard receives the other shards over NVLink in the order q+1, q+2, ..., q-1.  Every query group must
    therefore sweep the key tiles as ONE rotation that starts on a tile lying fully inside the local rows and runs upwards
    with wrap-around -- the tile straddling the start of the local shard (it needs rows of rank q-1) comes after all others."""
    import numpy as np
    info, pieces, start, slots, groups = _plan(lib, nq, nk, q0, dp, k)
    n_tiles = -(-nk // 256)
    first_full = -(-q0 // 256)
    last_full = (q0 + nq) // 256 - 1
    per_group = {}
    for g, slot, t_lo, cnt, shift, i_lo, i_cnt, _ in pieces:
        i = np.arange(i_lo, i_lo + i_cnt) + shift
        tiles = (np.where(i >= cnt, i - cnt, i) + t_lo) % n_tiles
        per_group.setdefault(int(g), []).append((int(slot), tiles))
    for g, lst in per_group.items():
        seq = np.concatenate([t for _, t in sorted(lst, key=lambda x: x[0])])      # slots are handed out in sweep order
        assert len(seq) == n_tiles
        assert ((seq[1:] - seq[:-1]) % n_tiles == 1).all(), (g, seq[:8])
        if first_full <= last_full:
            assert first_full <= seq[0] <= last_full, (g, seq[0], first_full, last_full)
            if q0 % 256:
                # the head straddler is behind every tile of the other shards
                pos = int(np.flatnonzero(seq == first_full - 1)[0])
                foreign = [int(np.flatnonzero(seq == t)[0]) for t in range(n_tiles) if t < first_full - 1 or t > last_full + 1]
                assert not foreign or pos > max(foreign)


def test_knn_piece_table_random_shapes(lib):
    """Randomised shapes (ragged shards of 1..8 ranks, arbitrary query sub-ranges, 8..148 SMs, every list width): every
    (query group, key tile) pair exactly once, every piece in its own candidate slot, at most 512 candidates per row."""
    import random
    import numpy as np
    rnd = random.Random(5)
    for _ in range(120):
        nk = rnd.choice([600, 1000, 3000, 7777, 20011, 50000, 123457])
        world = rnd.choice([1, 2, 3, 4, 5, 8])
        per = -(-nk // world)
        q0 = min(rnd.randrange(world) * per, nk - 1)
        nq = max(1, min(per, nk - q0))
        if rnd.random() < 0.2:
            q0 = rnd.randrange(0, nk)
            nq = rnd.randrange(1, nk - q0 + 1)
        dp = rnd.choice([64, 1088, 1280, 5120])
        k = min(rnd.choice([1, 2, 5, 15, 24, 40, 60]), nk)
        sm = rnd.choice([148, 132, 8])
        info, pieces, start, slots, groups = _plan(lib, nq, nk, q0, dp, k, sm)
        n_tiles = -(-nk // 256)
        cover = np.zeros((groups, n_tiles), dtype=np.int32)
        seen = set()
        for g, slot, t_lo, cnt, shift, i_lo, i_cnt, _pad in pieces:
            assert (g, slot) not in seen and 0 <= slot < slots[g] <= info["slots"]
            seen.add((g, slot))
            assert 0 <= i_lo and i_lo + i_cnt <= cnt and i_cnt >= 1 and 0 <= shift < cnt and 0 <= t_lo < n_tiles
            i = np.arange(i_lo, i_lo + i_cnt) + shift
            cover[g, (np.where(i >= cnt, i - cnt, i) + t_lo) % n_tiles] += 1
        assert (cover == 1).all(), (nq, nk, q0, dp, k, sm, info)
        assert info["slots"] * info["kp"] <= 512
