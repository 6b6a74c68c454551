"""K11, MCL of many groups in one call: the oracle's definition on the CPU (known answers, invariants, the numba twin and
the block-diagonal batch against the plain-Python reference, pruning branches, refusals), and (GPU) kb_mcl_build
against the twin, bit for bit."""
import math
import shutil
import subprocess

import numpy as np
import pytest

from oracle import mcl_oracle as mo

CLIQUES = [(x, y, 1.0) for c in ("abcd", "efgh") for i, x in enumerate(c) for y in c[i + 1:]] + [("d", "e", 0.1)]
TRIANGLES = [("a", "b", 1.0), ("b", "c", 0.5), ("a", "c", 2.0), ("x", "y", 1.0), ("y", "z", 1.0), ("x", "z", 0.25)]
STAR = [("hub", "leaf%d" % i, 1.0 + 0.1 * i) for i in range(6)]
KNOWN = {
    "cliques": (CLIQUES, [list("abcd"), list("efgh")]),
    "edge": ([("u", "v", 3.0)], [["u", "v"]]),
    "triangles": (TRIANGLES, [list("abc"), list("xyz")]),
    "star": (STAR, [["hub"] + ["leaf%d" % i for i in range(6)]]),
}


def random_groups(seed, n_groups, lo=2, hi=300, ties=False):
    """Seeded groups of sizes lo..hi as one node set: edge arrays (a, b, w), group ids, and the node count.  Each group
    is a few dense communities joined by sparse edges; ``ties`` draws weights from four values."""
    rng = np.random.default_rng(seed)
    a, b, w, group = [], [], [], []
    n = 0
    for g in range(n_groups):
        size = int(rng.integers(lo, hi + 1))
        comm = max(1, size // int(rng.integers(3, 12)))
        label = rng.integers(0, comm, size)
        p_in, p_out = min(1.0, 4.0 / max(1, size / comm)), min(0.5, 1.5 / size)
        for i in range(size):
            for j in range(i + 1, size):
                if rng.random() < (p_in if label[i] == label[j] else p_out) or j == i + 1 and rng.random() < 0.3:
                    a.append(n + i)
                    b.append(n + j)
                    w.append(float(rng.choice([0.25, 0.5, 1.0, 2.0])) if ties else float(rng.random() * 2 + 1e-3))
        group.extend([g] * size)
        n += size
    perm = rng.permutation(len(a))                       # stream order is not sorted order
    flip = rng.random(len(a)) < 0.5
    a, b = np.array(a, np.int64)[perm], np.array(b, np.int64)[perm]
    a, b = np.where(flip, b, a), np.where(flip, a, b)
    return a.astype(np.int32), b.astype(np.int32), np.array(w)[perm], np.array(group, np.int32), n


def partition(clusters_names):
    return sorted(sorted(map(str, c)) for c in clusters_names)


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", sorted(KNOWN))
def test_known_answers(name):
    edges, want = KNOWN[name]
    got = mo.mcl_stream(edges)
    assert got["lines"] == want
    assert got["overlap"] == 0


def test_iterates_are_stochastic_and_converge_to_an_idempotent():
    a, b, w, group, n = random_groups(5, 6, 20, 80)
    seg = mo.segment(n, a, b, w, group, 6)
    worst = 0.0
    for g, stream in enumerate(seg["streams"]):
        size = int(seg["size"][g])

        def check(it, cols, chaos):
            for col in cols:
                assert abs(math.fsum(v for _, v in col) - 1.0) <= 1e-12

        cols, _ = mo.mcl_matrix(size, stream, on_iterate=check)
        m = np.zeros((size, size))
        for j, col in enumerate(cols):
            for i, v in col:
                m[i, j] = v
        worst = max(worst, float(np.abs(m @ m - m).max()))
    assert worst <= 1e-3, worst                   # observed: about 1e-5 (chaos < 1e-4 bounds the distance)


@pytest.mark.parametrize("ties", [False, True])
def test_twin_and_batch_equal_the_reference(ties):
    """The numba twin on the block-diagonal union, every group frozen on its own chaos, equals the plain-Python
    reference run on each group's stream separately, bit for bit (values, iterations, partitions, output order)."""
    a, b, w, group, n = random_groups(11 + ties, 14, 2, 300, ties)
    twin = mo.groups_oracle(n, a, b, w, group, 14, twin=True)
    ref = mo.groups_oracle(n, a, b, w, group, 14, twin=False)
    assert twin["iterations"].tolist() == ref["iterations"].tolist()
    assert [[(i, v.hex()) for i, v in c] for c in twin["columns"]] == [[(i, v.hex()) for i, v in c] for c in ref["columns"]]
    assert twin["cluster"].tolist() == ref["cluster"].tolist() and twin["clusters"] == ref["clusters"]
    # one group per call gives the same bits as all groups in one call
    for g in (0, 5, 13):
        keep = (group[a] == g)
        solo = mo.groups_oracle(n, a[keep], b[keep], w[keep], np.where(group == g, 0, -1).astype(np.int32), 1)
        lo, hi = twin["size"][:g].sum(), twin["size"][:g + 1].sum()
        assert solo["columns"] == twin["columns"][lo:hi] and solo["iterations"][0] == twin["iterations"][g]


def test_relabelling_keeps_the_partition():
    """Permuting and flipping the stream's edges renumbers the nodes and reorders every sum; the partition stays the
    same wherever no node reaches two attractor systems.  A node that does joins the system with the smaller number,
    and numbers follow labels (the unpinned overlap rule): on this seeded set 4 of 10 groups have one such node, and
    only those groups ever changed."""
    a, b, w, group, n = random_groups(21, 10, 5, 120)
    seg = mo.segment(n, a, b, w, group, 10)
    rng = np.random.default_rng(3)
    checked = overlapping = 0
    for g, stream in enumerate(seg["streams"]):
        names = [(g, i) for i in range(int(seg["size"][g]))]
        edges = [(names[x], names[y], v) for x, y, v in stream]
        ref = mo.mcl_stream(edges)
        for _ in range(2):
            perm = rng.permutation(len(edges))
            shuffled = [edges[i] if rng.random() < 0.5 else (edges[i][1], edges[i][0], edges[i][2]) for i in perm]
            got = mo.mcl_stream(shuffled)
            assert got["overlap"] == ref["overlap"]
            if ref["overlap"] == 0:
                assert partition(got["lines"]) == partition(ref["lines"])
                checked += 1
        overlapping += ref["overlap"] > 0
    assert checked == 12 and overlapping == 4


def _expanded_column(cols, j):
    acc = {}
    for k, mkj in cols[j]:
        for i, mik in cols[k]:
            acc[i] = acc.get(i, 0.0) + mik * mkj
    return sorted(acc.items())


def test_pruning_selection_on_a_near_uniform_clique():
    """Every column of a 950-clique with weights 1 +- 1 % has 950 entries of about 1/950 >= 1/7000 after the first
    expansion: selection keeps the 900 largest, whose mass (about 900/950) needs no recovery."""
    n = 950
    rng = np.random.default_rng(2)
    edges = [(i, j, 1.0 + 0.01 * rng.random()) for i in range(n) for j in range(i + 1, n)]
    cols = mo.initial_columns(n, edges)
    for j in (0, 477, 949):
        stats = []
        col = _expanded_column(cols, j)
        kept = mo.prune_column(col, stats)
        s = stats[0]
        assert s["entries"] == n and s["over_cutoff"] == n and s["selected"] and s["recovered"] == 0
        assert len(kept) == s["kept"] == mo.S
        assert 0.9 * s["mass"] <= s["kept_mass"] <= s["mass"] * 900 / 950 * 1.02
        values = sorted((v for _, v in col), reverse=True)
        assert s["kept_mass"] == pytest.approx(math.fsum(values[:mo.S]), rel=1e-12)
        assert abs(math.fsum(v for _, v in kept) - 1.0) <= 1e-12


def test_pruning_recovery_on_a_star():
    """The hub column of a 4000-leaf star spreads its mass over 4001 entries of about 1/4001 < 1/7000 after the first
    expansion: the cutoff keeps only the hub's own entry, and recovery adds the next largest until R entries are kept."""
    n = 4000
    edges = [(0, i, 1.0) for i in range(1, n + 1)]
    cols = mo.initial_columns(n + 1, edges)
    stats = []
    col = _expanded_column(cols, 0)
    kept = mo.prune_column(col, stats)
    s = stats[0]
    assert s["entries"] == n + 1 and s["over_cutoff"] == 1 and not s["selected"]
    assert s["kept"] == len(kept) == mo.R and s["recovered"] == mo.R - 1
    values = sorted((v for _, v in col), reverse=True)
    assert s["kept_mass"] == pytest.approx(math.fsum(values[:mo.R]), rel=1e-12) and s["kept_mass"] < 0.9 * s["mass"]
    # recovery that stops on the mass: one entry of 0.85 and 1500 of 1e-4 (below the cutoff)
    stats = []
    col = [(0, 0.85)] + [(i, 1e-4) for i in range(1, 1501)]
    mo.prune_column(col, stats)
    s = stats[0]
    assert s["over_cutoff"] == 1 and 1 < s["kept"] < mo.R
    assert s["kept_mass"] >= 0.9 * s["mass"] > s["kept_mass"] - 1e-4
    assert s["kept"] == 1 + math.ceil((0.9 * s["mass"] - 0.85) / 1e-4 - 1e-6)


def test_refusals_before_any_gpu_work():
    from karma_b200 import mcl as km
    import networkx as nx
    for edges in ([("a", "a", 1.0)], [("a", "b", 1.0), ("b", "a", 2.0)], [("a", "b", 0.0)], [("a", "b", -1.0)],
                  [("a", "b", float("nan"))], [("a", "b", float("inf"))]):
        with pytest.raises(ValueError):
            km.mcl_abc(edges, engine=object())
        with pytest.raises(ValueError):
            mo.mcl_stream(edges)
    for bad in (1.0, 0.5, float("nan"), float("inf"), True, "2"):
        with pytest.raises(ValueError):
            km.mcl_abc([("a", "b", 1.0)], inflation=bad, engine=object())
    g = nx.Graph()
    g.add_edge("a", "b", weight=1.0)
    g.add_edge("c", "c", weight=1.0)
    with pytest.raises(ValueError):
        km.mcl_groups(g, [["a", "b"], ["a"]], engine=object())          # a node in two groups
    with pytest.raises(ValueError):
        km.mcl_groups(g, [["a", "b", "c"]], engine=object())            # a self-edge inside a group
    g.add_edge("a", "d", weight=float("nan"))
    with pytest.raises(ValueError):
        km.mcl_groups(g, [["a", "d"]], engine=object())


@pytest.mark.skipif(shutil.which("mcl") is None, reason="no mcl binary on PATH")
def test_partitions_against_a_real_mcl_binary():
    a, b, w, group, n = random_groups(31, 8, 5, 150)
    seg = mo.segment(n, a, b, w, group, 8)
    for edges in [e for e, _ in KNOWN.values()] + [[("n%d" % x, "n%d" % y, v) for x, y, v in s] for s in seg["streams"]]:
        text = "".join("%s\t%s\t%r\n" % e for e in edges)
        out = subprocess.run(["mcl", "-", "--abc", "-o", "-"], input=text, capture_output=True, text=True, check=True).stdout
        assert partition(line.split("\t") for line in out.splitlines() if line) == partition(mo.mcl_stream(edges)["lines"])


# ------------------------------------------------------------------ GPU
def _device(engine, n, a, b, w, group, n_groups, inflation=2.0):
    import torch
    from karma_b200 import mcl as km
    dev = engine.device
    t = lambda x, dt: torch.from_numpy(np.ascontiguousarray(x)).to(dev, dt)      # noqa: E731
    return km.mcl_arrays(engine, n, t(a, torch.int32), t(b, torch.int32), t(w, torch.float64), t(group, torch.int32),
                         n_groups, inflation, columns=True)


def _columns(res):
    cp = res["colptr"]
    return [[(int(r), float(v)) for r, v in zip(res["rows"][cp[j]:cp[j + 1]], res["vals"][cp[j]:cp[j + 1]])]
            for j in range(len(cp) - 1)]


def _assert_equal(got, want, exact=True):
    assert got["local"].tolist() == want["local"].tolist()
    assert got["iterations"].tolist() == want["iterations"].tolist()
    assert got["cluster"].tolist() == want["cluster"].tolist()
    assert got["n_clusters"].tolist() == want["n_clusters"].tolist()
    assert got["overlap"].tolist() == want["overlap"].tolist()
    gc = _columns(got)
    if exact:
        assert [[(i, v.hex()) for i, v in c] for c in gc] == [[(i, v.hex()) for i, v in c] for c in want["columns"]]
    else:
        assert [[i for i, _ in c] for c in gc] == [[i for i, _ in c] for c in want["columns"]]
        for c, d in zip(gc, want["columns"]):
            for (_, x), (_, y) in zip(c, d):
                assert abs(x - y) <= 1e-12                  # columns sum to 1: relative to the column's mass


def _stream_arrays(edges):
    index = {}
    for u, v, _ in edges:
        for x in (u, v):
            index.setdefault(x, len(index))
    return (np.array([index[u] for u, _, _ in edges], np.int32), np.array([index[v] for _, v, _ in edges], np.int32),
            np.array([x for _, _, x in edges]), np.zeros(len(index), np.int32), len(index))


@pytest.mark.gpu
def test_gpu_known_answers(engine):
    from karma_b200 import mcl as km
    for name, (edges, want) in KNOWN.items():
        assert km.mcl_abc(edges, engine=engine) == want, name
        a, b, w, group, n = _stream_arrays(edges)
        _assert_equal(_device(engine, n, a, b, w, group, 1), mo.groups_oracle(n, a, b, w, group, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("ties", [False, True])
def test_gpu_two_thousand_groups_in_one_call(engine, ties):
    a, b, w, group, n = random_groups(41 + ties, 2000, 2, 60, ties)
    a2, b2, w2, g2, n2 = random_groups(43 + ties, 6, 257, 700, ties)          # groups on the CTA path too
    a = np.concatenate([a, a2 + n]); b = np.concatenate([b, b2 + n]); w = np.concatenate([w, w2])
    group = np.concatenate([group, g2 + 2000]).astype(np.int32)
    want = mo.groups_oracle(n + n2, a, b, w, group, 2006)
    got = _device(engine, n + n2, a, b, w, group, 2006)
    _assert_equal(got, want)
    again = _device(engine, n + n2, a, b, w, group, 2006)                     # determinism
    assert again["vals"].tobytes() == got["vals"].tobytes() and again["rows"].tobytes() == got["rows"].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("inflation", [1.5, 3.0])
def test_gpu_other_inflations(engine, inflation):
    """pow may differ from the host's in the last bit, and the difference compounds over the iterations: identical
    partitions, iterations and entries, values within 1e-12 of the column's mass (on a B200 at I = 1.5 the largest
    difference was 1.7e-17, 2.2e-12 relative to its entry)."""
    a, b, w, group, n = random_groups(47, 300, 2, 120)
    want = mo.groups_oracle(n, a, b, w, group, 300, inflation)
    _assert_equal(_device(engine, n, a, b, w, group, 300, inflation), want, exact=False)


def _communities(n, size, seed):
    rng = np.random.default_rng(seed)
    a, b = [], []
    for c0 in range(0, n, size):
        m = min(size, n - c0)
        for i in range(m):
            for j in range(i + 1, m):
                if rng.random() < 0.6:
                    a.append(c0 + i); b.append(c0 + j)
    extra = rng.integers(0, n, (n // 2, 2))
    pairs = set(zip(a, b))
    for x, y in extra.tolist():
        if x != y and (min(x, y), max(x, y)) not in pairs:
            pairs.add((min(x, y), max(x, y))); a.append(min(x, y)); b.append(max(x, y))
    perm = rng.permutation(len(a))
    return (np.array(a, np.int32)[perm], np.array(b, np.int32)[perm], rng.random(len(a))[perm] + 0.05)


@pytest.mark.gpu
def test_gpu_large_group_path(engine):
    """A 40 000-node group: beyond the shared-memory accumulator (16 384 rows), so its columns use the global one."""
    n = 40000
    a, b, w = _communities(n, 8, 5)
    group = np.zeros(n, np.int32)
    _assert_equal(_device(engine, n, a, b, w, group, 1), mo.groups_oracle(n, a, b, w, group, 1))


@pytest.mark.gpu
def test_gpu_selection_and_recovery_graphs(engine):
    rng = np.random.default_rng(2)
    n = 950
    iu = np.triu_indices(n, 1)
    a1, b1, w1 = iu[0].astype(np.int32), iu[1].astype(np.int32), 1.0 + 0.01 * rng.random(len(iu[0]))
    a2 = np.zeros(4000, np.int32) + n
    b2 = np.arange(n + 1, n + 4001, dtype=np.int32)
    a, b, w = np.concatenate([a1, a2]), np.concatenate([b1, b2]), np.concatenate([w1, np.ones(4000)])
    group = np.concatenate([np.zeros(n, np.int32), np.ones(4001, np.int32)])
    _assert_equal(_device(engine, n + 4001, a, b, w, group, 2), mo.groups_oracle(n + 4001, a, b, w, group, 2))


@pytest.mark.gpu
def test_gpu_edge_cases(engine):
    # group 0 empty, group 1 one edge, group 2 nodes without edges among them, nodes of group -1, an edge across groups
    a = np.array([1, 2, 4, 0, 5], np.int32)
    b = np.array([2, 3, 5, 6, 3], np.int32)
    w = np.array([0.5, 1.0, 2.0, 1.0, 1.0])
    group = np.array([-1, 1, 1, 2, -1, -1, 2], np.int32)
    want = mo.groups_oracle(7, a, b, w, group, 3)
    got = _device(engine, 7, a, b, w, group, 3)
    _assert_equal(got, want)
    assert got["n_clusters"].tolist() == [0, 1, 0] and got["local"].tolist() == [-1, 0, 1, -1, -1, -1, -1]
    empty = _device(engine, 3, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0), np.array([0, -1, 0], np.int32), 2)
    assert empty["cluster"].tolist() == [-1, -1, -1] and empty["iterations"].tolist() == [0, 0]


@pytest.mark.gpu
def test_gpu_read_graph_groups(engine, tmp_path):
    """The read graph of 200 k synthetic contigs, grouped by synthetic families (k-mer clusters of 2-10 contigs), plus
    one unlabeled-sized group of about 12 k contigs; then mcl_groups on the networkx graph."""
    from karma_b200 import mcl as km
    from karma_b200 import read_graph as rg
    from karma_b200 import rearrange as rr
    from oracle import readgraph_oracle as ro
    names, classes = ro.synth_eq_classes(200000, 1000000, seed=11, family=6, max_size=8)
    path = str(tmp_path / "eq.txt")
    ro.write_eq_file(path, names, classes)
    graph = rg.from_equivalence_classes(path, {">" + x: "" for x in names}, engine=engine)
    groups = synth_groups(list(graph.nodes()), seed=3)
    index, a, b, w = rr.graph_arrays(graph)
    from karma_b200.rearrange import _roles
    group, _, _ = _roles(index, groups, "groups")
    want = mo.groups_oracle(len(index), a, b, w, group, len(groups))
    got = _device(engine, len(index), a, b, w, group, len(groups))
    _assert_equal(got, want)
    nodes = list(index)
    by_group = km.mcl_groups(graph, groups, engine=engine)
    inv = {}
    for v in np.flatnonzero(want["local"] >= 0).tolist():
        inv[(int(group[v]), int(want["local"][v]))] = nodes[v]
    assert by_group == [[[inv[(g, i)] for i in c] for c in cg] for g, cg in enumerate(want["clusters"])]


def synth_groups(nodes, seed, unlabeled=12000):
    """k-mer-cluster-like groups: runs of 2-10 consecutive contigs (mostly one family), then one unlabeled group."""
    rng = np.random.default_rng(seed)
    groups, i = [], unlabeled
    while i < len(nodes):
        k = int(rng.integers(2, 11))
        groups.append(nodes[i:i + k])
        i += k
    groups.append(list(nodes[:unlabeled]))
    return groups


@pytest.mark.gpu
def test_gpu_c_abi_refusals(engine):
    import torch
    from ctypes import byref, c_int64
    from karma_b200 import _lib
    dev = engine.device
    t = lambda x, dt: torch.tensor(x, dtype=dt, device=dev)      # noqa: E731
    cases = [([0], [0], [1.0], [0, 0, 0], 2.0),                   # self-edge
             ([0, 1], [1, 0], [1.0, 1.0], [0, 0, 0], 2.0),        # the same pair twice
             ([0], [1], [0.0], [0, 0, 0], 2.0), ([0], [1], [float("nan")], [0, 0, 0], 2.0),
             ([0], [1], [float("inf")], [0, 0, 0], 2.0),
             ([0], [3], [1.0], [0, 0, 0], 2.0),                    # an index out of range
             ([0], [1], [1.0], [0, 5, 0], 2.0),                    # a group id out of range
             ([0], [1], [1.0], [0, 0, 0], 1.0), ([0], [1], [1.0], [0, 0, 0], float("nan"))]
    for a, b, w, g, inflation in cases:
        da, db, dw, dg = t(a, torch.int32), t(b, torch.int32), t(w, torch.float64), t(g, torch.int32)
        nc, nz = c_int64(), c_int64()
        rc = engine.lib.kb_mcl_build(engine.ctx, 3, len(a), _lib.ptr(da), _lib.ptr(db), _lib.ptr(dw), _lib.ptr(dg), 1,
                                     inflation, byref(nc), byref(nz))
        assert rc == _lib.KB_EINVAL, (a, b, w, g, inflation)
