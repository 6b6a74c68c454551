"""HDBSCAN (K9): the oracle's tree routines and canonical MST against scikit-learn 1.9.0, ``kb_hdbscan_labels`` through
ctypes and the hdbscan-0.8.22 mirror's host rules (CPU); core distances, the device MST, labels and probabilities
against the oracle and scikit-learn (-m gpu)."""
import numpy as np
import pytest
import torch

from oracle import hdbscan_oracle as ho
from oracle import umap_layout_oracle as lo


def _pts(n, dim, seed, n_blobs=8, coincident=0):
    """float32 blobs; ``coincident`` rows copy row 0 and as many copy the last row (zero distances, zero weights)."""
    x = lo.blobs(n, n_blobs, dim, seed=seed)[0].astype(np.float32)
    if coincident:
        x[1:1 + coincident] = x[0]
        x[n - 1 - coincident:n - 1] = x[n - 1]
    return x


def _bits_equal(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


# (n, n_blobs, coincident rows, core_k) -> the oracle's canonical MST
TREE_INPUTS = {
    "ties, one blob": (8000, 1, 0, 3),
    "eight blobs": (5000, 8, 0, 3),
    "coincident rows": (3000, 8, 40, 3),
    "core_k 16": (4000, 30, 0, 16),
    "tie-free, core_k 1": (3000, 8, 0, 1),
}


@pytest.fixture(scope="module")
def trees():
    out = {}
    for name, (n, blobs, coincident, core_k) in TREE_INPUTS.items():
        x = _pts(n, 10, seed=1, n_blobs=blobs, coincident=coincident)
        out[name] = ho.mst(x, core_k)
    return out


def test_ties_and_zero_weights_are_present(trees):
    w = trees["ties, one blob"][2]
    assert len(w) - len(np.unique(w)) > 100
    assert (trees["coincident rows"][2] == 0.0).sum() >= 78
    w = trees["tie-free, core_k 1"][2]
    assert len(np.unique(w)) == len(w)


@pytest.mark.parametrize("allow_single", [False, True])
@pytest.mark.parametrize("mcs", [2, 5, 15])
@pytest.mark.parametrize("name", list(TREE_INPUTS))
def test_tree_port_equals_sklearn(trees, name, mcs, allow_single):
    _, edges, weights = trees[name]
    labels, probs, n_clusters = ho.tree_to_labels(edges, weights, mcs, allow_single)
    ref_labels, ref_probs = ho.sklearn_tree_to_labels(edges, weights, mcs, allow_single)
    assert np.array_equal(labels, ref_labels) and _bits_equal(probs, ref_probs)
    assert n_clusters == len(set(ref_labels.tolist()) - {-1})


def test_tree_port_single_cluster_by_hand():
    """Two points: with allow_single_cluster both belong to the root at probability 1, otherwise both are noise."""
    edges, weights = np.array([[0, 1]], np.int32), np.array([2.0])
    assert [a.tolist() for a in ho.tree_to_labels(edges, weights, 2, True)[:2]] == [[0, 0], [1.0, 1.0]]
    assert [a.tolist() for a in ho.tree_to_labels(edges, weights, 2, False)[:2]] == [[-1, -1], [0.0, 0.0]]


@pytest.mark.parametrize("n,dim,coincident", [(300, 10, 0), (257, 2, 30), (200, 1, 20)])
@pytest.mark.parametrize("core_k", [1, 3, 16])
def test_prim_port_twin_kruskal_and_sklearn(n, dim, coincident, core_k):
    x = _pts(n, dim, seed=n + core_k, coincident=coincident)
    core = ho.core_distances(x, core_k)
    pe, pw = ho.prim_mst_port(x, core)
    te, tw = ho.prim_mst(x, core)
    assert np.array_equal(pe, te) and _bits_equal(pw, tw)
    ke, kw = ho.kruskal_mst(x, core)
    assert np.array_equal(ke, te) and _bits_equal(kw, tw)
    assert _bits_equal(np.sort(ho.sklearn_prim(x, core)[1]), tw)


def test_prim_twin_weights_equal_sklearn_at_5000(trees):
    x = _pts(5000, 10, seed=1, n_blobs=8)
    core, _, w = trees["eight blobs"]
    assert _bits_equal(np.sort(ho.sklearn_prim(x, core)[1]), w)


@pytest.mark.parametrize("n,dim,coincident", [(2, 3, 0), (129, 10, 20), (3000, 10, 40), (1000, 64, 10)])
def test_oracle_core_distances_equal_kneighbors(n, dim, coincident):
    from sklearn.neighbors import NearestNeighbors
    x = _pts(n, dim, seed=3, coincident=coincident)
    k = min(n, 128)
    ref = NearestNeighbors(n_neighbors=k, algorithm="kd_tree").fit(x.astype(np.float64)).kneighbors(x.astype(np.float64), k)[0]
    for core_k in (1, 2, 3, 16, 128):
        if core_k <= n:
            assert _bits_equal(ho.core_distances(x, core_k), ref[:, core_k - 1]), core_k


# ---------------------------------------------------------------------------------------------
# kb_hdbscan_labels through ctypes (no GPU)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("allow_single", [False, True])
@pytest.mark.parametrize("mcs", [2, 5, 15])
@pytest.mark.parametrize("name", list(TREE_INPUTS))
def test_native_labels_equal_the_oracle(trees, name, mcs, allow_single):
    from karma_b200.hdbscan_ import tree_labels
    _, edges, weights = trees[name]
    labels, probs, n_clusters = tree_labels(edges, weights, mcs, allow_single)
    ref_labels, ref_probs, ref_n = ho.tree_to_labels(edges, weights, mcs, allow_single)
    assert labels.dtype == np.int32 and np.array_equal(labels, ref_labels)
    assert _bits_equal(probs, ref_probs) and n_clusters == ref_n


def test_native_labels_refusals(trees):
    from karma_b200 import _lib
    from karma_b200.hdbscan_ import tree_labels
    _, edges, weights = trees["eight blobs"]

    def refused(e, w, mcs=5):
        with pytest.raises(_lib.KarmaB200Error) as err:
            tree_labels(e, w, mcs)
        assert err.value.code == _lib.KB_EINVAL
        return str(err.value)

    e = edges.copy()
    e[10, 1] = len(weights) + 1                                   # index out of range
    refused(e, weights)
    e = edges.copy()
    e[10] = e[10, ::-1]                                           # not (min, max)
    refused(e, weights)
    e, w = edges.copy(), weights.copy()                           # two edges swapped
    e[[20, 21]], w[[20, 21]] = e[[21, 20]], w[[21, 20]]
    assert "order" in refused(e, w)
    tie = np.flatnonzero(weights[1:] == weights[:-1])
    e = edges.copy()                                              # equal weights, keys out of order
    e[[tie[0], tie[0] + 1]] = e[[tie[0] + 1, tie[0]]]
    assert "order" in refused(e, weights)
    for v in (np.nan, np.inf, -1.0):
        w = weights.copy()
        w[-1] = v
        refused(edges, w)
    w = weights.copy()
    w[0] = -0.5
    refused(edges, w)
    # a cycle: (0, 1), (1, 2), (0, 2) and a point left out
    cyc = np.array([[0, 1], [1, 2], [0, 2]], np.int32)
    assert "cycle" in refused(cyc, np.array([1.0, 2.0, 3.0]), mcs=2)
    refused(edges, weights, mcs=1)
    assert tree_labels(edges, weights, 5)[2] >= 1                 # still usable


# ---------------------------------------------------------------------------------------------
# the hdbscan-0.8.22 mirror, with a fake engine
# ---------------------------------------------------------------------------------------------
@pytest.fixture
def fake(monkeypatch):
    import types
    from karma_b200 import hdbscan_
    seen = {}

    def mst(engine, x, core_k):
        seen.update(core_k=core_k, x=x.numpy().copy())
        _, e, w = ho.mst(x.numpy(), core_k)
        return {"core": None, "edges": torch.from_numpy(e), "weights": torch.from_numpy(w)}

    monkeypatch.setattr(hdbscan_, "mutual_reachability_mst", mst)
    return hdbscan_, types.SimpleNamespace(device=torch.device("cpu")), seen


def test_mirror_min_samples_rules(fake):
    mod, eng, seen = fake
    x = _pts(300, 10, seed=2)
    for mcs, ms, want in ((5, None, 6), (2, None, 3), (15, 1, 2), (2, 7, 8), (400, None, 300), (2, 1000, 300)):
        mod.cluster_embedding(eng, x, mcs, ms)
        assert seen["core_k"] == want, (mcs, ms)
        assert mod.host_rules(300, mcs, ms) == ho.host_rules(300, mcs, ms) == (want - 1, want)
    assert mod.host_rules(2, 2) == ho.host_rules(2, 2) == (1, 2)
    assert ho.host_rules(1, 2) == (1, 2)                          # 0 is raised to 1
    assert ho.karma_kwargs(1) == {"allow_single_cluster": True} and ho.karma_kwargs(3) == {"min_cluster_size": 3}


def test_mirror_fit_equals_the_oracle(fake):
    mod, eng, seen = fake
    x = _pts(2000, 10, seed=4)
    c = mod.HDBSCAN(min_cluster_size=15, engine=eng).fit(x)
    _, e, w = ho.mst(x, 16)
    labels, probs, _ = ho.tree_to_labels(e, w, 15)
    assert c.labels_.dtype == np.intp and np.array_equal(c.labels_, labels) and _bits_equal(c.probabilities_, probs)
    assert np.array_equal(mod.HDBSCAN(allow_single_cluster=True, engine=eng).fit_predict(x),
                          ho.tree_to_labels(*ho.mst(x, 6)[1:], 5, True)[0])


def test_mirror_refuses_what_it_does_not_serve(fake):
    mod, eng, _ = fake
    for kw in ({"metric": "manhattan"}, {"alpha": 0.5}, {"cluster_selection_method": "leaf"}, {"prediction_data": True},
               {"approx_min_span_tree": False}, {"cluster_selection_epsilon": 0.1}, {"max_cluster_size": 10}):
        with pytest.raises(ValueError, match=next(iter(kw))):
            mod.HDBSCAN(engine=eng, **kw)
    mod.HDBSCAN(engine=eng, metric="euclidean", alpha=1.0, algorithm="best", leaf_size=40)
    for kw in ({"min_cluster_size": 1}, {"min_cluster_size": 0}, {"min_samples": 0}, {"min_cluster_size": 2.5}):
        with pytest.raises(ValueError):
            mod.HDBSCAN(engine=eng, **kw)


def test_mirror_input_types(fake):
    mod, eng, seen = fake
    x = _pts(200, 10, seed=5)
    a = mod.HDBSCAN(min_cluster_size=5, engine=eng).fit(x).labels_
    b = mod.HDBSCAN(min_cluster_size=5, engine=eng).fit(x.astype(np.float64)).labels_
    c = mod.HDBSCAN(min_cluster_size=5, engine=eng).fit(torch.from_numpy(x)).labels_
    assert np.array_equal(a, b) and np.array_equal(a, c) and seen["x"].dtype == np.float32
    bad = x.astype(np.float64)
    bad[3, 4] += 1e-12                                            # not a float32 value
    with pytest.raises(ValueError, match="float32"):
        mod.HDBSCAN(engine=eng).fit(bad)
    for wrong in (x.astype(np.float16), x.astype(np.int32), torch.from_numpy(x).half()):
        with pytest.raises(ValueError):
            mod.HDBSCAN(engine=eng).fit(wrong)


# ---------------------------------------------------------------------------------------------
# device (K9)
# ---------------------------------------------------------------------------------------------
def _dev(engine, x):
    return torch.from_numpy(x).to(engine.device)


def _device_mst(engine, x, core_k):
    from karma_b200.hdbscan_ import mutual_reachability_mst
    r = mutual_reachability_mst(engine, _dev(engine, x), core_k)
    return r["core"].cpu().numpy(), r["edges"].cpu().numpy(), r["weights"].cpu().numpy()


def _grid_points(n, dim):
    return _pts(n, dim, seed=n + dim, coincident=min(n // 10, 50) if n > 20 else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [1, 2, 10, 64])
@pytest.mark.parametrize("n", [2, 3, 129, 4097, 20000])
def test_device_core_and_mst(engine, n, dim):
    """Core distances bit-identical to kneighbors at every (n, dim, core_k).  The MST edge for edge (order, orientation,
    weight bits) the oracle's canonical MST at every case up to 4097 points, and at 20 000 points for dim 2 and 10 with
    core_k 1, 3 and 16; its sorted weights equal sklearn's Prim MST's up to 4097 points.  Labels and probabilities of
    kb_hdbscan_labels equal the oracle's at min_cluster_size 2 up to 4097 points.  The reductions at 20 000 points keep
    the CPU references (single-threaded O(N^2 dim) Prim, the pure-Python tree) within minutes; the S1 50 k, tie-free
    end-to-end, HDBSCAN.fit and 1 M tests below cover the larger sizes and the other min_cluster_size values."""
    from sklearn.neighbors import NearestNeighbors
    x = _grid_points(n, dim)
    x64 = x.astype(np.float64)
    k = min(n, 128)
    ref = NearestNeighbors(n_neighbors=k, algorithm="kd_tree", n_jobs=-1).fit(x64).kneighbors(x64, k)[0]
    for core_k in (1, 2, 3, 16, 128):
        if core_k > n:
            continue
        core, edges, weights = _device_mst(engine, x, core_k)
        assert _bits_equal(core, ref[:, core_k - 1]), core_k
        if n <= 4097 or (dim in (2, 10) and core_k in (1, 3, 16)):
            e, w = ho.prim_mst(x, core)
            assert np.array_equal(edges, e) and _bits_equal(weights, w), core_k
            if n <= 4097:
                assert _bits_equal(np.sort(ho.sklearn_prim(x, core)[1]), weights), core_k
        labels, probs, nc = ho.tree_to_labels(edges, weights, 2) if n <= 4097 else (None, None, None)
        if labels is not None:
            from karma_b200.hdbscan_ import tree_labels
            got = tree_labels(edges, weights, 2)
            assert np.array_equal(got[0], labels) and _bits_equal(got[1], probs) and got[2] == nc


@pytest.mark.gpu
@pytest.mark.parametrize("allow_single", [False, True])
@pytest.mark.parametrize("mcs", [2, 5, 15])
def test_device_hdbscan_fit_equals_the_oracle(engine, mcs, allow_single):
    """The drop-in with the real engine: HDBSCAN.fit and cluster_embedding against the oracle's core distances,
    canonical MST and tree port, on blobs with coincident rows and on one blob (heavy ties)."""
    from karma_b200.hdbscan_ import HDBSCAN, cluster_embedding
    for x in (_pts(4000, 10, seed=21, coincident=40), _pts(3000, 10, seed=22, n_blobs=1)):
        _, core_k = ho.host_rules(len(x), mcs)
        core, e, w = ho.mst(x, core_k)
        labels, probs, nc = ho.tree_to_labels(e, w, mcs, allow_single)
        c = HDBSCAN(min_cluster_size=mcs, allow_single_cluster=allow_single, engine=engine).fit(x)
        assert np.array_equal(c.labels_, labels) and _bits_equal(c.probabilities_, probs)
        res = cluster_embedding(engine, _dev(engine, x), mcs, allow_single_cluster=allow_single)
        assert np.array_equal(res["labels"], labels) and _bits_equal(res["probabilities"], probs) and res["n_clusters"] == nc
        assert _bits_equal(res["mst"]["core"].cpu().numpy(), core)
        assert np.array_equal(res["mst"]["edges"].cpu().numpy(), e) and _bits_equal(res["mst"]["weights"].cpu().numpy(), w)


@pytest.fixture(scope="module")
def s1_embedding(engine):
    """The K8 embedding of a 50 k S1 pass: device_pass -> K7 -> K8 (200 epochs, dim 10, random init, seed 42)."""
    from karma_b200 import synth
    from karma_b200.engine import device_pass
    from karma_b200.umap_graph import build_graph
    from karma_b200.umap_layout import find_ab_params, layout_graph
    n = 50000
    asm = synth.make("S1", n)
    d_bases, d_offsets, d_key_len = engine.upload(asm.bases, asm.offsets, asm.key_len)
    r = device_pass(engine, d_bases, d_offsets, d_key_len, n, "5p6", n_neighbors=15, want_profile=False)
    g = build_graph(engine, r["idx"].contiguous(), r["dist"].contiguous())
    a, b = find_ab_params(1.0, 0.1)
    init = torch.rand(n, 10, device=engine.device, generator=torch.Generator(engine.device).manual_seed(42)) * 20 - 10
    return layout_graph(engine, g, init, 200, a, b, 42).cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("mcs", [2, 15])
def test_device_s1_embedding(engine, s1_embedding, mcs):
    from karma_b200.hdbscan_ import cluster_embedding
    x = s1_embedding
    res = cluster_embedding(engine, _dev(engine, x), mcs)
    core = res["mst"]["core"].cpu().numpy()
    edges, weights = res["mst"]["edges"].cpu().numpy(), res["mst"]["weights"].cpu().numpy()
    assert _bits_equal(core, ho.core_distances(x, mcs + 1))
    e, w = ho.prim_mst(x, core)
    assert np.array_equal(edges, e) and _bits_equal(weights, w)
    assert _bits_equal(np.sort(ho.sklearn_prim(x, core)[1]), weights)
    labels, probs, nc = ho.tree_to_labels(edges, weights, mcs)
    assert np.array_equal(res["labels"], labels) and _bits_equal(res["probabilities"], probs) and res["n_clusters"] == nc
    print("S1 50 k K8 embedding, min_cluster_size %d: %d clusters, %d noise" % (mcs, nc, int((labels == -1).sum())))


@pytest.mark.gpu
@pytest.mark.parametrize("n,blobs,mcs", [(5000, 8, 5), (20000, 30, 15), (3000, 1, 2)])
def test_device_end_to_end_against_sklearn_hdbscan(engine, n, blobs, mcs):
    """Tie-free inputs (core_k = 1, distinct MST weights): labels equal up to a bijection, probabilities bit-identical."""
    from sklearn.cluster import HDBSCAN as SkHDBSCAN
    from karma_b200.hdbscan_ import tree_labels
    x = _pts(n, 10, seed=7, n_blobs=blobs)
    _, edges, weights = _device_mst(engine, x, 1)
    assert len(np.unique(weights)) == len(weights)
    labels, probs, nc = tree_labels(edges, weights, mcs)
    sk = SkHDBSCAN(min_cluster_size=mcs, min_samples=1, algorithm="kd_tree").fit(x.astype(np.float64))
    assert _bits_equal(probs, sk.probabilities_)
    pairs = set(zip(labels.tolist(), sk.labels_.tolist()))
    assert len(pairs) == len(set(labels.tolist())) == len(set(sk.labels_.tolist()))
    assert (-1, -1) in pairs or -1 not in labels
    assert nc == len(set(sk.labels_.tolist()) - {-1})


@pytest.mark.gpu
def test_device_is_deterministic(engine):
    x = _pts(20000, 10, seed=9, n_blobs=1, coincident=50)
    first = [a.tobytes() for a in _device_mst(engine, x, 3)]
    assert [a.tobytes() for a in _device_mst(engine, x, 3)] == first
    _device_mst(engine, _pts(3000, 2, seed=1), 16)
    assert [a.tobytes() for a in _device_mst(engine, x, 3)] == first


@pytest.mark.gpu
def test_device_1m(engine):
    """1 M x 10 runs to the end; kb_hdbscan_labels accepts its N - 1 edges (a sorted spanning tree), and its labels and
    probabilities equal scikit-learn's tree_to_labels on the device MST."""
    from karma_b200.hdbscan_ import tree_labels
    x = _pts(1000000, 10, seed=11, n_blobs=30)
    core, edges, weights = _device_mst(engine, x, 3)
    assert edges.shape == (999999, 2) and np.isfinite(core).all()
    for mcs in (2, 15):
        labels, probs, nc = tree_labels(edges, weights, mcs)
        ref_labels, ref_probs = ho.sklearn_tree_to_labels(edges, weights, mcs)
        assert np.array_equal(labels, ref_labels) and _bits_equal(probs, ref_probs)
        print("1 M x 10, min_cluster_size %d: %d clusters, %d noise" % (mcs, nc, int((labels == -1).sum())))


@pytest.mark.gpu
def test_device_refusals(engine):
    from karma_b200 import _lib
    from karma_b200.hdbscan_ import mutual_reachability_mst
    x = _pts(300, 10, seed=2)

    def refused(code, pts, core_k):
        with pytest.raises(_lib.KarmaB200Error) as e:
            mutual_reachability_mst(engine, _dev(engine, pts), core_k)
        assert e.value.code == code

    for v in (np.nan, np.inf, -np.inf):
        bad = x.copy()
        bad[17, 3] = v
        refused(_lib.KB_EINVAL, bad, 3)
    refused(_lib.KB_EINVAL, x[:1], 1)
    refused(_lib.KB_EINVAL, x[:5], 6)
    refused(_lib.KB_EINVAL, x, 0)
    refused(_lib.KB_EUNSUPPORTED, _pts(300, 65, seed=2), 3)
    refused(_lib.KB_EUNSUPPORTED, x, 129)
    core, edges, weights = _device_mst(engine, x, 3)             # the context is usable afterwards
    assert np.array_equal(edges, ho.prim_mst(x, core)[0])
