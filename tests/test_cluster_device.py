"""KmerClustering's device route: K7 -> K10 -> K8 -> K9 from the pass's own lists (karma_b200.cluster)."""
import functools
import os
import sys
import types
import warnings

import numpy as np
import pytest
import scipy.sparse
import torch

from karma_b200 import cluster
from karma_b200.kmer import KmerClustering

FAKE = types.SimpleNamespace(device=torch.device("cpu"))


def _state(rs):
    st = rs.get_state()
    return st[1].tobytes(), st[2], st[3], st[4]


# ---------------------------------------------------------------------------------------------
# route selection


def test_route_from_keyword_environment_and_default(monkeypatch, tmp_path):
    monkeypatch.delenv("KARMA_B200_CLUSTER", raising=False)
    assert KmerClustering({}, str(tmp_path), "5p6", 1).cluster_on == "host"
    assert KmerClustering({}, str(tmp_path), "5p6", 1, cluster_on="device").cluster_on == "device"
    monkeypatch.setenv("KARMA_B200_CLUSTER", "device")
    assert KmerClustering({}, str(tmp_path), "5p6", 1).cluster_on == "device"
    assert KmerClustering({}, str(tmp_path), "5p6", 1, cluster_on="host").cluster_on == "host"   # the keyword wins
    monkeypatch.setenv("KARMA_B200_CLUSTER", "")
    assert KmerClustering({}, str(tmp_path), "5p6", 1).cluster_on == "host"
    monkeypatch.setenv("KARMA_B200_CLUSTER", "gpu")
    with pytest.raises(ValueError, match="KARMA_B200_CLUSTER"):
        KmerClustering({}, str(tmp_path), "5p6", 1)
    monkeypatch.delenv("KARMA_B200_CLUSTER")
    with pytest.raises(ValueError, match="cluster_on"):
        KmerClustering({}, str(tmp_path), "5p6", 1, cluster_on="Device")


# ---------------------------------------------------------------------------------------------
# cluster_from_lists' host rules, with the stages stubbed


@pytest.fixture
def stages(monkeypatch):
    """The device stages of cluster_from_lists replaced by CPU stubs that record their arguments and the generator's
    state.  The spectral stub draws what 0.3.9's spectral_layout (uniform fallback) and _init_embedding draw."""
    seen = {}

    def build_graph(engine, idx, dist, local_connectivity=1.0, set_op_mix_ratio=1.0):
        seen["graph"] = dict(n=idx.shape[0], local_connectivity=local_connectivity, set_op_mix_ratio=set_op_mix_ratio,
                             state=_state(seen["rs"]) if "rs" in seen else None)
        return "GRAPH"

    def spectral_init(engine, graph, dim, n_epochs, random_state, data=None, return_build=False):
        n = seen["graph"]["n"]
        seen["spectral"] = dict(graph=graph, dim=dim, n_epochs=n_epochs, data=data, state=_state(random_state))
        u = random_state.random_sample((n, dim))
        init = (u * (10.0 / np.abs(u).max())).astype(np.float32) + \
            random_state.normal(scale=0.0001, size=[n, dim]).astype(np.float32)
        return torch.from_numpy(init), {"n_comp": 1, "stats": np.arange(6)}

    def layout_graph(engine, graph, embedding, n_epochs, a, b, seed, gamma=1.0, initial_alpha=1.0,
                     negative_sample_rate=5.0):
        seen["layout"] = dict(n_epochs=n_epochs, a=a, b=b, seed=seed, gamma=gamma, initial_alpha=initial_alpha,
                              negative_sample_rate=negative_sample_rate)
        return embedding

    def mutual_reachability_mst(engine, x, core_k):
        seen["core_k"] = core_k
        n = x.shape[0]
        return {"edges": torch.zeros((n - 1, 2), dtype=torch.int32), "weights": torch.zeros(n - 1, dtype=torch.float64)}

    def tree_labels(edges, weights, min_cluster_size, allow_single_cluster=False):
        seen["hdbscan"] = dict(min_cluster_size=min_cluster_size, allow_single_cluster=allow_single_cluster)
        n = edges.shape[0] + 1
        return np.arange(n, dtype=np.int32) % 3 - 1, np.linspace(0, 1, n), 2

    for name, fn in (("build_graph", build_graph), ("spectral_init", spectral_init), ("layout_graph", layout_graph),
                     ("mutual_reachability_mst", mutual_reachability_mst), ("tree_labels", tree_labels),
                     ("_synchronize", lambda engine: None)):
        monkeypatch.setattr(cluster, name, fn)
    return seen


def _lists(n, k, seed=0):
    rng = np.random.default_rng(seed)
    idx = np.concatenate([np.arange(n)[:, None], rng.integers(0, n, (n, k - 1))], axis=1).astype(np.int32)
    dst = np.sort(rng.random((n, k)).astype(np.float32), axis=1)
    dst[:, 0] = 0
    return idx, dst


def test_random_state_is_consumed_as_route_2_consumes_it(stages, monkeypatch):
    """The generator's state at each stage equals route 2's (umap_embedding through the 0.3.9 stubs, with the
    library's simplicial_set_embedding mirror and a spectral_layout stub drawing as the device stub draws)."""
    from karma_b200 import umap_layout
    from karma_b200.kmer import umap_embedding
    from karma_b200.umap_layout import fold_seed
    from tests.test_host_logic import _fake_umap_039

    n, k, dim = 40, 3, 4
    idx, dst = _lists(n, k)
    prof = np.random.default_rng(1).random((n, 7))
    route2 = {}
    fake = _fake_umap_039({})

    def fss(X, n_neighbors, random_state, metric, metric_kwds={}, knn_indices=None, knn_dists=None, angular=False,
            set_op_mix_ratio=1.0, local_connectivity=1.0, verbose=False):
        route2["graph"] = _state(random_state)
        ring = np.arange(n)
        return scipy.sparse.csr_matrix((np.full(n, 0.5), (ring, (ring + 1) % n)), shape=(n, n))

    def spectral_layout(data, graph, dim, random_state, metric="euclidean", metric_kwds={}):
        route2["spectral"] = _state(random_state)
        return random_state.random_sample((graph.shape[0], dim))

    def layout(engine, graph, embedding, n_epochs, a, b, seed, gamma, initial_alpha, negative_sample_rate):
        route2["seed"], route2["init"] = seed, embedding.numpy().copy()
        return embedding

    monkeypatch.setattr(umap_layout, "layout_graph", layout)
    fake.umap_.fuzzy_simplicial_set = fss
    fake.umap_.simplicial_set_embedding = functools.partial(umap_layout.simplicial_set_embedding, engine=FAKE,
                                                            spectral_layout=spectral_layout)
    rs2 = np.random.RandomState(42)
    _, route = umap_embedding(prof, idx, dst, {"n_neighbors": k, "n_components": dim, "min_dist": 0, "random_state": rs2},
                              umap_module=fake)
    assert route == "fuzzy_simplicial_set"

    rs = np.random.RandomState(42)
    stages["rs"] = rs
    out = cluster.cluster_from_lists(FAKE, torch.from_numpy(idx), torch.from_numpy(dst), "PROFILE", dim, 0, rs, 2)
    assert stages["graph"]["state"] == route2["graph"] == _state(np.random.RandomState(42))
    assert stages["spectral"]["state"] == route2["spectral"]
    assert stages["layout"]["seed"] == route2["seed"]
    assert np.array_equal(out["embedding"].numpy(), route2["init"])
    assert _state(rs) == _state(rs2)
    # the seed is the fold of the three words drawn right after the initialisation
    ref = np.random.RandomState(42)
    ref.random_sample((n, dim))
    ref.normal(scale=0.0001, size=[n, dim])
    assert stages["layout"]["seed"] == fold_seed(ref.randint(umap_layout.INT32_MIN, umap_layout.INT32_MAX, 3))
    # karma's UMAP arguments: the fixed values route 2 passes
    assert stages["graph"]["local_connectivity"] == 1.0 and stages["graph"]["set_op_mix_ratio"] == 1.0
    assert stages["spectral"]["data"] == "PROFILE" and stages["spectral"]["dim"] == dim
    lay = stages["layout"]
    assert (lay["gamma"], lay["initial_alpha"], lay["negative_sample_rate"]) == (1.0, 1.0, 5)
    assert (lay["a"], lay["b"]) == umap_layout.find_ab_params(1.0, 0)
    # an integer seed builds the same generator (sklearn's check_random_state, as UMAP.fit)
    again = cluster.cluster_from_lists(FAKE, torch.from_numpy(idx), torch.from_numpy(dst), None, dim, 0, 42, 2)
    assert again["embedding"].numpy().tobytes() == out["embedding"].numpy().tobytes()


@pytest.mark.parametrize("n,epochs", [(10000, 500), (10001, 200)])
def test_n_epochs_rule(stages, n, epochs):
    idx, dst = _lists(n, 2)
    out = cluster.cluster_from_lists(FAKE, torch.from_numpy(idx), torch.from_numpy(dst), None, 2, 0, 1, 2)
    assert stages["spectral"]["n_epochs"] == stages["layout"]["n_epochs"] == out["n_epochs"] == epochs
    assert set(out["ms"]) == {"graph", "spectral", "layout", "hdbscan_mst", "hdbscan_tree"}
    assert out["spectral"] == {"n_comp": 1, "lanczos_steps": 0, "restarts": 1, "meta_steps": 2, "meta_restarts": 3}


@pytest.mark.parametrize("mcs,want", [(1, (5, True, 6)), (2, (2, False, 3)), (15, (15, False, 16))])
def test_min_cluster_size_rule(stages, mcs, want):
    """karma: min_cluster_size 1 -> HDBSCAN(allow_single_cluster=True) at hdbscan's default size 5."""
    idx, dst = _lists(50, 2)
    out = cluster.cluster_from_lists(FAKE, torch.from_numpy(idx), torch.from_numpy(dst), None, 2, 0, 1, mcs)
    got = stages["hdbscan"]
    assert (got["min_cluster_size"], got["allow_single_cluster"], stages["core_k"]) == want
    assert out["labels"].dtype == np.intp and out["probabilities"].dtype == np.float64 and out["n_clusters"] == 2


# ---------------------------------------------------------------------------------------------
# KmerClustering.run on the device route, with the pass and the clustering stubbed

SEQS = {">c0 len=5": "ACGTA", ">c1": "ACGTT", ">c2": "GGGGG", ">c3": "TTTTT", ">c4 x": "AAAAC"}
LABELS = np.array([0, 0, -1, 1, 1])
PROBS = np.array([1.0, 0.5, 0.0, 1.0, 0.7])


def _device_clustering(monkeypatch, out_dir, seqs=SEQS, labels=LABELS, probs=PROBS):
    k = KmerClustering(seqs, str(out_dir), "5p6", 1, cluster_on="device")
    seen = {}

    def fake_profile(n_neighbors=None, host_profile=True):
        seen["profile"] = (n_neighbors, host_profile)
        n = len(seqs)
        k._d_knn = (torch.zeros((n, n_neighbors), dtype=torch.int32), torch.zeros((n, n_neighbors)))
        return "D_PROFILE"

    def fake_cluster(engine, d_idx, d_dist, d_profile, n_components, min_dist, random_state, min_cluster_size):
        seen["cluster"] = dict(k=d_idx.shape[1], d_profile=d_profile, n_components=n_components, min_dist=min_dist,
                               random_state=random_state, min_cluster_size=min_cluster_size)
        return {"labels": labels, "probabilities": probs, "n_clusters": int(labels.max()) + 1,
                "embedding": torch.zeros((len(seqs), n_components)), "n_epochs": 500, "ms": {"graph": 1.0},
                "spectral": {"n_comp": 1}}

    monkeypatch.setattr(k, "_KmerClustering__calc_kmer_profile", fake_profile)
    monkeypatch.setattr(k, "_get_engine", lambda: FAKE)
    monkeypatch.setattr(cluster, "cluster_from_lists", fake_cluster)
    return k, seen


def test_files_are_the_host_routes_given_the_same_labels(tmp_path, monkeypatch):
    host_dir, dev_dir = tmp_path / "host", tmp_path / "device"
    host_dir.mkdir()
    dev_dir.mkdir()

    class UMAP:
        def __init__(self, **kw):
            pass

        def fit_transform(self, x):
            return x[:, :2]

    class HDBSCAN:
        def __init__(self, **kw):
            pass

        def fit(self, emb):
            self.labels_, self.probabilities_ = LABELS.astype(np.intp), PROBS
            return self

    monkeypatch.setitem(sys.modules, "umap", types.SimpleNamespace(UMAP=UMAP))
    monkeypatch.setitem(sys.modules, "hdbscan", types.SimpleNamespace(HDBSCAN=HDBSCAN))
    host = KmerClustering(SEQS, str(host_dir), "5p6", 1, cluster_on="host")

    def fake_profile(n_neighbors=None):
        host.knn_indices = np.zeros((5, n_neighbors), dtype=np.int32)
        host.knn_dists = np.zeros((5, n_neighbors), dtype=np.float32)
        return np.eye(5)
    monkeypatch.setattr(host, "_KmerClustering__calc_kmer_profile", fake_profile)
    host.run(neighbors=2, components=10, dist=0, r_state=42, min_cluster_size=2)

    dev, seen = _device_clustering(monkeypatch, dev_dir, labels=LABELS.astype(np.intp))
    dev.run(neighbors=2, components=10, dist=0, r_state=42, min_cluster_size=2)
    assert seen["profile"] == (2, False)
    assert seen["cluster"] == dict(k=2, d_profile="D_PROFILE", n_components=10, min_dist=0, random_state=42,
                                   min_cluster_size=2)
    for name in ("cluster.txt", "eval.txt"):
        assert (host_dir / name).read_bytes() == (dev_dir / name).read_bytes(), name
    assert dev.clusters == host.clusters and dev.unlabeled_cluster == host.unlabeled_cluster
    assert dev.umap_route == "device" and dev.embedding.shape == (5, 10) and dev.embedding.dtype == np.float32
    assert set(dev.stage_ms) == {"pass", "graph", "files"} and dev._d_knn is None
    # a second run resumes from cluster.txt, as the host route does
    again = KmerClustering(SEQS, str(dev_dir), "5p6", 1, cluster_on="device")
    again.run(neighbors=2, components=10, dist=0, r_state=42, min_cluster_size=2)
    assert again.clusters == dev.clusters and again.unlabeled_cluster == dev.unlabeled_cluster


def test_n_neighbors_at_least_n_is_truncated_with_umaps_warning(tmp_path, monkeypatch):
    k, seen = _device_clustering(monkeypatch, tmp_path)
    with pytest.warns(UserWarning, match=r"^n_neighbors is larger than the dataset size; truncating to X.shape\[0\] - 1$"):
        k.run(neighbors=5, components=2, dist=0, r_state=1, min_cluster_size=2)
    assert seen["profile"] == (4, False) and seen["cluster"]["k"] == 4
    assert open(k.output_eval).read().split("\n")[1].split("\t")[1] == "5"     # eval.txt keeps the value given
    assert cluster.check_arguments(5, 4, 2, 2) == 4


@pytest.mark.parametrize("seqs,neighbors,components,mcs,match", [
    ({">a": "ACGTA"}, 2, 2, 2, "at least 2"),
    ({}, 2, 2, 2, "at least 2"),
    (SEQS, 2.0, 2, 2, "n_neighbors"),
    (SEQS, True, 2, 2, "n_neighbors"),
    (SEQS, 0, 2, 2, "n_neighbors"),
    (SEQS, 2, 0, 2, "n_components"),
    (SEQS, 2, 65, 2, "n_components"),
    (SEQS, 2, 2.0, 2, "n_components"),
    (SEQS, 2, 2, 0, "min_cluster_size"),
])
def test_argument_errors_before_any_gpu_work(tmp_path, seqs, neighbors, components, mcs, match):
    k = KmerClustering(seqs, str(tmp_path), "5p6", 1, cluster_on="device")

    def no_pass(*a, **kw):
        raise AssertionError("the pass must not start")
    k._KmerClustering__calc_kmer_profile = no_pass
    k._get_engine = no_pass
    with pytest.raises(ValueError, match=match):
        k.run(neighbors=neighbors, components=components, dist=0, r_state=1, min_cluster_size=mcs)
    assert not os.path.exists(k.output_file)


# ---------------------------------------------------------------------------------------------
# GPU


@pytest.fixture(scope="module")
def assemblies():
    from karma_b200 import synth
    cache = {}

    def get(n):
        if n not in cache:
            cache[n] = synth.make("S1", n).as_dict()
        return cache[n]
    return get


def _mirror_modules(engine):
    """The library's own mirrors as umap-learn 0.3.9 and hdbscan 0.8.22: run() on the host route then goes through
    umap_embedding's route 2 (fuzzy_simplicial_set, then simplicial_set_embedding) and the HDBSCAN mirror."""
    from karma_b200 import hdbscan_, umap_graph, umap_layout, umap_spectral
    from tests.test_host_logic import _fake_umap_039
    umap_ = types.SimpleNamespace(
        fuzzy_simplicial_set=functools.partial(umap_graph.fuzzy_simplicial_set, engine=engine),
        simplicial_set_embedding=functools.partial(
            umap_layout.simplicial_set_embedding, engine=engine,
            spectral_layout=functools.partial(umap_spectral.spectral_layout, engine=engine)),
        find_ab_params=umap_layout.find_ab_params)
    umap = types.SimpleNamespace(UMAP=_fake_umap_039({}).UMAP, umap_=umap_)
    return umap, types.SimpleNamespace(HDBSCAN=functools.partial(hdbscan_.HDBSCAN, engine=engine))


def _run(engine, seqs, out_dir, route, kmer_size="5p6", neighbors=2, components=10, mcs=2, r_state=42):
    os.makedirs(out_dir, exist_ok=True)
    k = KmerClustering(seqs, str(out_dir), kmer_size, 1, cluster_on=route)
    k._engine = engine
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")             # umap's meta-embedding notice
        k.run(neighbors=neighbors, components=components, dist=0, r_state=r_state, min_cluster_size=mcs)
    files = tuple(open(os.path.join(out_dir, f), "rb").read() for f in ("cluster.txt", "eval.txt"))
    return k, files


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5000, 20000])
@pytest.mark.parametrize("neighbors", [2, 15])
@pytest.mark.parametrize("components", [2, 10])
@pytest.mark.parametrize("mcs", [1, 2, 15])
def test_same_bytes_as_route_2(engine, assemblies, tmp_path, monkeypatch, n, neighbors, components, mcs):
    umap, hdbscan = _mirror_modules(engine)
    monkeypatch.setitem(sys.modules, "umap", umap)
    monkeypatch.setitem(sys.modules, "hdbscan", hdbscan)
    seqs = assemblies(n)
    host, want = _run(engine, seqs, tmp_path / "host", "host", neighbors=neighbors, components=components, mcs=mcs)
    assert host.umap_route == "fuzzy_simplicial_set"
    _, got = _run(engine, seqs, tmp_path / "device", "device", neighbors=neighbors, components=components, mcs=mcs)
    assert got[0] == want[0] and got[1] == want[1]


@pytest.mark.gpu
def test_same_bytes_as_route_2_integer_k(engine, assemblies, tmp_path, monkeypatch):
    umap, hdbscan = _mirror_modules(engine)
    monkeypatch.setitem(sys.modules, "umap", umap)
    monkeypatch.setitem(sys.modules, "hdbscan", hdbscan)
    seqs = assemblies(5000)
    host, want = _run(engine, seqs, tmp_path / "host", "host", kmer_size=6)
    assert host.umap_route == "fuzzy_simplicial_set"
    _, got = _run(engine, seqs, tmp_path / "device", "device", kmer_size=6)
    assert got == want


def _device_lists(engine, seqs, kmer_size, k):
    from karma_b200.engine import profile_and_knn
    probe = KmerClustering(seqs, "/nonexistent", kmer_size, 1)
    bases, offsets, key_len = probe._pack()
    return profile_and_knn(engine, bases, offsets, key_len, kmer_size, n_neighbors=k, host_profile=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n,neighbors,components,mcs", [(5000, 15, 10, 1), (20000, 2, 10, 2)])
def test_composition_equals_the_stages_one_by_one(engine, assemblies, n, neighbors, components, mcs):
    from karma_b200.hdbscan_ import cluster_embedding
    from karma_b200.umap_graph import build_graph
    from karma_b200.umap_layout import INT32_MAX, INT32_MIN, find_ab_params, fold_seed, layout_graph
    from karma_b200.umap_spectral import spectral_init
    res = _device_lists(engine, assemblies(n), "5p6", neighbors)
    assert res["profile"] is None and res["knn_idx"].shape == (n, neighbors)
    assert res["d_idx"].is_cuda and res["d_dist"].is_cuda and res["d_profile"].dtype == torch.float64
    assert np.array_equal(res["d_idx"].cpu().numpy(), res["knn_idx"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = cluster.cluster_from_lists(engine, res["d_idx"], res["d_dist"], res["d_profile"], components, 0,
                                         np.random.RandomState(42), mcs)
        rs = np.random.RandomState(42)
        a, b = find_ab_params(1.0, 0)
        g = build_graph(engine, res["d_idx"], res["d_dist"])
        epochs = 500 if n <= 10000 else 200
        init = spectral_init(engine, g, components, epochs, rs, data=res["d_profile"])
        emb = layout_graph(engine, g, init, epochs, a, b, fold_seed(rs.randint(INT32_MIN, INT32_MAX, 3)))
        ref = cluster_embedding(engine, emb, 5 if mcs == 1 else mcs, allow_single_cluster=(mcs == 1))
    assert torch.equal(out["embedding"], emb)
    assert np.array_equal(out["labels"], ref["labels"]) and out["n_clusters"] == ref["n_clusters"]
    assert out["probabilities"].tobytes() == ref["probabilities"].tobytes()
    print("S1 %d k=%d dim=%d mcs=%d: %d clusters, ms %s, spectral %s"
          % (n, neighbors, components, mcs, out["n_clusters"], out["ms"], out["spectral"]))


@pytest.mark.gpu
def test_two_runs_give_identical_files(engine, assemblies, tmp_path):
    seqs = assemblies(20000)
    a, fa = _run(engine, seqs, tmp_path / "a", "device")
    b, fb = _run(engine, seqs, tmp_path / "b", "device")
    assert fa == fb and a.embedding.tobytes() == b.embedding.tobytes()


def _gene(name):
    return name.split("_")[1]                      # TRINITY_DN{gene}_c0_g1_i{iso}


@pytest.mark.gpu
def test_quality_on_known_gene_families(engine, assemblies, tmp_path):
    """S1 20 k at karma's defaults (n_neighbors 2, 10 components, min_dist 0, random_state 42, min_cluster_size 2).
    Purity: the share of clustered contigs whose cluster's most frequent gene is their own gene.  The bounds were set
    from the first B200 run (4 430 clusters, purity 0.8703, noise fraction 0.0697) with a small margin: the route is
    deterministic, so a change beyond the margin is a change of the result, not noise."""
    k, _ = _run(engine, assemblies(20000), tmp_path, "device")
    clustered = sum(len(c) for c in k.clusters)
    agree = sum(max(np.unique([_gene(m) for m in c], return_counts=True)[1]) for c in k.clusters)
    purity = agree / clustered
    noise = len(k.unlabeled_cluster[0]) / 20000
    print("S1 20k: %d clusters, purity %.4f, noise fraction %.4f" % (len(k.clusters), purity, noise))
    assert purity >= 0.85 and noise <= 0.08


@pytest.mark.gpu
def test_exotic_bytes_take_the_general_path_and_still_cluster(engine, assemblies, tmp_path, monkeypatch):
    seqs = dict(assemblies(5000))
    for i, name in enumerate(list(seqs)[::97]):
        s = seqs[name]
        seqs[name] = s[:50] + "N" + s[51:100] + "acgt" + s[104:] if i % 2 else s[:30] + "NNRY" + s[34:]
    umap, hdbscan = _mirror_modules(engine)
    monkeypatch.setitem(sys.modules, "umap", umap)
    monkeypatch.setitem(sys.modules, "hdbscan", hdbscan)
    host, want = _run(engine, seqs, tmp_path / "host", "host")
    assert host.umap_route == "fuzzy_simplicial_set" and any(not set(c) <= set("ACGT") for c in host.kmers)
    dev, got = _run(engine, seqs, tmp_path / "device", "device")
    assert got == want and len(dev.clusters) > 0


@pytest.mark.gpu
def test_more_components_than_the_meta_embedding_serves_are_refused(engine):
    """Self-only lists give a graph without edges: every one of 70 000 rows is its own component."""
    from karma_b200 import _lib
    n = 70000
    d_idx = torch.arange(n, dtype=torch.int32, device=engine.device)[:, None].contiguous()
    d_dist = torch.zeros((n, 1), dtype=torch.float32, device=engine.device)
    prof = torch.rand((n, 4), dtype=torch.float64, device=engine.device)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        with pytest.raises(_lib.KarmaB200Error) as e:
            cluster.cluster_from_lists(engine, d_idx, d_dist, prof, 2, 0, 42, 2)
    assert e.value.code == _lib.KB_EUNSUPPORTED and "65536" in str(e.value)
