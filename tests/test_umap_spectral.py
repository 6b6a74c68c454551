"""K10: UMAP's spectral initialisation (umap-learn 0.3.9 spectral_layout) on the device, disconnected graphs included."""
import sys
import types
import warnings

import numpy as np
import pytest
import scipy.sparse
import scipy.sparse.linalg
import torch

from oracle import umap_spectral_oracle as so


def _cliques(sizes, order=None):
    """Disjoint cliques of the given sizes (weights 0.5); vertices renumbered by ``order``."""
    n = sum(sizes)
    rows, cols, o = [], [], 0
    for s in sizes:
        for a in range(o, o + s):
            for b in range(o, o + s):
                if a != b:
                    rows.append(a)
                    cols.append(b)
        o += s
    order = np.arange(n) if order is None else np.asarray(order)
    return scipy.sparse.csr_matrix((np.full(len(rows), 0.5), (order[rows], order[cols])), shape=(n, n))


def _weighted(sizes, seed):
    """Disjoint components of the given sizes, each a ring with random chords and random weights (distinct eigenvalues),
    vertices shuffled."""
    rs = np.random.RandomState(seed)
    n = sum(sizes)
    order = rs.permutation(n)
    rows, cols, o = [], [], 0
    for s in sizes:
        if s > 1:
            i = np.arange(s)
            a, b = np.r_[i, rs.randint(0, s, 2 * s)], np.r_[(i + 1) % s, rs.randint(0, s, 2 * s)]
            keep = a != b
            rows.append(o + a[keep])
            cols.append(o + b[keep])
        o += s
    a, b = np.concatenate(rows), np.concatenate(cols)
    g = scipy.sparse.coo_matrix((rs.uniform(0.1, 1.0, a.size), (order[a], order[b])), shape=(n, n)).tocsr()
    return (g + g.T).tocsr()


def _ring(n):
    i = np.arange(n)
    return scipy.sparse.csr_matrix((np.full(2 * n, 0.5), (np.r_[i, i], np.r_[(i + 1) % n, (i - 1) % n])), shape=(n, n))


def _exact_solve(g, dim, rows):
    return so.exact_eigenvectors(g, dim)[0]


# ---------------------------------------------------------------------------------------------
# the oracle's rules on hand graphs
# ---------------------------------------------------------------------------------------------
def test_uniform_is_low_plus_range_times_random_sample():
    """The device takes random_sample draws and applies numpy's uniform arithmetic, low + (high - low) * u."""
    for r in (0.37, 1e-3, 3.3e-10, 10.0):
        a, b = np.random.RandomState(5), np.random.RandomState(5)
        x = a.uniform(low=-r, high=r, size=(7, 3))
        assert np.array_equal(x, -r + (r - (-r)) * b.random_sample((7, 3)))
        assert a.random_sample() == b.random_sample()


def test_two_components_take_the_plus_minus_eye_meta():
    g = _cliques([6, 5], order=np.random.RandomState(0).permutation(11))
    assert np.array_equal(so.eye_meta(2, 2), [[1.0, 0.0], [-1.0, 0.0]])
    with pytest.warns(UserWarning, match="2 separate connected components"):
        out = so.spectral_layout_exact(None, g, 2, np.random.RandomState(1))
    _, labels = so.components(g)
    ranges = so.data_range_exact(so.eye_meta(2, 2))
    assert np.array_equal(ranges, [1.0, 1.0])
    for c, meta in enumerate(so.eye_meta(2, 2)):
        rows = np.flatnonzero(labels == c)
        v = so.exact_eigenvectors(g[rows][:, rows], 2)[0]
        want = (v * (1.0 / np.abs(v).max()) + meta).astype(np.float32)
        assert np.array_equal(out[rows], want)


def test_small_components_take_draws_in_label_order():
    dim = 2
    order = np.random.RandomState(3).permutation(9)
    g = _cliques([1, 2, 6], order=order)                # 2 * dim = 4: the first two draw, the third is solved
    n_comp, labels = so.components(g)
    assert n_comp == 3
    rs, ref = np.random.RandomState(7), np.random.RandomState(7)
    with pytest.warns(UserWarning):
        out = so.spectral_layout_exact(None, g, dim, rs)
    meta = so.eye_meta(3, dim)
    ranges = so.data_range_exact(meta)
    sizes = np.bincount(labels)
    assert sorted(sizes) == [1, 2, 6] and sizes[0] == 6     # labels follow the smallest vertex, not the construction
    for c in np.flatnonzero(sizes < 2 * dim):
        rows = np.flatnonzero(labels == c)
        want = (ref.uniform(low=-ranges[c], high=ranges[c], size=(rows.size, dim)) + meta[c]).astype(np.float32)
        assert np.array_equal(out[rows], want)
    assert rs.random_sample() == ref.random_sample()      # the solved component draws nothing


def test_more_than_two_dim_components_take_component_layout():
    dim = 2
    data = np.random.RandomState(0).rand(10, 6).astype(np.float32)
    calls = []

    def meta_fn(data, n_comp, labels, dim):
        calls.append(n_comp)
        return so.component_layout(data, n_comp, labels, dim)
    with pytest.warns(UserWarning):
        so.spectral_layout_flow(data[:8], _cliques([2, 2, 2, 2]), dim, np.random.RandomState(0), _exact_solve, meta_fn,
                                lambda m, c: so.data_range_exact(m)[c])
        assert calls == []                                 # 4 = 2 * dim components: +-eye
        so.spectral_layout_flow(data, _cliques([2, 2, 2, 2, 2]), dim, np.random.RandomState(0), _exact_solve, meta_fn,
                                lambda m, c: so.data_range_exact(m)[c])
    assert calls == [5]
    meta = so.component_layout(data, 5, np.repeat(np.arange(5), 2), dim)
    assert meta.max() == 1.0 and meta.shape == (5, dim)


def test_centroids_are_numpys_float32_mean():
    rs = np.random.RandomState(1)
    data = rs.rand(300, 7).astype(np.float32)
    labels = rs.randint(0, 9, 300)
    cent = so.centroids(data, labels, 9)
    for c in range(9):
        assert np.array_equal(cent[c], data[labels == c].mean(axis=0).astype(np.float64))
        acc = np.zeros(7, np.float32)
        for row in data[labels == c]:
            acc = acc + row                                  # the float32 sum in row order the device takes
        assert np.array_equal(cent[c], (acc.astype(np.float64) / (labels == c).sum()).astype(np.float32))


def test_sign_rule_is_sklearns():
    from sklearn.utils.extmath import _deterministic_vector_sign_flip
    rs = np.random.RandomState(2)
    for _ in range(20):
        u = rs.randn(40, 5)
        u[rs.randint(40), 0] = -np.abs(u).max() - 1.0        # a negative extreme
        u[3, 1], u[7, 1] = -5.0, 5.0                         # a tie: the first occurrence decides
        u[3, 1] = -np.abs(u[:, 1]).max() - 1.0
        u[7, 1] = -u[3, 1]
        assert np.array_equal(so.sign_flip(u), _deterministic_vector_sign_flip(u.T).T)
        assert so.sign_flip(u)[3, 1] > 0


def test_exact_eigenvectors_on_a_clique_pair_are_unit_and_signed():
    g = _cliques([40])
    g = g + scipy.sparse.random(40, 40, density=0.2, random_state=np.random.RandomState(4))
    g = (g + g.T).tocsr()
    v, w = so.exact_eigenvectors(g, 3)
    lap = so.laplacian(g).toarray()
    assert np.allclose(np.linalg.norm(v, axis=0), 1.0, atol=1e-14)
    for k in range(3):
        assert np.abs(lap @ v[:, k] - w[k + 1] * v[:, k]).max() < 1e-12
        assert v[np.argmax(np.abs(v[:, k])), k] > 0


@pytest.fixture(scope="module")
def s1_5k_k2():
    """S1 5 k, exact sklearn kNN at n_neighbors 2, the oracle's K7 graph pruned at max / 500, and its meta points."""
    from sklearn.neighbors import NearestNeighbors
    from karma_b200 import synth
    from oracle import kmer_oracle as ko
    from oracle import umap_graph_oracle as ugo
    asm = synth.make("S1", 5000)
    c, _ = ko.counts_mode(asm.bases, asm.offsets, "5p6")
    prof = (c / asm.key_len[:, None]).astype(np.float32)
    d, i = NearestNeighbors(n_neighbors=2).fit(prof).kneighbors(prof)
    g = so.prune(ugo.fuzzy_graph(i.astype(np.int64), d.astype(np.float32))["csr"], 500)
    n_comp, labels = so.components(g)
    return prof, g, n_comp, labels, so.component_layout(prof, n_comp, labels, 10)


def test_reference_data_range_picks_a_self_distance(s1_5k_k2):
    """0.3.9 takes data_range from pairwise_distances, whose dot-product expansion often leaves a point's distance to
    itself positive: the reference then halves that self-distance.  The exact rule never does."""
    from sklearn.metrics import pairwise_distances
    _, _, n_comp, _, meta = s1_5k_k2
    exact = so.data_range_exact(meta)
    picked = []
    for c in range(n_comp):
        d = pairwise_distances([meta[c]], meta)[0]
        ref = so.data_range_reference(meta, c)
        if d[c] > 0.0 and d[c] / 2.0 == ref:
            picked.append(c)
            assert exact[c] > ref
    print("S1 5k, n_neighbors 2: %d components, the reference halves a self-distance for %d" % (n_comp, len(picked)))
    assert n_comp > 2 * 10 and len(picked) > 0
    assert np.all(exact > 0.0)


# ---------------------------------------------------------------------------------------------
# the mirror's host rules, with a fake engine
# ---------------------------------------------------------------------------------------------
FAKE = types.SimpleNamespace(device=torch.device("cpu"))


def _fake_res(graph, dim, status):
    n_comp, labels = so.components(graph)
    n = graph.shape[0]
    vectors = np.zeros((n, dim))
    for c in range(n_comp):
        if status[c] == 1:
            rows = np.flatnonzero(labels == c)
            vectors[rows] = so.exact_eigenvectors(graph[rows][:, rows], dim)[0]
    meta = so.eye_meta(n_comp, dim) if n_comp > 1 else None
    ranges = so.data_range_exact(meta) if n_comp > 1 else np.full(1, 10.0)
    return {"n": n, "dim": dim, "n_comp": n_comp, "size": np.bincount(labels).astype(np.int32),
            "status": np.asarray(status, np.int32), "range": ranges, "stats": np.zeros(6, np.int64),
            "labels": torch.from_numpy(labels.astype(np.int32)), "vectors": torch.from_numpy(vectors),
            "meta": None if meta is None else torch.from_numpy(meta), "centroids": None}


def _fake_assemble(engine, res, u):
    """sp_assemble's arithmetic in numpy."""
    labels = res["labels"].numpy()
    vec, meta = res["vectors"].numpy(), res["meta"]
    out = np.empty((res["n"], res["dim"]), np.float32)
    for c in range(res["n_comp"]):
        rows = np.flatnonzero(labels == c)
        r = res["range"][c]
        if res["status"][c] == 1:
            v = vec[rows]
            v = v * (r / np.abs(v).max()) if meta is not None else v
        else:
            v = -r + (r - (-r)) * u[rows]
        out[rows] = v + meta[c].numpy() if meta is not None else v
    return torch.from_numpy(out)


@pytest.fixture
def fake(monkeypatch):
    from karma_b200 import umap_spectral
    state = {}

    def spectral_build(engine, graph, dim, n_epochs, data=None):
        if "build" in state:
            return state["build"](engine, graph, dim, n_epochs, data)
        csr = scipy.sparse.csr_matrix((graph["data"].numpy(), graph["indices"].numpy(), graph["indptr"].numpy()))
        state["n_epochs"] = n_epochs
        return _fake_res(csr, dim, state["status"](so.components(csr)[0]))

    monkeypatch.setattr(umap_spectral, "spectral_build", spectral_build)
    monkeypatch.setattr(umap_spectral, "assemble", _fake_assemble)
    return umap_spectral, state


def test_mirror_consumes_random_state_as_umap_with_fallbacks(fake):
    """Draws for small and non-converged components in label order, with umap's warnings; the solved ones draw nothing."""
    mod, state = fake
    dim = 2
    g = _cliques([1, 6, 2, 5], order=np.random.RandomState(8).permutation(14))
    sizes = np.bincount(so.components(g)[1])
    state["status"] = lambda n_comp: [0 if s < 2 * dim else 2 if s == 5 else 1 for s in sizes]   # the 5 fails

    def solve(gc, d, rows):                                # the oracle with the same component failing
        return None if rows.size == 5 else so.exact_eigenvectors(gc, d)[0]
    rs, ref = np.random.RandomState(11), np.random.RandomState(11)
    with warnings.catch_warnings(record=True) as got:
        warnings.simplefilter("always")
        out = mod.spectral_layout(None, g, dim, rs, engine=FAKE)
    with warnings.catch_warnings(record=True) as want_w:
        warnings.simplefilter("always")
        want = so.spectral_layout_flow(None, g, dim, ref, solve, None, lambda m, c: so.data_range_exact(m)[c])
    assert [str(w.message) for w in got] == [str(w.message) for w in want_w] and len(got) == 2
    assert out.dtype == np.float32 and np.array_equal(out, want)
    assert rs.random_sample() == ref.random_sample()
    assert state["n_epochs"] == 0                          # the mirror's graph is pruned already


@pytest.mark.parametrize("converged", [True, False])
def test_mirror_draws_and_discards_lobpcgs_block_at_two_million_rows(fake, converged):
    mod, state = fake
    n, dim = so.LOBPCG_ROWS, 2
    g = _ring(n)

    def build(engine, graph, dim, n_epochs, data=None):                 # connected: no eigensolve at 2 M rows here
        return {"n": n, "dim": dim, "n_comp": 1, "size": np.array([n], np.int32),
                "status": np.array([1 if converged else 2], np.int32), "range": np.full(1, 10.0),
                "stats": np.zeros(6, np.int64), "labels": torch.zeros(n, dtype=torch.int32),
                "vectors": torch.zeros((n, dim), dtype=torch.float64), "meta": None, "centroids": None}
    state["build"] = build
    rs, ref = np.random.RandomState(4), np.random.RandomState(4)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = mod.spectral_layout(None, g, dim, rs, engine=FAKE)
        want = so.spectral_layout_flow(None, g, dim, ref, lambda gc, d, rows: np.zeros((n, d)) if converged else None,
                                       None, None)
    assert out.dtype == np.float64 and np.array_equal(out, want)
    assert rs.random_sample() == ref.random_sample()


def test_mirror_refusals():
    from karma_b200 import umap_spectral
    g = _ring(30)
    with pytest.raises(ValueError, match="euclidean"):
        umap_spectral.spectral_layout(None, g, 2, np.random.RandomState(0), metric="cosine", engine=FAKE)
    with pytest.raises(ValueError, match="square"):
        umap_spectral.spectral_layout(None, scipy.sparse.csr_matrix(np.ones((3, 4))), 2, np.random.RandomState(0),
                                      engine=FAKE)
    with pytest.raises(ValueError, match="RandomState"):
        umap_spectral.spectral_init(FAKE, {}, 2, 200, 42)
    with pytest.raises(ValueError, match="dim"):
        umap_spectral.spectral_build(FAKE, {}, 0, 200)


def test_simplicial_set_embedding_spectral_layout_keyword(monkeypatch):
    """spectral_layout= replaces umap.spectral.spectral_layout; without it the mirror still needs umap-learn."""
    from karma_b200 import umap_layout
    seen = {}

    def layout_graph(engine, graph, embedding, n_epochs, a, b, seed, gamma, initial_alpha, negative_sample_rate):
        seen["init"] = embedding.numpy().copy()
        return embedding

    monkeypatch.setattr(umap_layout, "layout_graph", layout_graph)
    monkeypatch.setitem(sys.modules, "umap", None)
    got = {}

    def spectral_layout(data, graph, dim, random_state, metric="euclidean", metric_kwds={}):
        got["nnz"] = graph.nnz
        return random_state.normal(size=(graph.shape[0], dim)).astype(np.float32)

    args = (None, _ring(60), 3, 1.0, 1.58, 0.9, 1.0, 5.0, 10, "spectral")
    rs, ref = np.random.RandomState(2), np.random.RandomState(2)
    umap_layout.simplicial_set_embedding(*args, rs, "euclidean", {}, engine=FAKE, spectral_layout=spectral_layout)
    assert got["nnz"] == 120
    assert np.array_equal(seen["init"], so.init_embedding(ref.normal(size=(60, 3)).astype(np.float32), ref))
    with pytest.raises(ValueError, match="spectral"):
        umap_layout.simplicial_set_embedding(*args, np.random.RandomState(2), "euclidean", {}, engine=FAKE)


# ---------------------------------------------------------------------------------------------
# device (K10)
# ---------------------------------------------------------------------------------------------
N_EPOCHS = 200                                             # umap's default above 10 000 rows
EXACT_MAX = 3000                                           # components checked against the dense exact eigenvectors
ARPACK_NCV, ARPACK_RESTARTS = 128, 300                     # the larger ones against ARPACK, in bounded time


def _csr(g):
    return scipy.sparse.csr_matrix((g["data"].cpu().numpy(), g["indices"].cpu().numpy(), g["indptr"].cpu().numpy()))


def _to_dev(engine, csr):
    return {"indptr": torch.from_numpy(csr.indptr.astype(np.int64)).to(engine.device),
            "indices": torch.from_numpy(csr.indices.astype(np.int32)).to(engine.device),
            "data": torch.from_numpy(csr.data.astype(np.float64)).to(engine.device)}


@pytest.fixture(scope="module")
def s1_50k(engine):
    """S1 50 k: the device profile (float64) and the K7 graphs of the exact device lists at n_neighbors 2, 5, 15."""
    from karma_b200 import synth
    from karma_b200.engine import device_pass
    from karma_b200.umap_graph import build_graph
    asm = synth.make("S1", 50000)
    d_bases, d_offsets, d_key_len = engine.upload(asm.bases, asm.offsets, asm.key_len)
    out = {}
    for k in (2, 5, 15):
        r = device_pass(engine, d_bases, d_offsets, d_key_len, asm.n, "5p6", n_neighbors=k, want_profile=(k == 2))
        if k == 2:
            out["profile"] = r["profile"].contiguous()
        out[k] = build_graph(engine, r["idx"].contiguous(), r["dist"].contiguous())
    return out


def _check_build(engine, s1_50k, k, dim):
    from karma_b200.umap_spectral import SOLVED, spectral_build
    prof = s1_50k["profile"]
    res = spectral_build(engine, s1_50k[k], dim, N_EPOCHS, data=prof)
    pruned = so.prune(_csr(s1_50k[k]), N_EPOCHS)
    n_comp, labels = so.components(pruned)
    assert res["n_comp"] == n_comp
    assert np.array_equal(res["labels"].cpu().numpy(), labels.astype(np.int32))
    assert np.array_equal(res["size"], np.bincount(labels))
    assert np.array_equal(res["status"], [SOLVED if (n_comp == 1 or s >= 2 * dim) else 0 for s in res["size"]])
    x32 = prof.cpu().numpy().astype(np.float32)
    if n_comp > 2 * dim:
        assert np.array_equal(res["centroids"].cpu().numpy(), so.centroids(x32, labels, n_comp))
    if n_comp > 1:
        meta = res["meta"].cpu().numpy()
        assert np.array_equal(res["range"], so.data_range_exact(meta))
        if n_comp <= 2 * dim:
            assert np.array_equal(meta, so.eye_meta(n_comp, dim))
        elif n_comp <= 8000:
            ref = so.component_layout(x32, n_comp, labels, dim)
            err = np.abs(meta - ref).max()
            print("k=%d dim=%d: %d components, meta max |device - sklearn| = %.3g" % (k, dim, n_comp, err))
            assert err <= 1e-6
    # every solved component: residual, and agreement with the exact eigenvectors
    vec = res["vectors"].cpu().numpy()
    worst_res, worst_cos = 0.0, 0.0
    order = np.argsort(labels, kind="stable")
    off = np.concatenate(([0], np.cumsum(np.bincount(labels))))
    for c in np.flatnonzero(res["status"] == SOLVED):
        rows = order[off[c]:off[c + 1]]
        gc = pruned[rows][:, rows]
        v = vec[rows]
        lap = so.laplacian(gc)
        lam = np.einsum("ij,ij->j", v, lap @ v)
        worst_res = max(worst_res, np.linalg.norm(lap @ v - v * lam, axis=0).max())
        assert np.allclose(np.linalg.norm(v, axis=0), 1.0, atol=1e-12)
        assert np.all(v[np.argmax(np.abs(v), axis=0), np.arange(dim)] > 0)
        if rows.size > EXACT_MAX:
            # beyond dense eigh: ARPACK on M = I - L at a tight tolerance, with a bounded number of restarts
            m = scipy.sparse.identity(rows.size, format="csr") - lap
            w, ex = scipy.sparse.linalg.eigsh(m, dim + 2, which="LA", tol=1e-12, ncv=min(rows.size - 1, ARPACK_NCV),
                                              maxiter=ARPACK_RESTARTS)
            o = np.argsort(-w)
            w, ex = 1.0 - w[o], so.sign_flip(ex[:, o][:, 1:dim + 1])
        else:
            ex, w = so.exact_eigenvectors(gc, dim)
        gaps = np.minimum(np.diff(w)[:dim], np.diff(w)[1:dim + 1])
        for j in range(dim):
            if gaps[j] >= 1e-3:
                one_minus = 1.0 - abs(v[:, j] @ ex[:, j])
                worst_cos = max(worst_cos, one_minus)
                assert one_minus <= 1e-8, (c, j, one_minus, gaps[j])
        assert np.linalg.svd(v.T @ ex, compute_uv=False).min() > 1.0 - 1e-6
    print("k=%d dim=%d: %d components, %d solved, worst residual %.3g, worst 1-|cos| %.3g, stats %s"
          % (k, dim, n_comp, (res["status"] == SOLVED).sum(), worst_res, worst_cos, res["stats"].tolist()))
    assert worst_res <= 2e-9
    return res, pruned, x32


@pytest.mark.gpu
@pytest.mark.parametrize("k,dim", [(2, 10), (5, 10), (15, 10), (15, 2)])
def test_device_build_matches_the_oracle(engine, s1_50k, k, dim):
    _check_build(engine, s1_50k, k, dim)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 15])
def test_device_init_equals_the_oracles_and_is_deterministic(engine, s1_50k, k):
    from karma_b200.umap_spectral import spectral_build, spectral_init
    dim = 10
    res = spectral_build(engine, s1_50k[k], dim, N_EPOCHS, data=s1_50k["profile"])
    vec = res["vectors"].cpu().numpy()
    meta = None if res["meta"] is None else res["meta"].cpu().numpy()
    pruned = so.prune(_csr(s1_50k[k]), N_EPOCHS)
    ranges = None if meta is None else so.data_range_exact(meta)       # once: the flow asks per component
    rs = np.random.RandomState(42)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        got = spectral_init(engine, s1_50k[k], dim, N_EPOCHS, rs, data=s1_50k["profile"]).cpu().numpy()
        again = spectral_init(engine, s1_50k[k], dim, N_EPOCHS, np.random.RandomState(42),
                              data=s1_50k["profile"]).cpu().numpy()
        ref = np.random.RandomState(42)
        layout = so.spectral_layout_flow(None, pruned, dim, ref, lambda gc, d, rows: vec[rows], lambda *a: meta,
                                         lambda m, c: ranges[c])
        want = so.init_embedding(layout, ref)
    assert got.tobytes() == again.tobytes()
    assert np.array_equal(got, want)
    assert rs.random_sample() == ref.random_sample()


@pytest.mark.gpu
def test_sign_flip_of_an_init_column_mirrors_k8_and_keeps_k9(engine, s1_50k):
    from karma_b200.hdbscan_ import cluster_embedding
    from karma_b200.umap_layout import find_ab_params, layout_graph
    from karma_b200.umap_spectral import spectral_init
    g = s1_50k[15]
    init = spectral_init(engine, g, 10, N_EPOCHS, np.random.RandomState(0), data=s1_50k["profile"])
    flip = init.clone()
    flip[:, 3] = -flip[:, 3]
    a, b = find_ab_params(1.0, 0.1)
    e0 = layout_graph(engine, g, init, N_EPOCHS, a, b, seed=7)
    e1 = layout_graph(engine, g, flip, N_EPOCHS, a, b, seed=7)
    want = e0.clone()
    want[:, 3] = -want[:, 3]
    assert torch.equal(e1, want)
    l0 = cluster_embedding(engine, e0, 15)["labels"]
    l1 = cluster_embedding(engine, e1, 15)["labels"]
    assert np.array_equal(l0, l1)


@pytest.mark.gpu
def test_device_refusals(engine):
    from karma_b200 import _lib
    from karma_b200.umap_spectral import spectral_build
    g = _cliques([30, 30])
    bad = _to_dev(engine, g)
    bad["data"][5] = float("nan")
    with pytest.raises(_lib.KarmaB200Error) as e:
        spectral_build(engine, bad, 2, 0)
    assert e.value.code == _lib.KB_EINVAL
    with pytest.raises(_lib.KarmaB200Error) as e:
        spectral_build(engine, _to_dev(engine, g), 65, 0)
    assert e.value.code == _lib.KB_EUNSUPPORTED
    many = scipy.sparse.csr_matrix((70000, 70000))             # every vertex alone: 70 000 components
    with pytest.raises(_lib.KarmaB200Error) as e:
        spectral_build(engine, _to_dev(engine, many), 2, 0, data=torch.zeros((70000, 3), device=engine.device))
    assert e.value.code == _lib.KB_EUNSUPPORTED
    with pytest.raises(_lib.KarmaB200Error) as e:                # 60 components > 2 * dim need the data
        spectral_build(engine, _to_dev(engine, _cliques([2] * 30)), 2, 0)
    assert e.value.code == _lib.KB_EINVAL


@pytest.mark.gpu
def test_device_mirror_equals_exact_oracle_on_hand_graphs(engine):
    from karma_b200.umap_spectral import spectral_layout
    g = _weighted([1, 6, 2, 50, 3, 9], seed=8)
    data = np.random.RandomState(9).rand(71, 5).astype(np.float32)
    for dim in (2, 3):                                        # 6 components: meta-embedding at dim 2, +-eye at dim 3
        rs, ref = np.random.RandomState(3), np.random.RandomState(3)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out = spectral_layout(data, g, dim, rs, engine=engine)
            want = so.spectral_layout_exact(data, g, dim, ref)
        assert out.dtype == np.float32 and out.shape == (71, dim)
        assert np.abs(out - want).max() <= 1e-6
        assert rs.random_sample() == ref.random_sample()
    ring = _weighted([500], seed=1)                           # connected: the eigenvectors themselves, float64
    out = spectral_layout(None, ring, 2, np.random.RandomState(0), engine=engine)
    lap = so.laplacian(ring)
    lam = np.einsum("ij,ij->j", out, lap @ out)
    assert out.dtype == np.float64 and np.linalg.norm(lap @ out - out * lam, axis=0).max() <= 2e-9


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 15])
def test_full_chain_s1_50k(engine, s1_50k, k):
    """S1 50 k -> K7 -> K10 -> K8 -> K9, all on the device."""
    from karma_b200.hdbscan_ import cluster_embedding
    from karma_b200.umap_layout import INT32_MAX, INT32_MIN, find_ab_params, fold_seed, layout_graph
    from karma_b200.umap_spectral import spectral_init
    rs = np.random.RandomState(42)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        init = spectral_init(engine, s1_50k[k], 10, N_EPOCHS, rs, data=s1_50k["profile"])
    a, b = find_ab_params(1.0, 0.1)
    emb = layout_graph(engine, s1_50k[k], init, N_EPOCHS, a, b, fold_seed(rs.randint(INT32_MIN, INT32_MAX, 3)))
    assert torch.isfinite(emb).all()
    res = cluster_embedding(engine, emb, 2)
    print("S1 50k, n_neighbors %d: %d clusters, %d noise points" % (k, res["n_clusters"], int((res["labels"] < 0).sum())))
    assert res["n_clusters"] >= 1
