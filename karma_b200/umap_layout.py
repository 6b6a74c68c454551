"""UMAP's layout optimisation on the GPU, from the fuzzy graph (K8, ``kb_umap_layout``).

The last numerical stage of umap-learn 0.3.9's ``UMAP.fit`` (``simplicial_set_embedding``: pruning, the per-edge
epoch schedule, ``optimize_layout``).  It runs on the device, on a graph that may never have left it::

    from karma_b200.umap_graph import build_graph
    from karma_b200.umap_layout import find_ab_params, layout_graph
    g = build_graph(engine, plan.all_idx[:n], plan.all_dist[:n])                       # K7: device CSR
    a, b = find_ab_params(1.0, 0.1)
    init = (torch.rand(n, 10, device=engine.device) * 20 - 10)
    emb = layout_graph(engine, g, init, 200, a, b, seed=42)                             # K8: device [n, 10] float32

The device loop is epoch-synchronous and deterministic (same inputs and seed, same bits): umap's schedule, every sample
of an epoch reads the positions of the epoch's start, and a vertex's moves within an epoch are summed exactly in fixed
point rather than applied one by one as umap 0.3.9's sequential loop applies them.  The rules are frozen in
oracle/umap_layout_oracle.py (``optimize_layout_sync``).
"""
from ctypes import byref, c_int64

import numpy as np
import torch

from ._lib import check, ptr

INT32_MIN = np.iinfo(np.int32).min + 1
INT32_MAX = np.iinfo(np.int32).max - 1
_M64 = (1 << 64) - 1

# umap-learn 0.3.9's named distances (umap.distances.named_distances): the metrics simplicial_set_embedding accepts
METRICS = frozenset((
    "euclidean", "l2", "manhattan", "taxicab", "l1", "chebyshev", "linfinity", "linfty", "linf", "minkowski",
    "seuclidean", "standardised_euclidean", "wminkowski", "weighted_minkowski", "mahalanobis", "canberra", "cosine",
    "correlation", "haversine", "braycurtis", "hamming", "jaccard", "dice", "matching", "kulsinski", "rogerstanimoto",
    "russellrao", "sokalsneath", "sokalmichener", "yule"))


def _mix64(z):
    z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & _M64
    z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & _M64
    return z ^ (z >> 31)


def fold_seed(rng_state):
    """The device seed of umap's ``rng_state`` (the three int64 of ``random_state.randint(INT32_MIN, INT32_MAX, 3)``)."""
    s = [int(x) & 0xffffffff for x in rng_state]
    return _mix64(_mix64(_mix64(s[0]) ^ s[1]) ^ s[2])


def find_ab_params(spread, min_dist):
    """umap's ``find_ab_params``: fit 1 / (1 + a x^(2b)) to the offset exponential of ``spread`` / ``min_dist``."""
    from scipy.optimize import curve_fit

    def curve(x, a, b):
        return 1.0 / (1.0 + a * x ** (2 * b))

    xv = np.linspace(0, spread * 3, 300)
    yv = np.zeros(xv.shape)
    yv[xv < min_dist] = 1.0
    yv[xv >= min_dist] = np.exp(-(xv[xv >= min_dist] - min_dist) / spread)
    params, _ = curve_fit(curve, xv, yv)
    return params[0], params[1]


def layout_graph(engine, graph, embedding, n_epochs, a, b, seed, gamma=1.0, initial_alpha=1.0, negative_sample_rate=5.0,
                 return_samples=False):
    """Device graph in, device embedding out.  ``graph``: ``build_graph``'s dict (indptr int64[N+1], indices int32,
    data float64, all on the engine's GPU); ``embedding``: float32 [N, dim] on that GPU, the initial layout (not
    modified).  Returns a new float32 [N, dim] device tensor; with ``return_samples`` also the int64 [nnz_kept, 2]
    positive / negative sample counts of every kept edge, in CSR order.  ``seed``: a uint64."""
    indptr, indices, data = graph["indptr"], graph["indices"], graph["data"]
    if indptr.dtype != torch.int64 or indices.dtype != torch.int32 or data.dtype != torch.float64:
        raise ValueError("the graph must be indptr int64, indices int32, data float64")
    if embedding.dim() != 2 or embedding.dtype != torch.float32:
        raise ValueError("the embedding must be a float32 [N, dim] tensor")
    n, dim = embedding.shape
    if indptr.numel() != n + 1 or indices.numel() != data.numel():
        raise ValueError("the graph has %d rows and the embedding %d" % (indptr.numel() - 1, n))
    for t in (indptr, indices, data, embedding):
        if t.device != engine.device:
            raise ValueError("the graph and the embedding must live on the engine's device %s" % engine.device)
    out = embedding.contiguous().clone()
    samples = torch.empty((max(indices.numel(), 1), 2), dtype=torch.int64, device=engine.device) if return_samples else None
    engine._bind_stream()
    kept = c_int64()
    check(engine.lib.kb_umap_layout(engine.ctx, n, indices.numel(), ptr(indptr.contiguous()), ptr(indices.contiguous()),
                                    ptr(data.contiguous()), dim, int(n_epochs), float(a), float(b), float(gamma),
                                    float(initial_alpha), float(negative_sample_rate), int(seed) & _M64, ptr(out),
                                    ptr(samples), byref(kept)))
    if return_samples:
        return out, samples[:kept.value]
    return out


def _init_embedding(data, graph, n_components, init, random_state, metric, metric_kwds, spectral_layout=None):
    """umap 0.3.9's initial layout, drawing from ``random_state`` as umap does.  ``spectral_layout``: the function
    init="spectral" calls (default: ``umap.spectral.spectral_layout``)."""
    n = graph.shape[0]
    if isinstance(init, str) and init == "random":
        return random_state.uniform(low=-10.0, high=10.0, size=(n, n_components)).astype(np.float32)
    if isinstance(init, str) and init == "spectral":
        if spectral_layout is None:
            try:
                from umap.spectral import spectral_layout
            except ImportError:
                raise ValueError("init='spectral' needs umap-learn (umap.spectral.spectral_layout), which is not "
                                 "importable; pass init='random', an array, or spectral_layout=") from None
        initialisation = spectral_layout(data, graph, n_components, random_state, metric=metric, metric_kwds=metric_kwds)
        expansion = 10.0 / np.abs(initialisation).max()
        return (initialisation * expansion).astype(np.float32) + random_state.normal(
            scale=0.0001, size=[n, n_components]).astype(np.float32)
    if isinstance(init, str):
        raise ValueError("init must be 'random', 'spectral' or an array, got %r" % (init,))
    init_data = np.array(init)
    if init_data.shape != (n, n_components):
        raise ValueError("init has shape %s, expected (%d, %d)" % (init_data.shape, n, n_components))
    if np.unique(init_data, axis=0).shape[0] < init_data.shape[0]:
        # umap 0.3.9 jitters duplicate rows with numpy's global generator, not random_state
        from sklearn.neighbors import KDTree
        dist, _ = KDTree(init_data).query(init_data, k=2)
        nndist = np.mean(dist[:, 1])
        init_data = init_data + np.random.normal(scale=0.001 * nndist, size=init_data.shape).astype(np.float32)
    return np.ascontiguousarray(init_data, dtype=np.float32)


def simplicial_set_embedding(data, graph, n_components, initial_alpha, a, b, gamma, negative_sample_rate, n_epochs, init,
                             random_state, metric, metric_kwds, verbose=False, engine=None, spectral_layout=None):
    """Drop-in for ``umap.umap_.simplicial_set_embedding`` of umap-learn 0.3.9: the same signature and host rules
    (n_epochs <= 0 -> 500 up to 10 000 rows, else 200; pruning; the initial layout from the pruned graph; ``rng_state``
    drawn last), the layout on
    the device.  Returns float32 [N, n_components].  ``random_state`` is a numpy RandomState, consumed exactly as umap
    consumes it.  ``engine``: the GPU context (default: a new one).  ``spectral_layout``: the function init="spectral"
    calls instead of ``umap.spectral.spectral_layout``, with its signature (e.g. ``umap_spectral.spectral_layout``)."""
    import scipy.sparse
    if not (callable(metric) or metric in METRICS):
        raise ValueError("unknown metric %r" % (metric,))
    if not scipy.sparse.issparse(graph) or graph.ndim != 2 or graph.shape[0] != graph.shape[1]:
        raise ValueError("graph must be a square scipy sparse matrix")
    graph = graph.tocoo(copy=True)
    graph.sum_duplicates()
    n = graph.shape[0]
    if n_epochs <= 0:
        n_epochs = 500 if n <= 10000 else 200
    # umap's pruning, before the initial layout: spectral_layout sees the pruned graph.  The device prunes again with the
    # same max, which keeps every remaining edge.
    graph.data[graph.data < (graph.data.max() / float(n_epochs))] = 0.0
    graph.eliminate_zeros()
    embedding = _init_embedding(data, graph, n_components, init, random_state, metric, metric_kwds, spectral_layout)
    rng_state = random_state.randint(INT32_MIN, INT32_MAX, 3).astype(np.int64)
    csr = graph.tocsr()
    if engine is None:
        from .engine import Engine
        engine = Engine()
    dev = engine.device
    g = {"indptr": torch.from_numpy(csr.indptr.astype(np.int64)).to(dev),
         "indices": torch.from_numpy(csr.indices.astype(np.int32)).to(dev),
         "data": torch.from_numpy(csr.data.astype(np.float64)).to(dev)}
    out = layout_graph(engine, g, torch.from_numpy(embedding).to(dev), n_epochs, a, b, fold_seed(rng_state), gamma,
                       initial_alpha, negative_sample_rate)
    if verbose:
        print("\tcompleted ", n_epochs, " / ", n_epochs, "epochs")
    return out.cpu().numpy()
