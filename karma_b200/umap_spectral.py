"""UMAP's spectral initialisation on the GPU, disconnected graphs included (K10, ``kb_spectral_build`` and
``kb_spectral_assemble``).

The initial layout of umap-learn 0.3.9's ``UMAP.fit`` (``init="spectral"``, ``umap.spectral.spectral_layout``), from
the pruned fuzzy graph.  With it the whole chain stays on the device::

    from karma_b200.umap_graph import build_graph
    from karma_b200.umap_spectral import spectral_init
    from karma_b200.umap_layout import find_ab_params, layout_graph
    g = build_graph(engine, idx, dist)                                              # K7
    init = spectral_init(engine, g, 10, 200, np.random.RandomState(42), data=prof)  # K10: device [n, 10] float32
    emb = layout_graph(engine, g, init, 200, a, b, seed)                            # K8

A connected graph, and every component of at least 2 * dim vertices of a disconnected one, gets the exact unit
eigenvectors of its normalised Laplacian's dim smallest non-trivial eigenvalues, sign fixed so that the largest-|.|
entry is positive (0.3.9's ARPACK call stops at tol 1e-4 with an arbitrary sign).  Components are placed around meta
points (the spectral embedding of their centroids, or +-unit vectors), and every other component is a uniform draw
from ``random_state``, taken here on the host exactly where 0.3.9 takes it.  The rules are frozen in
oracle/umap_spectral_oracle.py; DESIGN §3 K10 records where the reference itself depends on BLAS rounding.
"""
import warnings
from ctypes import byref, c_int64

import numpy as np
import torch

from ._lib import check, ptr

DRAW, SOLVED, NOT_CONVERGED = 0, 1, 2
LOBPCG_ROWS = 2000000                   # 0.3.9 switches a connected graph from eigsh to lobpcg at this many rows
DIM_MAX = 64


def _graph(engine, graph):
    indptr, indices, data = graph["indptr"], graph["indices"], graph["data"]
    if indptr.dtype != torch.int64 or indices.dtype != torch.int32 or data.dtype != torch.float64:
        raise ValueError("the graph must be indptr int64, indices int32, data float64")
    for t in (indptr, indices, data):
        if t.device != engine.device:
            raise ValueError("the graph must live on the engine's device %s" % engine.device)
    if indices.numel() != data.numel():
        raise ValueError("indices and data differ in length")
    return indptr.contiguous(), indices.contiguous(), data.contiguous()


def spectral_build(engine, graph, dim, n_epochs, data=None):
    """The device half before the draws.  ``graph``: ``build_graph``'s dict (device CSR); ``n_epochs`` prunes
    w < max / n_epochs as K8 does (0: no pruning); ``data``: device or host float32 / float64 [N, D], needed when the
    graph has more than 2 * dim components.  Returns a dict: ``n_comp``, numpy ``size``, ``status``, ``range``,
    ``stats`` and device ``labels`` (int32 [N]), ``vectors`` (float64 [N, dim]), ``meta`` (float64 [n_comp, dim] or
    None), ``centroids`` (float64 [n_comp, D] or None)."""
    if isinstance(dim, bool) or not isinstance(dim, (int, np.integer)) or dim < 1:
        raise ValueError("dim must be an integer >= 1, got %r" % (dim,))
    indptr, indices, values = _graph(engine, graph)
    n = indptr.numel() - 1
    x, x_dtype, x_cols = None, 0, 0
    if data is not None:
        x = data if isinstance(data, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(data))
        if x.dim() != 2 or x.shape[0] != n or x.dtype not in (torch.float32, torch.float64):
            raise ValueError("data must be float32 or float64 [N, D] with N = %d graph rows" % n)
        x = x.to(engine.device).contiguous()
        x_dtype, x_cols = (1 if x.dtype == torch.float32 else 2), x.shape[1]
    engine._bind_stream()
    n_comp = c_int64()
    check(engine.lib.kb_spectral_build(engine.ctx, n, indices.numel(), ptr(indptr), ptr(indices), ptr(values),
                                       int(n_epochs), int(dim), ptr(x), x_dtype, x_cols, byref(n_comp)))
    nc = n_comp.value
    size, status = np.empty(nc, np.int32), np.empty(nc, np.int32)
    rng, stats = np.empty(nc, np.float64), np.empty(6, np.int64)
    dev = engine.device
    labels = torch.empty(n, dtype=torch.int32, device=dev)
    vectors = torch.empty((n, dim), dtype=torch.float64, device=dev)
    meta = torch.empty((nc, dim), dtype=torch.float64, device=dev) if nc > 1 else None
    cent = torch.empty((nc, x_cols), dtype=torch.float64, device=dev) if nc > 2 * dim else None
    check(engine.lib.kb_spectral_fetch(engine.ctx, size.ctypes.data, status.ctypes.data, rng.ctypes.data,
                                       stats.ctypes.data, ptr(labels), ptr(meta), ptr(vectors), ptr(cent)))
    return {"n": n, "dim": dim, "n_comp": nc, "size": size, "status": status, "range": rng, "stats": stats,
            "labels": labels, "vectors": vectors, "meta": meta, "centroids": cent}


def draws(res, random_state):
    """Consume ``random_state`` as umap 0.3.9's spectral_layout does, given the build's components.  Returns float64
    [N, dim] uniform [0, 1) draws (row i for vertex i; zero rows for solved components), or None when nothing is
    drawn.  ``res``: ``spectral_build``'s dict (``labels`` may be a tensor or an array)."""
    n, dim, nc, status = res["n"], res["dim"], res["n_comp"], res["status"]
    u = None
    if nc == 1:
        if n >= LOBPCG_ROWS:
            random_state.normal(size=(n, dim + 1))            # lobpcg's start block: drawn, then unused
        if status[0] != SOLVED:
            warnings.warn("WARNING: spectral initialisation failed! The eigenvector solver\n"
                          "failed. This is likely due to too small an eigengap. Consider\n"
                          "adding some noise or jitter to your data.\n\n"
                          "Falling back to random initialisation!")
            u = random_state.random_sample((n, dim))
        return u
    warnings.warn("Embedding a total of {} separate connected components using meta-embedding (experimental)".format(nc))
    labels = res["labels"]
    labels = labels.cpu().numpy() if isinstance(labels, torch.Tensor) else np.asarray(labels)
    order = np.argsort(labels, kind="stable")
    off = np.concatenate(([0], np.cumsum(res["size"])))
    for c in range(nc):
        if status[c] == SOLVED:
            continue
        if status[c] == NOT_CONVERGED:
            warnings.warn("WARNING: spectral initialisation failed! The eigenvector solver\n"
                          "failed. This is likely due to too small an eigengap. Consider\n"
                          "adding some noise or jitter to your data.\n\n"
                          "Falling back to random initialisation!")
        if u is None:
            u = np.zeros((n, dim))
        u[order[off[c]:off[c + 1]]] = random_state.random_sample((int(res["size"][c]), dim))
    return u


def assemble(engine, res, u):
    """The float32 [N, dim] device layout spectral_layout returns, from the build and the host draws."""
    out = torch.empty((res["n"], res["dim"]), dtype=torch.float32, device=engine.device)
    d_u = None if u is None else torch.from_numpy(np.ascontiguousarray(u, dtype=np.float64)).to(engine.device)
    engine._bind_stream()
    check(engine.lib.kb_spectral_assemble(engine.ctx, ptr(d_u), ptr(out)))
    if d_u is not None:
        torch.cuda.current_stream(engine.device).synchronize()    # d_u is freed on return
    return out


def _layout(engine, res, random_state):
    """0.3.9's spectral_layout result on the device: float64 for a connected graph (eigsh's vectors, or the uniform
    fallback), float32 otherwise (its multi-component result array)."""
    u = draws(res, random_state)
    if res["n_comp"] == 1:
        if u is None:
            return res["vectors"]
        return torch.from_numpy(-10.0 + 20.0 * u).to(engine.device)
    return assemble(engine, res, u)


def spectral_init(engine, graph, dim, n_epochs, random_state, data=None, return_build=False):
    """K7's device graph in, the device float32 [N, dim] initial layout for ``layout_graph`` out: umap 0.3.9's
    spectral_layout on the graph pruned at max / n_epochs, then ``_init_embedding``'s expansion to 10 / max|.| and its
    ``normal(scale=1e-4)`` noise.  ``random_state`` (a numpy RandomState) is consumed exactly as umap consumes it.
    With ``return_build`` also ``spectral_build``'s dict (components, status, Lanczos statistics)."""
    if not isinstance(random_state, np.random.RandomState):
        raise ValueError("random_state must be a numpy RandomState")
    res = spectral_build(engine, graph, dim, n_epochs, data)
    init = _layout(engine, res, random_state)
    n = res["n"]
    if init.dtype == torch.float64:
        # float64 array times a Python float, then the float32 cast
        init = (init * (10.0 / init.abs().max().item())).to(torch.float32)
    else:
        expansion = np.float32(10.0) / np.float32(init.abs().max().item())
        init = init * torch.tensor(expansion, dtype=torch.float32, device=engine.device)
    noise = random_state.normal(scale=0.0001, size=[n, dim]).astype(np.float32)
    init = init + torch.from_numpy(noise).to(engine.device)
    return (init, res) if return_build else init


def spectral_layout(data, graph, dim, random_state, metric="euclidean", metric_kwds={}, engine=None):
    """Drop-in for ``umap.spectral.spectral_layout`` of umap-learn 0.3.9, for ``simplicial_set_embedding``'s
    ``spectral_layout=`` keyword: ``graph`` is the pruned scipy sparse graph, ``data`` the float32 [N, D] points.
    Returns a numpy array as 0.3.9 does (float64 for a connected graph, float32 otherwise).  Metric euclidean only."""
    import scipy.sparse
    if metric not in ("euclidean", "l2"):
        raise ValueError("spectral_layout serves metric 'euclidean' only, got %r" % (metric,))
    if not scipy.sparse.issparse(graph) or graph.ndim != 2 or graph.shape[0] != graph.shape[1]:
        raise ValueError("graph must be a square scipy sparse matrix")
    if engine is None:
        from .engine import Engine
        engine = Engine()
    csr = graph.tocsr()
    csr.sum_duplicates()
    dev = engine.device
    g = {"indptr": torch.from_numpy(csr.indptr.astype(np.int64)).to(dev),
         "indices": torch.from_numpy(csr.indices.astype(np.int32)).to(dev),
         "data": torch.from_numpy(csr.data.astype(np.float64)).to(dev)}
    x = None
    if data is not None:
        x = np.asarray(data)
        if x.dtype not in (np.float32, np.float64):
            x = x.astype(np.float32)
    res = spectral_build(engine, g, dim, 0, x)
    return _layout(engine, res, random_state).cpu().numpy()
