"""Frozen rules of K10: umap-learn 0.3.9's spectral initialisation (umap.spectral.spectral_layout), restated.

Two formulations:
  * the reference (``spectral_layout_reference``): 0.3.9's code path as restated from memory (unpinned, like K9's
    min_samples rules): scipy's eigsh with umap's arguments (tol 1e-4, v0 ones, arbitrary sign), scikit-learn's
    SpectralEmbedding for the meta points, and data_range from pairwise_distances (dot-product expansion);
  * the exact formulation the device equals (``spectral_layout_exact``): the same control flow and the same draws
    from random_state, with exact eigenvectors (dense eigh, unit norm, largest-|.| entry positive),
    the same meta points, and data_range from euclidean distances in fp64 coordinate order (``data_range_exact``).
"""
import warnings

import numpy as np
import scipy.sparse
import scipy.sparse.csgraph
import scipy.sparse.linalg

LOBPCG_ROWS = 2000000


def prune(graph, n_epochs):
    """umap 0.3.9's pruning in simplicial_set_embedding: weights below max / n_epochs dropped."""
    g = graph.tocoo(copy=True)
    g.sum_duplicates()
    g.data[g.data < (g.data.max() / float(n_epochs))] = 0.0
    g.eliminate_zeros()
    return g.tocsr()


def components(graph):
    return scipy.sparse.csgraph.connected_components(graph)


def sign_flip(u):
    """scikit-learn's _deterministic_vector_sign_flip on the columns of u: each column's largest-|.| entry (the first on
    ties) made positive."""
    u = np.array(u, dtype=np.float64, copy=True)
    rows = np.argmax(np.abs(u), axis=0)
    u *= np.sign(u[rows, np.arange(u.shape[1])])
    return u


def centroids(data, labels, n_comp):
    """component_layout's centroids: numpy's float32 mean of each component's rows, stored into float64."""
    data = np.asarray(data, dtype=np.float32)
    out = np.empty((n_comp, data.shape[1]), dtype=np.float64)
    order = np.argsort(labels, kind="stable")
    off = np.concatenate(([0], np.cumsum(np.bincount(labels, minlength=n_comp))))
    for c in range(n_comp):
        out[c] = data[order[off[c]:off[c + 1]]].mean(axis=0)
    return out


def component_layout(data, n_comp, labels, dim):
    """0.3.9's component_layout: scikit-learn's SpectralEmbedding of exp(-d^2) between the centroids, over its max."""
    from sklearn.manifold import SpectralEmbedding
    from sklearn.metrics import pairwise_distances
    affinity = np.exp(-pairwise_distances(centroids(data, labels, n_comp)) ** 2)
    emb = SpectralEmbedding(n_components=dim, affinity="precomputed").fit_transform(affinity)
    return emb / emb.max()


def eye_meta(n_comp, dim):
    k = int(np.ceil(n_comp / 2.0))
    base = np.hstack([np.eye(k), np.zeros((k, dim - k))])
    return np.vstack([base, -base])[:n_comp]


def data_range_reference(meta, c):
    from sklearn.metrics import pairwise_distances
    d = pairwise_distances([meta[c]], meta)
    return d[d > 0.0].min() / 2.0


def data_range_exact(meta):
    """Half the smallest positive euclidean distance from every meta point to the others: fp64, coordinate order."""
    meta = np.asarray(meta, dtype=np.float64)
    n, dim = meta.shape
    out = np.empty(n)
    for a0 in range(0, n, 512):
        blk = meta[a0:a0 + 512]
        d2 = np.zeros((blk.shape[0], n))
        for j in range(dim):
            df = blk[:, j:j + 1] - meta[None, :, j]
            d2 = d2 + df * df
        d2[d2 <= 0.0] = np.inf
        out[a0:a0 + 512] = np.sqrt(d2.min(axis=1)) / 2.0
    return out


def laplacian(graph):
    """L = I - D^-1/2 W D^-1/2, D the column sums (0.3.9)."""
    deg = np.asarray(graph.sum(axis=0)).ravel()
    d = scipy.sparse.spdiags(1.0 / np.sqrt(deg), 0, graph.shape[0], graph.shape[0])
    return scipy.sparse.identity(graph.shape[0], format="csr") - d @ graph @ d


def exact_eigenvectors(graph, dim):
    """Unit eigenvectors of the dim smallest non-trivial eigenvalues of L, sign fixed; and the dim + 2 smallest
    eigenvalues (for the gaps)."""
    lap = laplacian(scipy.sparse.csr_matrix(graph, dtype=np.float64))
    n = lap.shape[0]
    k = min(dim + 2, n)
    w, v = np.linalg.eigh(lap.toarray())
    vec = v[:, 1:dim + 1]
    vec = vec / np.linalg.norm(vec, axis=0)
    return sign_flip(vec), w[:k]


def _eigsh_umap(lap, dim, maxiter):
    k = dim + 1
    ncv = max(2 * k + 1, int(np.sqrt(lap.shape[0])))
    w, v = scipy.sparse.linalg.eigsh(lap, k, which="SM", ncv=ncv, tol=1e-4, v0=np.ones(lap.shape[0]), maxiter=maxiter)
    return v[:, np.argsort(w)[1:k]]


def _warn_fallback():
    warnings.warn("WARNING: spectral initialisation failed! The eigenvector solver\n"
                  "failed. This is likely due to too small an eigengap. Consider\n"
                  "adding some noise or jitter to your data.\n\n"
                  "Falling back to random initialisation!")


def assemble_component(result, rows, meta_c, data_range, vectors=None, random_state=None, dim=None):
    """0.3.9's arithmetic for one component of a disconnected graph, into the float32 result."""
    if vectors is None:
        result[rows] = random_state.uniform(low=-data_range, high=data_range, size=(rows.size, dim)) + meta_c
    else:
        expansion = data_range / np.max(np.abs(vectors))
        result[rows] = vectors * expansion + meta_c


def spectral_layout_flow(data, graph, dim, random_state, solve, meta_fn, range_fn):
    """0.3.9's spectral_layout control flow and random_state order.  ``solve(component_graph, dim, rows)`` returns the
    vectors of the component of vertices ``rows`` or None (ARPACK's failure); ``meta_fn(data, n_comp, labels, dim)``
    the meta points of more than 2 * dim components; ``range_fn(meta, c)`` the data range of component c."""
    n = graph.shape[0]
    n_comp, labels = components(graph)
    if n_comp == 1:
        if n >= LOBPCG_ROWS:
            random_state.normal(size=(n, dim + 1))
        v = solve(graph, dim, np.arange(n))
        if v is None:
            _warn_fallback()
            return random_state.uniform(low=-10.0, high=10.0, size=(n, dim))
        return v
    warnings.warn("Embedding a total of {} separate connected components using meta-embedding (experimental)".format(n_comp))
    meta = meta_fn(data, n_comp, labels, dim) if n_comp > 2 * dim else eye_meta(n_comp, dim)
    result = np.empty((n, dim), dtype=np.float32)
    csr = graph.tocsr()
    order = np.argsort(labels, kind="stable")
    off = np.concatenate(([0], np.cumsum(np.bincount(labels, minlength=n_comp))))
    for c in range(n_comp):
        rows = order[off[c]:off[c + 1]]
        r = range_fn(meta, c)
        if rows.size < 2 * dim:
            assemble_component(result, rows, meta[c], r, random_state=random_state, dim=dim)
            continue
        v = solve(csr[rows][:, rows], dim, rows)
        if v is None:
            _warn_fallback()
            assemble_component(result, rows, meta[c], r, random_state=random_state, dim=dim)
        else:
            assemble_component(result, rows, meta[c], r, vectors=v)
    return result


def spectral_layout_reference(data, graph, dim, random_state):
    """0.3.9 as restated: eigsh with umap's arguments, SpectralEmbedding, pairwise_distances' data_range."""
    def solve(g, dim, rows):
        try:
            return _eigsh_umap(laplacian(g), dim, g.shape[0] * 5)
        except scipy.sparse.linalg.ArpackError:
            return None
    return spectral_layout_flow(data, graph, dim, random_state, solve, component_layout, data_range_reference)


def spectral_layout_exact(data, graph, dim, random_state, meta_fn=component_layout):
    """The formulation the device equals, up to the eigensolver's residual: exact vectors, the exact data range."""
    ranges = {}

    def range_fn(meta, c):
        key = id(meta)
        if key not in ranges:
            ranges[key] = data_range_exact(meta)
        return ranges[key][c]
    return spectral_layout_flow(data, graph, dim, random_state, lambda g, d, rows: exact_eigenvectors(g, d)[0], meta_fn,
                                range_fn)


def init_embedding(layout, random_state):
    """The rest of 0.3.9's _init_embedding: expansion to 10 / max|.|, the float32 cast, normal(1e-4) noise."""
    n, dim = layout.shape
    expansion = 10.0 / np.abs(layout).max()
    return (layout * expansion).astype(np.float32) + random_state.normal(scale=0.0001, size=[n, dim]).astype(np.float32)
