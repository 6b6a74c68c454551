"""HDBSCAN on the GPU: clusters and membership probabilities from the UMAP embedding (K9, ``kb_hdbscan_mst`` and
``kb_hdbscan_labels``).

The last numerical stage of karma's ``KmerClustering.run``: ``hdbscan.HDBSCAN(min_cluster_size=m).fit(embedding)`` of
hdbscan 0.8.22 (metric euclidean, alpha 1, eom selection).  The mutual-reachability minimum spanning tree is built on
the device; the single-linkage tree, condensing, stability, selection, labels and probabilities run on the host in
the native library, over the N - 1 sorted edges::

    from karma_b200.hdbscan_ import HDBSCAN, cluster_embedding
    res = cluster_embedding(engine, emb, min_cluster_size=2)         # emb: device float32 [N, dim], e.g. from K8
    res["labels"], res["probabilities"], res["n_clusters"]
    clusterer = HDBSCAN(min_cluster_size=2).fit(emb)                 # the drop-in for karma's call

The tree is the exact MST under the total order (w, min(i, j), max(i, j)), so it is unique and does not depend on the
execution order.  hdbscan 0.8.22 defaults to an approximate tree and breaks ties in weight by its traversal order; on
inputs with tied weights its output, the number of clusters included, depends on that order (DESIGN §3 K9).
(The module is ``hdbscan_``: a bare ``hdbscan.py`` would shadow the real package when this directory is on sys.path.)
"""
from ctypes import byref, c_int64, c_void_p

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr

# hdbscan 0.8.22's HDBSCAN keywords other than min_cluster_size, min_samples and allow_single_cluster, at their defaults:
# the only values served
DEFAULTS = {"metric": "euclidean", "alpha": 1.0, "p": None, "algorithm": "best", "leaf_size": 40, "memory": None,
            "approx_min_span_tree": True, "gen_min_span_tree": False, "core_dist_n_jobs": 4,
            "cluster_selection_method": "eom", "prediction_data": False, "match_reference_implementation": False}


def host_rules(n, min_cluster_size, min_samples=None):
    """(min_samples, core_k) as hdbscan 0.8.22 derives them for N points: min_samples defaults to min_cluster_size, is
    clamped to N - 1 and raised to 1 if that gives 0; hdbscan's min_samples does not count the point itself, so the
    core distance is the (min_samples + 1)-th smallest distance including d(i, i) = 0.  (Rules as remembered from
    0.8.22; they are frozen in oracle/hdbscan_oracle.py.)"""
    if isinstance(min_cluster_size, bool) or not isinstance(min_cluster_size, (int, np.integer)) or min_cluster_size < 2:
        raise ValueError("min_cluster_size must be an integer >= 2, got %r" % (min_cluster_size,))
    if min_samples is not None and (isinstance(min_samples, bool) or not isinstance(min_samples, (int, np.integer))
                                    or min_samples < 1):
        raise ValueError("min_samples must be None or an integer >= 1, got %r" % (min_samples,))
    ms = int(min_cluster_size if min_samples is None else min_samples)
    ms = min(n - 1, ms)
    if ms == 0:
        ms = 1
    return ms, ms + 1


def mutual_reachability_mst(engine, x, core_k):
    """Device float32 [N, dim] in (N >= 2, dim <= 64, 1 <= core_k <= min(N, 128)).  Returns a dict of device tensors:
    ``core`` float64 [N], ``edges`` int32 [N-1, 2] oriented (min, max) and ``weights`` float64 [N-1], sorted by
    (weight, min, max)."""
    if not isinstance(x, torch.Tensor) or x.dim() != 2 or x.dtype != torch.float32:
        raise ValueError("x must be a float32 [N, dim] tensor")
    if x.device != engine.device:
        raise ValueError("x must live on the engine's device %s" % engine.device)
    x = x.contiguous()
    n, dim = x.shape
    core = torch.empty(max(n, 1), dtype=torch.float64, device=engine.device)
    edges = torch.empty((max(n - 1, 1), 2), dtype=torch.int32, device=engine.device)
    weights = torch.empty(max(n - 1, 1), dtype=torch.float64, device=engine.device)
    engine._bind_stream()
    check(engine.lib.kb_hdbscan_mst(engine.ctx, n, dim, ptr(x), int(core_k), ptr(core), ptr(edges), ptr(weights)))
    return {"core": core[:n], "edges": edges[:n - 1], "weights": weights[:n - 1]}


def tree_labels(edges, weights, min_cluster_size, allow_single_cluster=False):
    """The host half (no GPU): numpy int32 [N-1, 2] edges and float64 [N-1] weights of a spanning tree sorted by
    (w, min, max) in; (labels int32 [N], probabilities float64 [N], n_clusters) out."""
    edges = np.ascontiguousarray(edges, dtype=np.int32)
    weights = np.ascontiguousarray(weights, dtype=np.float64)
    if edges.ndim != 2 or edges.shape[1] != 2 or weights.shape != (edges.shape[0],):
        raise ValueError("edges must be [N-1, 2] and weights [N-1]")
    n = edges.shape[0] + 1
    labels = np.empty(n, np.int32)
    probabilities = np.empty(n, np.float64)
    n_clusters = c_int64()
    check(_lib.load().kb_hdbscan_labels(n, c_void_p(edges.ctypes.data), c_void_p(weights.ctypes.data),
                                        int(min_cluster_size), 1 if allow_single_cluster else 0,
                                        c_void_p(labels.ctypes.data), c_void_p(probabilities.ctypes.data),
                                        byref(n_clusters)))
    return labels, probabilities, n_clusters.value


def _points(engine, x):
    """float32 [N, dim] on the engine's device, from a tensor or an array; float64 only if every value is a float32."""
    if isinstance(x, torch.Tensor):
        if x.dtype == torch.float64:
            x = x.detach().cpu().numpy()
        else:
            if x.dtype != torch.float32:
                raise ValueError("X must be float32 (or float64 holding float32 values), got %s" % x.dtype)
            return x.detach().to(engine.device)
    x = np.asarray(x)
    if x.dtype == np.float64:
        x32 = x.astype(np.float32)
        if not np.array_equal(x32.astype(np.float64), x, equal_nan=True):
            raise ValueError("X is float64 with values that are not float32: the device computes from float32 points")
        x = x32
    elif x.dtype != np.float32:
        raise ValueError("X must be float32 (or float64 holding float32 values), got %s" % x.dtype)
    if x.ndim != 2:
        raise ValueError("X must be [N, dim]")
    return torch.from_numpy(np.ascontiguousarray(x)).to(engine.device)


def cluster_embedding(engine, x, min_cluster_size, min_samples=None, allow_single_cluster=False):
    """hdbscan 0.8.22's clustering of ``x`` (device float32 [N, dim], or an array ``_points`` accepts).  Returns
    ``labels`` (numpy int32, -1 = noise), ``probabilities`` (numpy float64), ``n_clusters`` and ``mst`` (the device
    dict of ``mutual_reachability_mst``)."""
    x = _points(engine, x)
    n = x.shape[0]
    _, core_k = host_rules(n, min_cluster_size, min_samples)
    mst = mutual_reachability_mst(engine, x, core_k)
    labels, probabilities, n_clusters = tree_labels(mst["edges"].cpu().numpy(), mst["weights"].cpu().numpy(),
                                                    min_cluster_size, allow_single_cluster)
    return {"labels": labels, "probabilities": probabilities, "n_clusters": n_clusters, "mst": mst}


class HDBSCAN:
    """Drop-in for ``hdbscan.HDBSCAN`` of hdbscan 0.8.22 as karma uses it: ``fit`` / ``fit_predict`` set ``labels_``
    (int64, -1 = noise) and ``probabilities_``.  Keywords other than ``min_cluster_size``, ``min_samples`` and
    ``allow_single_cluster`` are served at their defaults only.  ``engine``: the GPU context (default: a new one)."""

    def __init__(self, min_cluster_size=5, min_samples=None, allow_single_cluster=False, engine=None, **kw):
        for name, value in kw.items():
            if name not in DEFAULTS:
                raise ValueError("unknown argument %r" % name)
            if not (value is DEFAULTS[name] or (DEFAULTS[name] is not None and value == DEFAULTS[name])):
                raise ValueError("%s=%r is not served (only %r)" % (name, value, DEFAULTS[name]))
        host_rules(2, min_cluster_size, min_samples)          # refuse bad values at construction, as hdbscan does at fit
        self.min_cluster_size = min_cluster_size
        self.min_samples = min_samples
        self.allow_single_cluster = allow_single_cluster
        self.engine = engine

    def fit(self, X, y=None):
        if self.engine is None:
            from .engine import Engine
            self.engine = Engine()
        res = cluster_embedding(self.engine, X, self.min_cluster_size, self.min_samples, self.allow_single_cluster)
        self.labels_ = res["labels"].astype(np.intp)
        self.probabilities_ = res["probabilities"]
        return self

    def fit_predict(self, X, y=None):
        return self.fit(X).labels_
