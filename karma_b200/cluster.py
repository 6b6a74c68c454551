"""karma's clustering on the device: the exact kNN lists in, HDBSCAN's labels and probabilities out.

What ``KmerClustering.run`` does after the GPU pass when umap-learn 0.3.9 takes the lists through
``fuzzy_simplicial_set`` (``kmer.umap_embedding``'s route 2) and hdbscan 0.8.22 clusters the embedding, with every
array kept on the device::

    from karma_b200.cluster import cluster_from_lists
    res = profile_and_knn(engine, bases, offsets, key_len, "5p6", n_neighbors=2, host_profile=False)
    out = cluster_from_lists(engine, res["d_idx"], res["d_dist"], res["d_profile"], 10, 0, 42, 2)
    out["labels"], out["probabilities"], out["n_clusters"]

The stages are K7 (``umap_graph.build_graph``), K10 (``umap_spectral.spectral_init``), K8
(``umap_layout.layout_graph``) and K9 (``hdbscan_``).  ``random_state`` is consumed exactly as route 2 consumes it: the
lists are given, so the graph draws nothing; the spectral initialisation draws what 0.3.9's ``spectral_layout`` and
``_init_embedding`` draw; then ``rng_state`` is drawn for the layout.  Both routes therefore give the same bits.
"""
import time
import warnings

import numpy as np
import torch

from .hdbscan_ import host_rules, mutual_reachability_mst, tree_labels
from .umap_graph import build_graph
from .umap_layout import INT32_MAX, INT32_MIN, find_ab_params, fold_seed, layout_graph
from .umap_spectral import DIM_MAX, spectral_init

HDBSCAN_DEFAULT_MIN_CLUSTER_SIZE = 5         # hdbscan 0.8.22's default, which karma keeps for min_cluster_size == 1


def n_epochs_for(n):
    """umap 0.3.9's default number of epochs for n rows (``simplicial_set_embedding`` with n_epochs <= 0)."""
    return 500 if n <= 10000 else 200


def hdbscan_args(min_cluster_size):
    """karma's HDBSCAN arguments: min_cluster_size 1 means hdbscan's default size with a single cluster
    allowed.  Returns (min_cluster_size, allow_single_cluster)."""
    if min_cluster_size == 1:
        return HDBSCAN_DEFAULT_MIN_CLUSTER_SIZE, True
    return min_cluster_size, False


def _is_int(x):
    return isinstance(x, (int, np.integer)) and not isinstance(x, bool)


def check_components(n_components):
    if not _is_int(n_components) or not 1 <= n_components <= DIM_MAX:
        raise ValueError("n_components must be an integer in 1..%d, got %r" % (DIM_MAX, n_components))


def check_arguments(n, n_neighbors, n_components, min_cluster_size):
    """Refuse what the device route does not serve, before any GPU work: fewer than 2 rows, a non-integer or
    non-positive ``n_neighbors``, ``n_components`` outside 1..64, a ``min_cluster_size`` hdbscan refuses.  Returns
    ``n_neighbors``, truncated to n - 1 with umap 0.3.9's warning when it is not below n (as ``UMAP.fit`` does)."""
    if n < 2:
        raise ValueError("clustering needs at least 2 contigs, got %d" % n)
    if not _is_int(n_neighbors) or n_neighbors < 1:
        raise ValueError("n_neighbors must be an integer >= 1, got %r" % (n_neighbors,))
    check_components(n_components)
    host_rules(n, hdbscan_args(min_cluster_size)[0])
    if n_neighbors >= n:
        warnings.warn("n_neighbors is larger than the dataset size; truncating to X.shape[0] - 1")
        n_neighbors = n - 1
    return int(n_neighbors)


def _synchronize(engine):
    torch.cuda.current_stream(engine.device).synchronize()


def cluster_from_lists(engine, d_idx, d_dist, d_profile, n_components, min_dist, random_state, min_cluster_size):
    """UMAP (n_components, min_dist, random_state as karma passes them to ``umap.UMAP``) and HDBSCAN
    (``min_cluster_size`` by karma's rule) on the device lists ``d_idx`` int32 [N, k] and ``d_dist`` float32 [N, k]
    of the device profile ``d_profile`` [N, D] (read by the spectral initialisation when the graph has more than
    2 * n_components components).  Returns a dict: ``labels`` (numpy intp, -1 = noise), ``probabilities`` (numpy
    float64), ``n_clusters``, ``embedding`` (device float32 [N, n_components]), ``n_epochs``, ``spectral`` (components
    and Lanczos statistics of K10) and ``ms`` (host-clock milliseconds of each stage, each ended by a device
    synchronise: graph, spectral, layout, hdbscan_mst, hdbscan_tree)."""
    from sklearn.utils import check_random_state
    check_components(n_components)
    n = d_idx.shape[0]
    if n < 2:
        raise ValueError("clustering needs at least 2 rows, got %d" % n)
    mcs, allow_single = hdbscan_args(min_cluster_size)
    _, core_k = host_rules(n, mcs)
    random_state = check_random_state(random_state)
    a, b = find_ab_params(1.0, min_dist)
    ms = {}
    t = [time.perf_counter()]

    def lap(name):
        _synchronize(engine)
        t.append(time.perf_counter())
        ms[name] = (t[-1] - t[-2]) * 1e3

    graph = build_graph(engine, d_idx, d_dist, local_connectivity=1.0, set_op_mix_ratio=1.0)
    lap("graph")
    n_epochs = n_epochs_for(n)
    init, build = spectral_init(engine, graph, n_components, n_epochs, random_state, data=d_profile, return_build=True)
    lap("spectral")
    rng_state = random_state.randint(INT32_MIN, INT32_MAX, 3).astype(np.int64)
    emb = layout_graph(engine, graph, init, n_epochs, a, b, fold_seed(rng_state), gamma=1.0, initial_alpha=1.0,
                       negative_sample_rate=5)
    lap("layout")
    # hdbscan_.cluster_embedding's two halves, timed apart: the device tree, then the host labelling
    mst = mutual_reachability_mst(engine, emb, core_k)
    edges, weights = mst["edges"].cpu().numpy(), mst["weights"].cpu().numpy()
    lap("hdbscan_mst")
    labels, probabilities, n_clusters = tree_labels(edges, weights, mcs, allow_single)
    lap("hdbscan_tree")
    st = build["stats"]
    return {"labels": labels.astype(np.intp), "probabilities": probabilities, "n_clusters": n_clusters,
            "embedding": emb, "n_epochs": n_epochs, "ms": ms,
            "spectral": {"n_comp": build["n_comp"], "lanczos_steps": int(st[0]), "restarts": int(st[1]),
                         "meta_steps": int(st[2]), "meta_restarts": int(st[3])}}
