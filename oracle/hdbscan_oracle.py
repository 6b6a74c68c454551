"""HDBSCAN as karma calls it (hdbscan 0.8.22: ``HDBSCAN(min_cluster_size=m).fit(embedding)``), frozen for K9.

The reference of record is scikit-learn 1.9.0's ``sklearn/cluster/_hdbscan`` (``_linkage.pyx``, ``_tree.pyx``), a port of
hdbscan's tree code.  This module freezes:
  * ``core_distances``: core_i = the core_k-th smallest of {d(i, j) : all j}, d(i, i) = 0 and duplicates counted, with
    d = RN(sqrt(sum_c (x_ic - x_jc)^2)) in fp64 from float32 coordinates, in coordinate order, no FMA (sklearn's
    ``EuclideanDistance64.rdist`` then ``sqrt``; ``core_k`` counts the point itself, like sklearn's ``min_samples``);
  * the exact MST of w(i, j) = max(core_i, core_j, d(i, j)) under the canonical total order (w, min(i, j), max(i, j)):
    ``prim_mst_port`` (plain Python) and ``prim_mst`` (its numba twin), plus ``kruskal_mst`` over all pairs;
  * ``tree_to_labels``: a pure-Python port of ``make_single_linkage``, ``_condense_tree``, ``_compute_stability``,
    ``_get_clusters`` (eom, ``allow_single_cluster``), ``_do_labelling`` and ``get_probabilities``, keeping their fp64
    operation and summation order;
  * ``host_rules``: hdbscan 0.8.22's ``min_samples`` rules.  They are as remembered from 0.8.22 and could not be checked
    against its source (unpinned): min_samples defaults to min_cluster_size, is clamped to N - 1 and raised to 1 if
    that gives 0; hdbscan's min_samples counts neighbours without the point, so core_k = min_samples + 1.
"""
import math

import numpy as np


# ---------------------------------------------------------------------------------------------
# host rules
# ---------------------------------------------------------------------------------------------
def karma_kwargs(min_cluster_size):
    """The arguments karma passes (kmer.py): ``allow_single_cluster=True`` alone when m == 1."""
    return {"allow_single_cluster": True} if min_cluster_size == 1 else {"min_cluster_size": min_cluster_size}


def host_rules(n, min_cluster_size=5, min_samples=None):
    """(min_samples, core_k) of hdbscan 0.8.22 for N points (unpinned)."""
    ms = min_cluster_size if min_samples is None else min_samples
    ms = min(n - 1, ms)
    if ms == 0:
        ms = 1
    return ms, ms + 1


# ---------------------------------------------------------------------------------------------
# core distances and the canonical MST
# ---------------------------------------------------------------------------------------------
def _as64(x):
    x = np.asarray(x)
    if x.dtype != np.float32:
        raise ValueError("points must be float32")
    return np.ascontiguousarray(x, dtype=np.float64)


def d2_rows(X, rows):
    """fp64 squared distances of ``rows`` to every point, summed in coordinate order."""
    d2 = np.zeros((len(rows), X.shape[0]))
    for c in range(X.shape[1]):
        df = X[rows, c][:, None] - X[None, :, c]
        d2 += df * df
    return d2


def core_distances(x, core_k, chunk=256):
    X = _as64(x)
    n = X.shape[0]
    out = np.empty(n)
    for r0 in range(0, n, chunk):
        rows = np.arange(r0, min(n, r0 + chunk))
        d2 = d2_rows(X, rows)
        out[rows] = np.sqrt(np.partition(d2, core_k - 1, axis=1)[:, core_k - 1])
    return out


def _dist(X, i, j):
    d2 = 0.0
    for c in range(X.shape[1]):
        df = X[i, c] - X[j, c]
        d2 += df * df
    return math.sqrt(d2)


def _less(w, a, b, w2, a2, b2):
    return w < w2 or (w == w2 and (a < a2 or (a == a2 and b < b2)))


def prim_mst_port(x, core):
    """Prim from vertex 0 under the canonical order; returns the edges as ``canonical_sort`` leaves them."""
    X = _as64(x)
    n = X.shape[0]
    in_tree = [False] * n
    bw, ba, bb = [math.inf] * n, [n] * n, [n] * n        # each outside vertex's best edge to the tree
    cur = 0
    edges, weights = [], []
    for _ in range(n - 1):
        in_tree[cur] = True
        sel = -1
        for j in range(n):
            if in_tree[j]:
                continue
            w = max(core[cur], core[j], _dist(X, cur, j))
            a, b = min(cur, j), max(cur, j)
            if _less(w, a, b, bw[j], ba[j], bb[j]):
                bw[j], ba[j], bb[j] = w, a, b
            if sel < 0 or _less(bw[j], ba[j], bb[j], bw[sel], ba[sel], bb[sel]):
                sel = j
        edges.append((ba[sel], bb[sel]))
        weights.append(bw[sel])
        cur = sel
    return canonical_sort(np.array(edges, np.int32).reshape(-1, 2), np.array(weights))


_NB = {}


def _build_numba():
    import numba

    @numba.njit(cache=False)
    def less(w, a, b, w2, a2, b2):
        return w < w2 or (w == w2 and (a < a2 or (a == a2 and b < b2)))

    @numba.njit(cache=False)
    def prim(X, core):
        n, dim = X.shape
        in_tree = np.zeros(n, np.bool_)
        bw = np.full(n, np.inf)
        ba = np.full(n, n, np.int64)
        bb = np.full(n, n, np.int64)
        edges = np.empty((n - 1, 2), np.int32)
        weights = np.empty(n - 1)
        cur = 0
        for e in range(n - 1):
            in_tree[cur] = True
            sel = -1
            for j in range(n):
                if in_tree[j]:
                    continue
                d2 = 0.0
                for c in range(dim):
                    df = X[cur, c] - X[j, c]
                    d2 += df * df
                w = max(core[cur], core[j], math.sqrt(d2))
                a, b = min(cur, j), max(cur, j)
                if less(w, a, b, bw[j], ba[j], bb[j]):
                    bw[j], ba[j], bb[j] = w, a, b
                if sel < 0 or less(bw[j], ba[j], bb[j], bw[sel], ba[sel], bb[sel]):
                    sel = j
            edges[e, 0], edges[e, 1], weights[e] = ba[sel], bb[sel], bw[sel]
            cur = sel
        return edges, weights

    return {"prim": prim}


def prim_mst(x, core):
    """The numba twin of ``prim_mst_port`` (no fastmath: bit for bit the port)."""
    if not _NB:
        _NB.update(_build_numba())
    edges, weights = _NB["prim"](_as64(x), np.ascontiguousarray(core, np.float64))
    return canonical_sort(edges, weights)


def kruskal_mst(x, core):
    """Kruskal over all pairs in the canonical order (small N)."""
    X = _as64(x)
    n = X.shape[0]
    i, j = np.triu_indices(n, 1)
    d = np.sqrt(d2_rows(X, np.arange(n))[i, j])
    w = np.maximum(np.maximum(core[i], core[j]), d)
    order = np.lexsort((j, i, w))
    parent = list(range(n))

    def find(v):
        while parent[v] != v:
            parent[v] = parent[parent[v]]
            v = parent[v]
        return v

    edges, weights = [], []
    for e in order:
        ra, rb = find(int(i[e])), find(int(j[e]))
        if ra != rb:
            parent[ra] = rb
            edges.append((i[e], j[e]))
            weights.append(w[e])
    return np.array(edges, np.int32), np.array(weights)


def canonical_sort(edges, weights):
    """Orient every edge (min, max) and sort by (w, min, max)."""
    edges = np.asarray(edges)
    a = np.minimum(edges[:, 0], edges[:, 1]).astype(np.int32)
    b = np.maximum(edges[:, 0], edges[:, 1]).astype(np.int32)
    weights = np.asarray(weights, np.float64)
    order = np.lexsort((b, a, weights))
    return np.stack([a[order], b[order]], axis=1), weights[order]


def mst(x, core_k):
    """(core, edges, weights): the frozen device result."""
    core = core_distances(x, core_k)
    edges, weights = prim_mst(x, core)
    return core, edges, weights


# ---------------------------------------------------------------------------------------------
# scikit-learn 1.9.0's tree routines, in plain Python
# ---------------------------------------------------------------------------------------------
def make_single_linkage(edges, weights):
    """_linkage.pyx make_single_linkage over edges in the given order: rows (left, right, value, size)."""
    m = len(weights)
    n = m + 1
    parent = [-1] * (2 * n - 1)
    size = [1] * n + [0] * (n - 1)
    next_label = n

    def fast_find(x):
        p = x
        while parent[x] != -1:
            x = parent[x]
        while parent[p] != x:
            p, parent[p] = parent[p], x
        return x

    out = []
    for e in range(m):
        a, b = fast_find(int(edges[e][0])), fast_find(int(edges[e][1]))
        if a == b:
            raise ValueError("edge %d closes a cycle" % e)
        out.append((a, b, float(weights[e]), size[a] + size[b]))
        parent[a] = parent[b] = next_label
        size[next_label] = size[a] + size[b]
        next_label += 1
    return out


def _bfs_from_hierarchy(hier, root):
    n = len(hier) + 1
    q, out = [root], []
    while q:
        out.extend(q)
        q = [x - n for x in q if x >= n]
        if q:
            nxt = []
            for node in q:
                nxt.extend([hier[node][0], hier[node][1]])
            q = nxt
    return out


def condense_tree(hier, min_cluster_size):
    """_tree.pyx _condense_tree: rows (parent, child, lambda, size)."""
    root = 2 * len(hier)
    n = len(hier) + 1
    next_label = n + 1
    node_list = _bfs_from_hierarchy(hier, root)
    relabel = [0] * (root + 1)
    relabel[root] = n
    ignore = [False] * len(node_list)
    out = []
    for node in node_list:
        if ignore[node] or node < n:
            continue
        left, right, distance, _ = hier[node - n]
        lam = 1.0 / distance if distance > 0.0 else math.inf
        lc = hier[left - n][3] if left >= n else 1
        rc = hier[right - n][3] if right >= n else 1
        if lc >= min_cluster_size and rc >= min_cluster_size:
            relabel[left] = next_label
            next_label += 1
            out.append((relabel[node], relabel[left], lam, lc))
            relabel[right] = next_label
            next_label += 1
            out.append((relabel[node], relabel[right], lam, rc))
            continue
        if lc < min_cluster_size and rc < min_cluster_size:
            shed = (left, right)
        elif lc < min_cluster_size:
            relabel[right] = relabel[node]
            shed = (left,)
        else:
            relabel[left] = relabel[node]
            shed = (right,)
        for side in shed:
            for sub in _bfs_from_hierarchy(hier, side):
                if sub < n:
                    out.append((relabel[node], sub, lam, 1))
                ignore[sub] = True
    return out


def compute_stability(ct):
    parents = [r[0] for r in ct]
    smallest, largest_parent = min(parents), max(parents)
    largest_child = max(max(r[1] for r in ct), smallest)
    births = [math.nan] * (largest_child + 1)
    for p, c, v, s in ct:
        births[c] = v
    births[smallest] = 0.0
    result = [0.0] * (largest_parent - smallest + 1)
    for p, c, v, s in ct:
        result[p - smallest] += (v - births[p]) * s
    return {i + smallest: result[i] for i in range(len(result))}


def _max_lambdas(ct):
    deaths = [0.0] * (max(r[0] for r in ct) + 1)
    cur, mx = ct[0][0], ct[0][2]
    for p, c, v, s in ct[1:]:
        if p == cur:
            mx = max(mx, v)
        else:
            deaths[cur] = mx
            cur, mx = p, v
    deaths[cur] = mx
    return deaths


def get_clusters(ct, stability, allow_single_cluster):
    """_get_clusters with eom, no epsilon, no max_cluster_size: (labels, probabilities, n_clusters)."""
    node_list = sorted(stability, reverse=True)
    if not allow_single_cluster:
        node_list = node_list[:-1]
    tree = [r for r in ct if r[3] > 1]
    is_cluster = {c: True for c in node_list}
    kids = {}
    for p, c, v, s in tree:
        kids.setdefault(p, []).append(c)
    for node in node_list:
        sub = 0.0
        for c in kids.get(node, []):
            sub = sub + stability[c]
        if sub > stability[node]:
            is_cluster[node] = False
            stability[node] = sub
        else:
            q = list(kids.get(node, []))
            while q:
                x = q.pop()
                is_cluster[x] = False
                q.extend(kids.get(x, []))
    clusters = sorted(c for c in is_cluster if is_cluster[c])
    cluster_map = {c: i for i, c in enumerate(clusters)}
    labels = _do_labelling(ct, set(clusters), cluster_map, allow_single_cluster)
    probs = _get_probabilities(ct, {i: c for c, i in cluster_map.items()}, labels)
    return labels, probs, len(clusters)


def _do_labelling(ct, clusters, cluster_map, allow_single_cluster):
    root = min(r[0] for r in ct)
    size = max(r[0] for r in ct) + 1
    par, rank = list(range(size)), [0] * size

    def find(x):
        r = x
        while par[r] != r:
            r = par[r]
        while par[x] != r:
            par[x], x = r, par[x]
        return r

    for p, c, v, s in ct:
        if c not in clusters:
            xr, yr = find(p), find(c)
            if rank[xr] < rank[yr]:
                par[xr] = yr
            elif rank[xr] > rank[yr]:
                par[yr] = xr
            else:
                par[yr] = xr
                rank[xr] += 1
    labels = np.empty(root, np.int64)
    threshold = None
    point_lambda = {r[1]: r[2] for r in ct if r[1] < root}
    for n in range(root):
        cluster = find(n)
        label = -1
        if cluster != root:
            label = cluster_map[cluster]
        elif len(clusters) == 1 and allow_single_cluster:
            lam = point_lambda[n]
            if threshold is None:
                threshold = max(r[2] for r in ct if r[0] == cluster)
            if lam >= threshold:
                label = cluster_map[cluster]
        labels[n] = label
    return labels


def _get_probabilities(ct, reverse_map, labels):
    out = np.zeros(len(labels))
    deaths = _max_lambdas(ct)
    root = min(r[0] for r in ct)
    for p, c, v, s in ct:
        if c >= root or labels[c] == -1:
            continue
        max_lambda = deaths[reverse_map[labels[c]]]
        if max_lambda == 0.0 or math.isinf(v):
            out[c] = 1.0
        else:
            out[c] = min(v, max_lambda) / max_lambda
    return out


def tree_to_labels(edges, weights, min_cluster_size, allow_single_cluster=False):
    """(labels int64, probabilities float64, n_clusters) of an MST whose edges are in the order to consume."""
    ct = condense_tree(make_single_linkage(edges, weights), min_cluster_size)
    return get_clusters(ct, compute_stability(ct), allow_single_cluster)


def sklearn_tree_to_labels(edges, weights, min_cluster_size, allow_single_cluster=False):
    """scikit-learn's own make_single_linkage + tree_to_labels over the edges in the given order."""
    from sklearn.cluster._hdbscan._linkage import MST_edge_dtype, make_single_linkage as msl
    from sklearn.cluster._hdbscan._tree import tree_to_labels as ttl
    m = np.empty(len(weights), dtype=MST_edge_dtype)
    m["current_node"], m["next_node"], m["distance"] = edges[:, 0], edges[:, 1], weights
    return ttl(msl(m), min_cluster_size, "eom", allow_single_cluster)


def sklearn_prim(x, core):
    """scikit-learn's own exact Prim MST (mst_from_data_matrix): (edges, weights) in its order."""
    from sklearn.cluster._hdbscan._linkage import mst_from_data_matrix
    from sklearn.metrics import DistanceMetric
    m = mst_from_data_matrix(_as64(x), np.ascontiguousarray(core, np.float64), DistanceMetric.get_metric("euclidean"), 1.0)
    return np.stack([m["current_node"], m["next_node"]], axis=1), m["distance"]
