"""MCL on the GPU: the read graph's sub-clusters of every k-mer cluster in one device call (K11, ``kb_mcl_build``).

karma runs ``mcl - --abc -o -`` once per k-mer cluster on that cluster's subgraph of the read graph, and once on the
unlabeled contigs.  Here all of those streams form one block-diagonal matrix that iterates on the device; each group
stops on its own convergence, so its result is what a run of its stream alone gives::

    from karma_b200.mcl import mcl_groups, mcl_abc
    subclusters = mcl_groups(full_graph, k.clusters + k.unlabeled_cluster, inflation=2.0)
    subclusters[g]          # group g's clusters, as lists of node names, in mcl's output order
    mcl_abc([("a", "b", 0.5), ("b", "c", 0.25)])      # one abc stream -> its lines, split at tabs

The arithmetic is the library's definition of MCL, frozen in oracle/mcl_oracle.py; DESIGN §3 K11 lists where it rests on
memory of mcl 14-137 rather than on its source (loop weight, pruning constants, convergence threshold, overlap rule,
output order).  Only the inflation is a parameter.  There is no CPU fallback.
"""
import math
from ctypes import byref, c_int64, c_void_p

import numpy as np
import torch

from ._lib import check, ptr
from .rearrange import _engine, _roles, graph_arrays


def _inflation(inflation):
    if isinstance(inflation, bool) or not isinstance(inflation, (int, float, np.integer, np.floating)) \
            or not math.isfinite(inflation) or inflation <= 1:
        raise ValueError("inflation must be a finite number > 1, got %r" % (inflation,))
    return float(inflation)


def check_streams(a, b, w, group):
    """The refusals of ``kb_mcl_build`` on host arrays, as ValueError: inside a group no self-edge, no pair twice, and
    weights finite and > 0."""
    a = np.asarray(a, np.int64)
    b = np.asarray(b, np.int64)
    w = np.asarray(w, np.float64)
    group = np.asarray(group)
    ga, gb = group[a], group[b]
    inside = (ga >= 0) & (ga == gb)
    if (inside & (a == b)).any():
        raise ValueError("self-edge inside a group (node %d)" % int(a[inside & (a == b)][0]))
    bad = inside & ~(np.isfinite(w) & (w > 0))
    if bad.any():
        i = int(np.flatnonzero(bad)[0])
        raise ValueError("edge (%d, %d): weight %r is not finite and > 0" % (int(a[i]), int(b[i]), float(w[i])))
    key = np.minimum(a, b)[inside] * (int(max(a.max(initial=0), b.max(initial=0))) + 1) + np.maximum(a, b)[inside]
    if len(np.unique(key)) != len(key):
        raise ValueError("the same pair of nodes is listed twice inside a group")


def mcl_arrays(engine, n_nodes, d_a, d_b, d_w, d_group, n_groups, inflation=2.0, columns=False):
    """Array level: device int32 edge ends, float64 weights and int32 group ids (-1 = no group) in.  Returns numpy
    ``local`` and ``cluster`` (int32 per node, -1 outside every stream: the node's index in its group's stream and its
    cluster number in output order), ``n_clusters``, ``iterations`` and ``overlap`` (int64 per group: nodes that reached
    attractors of several systems).  With ``columns``, also the final matrix: ``colptr`` (int64, one column per stream
    node, groups in order, local indices within), ``rows`` (int32 local rows) and ``vals`` (float64)."""
    inflation = _inflation(inflation)
    for name, t, dt in (("a", d_a, torch.int32), ("b", d_b, torch.int32), ("w", d_w, torch.float64), ("group", d_group, torch.int32)):
        if not isinstance(t, torch.Tensor) or t.dtype != dt or t.dim() != 1 or t.device != engine.device:
            raise ValueError("%s must be a 1-d %s tensor on %s" % (name, dt, engine.device))
    if not (len(d_a) == len(d_b) == len(d_w)) or len(d_group) != n_nodes:
        raise ValueError("edge arrays must have one length, and group one entry per node")
    d_a, d_b, d_w, d_group = (t.contiguous() for t in (d_a, d_b, d_w, d_group))
    engine._bind_stream()
    n_cols, nnz = c_int64(), c_int64()
    check(engine.lib.kb_mcl_build(engine.ctx, int(n_nodes), len(d_a), ptr(d_a), ptr(d_b), ptr(d_w), ptr(d_group),
                                  int(n_groups), inflation, byref(n_cols), byref(nnz)))
    out = {"local": np.empty(n_nodes, np.int32), "cluster": np.empty(n_nodes, np.int32),
           "n_clusters": np.empty(n_groups, np.int64), "iterations": np.empty(n_groups, np.int64),
           "overlap": np.empty(n_groups, np.int64)}
    extra = [None, None, None]
    if columns:
        out.update(colptr=np.empty(n_cols.value + 1, np.int64), rows=np.empty(nnz.value, np.int32),
                   vals=np.empty(nnz.value, np.float64))
        extra = [out["colptr"], out["rows"], out["vals"]]
    arrays = [out[k] for k in ("local", "cluster", "n_clusters", "iterations", "overlap")] + extra
    check(engine.lib.kb_mcl_fetch(engine.ctx, *(None if x is None else x.ctypes.data_as(c_void_p) for x in arrays)))
    return out


def _split(names, group, res, n_groups):
    """Per group, the clusters as lists of names: clusters in output order, members by stream index."""
    node = np.flatnonzero(res["cluster"] >= 0)
    order = node[np.lexsort((res["local"][node], res["cluster"][node], group[node]))]
    out = [[[] for _ in range(int(res["n_clusters"][g]))] for g in range(n_groups)]
    for v, g, c in zip(order.tolist(), group[order].tolist(), res["cluster"][order].tolist()):
        out[g][c].append(names[v])
    return out


def mcl_groups(graph, groups, inflation=2.0, engine=None):
    """MCL of every group's subgraph of a networkx read graph (e.g. ``read_graph.from_equivalence_classes``) in one
    device call.  ``groups``: lists of node names (e.g. ``k.clusters + k.unlabeled_cluster``); a name the graph does
    not know is skipped, a name in two groups is a ValueError.  Group g's stream is the edges with both ends in g, in
    ``graph.edges()`` order.  Returns per group its clusters as lists of names (empty for a group without edges)."""
    inflation = _inflation(inflation)
    index, a, b, w = graph_arrays(graph)
    group, _, _ = _roles(index, groups, "groups")
    n_groups = len(groups)
    if len(a):
        check_streams(a, b, w, group)
    engine = _engine(engine)
    dev = engine.device
    res = mcl_arrays(engine, len(index), torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev),
                     torch.from_numpy(w).to(dev), torch.from_numpy(group).to(dev), n_groups, inflation)
    return _split(list(index), group, res, n_groups)


def mcl_abc(edges, inflation=2.0, engine=None):
    """One abc stream: ``(u, v, w)`` tuples with node names in, the lines ``mcl - --abc -o -`` prints (split at tabs)
    out, under this library's definition of MCL.  Labels are numbered by first appearance (u before v)."""
    inflation = _inflation(inflation)
    index, a, b, w = {}, [], [], []
    for u, v, x in edges:
        for y in (u, v):
            if y not in index:
                index[y] = len(index)
        a.append(index[u])
        b.append(index[v])
        w.append(float(x))
    if not a:
        return []
    a, b, w = np.array(a, np.int32), np.array(b, np.int32), np.array(w, np.float64)
    group = np.zeros(len(index), np.int32)
    check_streams(a, b, w, group)
    engine = _engine(engine)
    dev = engine.device
    res = mcl_arrays(engine, len(index), torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev),
                     torch.from_numpy(w).to(dev), torch.from_numpy(group).to(dev), 1, inflation)
    return _split(list(index), group, res, 1)[0]
