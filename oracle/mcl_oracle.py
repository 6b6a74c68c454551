"""MCL (Markov clustering) as this library defines it, frozen for K11 (TEST INFRASTRUCTURE ONLY).

karma runs ``mcl - --abc -o -`` once per k-mer cluster (``Mcl.run_pipe``).  The semantics below are the library's
definition; where they rest on memory of mcl 14-137 rather than on its source they are marked "unpinned" (DESIGN §3
K11 lists them).  Everything is fp64, every product and sum rounded separately (no FMA), every sum a left fold from 0.0
in the order stated.

  * input: an abc stream, an ordered list of edges (u, v, w); labels are numbered by first appearance (u before v);
    refused (ValueError): u == v, the same unordered pair twice, w not finite or <= 0
  * A: symmetric adjacency plus loops A[j, j] = max_i A[i, j] (unpinned); M = A / column sum (ascending rows)
  * one iteration: expansion E[:, j] = sum over k ascending of M[:, k] * M[k, j]; a row is present iff its sum != 0;
    pruning per column (``prune_column``; P, S, R, pct unpinned); inflation x**I (x*x at I = 2) and renormalisation;
    chaos = max_j max(0, max_i M[i, j] / sum_i M[i, j]^2 - 1); the graph has converged when chaos < 1e-4 (unpinned),
    an error after 1000 iterations
  * interpretation (``interpret``): attractors M[a, a] > 0, systems = connected attractors, numbered by their smallest
    attractor; a node in several systems joins the smallest number (unpinned); a node reaching no attractor is alone
  * output: clusters by size descending, then smallest member; members ascending (unpinned)

``mcl_stream`` is the plain-Python reference of one stream; ``mcl_union`` is its numba twin on the block-diagonal union
of many groups, each group frozen when it converges (what the device computes); ``groups_oracle`` segments a graph's
edge arrays into groups as ``kb_mcl_build`` does.
"""
import math

import numpy as np

P, S, R, PCT = 7000, 900, 1000, 90          # mcl 14-137's default resource scheme, as remembered (unpinned)
CUTOFF = 1.0 / P
RECOVER = PCT / 100.0
CHAOS_EPS = 1e-4                              # unpinned
MAX_ITER = 1000
CAP = max(S, R)                               # entries a column can hold after pruning


class NotConverged(RuntimeError):
    pass


# ---------------------------------------------------------------------------------------------
# input
# ---------------------------------------------------------------------------------------------
def check_inflation(inflation):
    if isinstance(inflation, bool) or not isinstance(inflation, (int, float, np.integer, np.floating)) \
            or not math.isfinite(inflation) or inflation <= 1:
        raise ValueError("inflation must be a finite number > 1, got %r" % (inflation,))
    return float(inflation)


def label_stream(edges):
    """abc stream -> (labels in first-appearance order, [(u_local, v_local, w)]); refusals as ValueError."""
    index, labels, out, seen = {}, [], [], set()
    for u, v, w in edges:
        w = float(w)
        if u == v:
            raise ValueError("self-edge %r" % (u,))
        if not math.isfinite(w) or w <= 0:
            raise ValueError("edge (%r, %r): weight %r is not finite and > 0" % (u, v, w))
        for x in (u, v):
            if x not in index:
                index[x] = len(labels)
                labels.append(x)
        a, b = index[u], index[v]
        key = (min(a, b), max(a, b))
        if key in seen:
            raise ValueError("edge (%r, %r) is listed twice" % (u, v))
        seen.add(key)
        out.append((a, b, w))
    return labels, out


def _fold(xs):
    s = 0.0
    for x in xs:
        s += x
    return s


def initial_columns(n, edges):
    """M as columns of (row, value) in ascending row order."""
    cols = [dict() for _ in range(n)]
    for a, b, w in edges:
        cols[b][a] = w
        cols[a][b] = w
    out = []
    for j in range(n):
        cols[j][j] = max(cols[j].values())
        col = sorted(cols[j].items())
        s = _fold(v for _, v in col)
        out.append([(i, v / s) for i, v in col])
    return out


# ---------------------------------------------------------------------------------------------
# one iteration (plain Python)
# ---------------------------------------------------------------------------------------------
def prune_column(col, stats=None):
    """E's column (row, value) in ascending rows, values > 0 -> the kept entries in ascending rows, renormalised.
    The kept set is always a prefix of the entries ordered by (value desc, row asc): cutoff keeps those >= 1/P;
    selection keeps the S largest if more remain; recovery then adds the next largest while fewer than R are kept and
    the kept mass (the kept entries summed in ascending rows, then each recovered one added) is < pct/100 of the column's
    mass T (ascending rows).  The kept entries are divided by their sum in ascending rows."""
    vals = [v for _, v in col]
    m = len(col)
    total = _fold(vals)
    c = sum(1 for v in vals if v >= CUTOFF)
    order = None

    def sorted_order():
        return sorted(range(m), key=lambda i: (-vals[i], col[i][0]))

    def kept_by(b):
        vb, rb = vals[b], col[b][0]
        return [(r, v) for r, v in col if v > vb or (v == vb and r <= rb)]

    if c > S:
        order = sorted_order()
        k = S
        kept = kept_by(order[k - 1])
    else:
        k = c
        kept = [(r, v) for r, v in col if v >= CUTOFF]
    mass = _fold(v for _, v in kept)
    recovered = 0
    if k < R and k < m and mass < RECOVER * total:
        if order is None:
            order = sorted_order()
        while k < R and k < m and mass < RECOVER * total:
            mass += vals[order[k]]
            k += 1
            recovered += 1
        kept = kept_by(order[k - 1])
    if stats is not None:
        stats.append({"entries": m, "over_cutoff": c, "kept": k, "selected": c > S, "recovered": recovered,
                      "mass": total, "kept_mass": _fold(v for _, v in kept)})
    s = _fold(v for _, v in kept)
    return [(r, v / s) for r, v in kept]


def inflate_column(col, inflation):
    """(column with entries > 0 in ascending rows, its chaos)."""
    if inflation == 2.0:
        ys = [(r, x * x) for r, x in col]
    else:
        ys = [(r, math.pow(x, inflation)) for r, x in col]
    s = _fold(y for _, y in ys)
    zs = [(r, y / s) for r, y in ys if y / s > 0]
    mx = max(z for _, z in zs)
    sq = _fold(z * z for _, z in zs)
    return zs, max(0.0, mx / sq - 1.0)


def iterate(cols, inflation, stats=None):
    """One MCL iteration over a graph's columns -> (new columns, chaos)."""
    out, chaos = [], 0.0
    for colj in cols:
        acc = {}
        for k, mkj in colj:
            for i, mik in cols[k]:
                acc[i] = acc.get(i, 0.0) + mik * mkj
        e = [(i, a) for i, a in sorted(acc.items()) if a != 0]
        z, ch = inflate_column(prune_column(e, stats), inflation)
        out.append(z)
        chaos = max(chaos, ch)
    return out, chaos


def mcl_matrix(n, edges, inflation=2.0, on_iterate=None, stats=None):
    """(final columns, iterations) of a graph given as local edges."""
    cols = initial_columns(n, edges)
    for it in range(1, MAX_ITER + 1):
        cols, chaos = iterate(cols, inflation, stats)
        if on_iterate is not None:
            on_iterate(it, cols, chaos)
        if chaos < CHAOS_EPS:
            return cols, it
    raise NotConverged("graph did not converge in %d iterations" % MAX_ITER)


# ---------------------------------------------------------------------------------------------
# interpretation and output order
# ---------------------------------------------------------------------------------------------
def interpret(n, cols):
    """Final columns (local rows) -> (clusters as ascending local index lists in output order, overlap count)."""
    attractor = [any(i == j and v > 0 for i, v in cols[j]) for j in range(n)]
    parent = list(range(n))

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    for b in range(n):
        if attractor[b]:
            for a, v in cols[b]:
                if v > 0 and attractor[a]:
                    ra, rb = find(a), find(b)
                    if ra != rb:
                        parent[max(ra, rb)] = min(ra, rb)          # roots stay the smallest attractor
    system = [find(j) if attractor[j] else -1 for j in range(n)]
    members, overlap = {}, 0
    for j in range(n):
        s = {system[a] for a, v in cols[j] if v > 0 and attractor[a]}
        if len(s) > 1:
            overlap += 1
        key = min(s) if s else ("alone", j)
        members.setdefault(key, []).append(j)
    clusters = sorted(members.values(), key=lambda c: (-len(c), c[0]))
    return clusters, overlap


def mcl_stream(edges, inflation=2.0):
    """The plain-Python reference of one abc stream: dict(labels, clusters (local indices), lines (names), iterations,
    overlap, columns)."""
    inflation = check_inflation(inflation)
    labels, local = label_stream(edges)
    if not labels:
        return {"labels": [], "clusters": [], "lines": [], "iterations": 0, "overlap": 0, "columns": []}
    cols, it = mcl_matrix(len(labels), local, inflation)
    clusters, overlap = interpret(len(labels), cols)
    return {"labels": labels, "clusters": clusters, "lines": [[labels[i] for i in c] for c in clusters],
            "iterations": it, "overlap": overlap, "columns": cols}


# ---------------------------------------------------------------------------------------------
# many groups: segmentation as kb_mcl_build does it, and the numba twin on the block-diagonal union
# ---------------------------------------------------------------------------------------------
def segment(n_nodes, a, b, w, group, n_groups):
    """Edge arrays + group per node -> dict(local int32[n_nodes] (-1 outside every stream), size int64[n_groups],
    off int64[n_groups + 1], col_group int32[n_cols], streams [local edge list per group]).  An edge belongs to group g
    when both ends are in g; each group's local indices follow first appearance in its edges in the given order."""
    a, b, w, group = (np.asarray(x) for x in (a, b, w, group))
    local = np.full(n_nodes, -1, np.int32)
    size = np.zeros(n_groups, np.int64)
    streams = [[] for _ in range(n_groups)]
    seen = set()
    for u, v, x in zip(a.tolist(), b.tolist(), w.tolist()):
        g = int(group[u])
        if g < 0 or g != group[v]:
            continue
        if u == v:
            raise ValueError("self-edge at node %d" % u)
        if not math.isfinite(x) or x <= 0:
            raise ValueError("edge (%d, %d): weight %r is not finite and > 0" % (u, v, x))
        key = (min(u, v), max(u, v))
        if key in seen:
            raise ValueError("edge (%d, %d) is listed twice" % (u, v))
        seen.add(key)
        for y in (u, v):
            if local[y] < 0:
                local[y] = size[g]
                size[g] += 1
        streams[g].append((int(local[u]), int(local[v]), x))
    off = np.zeros(n_groups + 1, np.int64)
    off[1:] = np.cumsum(size)
    col_group = np.repeat(np.arange(n_groups, dtype=np.int32), size)
    return {"local": local, "size": size, "off": off, "col_group": col_group, "streams": streams}


_NB = {}


def _build_numba():
    import numba

    @numba.njit(cache=False)
    def fold(x, n):
        s = 0.0
        for i in range(n):
            s += x[i]
        return s

    @numba.njit(cache=False)
    def column(j, base, ptr, ln, rows, vals, acc, seen, touched, lrow, lval, inflation, orow, oval):
        """One column of one iteration; rows are union indices.  Returns (entries written, chaos)."""
        p0 = ptr[j]
        nt = 0
        for t in range(ln[j]):
            k = rows[p0 + t]
            mkj = vals[p0 + t]
            q0 = ptr[k]
            for u in range(ln[k]):
                i = rows[q0 + u] - base
                acc[i] = acc[i] + vals[q0 + u] * mkj
                if not seen[i]:
                    seen[i] = True
                    touched[nt] = i
                    nt += 1
        rs = np.sort(touched[:nt])
        m = 0
        for t in range(nt):
            i = rs[t]
            if acc[i] != 0.0:
                lrow[m] = i
                lval[m] = acc[i]
                m += 1
            acc[i] = 0.0
            seen[i] = False
        total = fold(lval, m)
        c = 0
        for i in range(m):
            if lval[i] >= 1.0 / 7000.0:
                c += 1
        kept = np.zeros(m, np.bool_)
        order = np.empty(0, np.int64)
        if c > 900:
            order = np.argsort(-lval[:m], kind="mergesort")
            k = 900
            b = order[k - 1]
            for i in range(m):
                kept[i] = lval[i] > lval[b] or (lval[i] == lval[b] and lrow[i] <= lrow[b])
        else:
            k = c
            for i in range(m):
                kept[i] = lval[i] >= 1.0 / 7000.0
        mass = 0.0
        for i in range(m):
            if kept[i]:
                mass += lval[i]
        lim = 0.9 * total
        if k < 1000 and k < m and mass < lim:
            if order.shape[0] == 0:
                order = np.argsort(-lval[:m], kind="mergesort")
            while k < 1000 and k < m and mass < lim:
                mass += lval[order[k]]
                k += 1
            b = order[k - 1]
            for i in range(m):
                kept[i] = lval[i] > lval[b] or (lval[i] == lval[b] and lrow[i] <= lrow[b])
        s = 0.0
        for i in range(m):
            if kept[i]:
                s += lval[i]
        sy = 0.0
        for i in range(m):
            if kept[i]:
                x = lval[i] / s
                y = x * x if inflation == 2.0 else math.pow(x, inflation)
                lval[i] = y
                sy += y
        n_out = 0
        mx = 0.0
        for i in range(m):
            if kept[i]:
                z = lval[i] / sy
                if z > 0:
                    orow[n_out] = lrow[i] + base
                    oval[n_out] = z
                    n_out += 1
                    if z > mx:
                        mx = z
        sq = 0.0
        for i in range(n_out):
            sq += oval[i] * oval[i]
        return n_out, max(0.0, mx / sq - 1.0)

    @numba.njit(cache=False)
    def union(ptr, ln0, rows0, vals0, col_group, off, n_groups, inflation, max_iter):
        n_cols = ptr.shape[0]
        rows = np.empty((2, rows0.shape[0]), np.int32)
        vals = np.empty((2, rows0.shape[0]))
        ln = np.empty((2, n_cols), np.int64)
        rows[0, :] = rows0
        vals[0, :] = vals0
        ln[0, :] = ln0
        maxg = 1
        for g in range(n_groups):
            maxg = max(maxg, off[g + 1] - off[g])
        acc = np.zeros(maxg)
        seen = np.zeros(maxg, np.bool_)
        touched = np.empty(maxg, np.int32)
        lrow = np.empty(maxg, np.int32)
        lval = np.empty(maxg)
        iters = np.zeros(n_groups, np.int64)
        active = np.zeros(n_groups, np.bool_)
        for g in range(n_groups):
            active[g] = off[g + 1] > off[g]
        chaos = np.zeros(n_groups)
        any_active = True
        t = 0
        while any_active:
            t += 1
            if t > max_iter:
                for g in range(n_groups):
                    if active[g]:
                        return rows, vals, ln, iters, g
            cur, nxt = (t - 1) % 2, t % 2
            chaos[:] = 0.0
            for j in range(n_cols):
                g = col_group[j]
                if not active[g]:
                    continue
                base = off[g]
                n_out, ch = column(j, base, ptr, ln[cur], rows[cur], vals[cur], acc, seen, touched, lrow, lval,
                                   inflation, rows[nxt, ptr[j]:], vals[nxt, ptr[j]:])
                ln[nxt, j] = n_out
                if ch > chaos[g]:
                    chaos[g] = ch
            any_active = False
            for g in range(n_groups):
                if active[g]:
                    if chaos[g] < 1e-4:
                        active[g] = False
                        iters[g] = t
                    else:
                        any_active = True
        return rows, vals, ln, iters, -1

    return {"union": union}


def union_csc(seg, a, b, w, group):
    """The block-diagonal M of ``segment``'s groups in the fixed-capacity layout: column j at ptr[j] with room for
    min(n_g, CAP) entries and at least its initial degree + 1; rows are union indices."""
    n_cols = int(seg["off"][-1])
    cols = [None] * n_cols
    for g, stream in enumerate(seg["streams"]):
        if not stream:
            continue
        base = int(seg["off"][g])
        for j, col in enumerate(initial_columns(int(seg["size"][g]), stream)):
            cols[base + j] = [(i + base, v) for i, v in col]
    cap = np.array([max(len(cols[j]), min(int(seg["size"][seg["col_group"][j]]), CAP)) for j in range(n_cols)], np.int64)
    ptr = np.zeros(n_cols, np.int64)
    if n_cols:
        ptr[1:] = np.cumsum(cap)[:-1]
    total = int(cap.sum())
    rows = np.zeros(total, np.int32)
    vals = np.zeros(total)
    ln = np.zeros(n_cols, np.int64)
    for j, col in enumerate(cols):
        ln[j] = len(col)
        for t, (i, v) in enumerate(col):
            rows[ptr[j] + t] = i
            vals[ptr[j] + t] = v
    return ptr, ln, rows, vals


def mcl_union(seg, a, b, w, group, inflation=2.0):
    """The numba twin on the union of ``segment``'s groups: dict(iterations int64[G], columns [per union column, (local
    row, value) in ascending rows]).  Raises NotConverged naming the group."""
    inflation = check_inflation(inflation)
    if not _NB:
        _NB.update(_build_numba())
    ptr, ln, rows, vals = union_csc(seg, a, b, w, group)
    n_groups = len(seg["size"])
    rows, vals, lns, iters, bad = _NB["union"](ptr, ln, rows, vals, seg["col_group"], seg["off"], n_groups, inflation,
                                                MAX_ITER)
    if bad >= 0:
        raise NotConverged("group %d did not converge in %d iterations" % (bad, MAX_ITER))
    cols = []
    for j in range(len(ptr)):
        g = int(seg["col_group"][j])
        buf = int(iters[g]) % 2
        base = int(seg["off"][g])
        p = int(ptr[j])
        cols.append([(int(rows[buf, p + t]) - base, float(vals[buf, p + t])) for t in range(int(lns[buf, j]))])
    return {"iterations": iters, "columns": cols}


def groups_oracle(n_nodes, a, b, w, group, n_groups, inflation=2.0, twin=True):
    """What ``kb_mcl_build`` + ``kb_mcl_fetch`` return, from the numba twin on the union (``twin``) or from the
    plain-Python reference run on each group's stream separately: dict(local, cluster int32[n_nodes], n_clusters,
    iterations, overlap int64[n_groups], columns, clusters [per group, lists of local indices in output order])."""
    inflation = check_inflation(inflation)
    seg = segment(n_nodes, a, b, w, group, n_groups)
    off = seg["off"]
    if twin:
        res = mcl_union(seg, a, b, w, group, inflation)
        iters, columns = res["iterations"], res["columns"]
    else:
        iters, columns = np.zeros(n_groups, np.int64), []
        for g, stream in enumerate(seg["streams"]):
            if stream:
                cols, iters[g] = mcl_matrix(int(seg["size"][g]), stream, inflation)
                columns.extend(cols)
    cluster = np.full(n_nodes, -1, np.int32)
    n_clusters = np.zeros(n_groups, np.int64)
    overlap = np.zeros(n_groups, np.int64)
    clusters = []
    node_of = np.full(int(off[-1]), -1, np.int64)
    inside = np.flatnonzero(seg["local"] >= 0)
    node_of[off[np.asarray(group)[inside]] + seg["local"][inside]] = inside
    for g in range(n_groups):
        cg, overlap[g] = interpret(int(seg["size"][g]), columns[off[g]:off[g + 1]])
        n_clusters[g] = len(cg)
        clusters.append(cg)
        for c, members in enumerate(cg):
            for i in members:
                cluster[node_of[off[g] + i]] = c
    return {"local": seg["local"], "cluster": cluster, "n_clusters": n_clusters, "iterations": iters,
            "overlap": overlap, "columns": columns, "clusters": clusters, "size": seg["size"]}
