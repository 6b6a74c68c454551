"""Inter-group connection weights (SURVEY 8f rank 4, `--rearrange`): the oracle pinned to goldens
produced by the real reference functions, the host logic, and (GPU) kb_links_build against both."""
import json
import os

import numpy as np
import pytest

from oracle import links_oracle as lo
from oracle import readgraph_oracle as ro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUTOFFS = (0, 0.25, 1.5)


@pytest.fixture(scope="module")
def lk_golden():
    with open(os.path.join(ROOT, "tests", "golden", "links_golden.json")) as f:
        return json.load(f)["cases"]


def _oracle_graph(c):
    """Adjacency of the read graph of a golden case, from the read-graph oracle (itself golden-pinned)."""
    r = ro.build(c["names"], [(f, ids, k) for f, ids, k in c["classes"]], c["fasta_keys"])
    nodes = r["nodes"]
    return nodes, lo.adjacency(nodes, [(nodes[a], nodes[b], w) for a, b, w in r["edges"]])


def _expand(rle):
    return [[a, b] for a, b, n in rle for _ in range(n)]


def test_oracle_matches_reference_golden(lk_golden):
    assert len(lk_golden) >= 4
    for c in lk_golden:
        _, adj = _oracle_graph(c)
        lookup = lo.lookup_dict(c["clusters_with_subcluster"])
        for cutoff in CUTOFFS:
            assert lo.connections_between_subclusters(adj, lookup, cutoff) == _expand(c["connections"][repr(cutoff)]), (c["name"], cutoff)
        table = {(a, b): (w, e, o) for a, b, w, e, o in lo.pair_table(adj, lookup, 0)}
        assert [[a, b, w.hex()] for (a, b), (w, _, _) in table.items()] == c["pair_weights"], c["name"]
        for t in c["two_lists"]:
            assert float(lo.distance_between_subgraphs(adj, t["nodes_a"], t["nodes_b"])).hex() == t["weight"], c["name"]


def test_roles_and_argument_errors():
    from karma_b200 import rearrange as rr
    index = {"a": 0, "b": 1, "c": 2, "d": 3}
    g, p, m = rr._roles(index, [["c", "zz", "a"], ["d"]], "t")
    assert g.tolist() == [0, -1, 0, 1] and p.tolist() == [2, -1, 0, 0] and m == 3
    with pytest.raises(ValueError):
        rr._roles(index, [["a", "b"], ["a"]], "t")
    with pytest.raises(NameError):                      # the reference's own failure mode, karma.py:114
        rr.calc_connections_between_mcl_subclusters({0: {"mcl_subcluster": ["a"]}})


# ------------------------------------------------------------------ GPU
def _gpu_graph(engine, c, tmp_path):
    from karma_b200 import read_graph as rg
    path = str(tmp_path / (c["name"] + ".txt"))
    ro.write_eq_file(path, c["names"], [(f, ids, k) for f, ids, k in c["classes"]])
    return rg.from_equivalence_classes(path, {k: "" for k in c["fasta_keys"]}, engine=engine)


@pytest.mark.gpu
def test_gpu_links_match_reference_golden(engine, lk_golden, tmp_path):
    from karma_b200 import rearrange as rr
    for c in lk_golden:
        graph = _gpu_graph(engine, c, tmp_path)
        lookup = lo.lookup_dict(c["clusters_with_subcluster"])
        for cutoff in CUTOFFS:
            got = rr.calc_connections_between_mcl_subclusters(lookup, weight_cutoff=cutoff, full_graph=graph, engine=engine)
            assert got == _expand(c["connections"][repr(cutoff)]), (c["name"], cutoff)
        keys, t = rr.subcluster_link_table(lookup, graph, 0, engine)
        assert [[keys[a], keys[b], float(w).hex()] for a, b, w in zip(t["group_a"].tolist(), t["group_b"].tolist(), t["weight"].tolist())] \
            == c["pair_weights"], c["name"]                                        # float64 sums bit for bit
        for tl in c["two_lists"]:
            got = rr.calc_distance_between_subgraphs(graph, tl["nodes_a"], tl["nodes_b"], engine=engine)
            assert float(got).hex() == tl["weight"], c["name"]


@pytest.mark.gpu
def test_gpu_links_larger_graph_against_oracle(engine, tmp_path):
    from karma_b200 import read_graph as rg
    from karma_b200 import rearrange as rr
    names, classes = ro.synth_eq_classes(3000, 40000, seed=17, family=6, max_size=8, p_cross=0.2)
    path = str(tmp_path / "eq.txt")
    ro.write_eq_file(path, names, classes)
    graph = rg.from_equivalence_classes(path, {">" + x: "" for x in names}, engine=engine)
    nodes = list(graph.nodes())
    adj = lo.adjacency(nodes, [(a, b, d["weight"]) for a, b, d in graph.edges(data=True)])
    rng = np.random.default_rng(23)
    order = [nodes[i] for i in rng.permutation(len(nodes))]
    subs, i = [], 0
    while i < len(order):
        k = int(rng.integers(1, 30))
        subs.append(order[i:i + k])
        i += k
    lookup = {10 * j + 3: {"previous_cluster": 1, "mcl_subcluster": s} for j, s in enumerate(subs)}   # keys need not be 0..S-1
    want = lo.pair_table(adj, lookup, 0.3)
    keys, t = rr.subcluster_link_table(lookup, graph, 0.3, engine)
    got = [(keys[a], keys[b], w, e, o) for a, b, w, e, o in zip(t["group_a"].tolist(), t["group_b"].tolist(), t["weight"].tolist(),
                                                                t["edges"].tolist(), t["over"].tolist())]
    assert len(got) == len(want) > 1000
    assert [(a, b, float(w).hex(), e, o) for a, b, w, e, o in got] == [(a, b, float(w).hex(), e, o) for a, b, w, e, o in want]
    assert sum(t["edges"].tolist()) <= graph.number_of_edges()
    # cached edge arrays are reused while the graph is unchanged and rebuilt after a change
    assert rr.graph_arrays(graph) is rr.graph_arrays(graph)
    before = rr.graph_arrays(graph)
    graph.add_edge(order[0], order[-1], weight=0.5) if not graph.has_edge(order[0], order[-1]) else graph.remove_edge(order[0], order[-1])
    assert rr.graph_arrays(graph) is not before


@pytest.mark.gpu
def test_gpu_links_degenerate_inputs(engine):
    import networkx as nx
    from karma_b200 import rearrange as rr
    g = nx.Graph()
    g.add_nodes_from(["a", "b", "c"])
    lookup = lo.lookup_dict([[["a"], ["b", "c"]]])
    assert rr.calc_connections_between_mcl_subclusters(lookup, full_graph=g, engine=engine) == []       # no edges at all
    g.add_edge("b", "c", weight=0.75)
    assert rr.calc_connections_between_mcl_subclusters(lookup, full_graph=g, engine=engine) == []       # only inside one group
    g.add_edge("a", "a", weight=0.5)                                                                    # self loop
    g.add_edge("a", "c", weight=0.25)
    assert rr.calc_connections_between_mcl_subclusters(lookup, full_graph=g, engine=engine) == [[0, 1]]
    assert rr.calc_connections_between_mcl_subclusters(lookup, weight_cutoff=0.25, full_graph=g, engine=engine) == []
    # two lists sharing nodes: product visits (a,a) once, (a,c) and (c,a)
    assert rr.calc_distance_between_subgraphs(g, ["a", "c"], ["c", "a"], engine=engine) == 0.25 + 0.5 + 0.25
    assert rr.calc_distance_between_subgraphs(g, [], ["a"], engine=engine) == 0
    with pytest.raises(ValueError):
        rr.calc_distance_between_subgraphs(g, ["a", "a"], ["c"], engine=engine)
