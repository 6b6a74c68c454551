"""Read-graph path (SURVEY 8f rank 3): oracle pinned to the real reference's goldens, the
native eq_classes parser, and (GPU) the device build against the oracle."""
import json
import os

import pytest

from oracle import readgraph_oracle as ro

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def rg_golden():
    with open(os.path.join(ROOT, "tests", "golden", "readgraph_golden.json")) as f:
        return json.load(f)["cases"]


def _classes(c):
    return [(f, ids, cnt) for f, ids, cnt in c["classes"]]


def test_oracle_matches_reference_golden(rg_golden):
    assert len(rg_golden) >= 5
    for c in rg_golden:
        r = ro.build(c["names"], _classes(c), c["fasta_keys"])
        n = len(c["names"])
        assert r["nodes"][:n] == c["nodes"][:n] and set(r["nodes"]) == set(c["nodes"]), c["name"]
        assert [[a, b, float(w).hex()] for a, b, w in r["edges"]] == c["edges"], c["name"]     # order + bit-exact weights
        assert all(r["adj"][int(k)] == v for k, v in c["adj"].items()), c["name"]


def test_native_parser_matches_python_parser(tmp_path, rg_golden):
    from karma_b200 import read_graph as rg
    for c in rg_golden:
        path = str(tmp_path / (c["name"] + ".txt"))
        ro.write_eq_file(path, c["names"], _classes(c))
        p = rg.parse(path)
        names, classes = ro.parse_eq_file(path)
        assert p["names"] == names
        off = p["class_off"].tolist()
        assert [p["ids"][off[i]:off[i + 1]].tolist() for i in range(len(classes))] == [ids for _, ids, _ in classes]
        assert p["counts"].tolist() == [cnt for _, _, cnt in classes]
        assert p["skip"].tolist() == [1 if f == "1" else 0 for f, _, _ in classes]


@pytest.mark.parametrize("threads", [1, 6])
@pytest.mark.parametrize("body,why", [
    ("2\t0\t5\t3\n", "contig id 5 out of range"),
    ("2\t0\t1\t3\n2\t0\t-1\t3\n", "negative contig id"),
    ("2\t0\t1\tx\n", "count is not an integer"),
    ("2\t0\t1\t\n", "empty count"),
    ("2\t0\t1\t4\n\n2\t0\t1\t4\n", "blank line (the reference fails to unpack it)"),
    ("2 0 1 4\n", "no tab at all"),
    ("2\t0\t1 \t4\n", "id with a trailing blank"),
])
def test_native_parser_rejects_bad_input(tmp_path, monkeypatch, body, why, threads):
    from karma_b200 import _lib, read_graph as rg
    monkeypatch.setenv("KB_HOST_THREADS", str(threads))
    monkeypatch.setenv("KB_EQ_MIN_CHUNK", "1")
    p = tmp_path / "bad.txt"
    p.write_text("2\n1\na\nb\n2\t0\t1\t7\n" + body + "1\t1\t2\n")
    with pytest.raises(_lib.KarmaB200Error):
        rg.parse(str(p))
    good = tmp_path / "good.txt"
    good.write_text("2\n1\na\nb\n2\t0\t1\t7\n1\t1\t2")         # last line without a newline
    got = rg.parse(str(good))
    assert got["names"] == ["a", "b"] and got["ids"].tolist() == [0, 1, 1] and got["counts"].tolist() == [7, 2]
    assert got["class_off"].tolist() == [0, 2, 3] and got["skip"].tolist() == [0, 1]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["golden", "large"])
def test_device_build_matches_oracle(engine, tmp_path, rg_golden, case):
    from karma_b200 import read_graph as rg
    if case == "golden":
        todo = [(c["names"], _classes(c), c["fasta_keys"]) for c in rg_golden]
    else:
        names, classes = ro.synth_eq_classes(20000, 300000, seed=5, family=6, max_size=9)
        names2, classes2 = ro.synth_eq_classes(300, 2000, seed=6, family=60, max_size=50, p_cross=0.3)   # big classes
        todo = [(names, classes, [">" + x for x in names] + [">only_in_fasta"]),
                (names2, classes2, [">" + x for x in names2])]
    for i, (names, classes, keys) in enumerate(todo):
        path = str(tmp_path / ("eq%d.txt" % i))
        ro.write_eq_file(path, names, classes)
        want = ro.build(names, classes, keys)
        g = rg.from_equivalence_classes(path, {k: "" for k in keys}, engine=engine)
        nodes = list(g.nodes())
        n = len(names)
        assert nodes[:n] == want["nodes"][:n] and set(nodes) == set(want["nodes"])
        idx = {k: j for j, k in enumerate(nodes)}
        got = [(idx[a], idx[b], d["weight"].hex()) for a, b, d in g.edges(data=True)]
        assert got == [(a, b, float(w).hex()) for a, b, w in want["edges"]]
        assert all([idx[x] for x in g.adj[nodes[k]]] == v for k, v in want["adj"].items() if k < n)
        tot, _, _, _ = rg.build_edges(engine, rg.parse(path))
        assert tot.tolist() == want["totals"]
