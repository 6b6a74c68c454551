"""K4 (SIMT and tcgen05) + K5 parity against the fp64 / exact-rational kNN oracle."""
import numpy as np
import pytest
import torch

from karma_b200 import _lib, synth
from karma_b200.engine import mode_of, profile_and_knn
from oracle import kmer_oracle as ko
from oracle import knn_oracle

pytestmark = pytest.mark.gpu

IMPLS = {"simt": _lib.KB_KNN_SIMT, "tc": _lib.KB_KNN_TC}


def _run(engine, asm, kmer_size, k, impl):
    return profile_and_knn(engine, asm.bases, asm.offsets, asm.key_len, kmer_size, n_neighbors=k, impl=IMPLS[impl])


@pytest.mark.parametrize("impl", ["simt", "tc"])
@pytest.mark.parametrize("kind,n,k", [("S1", 700, 2), ("S1", 700, 15), ("S0", 300, 5), ("S2", 900, 15), ("S1", 130, 24)])
def test_knn_parity_5p6(engine, impl, kind, n, k):
    asm = synth.make(kind, n)
    res = _run(engine, asm, "5p6", k, impl)
    cols, prof = ko.profile_np(asm.as_dict(), "5p6")
    assert res["columns"] == cols and res["profile"].tobytes() == prof.tobytes()
    rep = knn_oracle.check_knn(res["knn_idx"], res["knn_dist"], knn_oracle.d2_fp64(prof))
    assert knn_oracle.parity_ok(rep), rep


@pytest.mark.parametrize("impl", ["simt", "tc"])
@pytest.mark.parametrize("kmer_size", ["5+6", "4+5", 4, 7])
def test_knn_parity_other_modes(engine, impl, kmer_size):
    asm = synth.s1_families(400, seed=77)
    res = _run(engine, asm, kmer_size, 6, impl)
    counts, _ = ko.counts_mode(asm.bases, asm.offsets, kmer_size)
    if isinstance(kmer_size, int):
        counts = counts[:, counts.any(0)]             # kmer.py keeps observed columns only
    prof = counts / asm.key_len[:, None].astype(np.float64)
    assert res["profile"].tobytes() == prof.tobytes()
    rep = knn_oracle.check_knn(res["knn_idx"], res["knn_dist"], knn_oracle.d2_fp64(prof))
    assert knn_oracle.parity_ok(rep), rep


def test_knn_exact_rational_truth_under_ties(engine):
    """Duplicates and equal distances: the result must satisfy the tie rule against the
    exact-rational oracle, self first, distance 0 to exact duplicates."""
    asm = synth.s2_redundant(160, seed=4)
    res = _run(engine, asm, "5p6", 4, "tc")
    counts, _ = ko.counts_mode(asm.bases, asm.offsets, "5p6")
    i_e, d_e = knn_oracle.knn_exact(counts, asm.key_len, 4, rows=range(0, 160, 8))
    rows = np.arange(0, 160, 8)
    prof = counts / asm.key_len[:, None].astype(np.float64)
    rep = knn_oracle.check_knn(res["knn_idx"][rows], res["knn_dist"][rows], knn_oracle.d2_fp64(prof, rows), rows=rows)
    assert knn_oracle.parity_ok(rep), rep
    assert np.allclose(np.sqrt(d_e), res["knn_dist"][rows], rtol=1e-6, atol=0)
    assert (res["knn_idx"][:, 0] == np.arange(160)).all() and (res["knn_dist"][:, 0] == 0).all()


def test_tc_equals_simt_candidates(engine):
    """Same scores, same tie rule: both candidate kernels must lead to identical output."""
    asm = synth.s1_families(1500, seed=13)
    a = _run(engine, asm, "5p6", 15, "simt")
    b = _run(engine, asm, "5p6", 15, "tc")
    assert np.array_equal(a["knn_idx"], b["knn_idx"]) and np.array_equal(a["knn_dist"], b["knn_dist"])


def test_tensor_core_gram_is_exact(engine):
    """The design relies on the fp16 x fp16 -> fp32 tensor-core Gram of integer counts
    being exact below 2^24 (SURVEY 7 'verify on hardware'): the fp32 scores must then be
    bit-identical to the same formula evaluated from an int64 Gram on the CPU."""
    asm = synth.s1_families(384, seed=21)
    mode = mode_of("5p6")
    d_bases, d_offsets, d_len = engine.upload(asm.bases, asm.offsets, asm.key_len)
    counts, _, _ = engine.count(d_bases, d_offsets, asm.n, mode)
    _, operand, rowmeta = engine.normalise(counts, 1088, d_len, want_profile=False)
    k = 24
    idx, dist, d2 = engine.knn(operand, rowmeta, k, impl=_lib.KB_KNN_TC, want_d2=True)
    torch.cuda.synchronize()
    c = counts.cpu().numpy().view(np.uint32).astype(np.int64)
    gram = c @ c.T
    l = asm.key_len.astype(np.float64)
    num = np.diag(gram)[:, None] * (l[None, :] ** 2) + np.diag(gram)[None, :] * (l[:, None] ** 2) - 2 * gram * np.outer(l, l)
    truth = num / np.outer(l, l) ** 2
    rep = knn_oracle.check_knn(idx.cpu().numpy(), dist.cpu().numpy(), truth)
    assert knn_oracle.parity_ok(rep), rep
    got = d2.cpu().numpy()
    assert np.array_equal(got, truth[np.arange(asm.n)[:, None], idx.cpu().numpy()]), "rerank is not exact"


def test_query_shard_equals_full(engine):
    """Multi-GPU layout on one GPU: a query-row shard against all keys gives the same rows, also for a lone
    query block (at most 128 rows: a CTA pair whose second CTA has no live rows), the last one ending at the last key."""
    asm = synth.s1_families(1000, seed=31)
    mode = mode_of("5p6")
    d_bases, d_offsets, d_len = engine.upload(asm.bases, asm.offsets, asm.key_len)
    counts, _, _ = engine.count(d_bases, d_offsets, asm.n, mode)
    _, operand, rowmeta = engine.normalise(counts, 1088, d_len, want_profile=False)
    full_i, full_d, _ = engine.knn(operand, rowmeta, 5, impl=_lib.KB_KNN_TC)
    for q0, nq in ((250, 333), (250, 100), (0, 1), (872, 128)):
        part_i, part_d, _ = engine.knn(operand, rowmeta, 5, q_row0=q0, nq=nq, impl=_lib.KB_KNN_TC)
        assert torch.equal(full_i[q0:q0 + nq], part_i) and torch.equal(full_d[q0:q0 + nq], part_d), (q0, nq)


def test_full_size_knn_properties_50k(engine):
    """BASELINE config 2 (50k contigs, 5p6, n_neighbors=2) at full size: structural
    properties for all rows and the tie-rule check on a row sample against fp64 brute force."""
    asm = synth.s1_families(50000)
    res = _run(engine, asm, "5p6", 2, "tc")
    idx, dist = res["knn_idx"], res["knn_dist"]
    assert idx.shape == (50000, 2) and (idx[:, 0] == np.arange(50000)).all() and (dist[:, 0] == 0).all()
    assert (idx[:, 1] != idx[:, 0]).all() and (idx >= 0).all() and (idx < 50000).all() and np.isfinite(dist).all()
    prof = res["profile"]
    rows = np.arange(0, 50000, 1499)
    rep = knn_oracle.check_knn(idx[rows], dist[rows], knn_oracle.d2_fp64(prof, rows), rows=rows)
    assert knn_oracle.parity_ok(rep), rep


def _assembly_from(seqs):
    lens = np.array([len(s) for s in seqs], dtype=np.int64)
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    bases = np.frombuffer("".join(seqs).encode("ascii"), dtype=np.uint8).copy()
    n = len(seqs)
    return synth.Assembly(bases, off, np.arange(n, dtype=np.int64) // 3, np.arange(n, dtype=np.int64) % 3 + 1)


@pytest.mark.parametrize("k", [2, 6])
def test_exact_side_path_for_rows_beyond_the_tensor_range(engine, k):
    """Rows with a k-mer count > 2048 (long homopolymers) or sum c^2 >= 2^24 (contigs beyond
    ~130 kb) cannot be scored exactly by the fp16/fp32 Gram; they take the fp64 side path
    (K4x) as queries AND as keys of ordinary rows.  Result must still satisfy the tie rule."""
    rng = np.random.default_rng(17)

    def rnd(n):
        return "".join("ACGT"[i] for i in rng.integers(0, 4, n))
    base = synth.s1_families(240, seed=9).as_dict()
    seqs = list(base.values())
    long_a = rnd(150000)
    seqs += [long_a, long_a[:140000] + rnd(500), rnd(200000), "A" * 3000, "A" * 2990 + rnd(40), rnd(300) + "A" * 2500,
             "ACGT" * 2200]
    asm = _assembly_from(seqs)
    counts, _ = ko.counts_mode(asm.bases, asm.offsets, "5p6")
    assert (counts.max(1) > 2048).sum() >= 3 and ((counts.astype(np.int64) ** 2).sum(1) >= 2 ** 24).sum() >= 3
    res = _run(engine, asm, "5p6", k, "tc")
    prof = counts[:, counts.any(0)] / asm.key_len[:, None].astype(np.float64)
    assert res["profile"].tobytes() == prof.tobytes()
    rep = knn_oracle.check_knn(res["knn_idx"], res["knn_dist"], knn_oracle.d2_fp64(prof))
    assert knn_oracle.parity_ok(rep), rep
    # the two near-identical long contigs must find each other
    assert res["knn_idx"][240, 1] == 241 and res["knn_idx"][241, 1] == 240


def test_exact_side_path_with_wide_rows(engine):
    """The same side path for -k 7 (16384 columns: four u32 query rows no longer fit the shared memory, K4x then takes one
    query row per CTA) with homopolymer runs (a count > 2048) among ordinary contigs."""
    rng = np.random.default_rng(23)

    def rnd(n):
        return "".join("ACGT"[i] for i in rng.integers(0, 4, n))
    seqs = list(synth.s1_families(150, seed=4).as_dict().values())
    seqs += ["A" * 3000, "A" * 2990 + rnd(60), rnd(400) + "C" * 2600, rnd(900)]
    asm = _assembly_from(seqs)
    counts, _ = ko.counts_mode(asm.bases, asm.offsets, 7)
    assert (counts.max(1) > 2048).sum() == 3
    res = _run(engine, asm, 7, 4, "tc")
    prof = counts[:, counts.any(0)] / asm.key_len[:, None].astype(np.float64)
    assert res["profile"].tobytes() == prof.tobytes()
    rep = knn_oracle.check_knn(res["knn_idx"], res["knn_dist"], knn_oracle.d2_fp64(prof))
    assert knn_oracle.parity_ok(rep), rep
    assert res["knn_idx"][150, 1] == 151 and res["knn_idx"][151, 1] == 150


def test_dense_5120_k15_at_scale(engine):
    """BASELINE configs 3/4 shape on one GPU at reduced N: 5120 dense columns, n_neighbors=15."""
    asm = synth.s2_redundant(12000, seed=3)
    res = _run(engine, asm, "5+6", 15, "tc")
    idx, dist = res["knn_idx"], res["knn_dist"]
    assert idx.shape == (12000, 15) and (idx[:, 0] == np.arange(12000)).all() and (dist[:, 0] == 0).all()
    assert all(len(set(r)) == 15 for r in idx[::97].tolist()) and (np.diff(dist[:, 1:], axis=1) >= 0).all()
    rows = np.arange(0, 12000, 401)
    rep = knn_oracle.check_knn(idx[rows], dist[rows], knn_oracle.d2_fp64(res["profile"], rows), rows=rows)
    assert knn_oracle.parity_ok(rep), rep


# ---------------------------------------------------------------------------------------------
# wide candidate lists, any n_neighbors, and the certificate behind the candidate width
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", ["simt", "tc"])
@pytest.mark.parametrize("k", [27, 42, 60])
def test_knn_parity_wide_lists(engine, impl, k):
    """n_neighbors 27..60: candidate lists of 48 / 64 entries per row (cmd_parser.py:101-107 accepts any int)."""
    asm = synth.s1_families(700, seed=5)
    res = _run(engine, asm, "5p6", k, impl)
    cols, prof = ko.profile_np(asm.as_dict(), "5p6")
    assert res["profile"].tobytes() == prof.tobytes()
    rep = knn_oracle.check_knn(res["knn_idx"], res["knn_dist"], knn_oracle.d2_fp64(prof))
    assert knn_oracle.parity_ok(rep), rep


@pytest.mark.parametrize("k", [61, 150])
def test_knn_any_n_neighbors_takes_the_exact_pass(engine, k):
    """Beyond 60 neighbours there is no candidate kernel: every row goes through the exact pass over all keys."""
    asm = synth.s1_families(400, seed=6)
    res = _run(engine, asm, "5p6", k, "tc")
    assert res["uncertified"] == asm.n
    cols, prof = ko.profile_np(asm.as_dict(), "5p6")
    rep = knn_oracle.check_knn(res["knn_idx"], res["knn_dist"], knn_oracle.d2_fp64(prof))
    assert knn_oracle.parity_ok(rep), rep


def _exact_d2(counts, key_len, i, js):
    from fractions import Fraction
    ci, li = [int(v) for v in counts[i]], int(key_len[i])
    out = []
    for j in js:
        cj, lj = [int(v) for v in counts[j]], int(key_len[j])
        out.append(Fraction(sum((a * lj - b * li) ** 2 for a, b in zip(ci, cj)), (li * lj) ** 2))
    return out


def test_certificate_sends_mass_duplicates_to_the_exact_pass(engine):
    """More exact duplicates than the candidate list is wide: the fp32 candidate ranking cannot tell which of
    them it dropped, K5 must not certify those rows, and the exact pass returns the canonical answer
    (self, then (distance, index))."""
    rng = np.random.default_rng(23)

    def rnd(n):
        return "".join("ACGT"[i] for i in rng.integers(0, 4, n))
    dup = rnd(1800)
    seqs = [rnd(int(x)) for x in rng.integers(300, 2500, 300)]
    pos = sorted(rng.choice(300, 40, replace=False).tolist())
    for p_ in pos:
        seqs[p_] = dup
    asm = _assembly_from(seqs)
    asm.key_len[:] = 11                                    # equal header lengths: the duplicates' profile rows are identical
    res = profile_and_knn(engine, asm.bases, asm.offsets, asm.key_len, "5p6", n_neighbors=3, impl=IMPLS["tc"])
    assert res["uncertified"] >= 40
    idx = res["knn_idx"]
    for p_ in pos:
        others = [q for q in pos if q != p_][:2]
        assert idx[p_].tolist() == [p_] + others, (p_, idx[p_])
        assert (res["knn_dist"][p_] == 0).all()
    counts, _ = ko.counts_mode(asm.bases, asm.offsets, "5p6")
    prof = counts / asm.key_len[:, None].astype(np.float64)
    rep = knn_oracle.check_knn(idx, res["knn_dist"], knn_oracle.d2_fp64(prof))
    assert knn_oracle.parity_ok(rep), rep


def test_certificate_near_ties_of_long_contigs(engine):
    """Adversarial case of the candidate width: 48 variants of one 15 kb contig, one substitution each.  Their
    distances to each other differ in the 7th digit while the fp32 scores are of magnitude n/l, so the
    candidate ranking is noise.  Whatever K5 certifies or hands to the exact pass, the k distances returned
    must be EXACTLY the k smallest exact-rational distances."""
    rng = np.random.default_rng(29)

    def rnd(n):
        return "".join("ACGT"[i] for i in rng.integers(0, 4, n))
    base = rnd(15000)
    seqs = [rnd(int(x)) for x in rng.integers(300, 3000, 260)]
    fam = []
    for v in range(48):
        p_ = int(rng.integers(10, 14990))
        b = base[p_]
        seqs.append(base[:p_] + "ACGT"[("ACGT".index(b) + 1 + v % 3) % 4] + base[p_ + 1:])
        fam.append(len(seqs) - 1)
    asm = _assembly_from(seqs)
    k = 4
    res = profile_and_knn(engine, asm.bases, asm.offsets, asm.key_len, "5p6", n_neighbors=k, impl=IMPLS["tc"])
    counts, _ = ko.counts_mode(asm.bases, asm.offsets, "5p6")
    for i in fam[::3]:
        want_i, want_d = knn_oracle.knn_exact(counts, asm.key_len, k, rows=[i])
        got = res["knn_idx"][i].tolist()
        assert got[0] == i and len(set(got)) == k
        got_d = sorted(float(x) for x in _exact_d2(counts, asm.key_len, i, got))
        assert np.allclose(got_d, sorted(want_d[0].tolist()), rtol=1e-14, atol=0), (i, got, want_i)
    prof = counts / asm.key_len[:, None].astype(np.float64)
    rep = knn_oracle.check_knn(res["knn_idx"], res["knn_dist"], knn_oracle.d2_fp64(prof))
    assert knn_oracle.parity_ok(rep), rep


def test_redundant_merge_200k_5120_k15(engine):
    """BASELINE config 4's regime on one GPU: S2 (16-fold families, 10 % exact duplicates), 5120 dense columns,
    n_neighbors = 15, 200 000 contigs.  1 024 sampled rows are checked against distances computed from the
    integer counts (fp64 Gram of integers below 2^53: exact), every row structurally."""
    n = 200000
    asm = synth.s2_redundant(n, seed=11)
    res = _run(engine, asm, "5+6", 15, "tc")
    idx, dist = res["knn_idx"], res["knn_dist"]
    assert idx.shape == (n, 15) and (idx[:, 0] == np.arange(n)).all() and (dist[:, 0] == 0).all()
    assert (idx >= 0).all() and (idx < n).all() and (np.diff(dist[:, 1:], axis=1) >= 0).all()
    rows = np.sort(np.random.default_rng(1).choice(n, 1024, replace=False))
    prof = res["profile"]                                  # counts / len(key), bit-exact by the K1-K3 tests
    l = asm.key_len.astype(np.float64)
    c_rows = np.rint(prof[rows] * l[rows, None])
    sq = np.empty(n)
    gram = np.empty((len(rows), n))
    for lo in range(0, n, 20000):
        blk = np.rint(prof[lo:lo + 20000] * l[lo:lo + 20000, None])
        sq[lo:lo + 20000] = np.einsum("ij,ij->i", blk, blk)
        gram[:, lo:lo + 20000] = c_rows @ blk.T
    num = sq[rows][:, None] * (l[None, :] ** 2) + sq[None, :] * (l[rows][:, None] ** 2) - 2.0 * gram * np.outer(l[rows], l)
    truth = num / np.outer(l[rows], l) ** 2
    rep = knn_oracle.check_knn(idx[rows], dist[rows], truth, rows=rows)
    assert knn_oracle.parity_ok(rep), rep


def test_rerank_reads_the_gram_entry_out_of_the_score_or_recomputes_it(engine):
    """K5 recovers the exact integer Gram entry from a candidate's fp32 score when exactly one integer maps to that
    score, and recomputes it from the operand rows otherwise.  Ordinary assemblies never need the second path; huge
    key lengths against long contigs (score spacing coarser than 2/l_j) force it.  Both must give the exact distances."""
    asm = synth.make("S1", 1500, seed=21)
    res = _run(engine, asm, "5p6", 6, "tc")
    addr = engine.uncertified_word(asm.n, asm.n, 0, 1088, 6, _lib.KB_KNN_TC)
    assert int(engine.word_view(addr + 4).item()) == 0            # every Gram entry came out of its score
    counts, _ = ko.counts_mode(asm.bases, asm.offsets, "5p6")
    i_e, d_e = knn_oracle.knn_exact(counts, asm.key_len, 6, rows=range(0, asm.n, 300))
    assert np.allclose(np.sqrt(d_e), res["knn_dist"][::300], rtol=1e-6, atol=0)
    # long contigs (40 kb: sum c^2 ~ 2e6 < 2^24, unflagged), two rows with header keys of 50 000 characters
    rng = np.random.default_rng(8)
    n, length = 700, 40000
    fam = rng.integers(0, 4, size=(35, length), dtype=np.uint8)
    seqs = []
    for r in range(n):
        s = fam[r % 35].copy()
        mut = rng.random(length) < 0.02 * (1 + r // 35)
        s[mut] = rng.integers(0, 4, size=int(mut.sum()), dtype=np.uint8)
        seqs.append(np.frombuffer(b"ACGT", dtype=np.uint8)[s])
    bases = np.concatenate(seqs)
    offsets = np.arange(n + 1, dtype=np.int64) * length
    key_len = (700 + (np.arange(n) % 13)).astype(np.int32)
    key_len[[0, 448]] = 50000                                     # their neighbours are rows with ordinary keys
    res = profile_and_knn(engine, bases, offsets, key_len, "5p6", n_neighbors=6, impl=IMPLS["tc"])
    addr = engine.uncertified_word(n, n, 0, 1088, 6, _lib.KB_KNN_TC)
    assert int(engine.word_view(addr + 4).item()) > 0             # the operand-row path ran
    counts, _ = ko.counts_mode(bases, offsets, "5p6")
    prof = counts / key_len[:, None].astype(np.float64)
    assert res["profile"].tobytes() == prof.tobytes()
    ex = np.arange(0, n, 64)                                      # rows 0, 448 have the long keys
    i_e, d_e = knn_oracle.knn_exact(counts, key_len, 6, rows=ex)
    assert np.allclose(np.sqrt(d_e), res["knn_dist"][ex], rtol=1e-6, atol=0)
    rows = np.arange(0, n, 3)
    rep = knn_oracle.check_knn(res["knn_idx"][rows], res["knn_dist"][rows], knn_oracle.d2_fp64(prof, rows), rows=rows)
    assert knn_oracle.parity_ok(rep), rep
