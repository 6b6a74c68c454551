"""Comparison with the original project's karma/kmer.py through its stored output: oracle/make_golden.py ran the
original on seeded random FASTA of several alphabets and k-mer sizes and froze inputs, columns and float64
matrices in tests/golden/kmer_profile_golden.json."""
import pytest

from oracle import kmer_oracle as ko


def test_reference_own_test():
    # the original project's tests/test_kmer.py:6-8
    assert ko.is_palindrome("ACGT") is False and ko.is_palindrome("AAAA") is True


@pytest.mark.parametrize("alphabet,k", [("ACGT", "5p6"), ("ACGTN", "5p6"), ("ACGTacgtNRY", "5p6"), ("AC", "5p6"),
                                        ("ACGT", 3), ("ACGTN", 4), ("ACGT", 7)])
def test_randomised_against_reference(golden, alphabet, k):
    cases = [c for c in golden if c["name"].startswith("rand") and c["name"].endswith("_%s_k%s" % (alphabet, k))]
    assert cases
    for c in cases:
        seqs = dict(zip(c["keys"], c["seqs"]))
        for f in (ko.profile_port, ko.profile_np):
            c2, m2 = f(seqs, c["kmer_size"])
            assert c2 == c["columns"] and m2.tobytes().hex() == c["matrix_hex"], (c["name"], f.__name__)
