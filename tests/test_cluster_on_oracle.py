"""Clustering below 100 % identity on the CPU: the reference of tests/cluster_ref.c on planted pairs, the command line
with the reference standing in for the device, and ITSX_CLUSTER=vsearch still building the vsearch command."""
import numpy as np
import pytest

import cluster_cases as K
import cluster_ref as R
from itsxpress_b200 import SeqSample
from itsxpress_b200 import _lib


@pytest.fixture()
def on_ref(oracle, monkeypatch):
    ctx = R.ClusterOracleContext(oracle)
    monkeypatch.setattr(SeqSample, "get_context", lambda: ctx)
    SeqSample.reset_sessions()
    yield ctx
    SeqSample.reset_sessions()


def test_dtable_is_the_identity_rule():
    for X in (0.99, 0.995, 0.9999, 0.75):
        D = _lib.cluster_dtable(X, 7000)
        for L in range(1, 7001):
            e = int(D[L])
            assert (L - e) / L >= X and (e == L or (L - e - 1) / L < X)
    assert _lib.cluster_dtable(0.99, 250)[250] == 2 and _lib.cluster_dtable(0.995, 250)[250] == 1
    with pytest.raises(_lib.ItsxError):
        _lib.cluster_dtable(0.5, 10)


def test_reference_edit_distance():
    assert R.ed(b"ACGTACGT", b"ACGTACGT", 2) == 0
    assert R.ed(b"ACGTACGT", b"ACGAACGT", 2) == 1
    assert R.ed(b"ACGTACGT", b"CGTACGT", 2) == 1
    assert R.ed(b"ACGTACGT", b"acgtacgu", 2) == 0               # case and U = T
    assert R.ed(b"AAAA", b"TTTT", 2) == 3                         # d + 1 above the band
    assert R.ed(b"ACGTNCGT", b"ACGTACGT", 2) == 1                 # N is an ordinary symbol


def test_reference_greedy_on_a_chain():
    """a - b - c with ed 1 each, ed(a, c) = 2 at D = 1: a and c are centroids, b joins a (earliest tie)"""
    a = b"ACGT" * 50
    b = a[:100] + b"T" + a[101:]
    c = b[:150] + (b"A" if b[150:151] != b"A" else b"C") + b[151:]
    seq, off = K.pack([a, a, b, c])
    first = np.array([0, 2, 3], np.int32)
    nc, crow, strand, ed, uor = R.cluster(seq, off, first, np.array([0, 1, 2], np.int32), 0.995)
    assert nc == 2 and crow.tolist() == [0, 0, 1] and ed.tolist() == [0, 1, 0] and uor.tolist() == [0, 2]
    nc, crow, _, _, uor = R.cluster(seq, off, first, np.array([1, 0, 2], np.int32), 0.995)   # b first: takes a and c
    assert nc == 1 and crow.tolist() == [0, 0, 0] and uor.tolist() == [1]


def test_cluster_cli_on_the_reference(on_ref, tmp_path):
    K.check_cluster_cli(tmp_path)
    assert "cluster" in on_ref.calls


def test_no_accepted_pairs_equals_exact_on_the_reference(on_ref, tmp_path):
    K.check_no_accepted_pairs_equals_exact(tmp_path)


def test_paired_cluster_cli_on_the_reference(on_ref, tmp_path):
    K.check_paired_cluster_cli(tmp_path)


def test_vsearch_switch_builds_the_vsearch_argv(monkeypatch, tmp_path):
    seen = []
    monkeypatch.setenv("ITSX_CLUSTER", "vsearch")
    monkeypatch.setattr(SeqSample, "_external", lambda tool, argv, what: seen.append((tool, argv, what)))
    s = SeqSample.SeqSampleNotPaired(K.MERGED, str(tmp_path))
    s.cluster(threads="2", cluster_id=0.995)
    assert seen == [("Vsearch", ["vsearch", "--cluster_size", K.MERGED, "--centroids", str(tmp_path / "rep.fa"), "--uc",
                                 str(tmp_path / "uc.txt"), "--strand", "both", "--id", "0.995", "--threads", "2"],
                     "clustering")]
