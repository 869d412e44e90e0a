"""itsx_cluster on the B200 at the edges of its pigeonhole filter, against the brute-force reference (tests/cluster_ref.c):
every identity from 0.8 to 0.999, pairs built to be found through one segment at the extreme shifts and partner lengths
(tests/cluster_edge_cases.py), reads of 1-15 residues, low-complexity reads, the band cap D = 64, families of error
variants at 20-30 k classes, and a chain that resolves in thousands of rounds.  Beyond the assignment (centroid row,
strand, ed, unique of row, read -> row), every call's n_accepted must equal the number of accepted pairs counted by brute
force: a pair the index misses fails the test even when the final assignment does not depend on it."""
import json

import numpy as np
import pytest

import cluster_cases as K
import cluster_edge_cases as E
from itsxpress_b200 import _lib

pytestmark = pytest.mark.gpu


def gpu_vs_ref(ctx, case, group=None):
    """the device against the reference on the case; returns the stats and the device's (crow, strand, ed, uor)"""
    seq, off = K.pack(case.reads)
    _, _, nu = ctx.derep(seq, off)
    first, _ = ctx.derep_clusters(nu)
    _, _, class_uid = ctx.derep_map(len(case.reads))
    if case.claims:                                 # planted cases: every read its own class, unique index = read index
        assert np.array_equal(first, np.arange(len(case.reads)))
    nc = ctx.cluster(case.X, case.order)
    got = ctx.cluster_fetch(nu, nc)
    st = ctx.cluster_stats()
    want = E.reference(case, first, class_uid, group)
    assert nc == want[0]
    for g, w, name in zip(got, want[1:5], ("centroid row", "strand", "ed", "unique of row")):
        assert np.array_equal(g, w), name
    assert st.n_accepted == want[5]
    _, _, uid = ctx.derep_map(len(case.reads))
    assert np.array_equal(uid, got[0][class_uid])
    lmax = max(len(r) for r in case.reads)
    T = E.Tables(case.X, lmax)
    assert st.n_accepted <= st.n_verified <= st.n_candidates
    assert st.d_max == T.D[lmax] and st.n_len_slots == T.W
    crow, strand, ed, uor = got
    for c in case.claims:
        if c.d <= T.D[max(len(case.reads[c.u]), len(case.reads[c.v]))]:
            assert uor[crow[c.v]] == c.v and crow[c.u] == crow[c.v], c
            assert (ed[c.u], strand[c.u]) == (c.d, c.strand), c
        else:
            assert crow[c.u] != crow[c.v], c
    return st, got


def log_stats(name, st):
    keys = ("n_unique", "n_centroids", "n_segments", "n_candidates", "n_verified", "n_accepted", "n_rounds", "d_max",
            "n_len_slots", "ms_total")
    print("cluster stats %s %s" % (name, json.dumps({k: round(getattr(st, k), 3) for k in keys})))


@pytest.mark.parametrize("X", E.SWEEP_X)
def test_identity_sweep(gpu_ctx, X):
    st, _ = gpu_vs_ref(gpu_ctx, E.sweep(X, seed=int(X * 1000)))
    assert st.n_accepted > 0 or st.d_max == 0


@pytest.mark.parametrize("X,Lv,lmax", E.pigeonhole_params())
def test_pigeonhole_edge(gpu_ctx, X, Lv, lmax):
    case = E.pigeonhole(X, Lv, lmax, seed=int(X * 1000) + Lv)
    st, _ = gpu_vs_ref(gpu_ctx, case)
    assert st.n_accepted == len(case.claims)


@pytest.mark.parametrize("X", [0.51, 0.6, 0.75])
def test_tiny_reads(gpu_ctx, X):
    gpu_vs_ref(gpu_ctx, E.tiny(X, seed=int(X * 100)))


@pytest.mark.parametrize("X", [0.97, 0.9])
def test_low_complexity(gpu_ctx, X):
    gpu_vs_ref(gpu_ctx, E.low_complexity(X, seed=int(X * 100)))


@pytest.mark.parametrize("X", [0.99, 0.8])
def test_band_cap(gpu_ctx, X):
    case, over = E.band_cap(X, seed=int(X * 100))
    st, _ = gpu_vs_ref(gpu_ctx, case)
    assert st.d_max == E.MAXD and st.n_accepted == sum(c.d == E.MAXD for c in case.claims)
    seq, off = K.pack(case.reads + [over])
    gpu_ctx.derep(seq, off)
    with pytest.raises(_lib.ItsxError) as e:
        gpu_ctx.cluster(X)
    assert e.value.code == -6


@pytest.mark.parametrize("X", [0.97, 0.99])
def test_scale(gpu_ctx, X):
    """no two families are within D of each other, so the per-family reference is the whole reference, and the sum of
    the per-family accepted pairs is the device's n_accepted (a false edge between families would show there too)"""
    case, fam = E.scale(X, seed=int(X * 100))
    st, _ = gpu_vs_ref(gpu_ctx, case, group=fam)
    log_stats("scale X=%g" % X, st)
    assert 20_000 <= st.n_unique <= 30_000 and st.n_centroids < st.n_unique


def test_long_chain(gpu_ctx):
    st, got = gpu_vs_ref(gpu_ctx, E.chain(4))
    log_stats("chain X=0.995", st)
    assert st.n_centroids == 1500 and st.n_rounds >= 1000


def test_short_segment_keys(gpu_ctx):
    """the 0.97 sweep case with segment keys cut to 12 and 8 bits: many more candidates (the keys collide), the same
    result and the same accepted pairs"""
    case = E.sweep(0.97, seed=970)
    seq, off = K.pack(case.reads)
    _, _, nu = gpu_ctx.derep(seq, off)
    res, st = [], []
    try:
        for bits in (64, 12, 8):
            gpu_ctx.cluster_set_key_bits(bits)
            nc = gpu_ctx.cluster(case.X)
            res.append(gpu_ctx.cluster_fetch(nu, nc))
            st.append(gpu_ctx.cluster_stats())
    finally:
        gpu_ctx.cluster_set_key_bits(64)
    for r in res[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(res[0], r))
    assert st[0].n_accepted == st[1].n_accepted == st[2].n_accepted > 0
    assert st[0].n_candidates < st[1].n_candidates < st[2].n_candidates < 1 << 28
