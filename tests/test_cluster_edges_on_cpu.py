"""The clustering reference and the edge workloads of tests/cluster_edge_cases.py, on the CPU: the reference's banded
edit distance against an unbanded full-matrix Levenshtein, ref_accepted_pairs on hand-built sets, the restated host
tables, and every claim the generators make about what they build (the ed and strand of each planted pair, the
untouched segment and its shift)."""
import itertools
import time

import numpy as np
import pytest

import cluster_cases as K
import cluster_edge_cases as E
import cluster_ref as R
from itsxpress_b200 import _lib

ALPHABET = b"ACGTUNRYMKSWHBVDacgtunrymkswhbvd"


def levenshtein(a, b):
    """unit-cost edit distance, every cell of the matrix"""
    prev = list(range(len(b) + 1))
    for i in range(1, len(a) + 1):
        cur = [i] + [0] * len(b)
        for j in range(1, len(b) + 1):
            cur[j] = min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (a[i - 1] != b[j - 1]))
        prev = cur
    return prev[-1]


def plain_norm(s):
    return bytes(c - 32 if 97 <= c <= 122 else c for c in s).replace(b"U", b"T")


def plain_rc(s):
    comp = dict(zip(b"ACGTRYMKHDBV", b"TGCAYRKMDHVB"))
    return bytes(comp.get(c, c) for c in reversed(plain_norm(s)))


def test_reference_ed_equals_the_full_matrix():
    rng = np.random.default_rng(1)
    n = 0
    for _ in range(1500):
        alpha = [ALPHABET, b"ACGT", b"AC"][int(rng.integers(3))]
        la = int(rng.integers(0, 41))
        a = bytes(rng.choice(list(alpha), la).tolist())
        if rng.random() < 0.5:                              # a close relative of a, so small distances occur
            b = bytearray(a)
            for _ in range(int(rng.integers(0, 8))):
                op, p = int(rng.integers(3)), int(rng.integers(len(b) + 1))
                if op == 0 and p < len(b):
                    b[p] = alpha[int(rng.integers(len(alpha)))]
                elif op == 1 and len(b) < 40:
                    b.insert(p, alpha[int(rng.integers(len(alpha)))])
                elif p < len(b):
                    del b[p]
            b = bytes(b)
        else:
            b = bytes(rng.choice(list(alpha), int(rng.integers(0, 41))).tolist())
        fp = levenshtein(plain_norm(a), plain_norm(b))
        fm = levenshtein(plain_rc(a), plain_norm(b))
        for d in range(13):
            assert R.ed(a, b, d) == min(fp, d + 1), (a, b, d)
            assert R.ed(a, b, d, rc=True) == min(fm, d + 1), (a, b, d)
            n += fp <= d
    assert n > 3000


def test_reference_ed_on_every_short_pair():
    for la, lb in ((0, 3), (2, 3), (3, 3), (4, 2)):
        for a in itertools.product(b"ACG", repeat=la):
            for b in itertools.product(b"ACG", repeat=lb):
                a, b = bytes(a), bytes(b)
                full = levenshtein(a, b)
                for d in range(5):
                    assert R.ed(a, b, d) == min(full, d + 1)


def _pairs_by_brute_force(reads, X, group):
    n = 0
    for u, v in itertools.combinations(range(len(reads)), 2):
        if group[u] != group[v]:
            continue
        a, b = reads[u], reads[v]
        L = max(len(a), len(b))
        D = int(_lib.cluster_dtable(X, max(L, 1))[L])
        e = min(levenshtein(plain_norm(a), plain_norm(b)), levenshtein(plain_rc(a), plain_norm(b)))
        n += e <= D
    return n


def test_accepted_pairs_on_hand_built_sets():
    a = b"ACGTTGCAAC" * 10
    b = a[:40] + b"T" + a[41:]                      # 1 substitution
    c = a[:10] + a[11:]                            # 1 deletion (len 99)
    d = K.rc(a[:60] + b"GG" + a[62:])              # 2 substitutions, reverse strand
    e = a[:95]                                     # 5 shorter
    reads = [a, b, c, d, e]
    seq, off = K.pack(reads)
    first = np.arange(5, dtype=np.int32)
    # 0.99: D(100) = 1: a-b, a-c (ed 1); b-c ed 2, a-d ed 2, e 5 away
    assert R.accepted_pairs(seq, off, first, 0.99) == 2
    # 0.98: D(100) = 2 adds a-d (on the reverse strand) and b-c
    assert R.accepted_pairs(seq, off, first, 0.98) == _pairs_by_brute_force(reads, 0.98, [0] * 5) == 4
    n95 = R.accepted_pairs(seq, off, first, 0.95)
    assert n95 == _pairs_by_brute_force(reads, 0.95, [0] * 5) > 4
    # groups: pairs across groups never count; the order of the uniques does not matter
    g = np.array([0, 1, 0, 1, 0], np.int32)
    ng = R.accepted_pairs(seq, off, first, 0.95, g)
    assert ng == _pairs_by_brute_force(reads, 0.95, g) < n95
    perm = np.array([3, 0, 4, 2, 1], np.int32)
    assert R.accepted_pairs(seq, off, first[perm], 0.95, g[perm]) == ng
    assert R.accepted_pairs(seq, off, np.zeros(0, np.int32), 0.95) == 0


def test_accepted_pairs_on_random_sets():
    rng = np.random.default_rng(2)
    for X in (0.6, 0.8, 0.9):
        T = E.rand_seq(rng, 30)
        reads = list(dict.fromkeys([K.edit(rng, T, int(rng.integers(0, 6))) for _ in range(30)]))
        reads = [r for i, r in enumerate(reads) if r and min(E.norm(r), E.rcn(r)) not in
                 {min(E.norm(x), E.rcn(x)) for x in reads[:i]}]
        reads = [K.rc(r) if rng.random() < 0.3 else r for r in reads]
        g = rng.integers(0, 2, len(reads)).astype(np.int32)
        seq, off = K.pack(reads)
        first = np.arange(len(reads), dtype=np.int32)
        assert R.accepted_pairs(seq, off, first, X, g) == _pairs_by_brute_force(reads, X, g)


def test_restated_tables():
    """W and K as cluster_run builds them, against definitions by search: HI(L) is the longest partner of L within lmax,
    K(L) the largest D of any pair a class of length L is in; the issue's table of (X, D(250), K(250) + 1, W)"""
    for X, lmax, d250, k250, W in ((0.995, 600, 1, 2, 6), (0.99, 600, 2, 3, 12), (0.97, 600, 7, 8, 36),
                                   (0.94, 600, 15, 16, 70), (0.9, 600, 25, 28, 115), (0.8, 320, 50, 63, 116)):
        T = E.Tables(X, lmax)
        assert (T.D[250], T.K[250] + 1, T.W) == (d250, k250, W)
        for L in range(1, lmax + 1):
            partners = [Lp for Lp in range(1, lmax + 1) if abs(Lp - L) <= T.D[max(L, Lp)]]
            assert T.LO[L] == min(partners) and T.HI[L] == max(partners)
            assert T.K[L] == max(T.D[max(L, Lp)] for Lp in partners)
    T = E.Tables(0.51, 15)
    assert all(T.K[L] + 1 == L for L in range(1, 8))       # single-residue segments
    assert [E.d_lcap(X) for X in (0.8, 0.85, 0.9, 0.99)] == [324, 433, 649, 6499]
    assert E.sweep_lengths(0.8) == [80, 174, 269] and E.sweep_lengths(0.97) == [80, 340, 600]


@pytest.mark.parametrize("X,Lv,lmax", E.pigeonhole_params())
def test_pigeonhole_claims(X, Lv, lmax):
    T = E.Tables(X, lmax)
    case = E.pigeonhole(X, Lv, lmax, seed=int(X * 1000) + Lv)
    only_j = E.check_claims(case, lmax)
    Kv = T.K[Lv]
    assert [Kv for X_, L_, _ in E.pigeonhole_params() if X_ == X] == [Kv] and Kv in (1, 2, 7, 15, 25, 64)
    c = case.claims
    # every segment untouched in some pair; the shifts -d, 0, +d; u of length HI(Lv); both strands; untouched segment at
    # u's start and end
    assert {x.j for x in c if x.j is not None} == set(range(Kv + 1))
    assert {x.shift for x in c if x.j is not None} >= {-T.D[Lv], 0, Kv}
    assert any(len(case.reads[x.u]) == T.HI[Lv] and x.d == Kv for x in c)
    assert {x.strand for x in c} == {0, 1}
    assert any(x.j == 0 and x.shift == 0 for x in c)
    assert any(x.j == Kv and len(case.reads[x.u]) == T.HI[Lv] for x in c)
    assert any(x.j is None for x in c)                       # the palindrome
    # u of length HI(Lv) leaves j the only untouched segment: the lookup finds the pair through j at its shift alone
    # (but for chance matches of a short segment elsewhere in the window)
    hi = [t for x, t in zip(c, only_j) if x.j is not None and len(case.reads[x.u]) == T.HI[Lv]]
    if Kv < 30:                 # (4-residue segments at K = 64 match somewhere in a window of 129 shifts by chance)
        assert sum(hi) >= 0.9 * len(hi)
        assert any(t and x.shift == Kv for x, t in zip(c, only_j))  # the +d edge, through the last segment alone


def test_pigeonhole_reference_results():
    """the reference on every pigeonhole case: each u joins its v with the claimed ed and strand (the palindrome on
    '+'), and the accepted pairs are exactly the planted ones; each call well under 10 s"""
    for X, Lv, lmax in E.pigeonhole_params():
        case = E.pigeonhole(X, Lv, lmax, seed=int(X * 1000) + Lv)
        first = np.arange(len(case.reads), dtype=np.int32)
        t = time.time()
        nc, crow, strand, ed, uor, npairs = E.reference(case, first, first)
        assert time.time() - t < 10
        ok = [x for x in case.claims]
        assert npairs == len(ok)
        for x in ok:
            assert uor[crow[x.v]] == x.v and crow[x.u] == crow[x.v], x
            assert (ed[x.u], strand[x.u]) == (x.d, x.strand), x


@pytest.mark.parametrize("X", E.SWEEP_X)
def test_sweep_workload(X):
    case = E.sweep(X, seed=int(X * 1000))
    L = max(len(r) for r in case.reads)
    assert int(_lib.cluster_dtable(X, L)[L]) <= E.MAXD
    assert min(E.sweep_lengths(X)) == 80 and max(E.sweep_lengths(X)) <= 600
    first, cls = E.derep_first(case.reads)
    t = time.time()
    nc, crow, strand, ed, uor, npairs = E.reference(case, first, cls)
    assert time.time() - t < 10
    D = int(_lib.cluster_dtable(X, L)[L])
    assert npairs >= len(first) - nc and (nc < len(first) if D > 0 else npairs == 0)
    # ties (same length, and across lengths where X allows): u joins the earlier of its two equal-identity centroids
    assert (ed > 0).sum() > 0 or D == 0


def test_tie_workload_is_a_tie():
    """the tie reads of E.ties: both centroids accept u at the same identity (cross-multiplied), ed(c1, c2) > D"""
    for X in (0.8, 0.85, 0.9, 0.94, 0.99):
        rng = np.random.default_rng(3)
        reads = E.ties(rng, X, 250)
        groups = [reads[i:i + 6] for i in range(0, len(reads), 6)]
        assert len(groups) >= (4 if X <= 0.94 else 2)
        for g in groups:
            c1, c2, u = g[0], g[3], g[5]
            assert g[:3] == [c1] * 3 and g[3:5] == [c2] * 2
            L1, L2 = max(len(u), len(c1)), max(len(u), len(c2))
            D = _lib.cluster_dtable(X, max(L1, L2) + 1)
            e1 = min(R.ed(u, c1, D[L1] + 1), R.ed(u, c1, D[L1] + 1, rc=True))
            e2 = min(R.ed(u, c2, D[L2] + 1), R.ed(u, c2, D[L2] + 1, rc=True))
            assert e1 <= D[L1] and e2 <= D[L2] and (L1 - e1) * L2 == (L2 - e2) * L1
            L12 = max(len(c1), len(c2))
            assert R.ed(c1, c2, D[L12]) > D[L12] and R.ed(c1, c2, D[L12], rc=True) > D[L12]


@pytest.mark.parametrize("X", [0.51, 0.6, 0.75])
def test_tiny_workload(X):
    case = E.tiny(X, seed=int(X * 100))
    first, cls = E.derep_first(case.reads)
    t = time.time()
    ref = E.reference(case, first, cls)
    assert time.time() - t < 10 and ref[5] > len(first)


@pytest.mark.parametrize("X", [0.97, 0.9])
def test_low_complexity_workload(X):
    case = E.low_complexity(X, seed=int(X * 100))
    assert max(len(r) for r in case.reads) < 700
    assert E.norm(b"AC" * 75) in {E.norm(r) for r in case.reads} and b"A" * 154 in case.reads
    first, cls = E.derep_first(case.reads)
    ref = E.reference(case, first, cls)
    assert 0 < ref[0] < len(first)


@pytest.mark.parametrize("X", [0.99, 0.8])
def test_band_cap_workload(X):
    case, over = E.band_cap(X, seed=int(X * 100))
    E.check_band_cap(case)
    assert max(len(r) for r in case.reads) == E.d_lcap(X) == len(over) - 1
    assert int(_lib.cluster_dtable(X, len(over))[len(over)]) == E.MAXD + 1
    first = np.arange(len(case.reads), dtype=np.int32)
    t = time.time()
    nc, crow, strand, ed, uor, npairs = E.reference(case, first, first)
    assert time.time() - t < 10
    assert npairs == sum(x.d == E.MAXD for x in case.claims)
    for x in case.claims:
        joined = crow[x.u] == crow[x.v]
        assert joined == (x.d == E.MAXD)
        if joined:
            assert (ed[x.u], strand[x.u]) == (x.d, x.strand)


def test_chain_workload():
    case = E.chain(4)
    assert len(set(case.reads)) == 3000
    for i in range(2, 3000, 97):
        assert R.ed(case.reads[i], case.reads[i - 2], 2) == 2
    first = np.arange(3000, dtype=np.int32)
    t = time.time()
    nc, crow, strand, ed, uor, npairs = E.reference(case, first, first)
    assert time.time() - t < 10
    assert nc == 1500 and (uor == np.arange(0, 3000, 2)).all() and npairs >= 2999


@pytest.mark.parametrize("X", [0.97, 0.99])
def test_scale_workload(X):
    case, fam = E.scale(X, seed=int(X * 100))
    first, cls = E.derep_first(case.reads)
    assert 300 <= len(np.unique(fam)) <= 500 and 20_000 <= len(first) <= 30_000
    t = time.time()
    nc, crow, strand, ed, uor, npairs = E.reference(case, first, cls, group=fam)
    assert time.time() - t < 10 * 8
    assert 0 < nc < len(first) and npairs >= len(first) - nc
