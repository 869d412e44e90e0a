"""Clustering workloads aimed at the edges of itsx_cluster's pigeonhole filter (csrc/cluster.cu), shared by
tests/test_cluster_edges_on_cpu.py (their claims, checked against the reference tests/cluster_ref.c) and
tests/test_gpu_cluster_edges.py (the device against the reference).

To aim edits at segments, the generators restate the host tables of cluster_run from _lib.cluster_dtable: D(L), the
largest accepted ed at length L; HI(L), the longest partner length of a class of length L; K(L) = D(HI(L)), so that a
class of length L is cut into K(L) + 1 segments [seg_lo(j), seg_lo(j + 1)); and W, the widest partner-length window.
Each generator returns a Case: the reads, the order of the uniques (None: the default order) and, for planted pairs,
the claims the device must meet (u joins centroid v at that ed on that strand)."""
import concurrent.futures as cf
import os
from collections import namedtuple

import numpy as np

import cluster_cases as K
import cluster_ref as R
from itsxpress_b200 import _lib

MAXD = 64                                   # ITSX_CLUSTER_MAXD
SWEEP_X = (0.8, 0.85, 0.9, 0.94, 0.97, 0.98, 0.99, 0.995, 0.999)

Case = namedtuple("Case", "reads order claims X")
# u joins v (unique indices = read indices: every read of a planted case is its own class) with ed d on strand (0 '+',
# 1 '-'); j: the segment of v left untouched, found in u's strand at v's position + shift
Claim = namedtuple("Claim", "v u d strand j shift")


# ---- the host tables of cluster_run, restated ------------------------------------------------------------------------
class Tables:
    def __init__(self, X, lmax):
        self.X, self.lmax = X, lmax
        self.D = [int(x) for x in _lib.cluster_dtable(X, lmax)]
        D = self.D
        self.HI, self.LO, self.K = [0] * (lmax + 1), [0] * (lmax + 1), [0] * (lmax + 1)
        self.W = 1
        hi = 0
        for L in range(lmax + 1):
            # the longest L' <= lmax with L' - D(L') <= L (a longer partner needs L' - L <= D(L')); L' - D(L') is
            # non-decreasing
            while hi + 1 <= lmax and hi + 1 - D[hi + 1] <= L:
                hi += 1
            hi = max(hi, L)
            self.HI[L], self.LO[L] = hi, L - D[L]
            self.K[L] = D[hi]
            self.W = max(self.W, hi - self.LO[L] + 1)

    def segments(self, L):
        k = self.K[L] + 1
        return [(seg_lo(L, k, j), seg_lo(L, k, j + 1)) for j in range(k)]


def seg_lo(L, k, j):
    return j * L // k


def d_lcap(X):
    """the longest length L with D(L) <= 64"""
    D = _lib.cluster_dtable(X, int((MAXD + 1) / (1 - X)) + 2)
    return int(np.flatnonzero(D <= MAXD)[-1])


NORM = bytes.maketrans(b"abcdefghijklmnopqrstuvwxyzU", b"ABCDEFGHIJKLMNOPQRSTUVWXYZT")
RCOMP = bytes.maketrans(b"ACGTRYMKHDBV", b"TGCAYRKMDHVB")


def norm(s):
    return s.translate(NORM)


def rcn(s):
    """reverse complement of the normalised residues, as the derep and the kernels take it"""
    return norm(s).translate(RCOMP)[::-1]


def lookup_hits(u, v, d, k):
    """(j, q) for every segment j of v (k segments) that occurs exactly in u at a shift q - a within +-d: the lookups
    query_kernel makes for the pair (u on one strand, partner v)"""
    u, v = norm(u), norm(v)
    hits = set()
    for j in range(k):
        a, b = seg_lo(len(v), k, j), seg_lo(len(v), k, j + 1)
        for q in range(max(0, a - d), a + d + 1):
            if q + b - a <= len(u) and u[q:q + b - a] == v[a:b]:
                hits.add((j, q))
    return hits


def rand_seq(rng, L):
    return bytes(rng.choice(list(b"ACGT"), L).tolist())


def _other(rng, *avoid):
    return [c for c in b"ACGT" if c not in avoid][int(rng.integers(4 - len(set(avoid))))]


# ---- b. the pigeonhole edge -----------------------------------------------------------------------------------------
def plant(rng, v, segs, edits):
    """u from v with one edit per segment: edits[i] = (kind 's' / 'i' / 'd', at 'first' / 'last' residue) or None.
    An insertion goes inside the segment (after its first residue, or before its last), so that the segment's residues
    are never contiguous in u."""
    out = bytearray()
    for (a, b), e in zip(segs, edits):
        s = bytearray(v[a:b])
        if e:
            kind, at = e
            p = 0 if at == "first" else len(s) - 1
            if kind == "s":
                s[p] = _other(rng, s[p])
            elif kind == "d":
                del s[p]
            else:
                assert len(s) >= 2
                p = 1 if at == "first" else len(s) - 1
                s.insert(p, _other(rng, s[p - 1], s[p]))
        out += s
    return bytes(out)


def pigeonhole_params():
    """(X, Lv, lmax) with K(Lv) = 1, 2, 7, 15, 25 and 64 (lmax: the longest class of the call, HI(Lv) at most)"""
    out = []
    for X, kk in ((0.995, 1), (0.99, 2), (0.97, 7), (0.94, 15), (0.9, 25)):
        T = Tables(X, 700)
        Lv = min(L for L in range(200, 400) if T.K[L] == kk and T.HI[L] - T.D[T.HI[L]] == L)
        out.append((X, Lv, T.HI[Lv]))
    lcap = d_lcap(0.8)
    out.append((0.8, lcap - MAXD, lcap))                 # HI(260) = 325 uncapped; capped at 324, D(324) = 64
    return out


def pigeonhole(X, Lv, lmax, seed):
    """For every segment j of v (K(Lv) + 1 of them): u with exactly d = D(max(Lu, Lv)) edits, one in each of d segments
    other than j, on the first or last residue of the segment, in three shapes:
      hi     Lu = HI(Lv), so d = K(Lv) and j is the only untouched segment; insertions before j first (shift up to +d)
      minus  Lu = Lv - D(Lv): D(Lv) deletions before j (shift -d), where j >= D(Lv)
      zero   Lu = Lv: substitutions, and a balanced insertion / deletion before j where there is room (shift 0)
    each on both strands (u reverse-complemented).  Every pair has its own random template; u is stored before v and
    the order puts v before u.  One pair has a reverse-complement palindrome v, where ed(+) = ed(-), and '+' wins."""
    rng = np.random.default_rng(seed)
    T = Tables(X, lmax)
    segs = T.segments(Lv)
    k = len(segs)
    Kv = k - 1
    assert T.K[Lv] == Kv and T.HI[Lv] <= lmax
    pairs = []                                         # (u, v, d, strand, j, shift)
    for j in range(k):
        others = [i for i in range(k) if i != j]
        for strand in (0, 1):
            at = lambda: ("first", "last")[int(rng.integers(2))]   # noqa: E731
            # hi
            Lu = T.HI[Lv]
            d = T.D[Lu]
            n_ins = Lu - Lv
            order_ins = [i for i in others if i < j] + [i for i in others if i > j]
            ins = set(order_ins[:n_ins])
            edits = [None] * k
            for i in others:
                edits[i] = ("i" if i in ins else "s", at())
            assert len(others) == d
            pairs.append((edits, d, strand, j, sum(1 for i in ins if i < j)))
            # minus and zero: both strands; at K(Lv) >= 30 (hundreds of pairs) one strand each, alternating with j
            dv = T.D[Lv]
            if j >= dv and dv > 0 and (Kv < 30 or strand == j % 2):
                edits = [None] * k
                for i in rng.choice(j, dv, replace=False):
                    edits[int(i)] = ("d", at())
                pairs.append((edits, dv, strand, j, -dv))
            if dv > 0 and (Kv < 30 or strand != j % 2):
                edits = [None] * k
                pick = [int(i) for i in rng.choice(others, dv, replace=False)]
                for i in pick:
                    edits[i] = ("s", at())
                before = [i for i in pick if i < j]
                if len(before) >= 2:                       # a balanced insertion / deletion ahead of j
                    edits[before[0]] = ("i", at())
                    edits[before[1]] = ("d", at())
                pairs.append((edits, dv, strand, j, 0))
    reads, claims = [], []
    for edits, d, strand, j, shift in pairs:
        for _ in range(100):        # a new template until no cheaper alignment undoes an edit (rare but possible)
            v = rand_seq(rng, Lv)
            u = plant(rng, v, segs, edits)
            if R.ed(u, v, d) == d and R.ed(u, v, d, rc=True) > d:
                break
        assert d == T.D[max(len(u), Lv)]
        reads += [K.rc(u) if strand else u, v]
        claims.append(Claim(len(reads) - 1, len(reads) - 2, d, strand, j, shift))
    # the palindrome: v = h + rc(h) (Lv rounded down to even), u with D substitutions; ed(+) = ed(-) = d, '+' wins
    h = rand_seq(rng, Lv // 2)
    v = h + K.rc(h)
    d = T.D[len(v)]
    if d > 0:
        while True:
            u = bytearray(v)
            for p in rng.choice(len(v) // 2, d, replace=False):
                u[int(p)] = _other(rng, u[int(p)])
            u = bytes(u)
            if R.ed(u, v, d) == d:
                break
        reads += [u, v]
        claims.append(Claim(len(reads) - 1, len(reads) - 2, d, 0, None, None))
    reads.append(rand_seq(rng, lmax))                  # pins the call's longest class (and so HI and K) at lmax
    order = np.arange(len(reads), dtype=np.int32)
    order[:-1] = order[:-1].reshape(-1, 2)[:, ::-1].ravel()     # every v before its u
    return Case(reads, order, claims, X)


def check_claims(case, lmax):
    """On the CPU: every read is its own class, and every claim holds -- u's ed against v is d on its strand and above d
    on the other (equal for the palindrome), d = D(max(Lu, Lv)), segment j of v is in u's strand at v's position + shift
    and is found by the lookup.  Returns, per claim, whether the lookup finds the pair through segment j alone (at
    v's position + shift)."""
    T = Tables(case.X, lmax)
    assert max(len(r) for r in case.reads) == lmax
    keys = [min(norm(r), rcn(r)) for r in case.reads]
    assert len(set(keys)) == len(keys)
    only_j = []
    for c in case.claims:
        u, v = case.reads[c.u], case.reads[c.v]
        up = rcn(u) if c.strand else norm(u)
        assert c.d == T.D[max(len(u), len(v))]
        assert R.ed(u, v, c.d + 1, rc=bool(c.strand)) == c.d
        other = R.ed(u, v, c.d, rc=not c.strand)
        if c.j is None:
            assert other == c.d and rcn(v) == norm(v)
            only_j.append(False)
            continue
        assert other == c.d + 1
        segs = T.segments(len(v))
        a, b = segs[c.j]
        assert up[a + c.shift:b + c.shift] == v[a:b]
        hits = lookup_hits(up, v, c.d, len(segs))
        assert (c.j, a + c.shift) in hits
        only_j.append(hits == {(c.j, a + c.shift)})
    return only_j


# ---- a. identity sweep ----------------------------------------------------------------------------------------------
def sweep_lengths(X):
    """template lengths from 80 bp up to 600 bp, or to the longest whose variants (up to D(L) + 1 longer) keep
    D(lmax) <= 64"""
    lcap = d_lcap(X)
    D = _lib.cluster_dtable(X, 600)
    top = max(L for L in range(80, 601) if L + D[L] + 1 <= lcap)
    return sorted({80, (80 + top) // 2, top})


def ties(rng, X, L):
    """Reads whose best centroids tie in identity: u with e substitutions from each of two centroids c1, c2 of its own
    length (ed(c1, c2) = 2e > D), in both orders of c1 and c2 (abundance 3 / 2 / 1 sets the order: u joins the earlier);
    and, where X allows it at these lengths, a tie across lengths: c1 = u with e1 substitutions (len n * e1), c2 = u with n
    insertions and one substitution (e2 = e1 + 1), (n e1 - e1) / (n e1) = (n e1 + n - e1 - 1) / (n e1 + n)."""
    reads = []
    D = int(_lib.cluster_dtable(X, L)[L])
    if D >= 1:
        e = (D + 2) // 2
        for first_c1 in (True, False):
            for _ in range(1000):
                u = bytearray(rand_seq(rng, L))
                pos = [int(p) for p in rng.choice(L, 2 * e, replace=False)]
                c1, c2 = bytearray(u), bytearray(u)
                for p in pos[:e]:
                    c1[p] = _other(rng, u[p])
                for p in pos[e:]:
                    c2[p] = _other(rng, u[p])
                u, c1, c2 = bytes(u), bytes(c1), bytes(c2)
                if R.ed(u, c1, D) == e == R.ed(u, c2, D) and R.ed(c1, c2, D) > D:
                    break
            else:
                raise AssertionError("no tie at X = %g, L = %d" % (X, L))
            a, b = (c1, c2) if first_c1 else (c2, c1)
            reads += [bytes(a)] * 3 + [bytes(b)] * 2 + [K.rc(bytes(u)) if rng.random() < 0.5 else bytes(u)]
    n = int(np.ceil(1 / (1 - X) + 1e-9)) + 1
    while (n - 1) / n < X:
        n += 1
    if 1 - 1 / n < (1 + X) / 2 - 0.01 and n * n <= 600:
        e1 = n - 1
        L1 = n * e1
        L2 = L1 + n
        D2 = int(_lib.cluster_dtable(X, L2)[L2])
        for c1_first in (True, False):
            for _ in range(1000):
                u = bytearray(rand_seq(rng, L1))
                c1 = bytearray(u)
                for p in rng.choice(L1 // 2, e1, replace=False):
                    c1[int(p)] = _other(rng, u[int(p)])
                c2 = bytearray(u)
                q = L1 // 2 + int(rng.integers(L1 // 4))
                c2[q] = _other(rng, u[q])
                for p in sorted(rng.choice(np.arange(L1 // 2, L1 - 1), n, replace=False), reverse=True):
                    c2.insert(int(p) + 1, _other(rng, c2[int(p)], c2[int(p) + 1]))
                u, c1, c2 = bytes(u), bytes(c1), bytes(c2)
                if R.ed(u, c1, D2) == e1 and R.ed(u, c2, D2) == e1 + 1 and R.ed(c1, c2, D2) > D2:
                    break
            else:
                raise AssertionError("no tie across lengths at X = %g" % X)
            a, b = (c1, c2) if c1_first else (c2, c1)
            reads += [bytes(a)] * 3 + [bytes(b)] * 2 + [bytes(u)]
    return reads


def sweep(X, seed):
    """K.planted at three template lengths with the D(L) of X at each, and the ties above; default order"""
    rng = np.random.default_rng(seed)
    reads = []
    for i, L in enumerate(sweep_lengths(X)):
        D = int(_lib.cluster_dtable(X, L)[L])
        reads += K.planted(seed * 10 + i, L=L, ntemplates=4, D=D)
        reads += ties(rng, X, L)
    return Case(reads, None, [], X)


# ---- c. tiny reads, d. low complexity, e. the band cap --------------------------------------------------------------
def tiny(X, seed):
    """every ACGT string of length 1-5 and random reads of 6-15 residues"""
    import itertools
    rng = np.random.default_rng(seed)
    reads = [bytes(p) for n in range(1, 6) for p in itertools.product(b"ACGT", repeat=n)]
    reads += [rand_seq(rng, int(rng.integers(6, 16))) for _ in range(400)]
    return Case([reads[i] for i in rng.permutation(len(reads))], None, [], X)


def low_complexity(X, seed):
    """homopolymers, di- and trinucleotide repeats and ITS-like microsatellites (a repeat between random flanks), with
    the repeat lengthened or shortened by whole units and a few substitutions"""
    rng = np.random.default_rng(seed)
    reads = []
    for unit in (b"A", b"C", b"AC", b"AG", b"CT", b"AAT", b"CAG", b"GTT"):
        for L in (60, 150, 300):
            n = L // len(unit)
            for dn in range(-4, 5):
                reads.append(unit * (n + dn))
            s = bytearray(unit * n)
            for p in rng.choice(len(s), 3, replace=False):
                s[int(p)] = _other(rng, s[int(p)])
            reads.append(bytes(s))
    for _ in range(12):
        unit = [b"CT", b"GA", b"TTG", b"A", b"CA", b"AATG"][int(rng.integers(6))]
        left, right = rand_seq(rng, int(rng.integers(60, 200))), rand_seq(rng, int(rng.integers(60, 200)))
        n = int(rng.integers(8, 30))
        for dn in range(-3, 4):
            reads += [left + unit * (n + dn) + right] * int(rng.integers(1, 4))
        x = bytearray(left + unit * n + right)
        x[int(rng.integers(len(x)))] = ord("G")
        reads.append(bytes(x))
    return Case([reads[i] for i in rng.permutation(len(reads))], None, [], X)


def scatter(rng, v, n_sub, n_ins, n_del):
    """v with edits at distinct positions at least 3 apart (so that none of them merge into a cheaper alignment)"""
    n = n_sub + n_ins + n_del
    pos = np.sort(rng.choice(len(v) // 3 - 2, n, replace=False)) * 3 + 3
    kinds = ["s"] * n_sub + ["i"] * n_ins + ["d"] * n_del
    kinds = [kinds[i] for i in rng.permutation(n)]
    s = bytearray(v)
    for p, kd in sorted(zip(pos.tolist(), kinds), reverse=True):
        if kd == "s":
            s[p] = _other(rng, s[p])
        elif kd == "d":
            del s[p]
        else:
            s.insert(p, _other(rng, s[p - 1], s[p]))
    return bytes(s)


def band_cap(X, seed):
    """Classes of length lcap, the longest with D = 64, and variants at ed 64 (substitutions on either strand, deletions
    only, balanced insertions and deletions) and 65 (rejected); no class longer than lcap.  Returns the case and one
    read of length lcap + 1 (D = 65), which makes the call return ITSX_ELIMIT."""
    rng = np.random.default_rng(seed)
    L = d_lcap(X)
    reads, claims = [], []
    for strand, n_sub, n_ins, n_del, ok in ((0, 64, 0, 0, True), (1, 64, 0, 0, True), (0, 0, 0, 64, True),
                                            (1, 0, 32, 32, True), (0, 32, 16, 16, True), (0, 65, 0, 0, False),
                                            (1, 65, 0, 0, False), (0, 1, 0, 64, False), (1, 33, 16, 16, False)):
        e = n_sub + n_ins + n_del
        while True:
            v = rand_seq(rng, L)
            u = scatter(rng, v, n_sub, n_ins, n_del)
            if R.ed(u, v, e) == e and R.ed(u, v, MAXD, rc=True) > MAXD:
                break
        reads += [v, K.rc(u) if strand else u]
        if ok:
            claims.append(Claim(len(reads) - 2, len(reads) - 1, 64, strand, None, None))
        else:
            claims.append(Claim(len(reads) - 2, len(reads) - 1, 65, strand, None, None))
    return Case(reads, None, claims, X), rand_seq(rng, L + 1)


def check_band_cap(case):
    T = Tables(case.X, max(len(r) for r in case.reads))
    assert T.D[T.lmax] == MAXD and int(_lib.cluster_dtable(case.X, T.lmax + 1)[T.lmax + 1]) == MAXD + 1
    for c in case.claims:
        u, v = case.reads[c.u], case.reads[c.v]
        assert R.ed(u, v, MAXD + 1, rc=bool(c.strand)) == c.d
        assert R.ed(u, v, MAXD, rc=not c.strand) == MAXD + 1


# ---- f. scale, g. a long chain -------------------------------------------------------------------------------------
def _hp_indel(rng, s):
    """s with one homopolymer run (>= 3) lengthened or shortened by one; None without such a run"""
    runs = [i for i in range(len(s) - 2) if s[i] == s[i + 1] == s[i + 2]]
    if not runs:
        return None
    i = runs[int(rng.integers(len(runs)))]
    return s[:i] + s[i + 1:] if rng.random() < 0.5 else s[:i] + s[i:i + 1] + s[i:]


def scale(X, seed, n_families=480):
    """Families of an abundant random template (200-550 bp, Zipf abundance) and 10-80 error variants each: 1-4
    substitutions biased to the 3' end, homopolymer +-1 indels, some with both, some reverse-complemented.  Returns the
    case and the family of every read."""
    rng = np.random.default_rng(seed)
    reads, fam = [], []
    for f in range(n_families):
        T = rand_seq(rng, int(rng.integers(200, 551)))
        fr = [T] * int(min(5 + rng.zipf(1.6), 2000))
        for _ in range(int(rng.integers(10, 81))):
            s = T
            kind = rng.random()
            if kind < 0.7:
                s = bytearray(s)
                for _ in range(int(rng.integers(1, 5))):
                    p = int(len(s) - 1 - min(rng.exponential(len(s) / 3), len(s) - 1))
                    s[p] = _other(rng, s[p])
                s = bytes(s)
            if kind > 0.5:
                s = _hp_indel(rng, s) or s
            if rng.random() < 0.1:
                s = K.rc(s)
            fr += [s] * int(min(rng.zipf(2.5), 20))
        reads += fr
        fam += [f] * len(fr)
    perm = rng.permutation(len(reads))
    return Case([reads[i] for i in perm], None, [], X), np.asarray(fam, np.int32)[perm]


def chain(seed, n=3000, L=250):
    """n classes, each one substitution from the previous (never at the position just changed, so any two classes two
    links apart are two substitutions apart), in chain order: at 0.995 (D(250) = 1) the greedy alternates centroid and
    member, and only a long run of resolution rounds decides the last link"""
    rng = np.random.default_rng(seed)
    s = bytearray(rand_seq(rng, L))
    reads, last = [bytes(s)], -1
    while len(reads) < n:
        p = int(rng.integers(L))
        if p == last:
            continue
        s[p] = _other(rng, s[p])
        last = p
        reads.append(bytes(s))
    return Case(reads, np.arange(n, dtype=np.int32), [], 0.995)


# ---- the reference on whole workloads --------------------------------------------------------------------------------
def derep_first(reads):
    """(first, class_of_read): the first read of every class (normalised residues, either strand), in first-occurrence
    order, as the derep numbers its uniques"""
    key, first, cls = {}, [], []
    for i, r in enumerate(reads):
        k = min(norm(r), rcn(r))
        if k not in key:
            key[k] = len(first)
            first.append(i)
        cls.append(key[k])
    return np.asarray(first, np.int32), np.asarray(cls, np.int32)


def reference(case, first, class_uid, group=None, workers=None):
    """(n_centroids, crow, strand, ed, unique_of_row, accepted pairs) of the reference on the case, given the derep
    (first: unique -> first read, class_uid: read -> unique).  With a group per read (one family of scale()), every group
    is clustered and counted on its own, in parallel; the groups must have no accepted pair between them."""
    import cluster_samples_cases as S
    seq, off = K.pack(case.reads)
    rep = first[class_uid] if len(class_uid) else class_uid
    order = R.default_order(rep) if case.order is None else case.order
    if group is None:
        want = R.cluster(seq, off, first, order, case.X)
        return want + (R.accepted_pairs(seq, off, first, case.X),)
    want = S.per_sample_reference(seq, off, first, class_uid, group, case.X, order)
    gu = group[first]
    with cf.ThreadPoolExecutor(workers or os.cpu_count()) as ex:
        n = sum(ex.map(lambda k: R.accepted_pairs(seq, off, first[gu == k], case.X), np.unique(gu)))
    return want + (n,)
