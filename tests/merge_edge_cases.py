"""Edge workloads for the paired-end merge (csrc/merge.cu, itsx_merge_pairs): pairs built from an explicit fragment,
explicit qualities and an explicit overlap, so that each lands on one decision edge of the algorithm -- the
expected-error band around maxee, each threshold on both sides, pairs that fail several rules at once, the options the
command line never passes, read lengths around the 32-bit words of the 5-mer planes and at the shared-memory staging
limit, and every consensus branch.

Every constructor returns a Case (fs, fq, fo, rs, rq, ro, params, expect): the concatenated R1 / R2 bases and
qualities with their offsets (R2 as read from the file), the merge options (keyword arguments of merge_params,
allow_stagger included) and, per pair, a dict naming the edge the pair is meant to hit and the reason it must end with.
Where a value has to land next to a threshold (a score or a drop near 16 bits) candidates are generated from a fixed
seed and the first one the float64 arithmetic puts inside the window is kept.  tests/test_merge_edges_on_cpu.py proves
every claim against the C oracle and the Python statement of tests/golden/make_merge_golden.py;
tests/test_gpu_merge_edges.py runs the cases on the device."""
import importlib.util
import math
import os
from collections import namedtuple

import numpy as np

_spec = importlib.util.spec_from_file_location(
    "make_merge_golden", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_merge_golden.py"))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)

Case = namedtuple("Case", "fs fq fo rs rq ro params expect")
REASONS = ("ok", "repeat", "staggered", "maxdiffs", "maxdiffpct", "nokmers", "minscore", "minovlen", "maxee", "badqual")
RULES = REASONS[1:9]                     # the order in which the rules are tested; the first failing one is reported

MG_WARPS = 4                             # warps (pairs in flight) per CTA of merge_kernel
SMEM_LIMIT = 200 * 1024                  # bytes of shared-memory staging the merge accepts per CTA
B200_WARPS = 148 * MG_WARPS              # resident warps on a 148-SM B200 at one CTA per SM
Q40 = 40
LENS = (0, 1, 4, 5, 31, 32, 33, 63, 64, 65, 96, 97)
_COMP = bytes.maketrans(b"ACGTURYSWKMBDHVN", b"TGCAAYRSWMKVHDBN")


def revcomp(s):
    return s.translate(_COMP)[::-1]


def rnd(rng, n, alphabet=b"ACGT"):
    return bytes(rng.choice(np.frombuffer(alphabet, np.uint8), n)) if n else b""


def other(b):
    """a plain base different from b"""
    return {ord("A"): b"C", ord("C"): b"G", ord("G"): b"T", ord("T"): b"A"}[b]


def staging_bytes(maxF, maxR):
    """shared memory merge_kernel needs for a batch whose longest reads are maxF / maxR bases (merge.cu: four warps,
    per warp four forward bit planes of WF words, four rc planes of WR + 2 words, bases / qualities / rc bases / rc
    qualities / merged qualities padded to a multiple of four)"""
    WF, WR = max(1, (maxF + 31) // 32), max(1, (maxR + 31) // 32)
    LF, LR = (maxF + 3) & ~3, (maxR + 3) & ~3
    return (16 * (WF + WR + 2) + 3 * (LF + LR)) * MG_WARPS


def largest_equal_len():
    """the largest F = R the staging accepts"""
    L = 1
    while staging_bytes(L + 1, L + 1) <= SMEM_LIMIT:
        L += 1
    return L


def largest_f_for(R):
    F = 1
    while staging_bytes(F + 1, R) <= SMEM_LIMIT:
        F += 1
    return F


# ---- pairs ------------------------------------------------------------------------------------------------------------

def pair(r1, q1, rcb, rcq):
    """R1 bases / Q values and the reverse complement of R2 with its Q values (forward orientation): the R2 record as
    the file holds it"""
    assert len(r1) == len(q1) and len(rcb) == len(rcq)
    return r1, list(q1), revcomp(rcb), list(rcq)[::-1]


def shifted(rng, F, R, sh, q1=None, rcq=None):
    """R1 and rc(R2) cut from one random sequence, rc(R2) starting sh bases after R1 (negative: before it): forward
    position p pairs with rc position p - sh, i.e. the pair overlaps on diagonal i = F - sh"""
    lo, hi = min(0, sh), max(F, sh + R)
    u = rnd(rng, hi - lo)
    r1, rcb = u[-lo:-lo + F], u[sh - lo:sh - lo + R]
    q1 = [Q40] * F if q1 is None else q1
    rcq = [Q40] * R if rcq is None else rcq
    return pair(r1, q1, rcb, rcq)


def overlap_pair(rng, pattern, left=20, right=20, mq=2, nq=Q40):
    """R1 = `left` random bases + the overlap + nothing; rc(R2) = the overlap + `right` random bases.  pattern gives the
    overlap position by position: 'M' the same base in both (Q40), 'x' different bases (Q mq in both), 'N' N in both"""
    ov = rnd(rng, len(pattern))
    a, b, qa, qb = bytearray(ov), bytearray(ov), [], []
    for k, c in enumerate(pattern):
        if c == "x":
            a[k] = other(ov[k])[0]
            qa.append(mq); qb.append(mq)
        elif c == "N":
            a[k] = b[k] = ord("N")
            qa.append(nq); qb.append(nq)
        else:
            qa.append(Q40); qb.append(Q40)
    r1 = rnd(rng, left) + bytes(a)
    rcb = bytes(b) + rnd(rng, right)
    return pair(r1, [Q40] * left + qa, rcb, qb + [Q40] * right)


def pack(pairs, params=None, expect=None, ascii=33):
    """a Case from (r1, q1, r2, q2) tuples (Q values as integers)"""
    fo, ro = np.zeros(len(pairs) + 1, np.int64), np.zeros(len(pairs) + 1, np.int64)
    fo[1:] = np.cumsum([len(p[0]) for p in pairs])
    ro[1:] = np.cumsum([len(p[2]) for p in pairs])
    cat = lambda k: np.frombuffer(b"".join(p[k] for p in pairs), np.uint8).copy()      # noqa: E731
    catq = lambda k: np.array([q + ascii for p in pairs for q in p[k]], np.uint8)       # noqa: E731
    params = dict(params or {})
    if ascii != 33:
        params["ascii"] = ascii
    return Case(cat(0), catq(1), fo, cat(2), catq(3), ro, params, expect or [{} for _ in pairs])


def records(case):
    """per pair (r1, q1, r2, q2) as bytes (quality characters), the form the Python statement takes"""
    out = []
    for i in range(len(case.fo) - 1):
        f, r = slice(case.fo[i], case.fo[i + 1]), slice(case.ro[i], case.ro[i + 1])
        out.append((case.fs[f].tobytes(), case.fq[f].tobytes(), case.rs[r].tobytes(), case.rq[r].tobytes()))
    return out


def reference(case):
    """per pair (merged, reason, info) from the Python statement under the case's options"""
    kw = dict(case.params)
    kw["stagger"] = bool(kw.pop("allow_stagger", False))
    out = []
    for r1, q1, r2, q2 in records(case):
        info = {}
        merged, why = G.merge_pair(r1, q1, r2, q2, info=info, **kw)
        out.append((merged, why, info))
    return out


def strided_ee(quals, ascii=33):
    """expected errors of a merged read summed as merge_kernel sums them: lane l adds the error probabilities of
    positions m = l, l + 32, ... in order, then the 32 partial sums are combined by xor shuffles at 16, 8, 4, 2, 1"""
    part = [0.0] * 32
    for m, q in enumerate(quals):
        part[m % 32] += G.P[q - ascii]
    for o in (16, 8, 4, 2, 1):
        part = [part[lane] + part[lane ^ o] for lane in range(32)]
    return part[0]


def read_order_ee(quals, ascii=33):
    ee = 0.0
    for q in quals:
        ee += G.P[q - ascii]
    return ee


def in_band(part, maxee):
    """merge_kernel replays the sum in read order only when the strided sum lies this close to maxee"""
    return abs(part - maxee) <= 1e-9 * (1.0 + abs(part))


def failing_rules(info, params):
    """every rule the pair breaks, in the order they are tested (the merged read's expected errors included)"""
    stag = params.get("allow_stagger", False)
    out = []
    if info["hits"] > 1:
        out.append("repeat")
    if not stag and info["best_i"] > info["F"]:
        out.append("staggered")
    if info["best_diffs"] > params.get("maxdiffs", 40):
        out.append("maxdiffs")
    if info["best_i"] and 100.0 * info["best_diffs"] / info["best_i"] > params.get("maxdiffpct", 100.0):
        out.append("maxdiffpct")
    if not info["kmers"]:
        out.append("nokmers")
    if info["best_score"] < 16.0:
        out.append("minscore")
    if info["best_i"] < params.get("minovlen", 10):
        out.append("minovlen")
    if "ee" in info and info["ee"] > params.get("maxee", 2.0):
        out.append("maxee")
    return out


# ---- expected-error band ----------------------------------------------------------------------------------------------

def _merged_quals_clean(q1, rcq, sh):
    """qualities of the merged read of an error-free, N-free overlap on shift sh >= 0 (default options)"""
    F, R = len(q1), len(rcq)
    ov = min(F - sh, R)
    return (list(q1[:sh]) + [G.SAME[a][b] - 33 for a, b in zip(q1[sh:sh + ov], rcq[:ov])] + list(rcq[ov:]))


def ee_band(lengths=(40, 150, 333, 700), seed=1):
    """For each merged length: one pair whose merged read must merge with maxee equal to its read-order expected errors
    and fail one ulp below, each as its own case.  Qualities are Q20 (p = 0.01, not a binary fraction) with a sprinkle
    of Q13 / Q30 from a fixed seed; the candidates are walked until the strided sum merge_kernel takes first differs
    from the read-order sum, so that one of the two cases of the length sits on the side where only the read-order
    replay decides correctly.  The last length is the longest merged read the staging allows."""
    rng = np.random.default_rng(seed)
    L = largest_equal_len()
    out = []
    for n in list(lengths) + [2 * L - 20]:
        if n > 2 * L - 100:
            F = R = L
        else:
            F = R = (n + 20) // 2
        sh = n - R                                          # overlap F - sh
        for attempt in range(200):
            q1 = [int(x) for x in rng.choice([20, 20, 20, 20, 13, 30], F)]
            rcq = [int(x) for x in rng.choice([20, 20, 20, 20, 13, 30], R)]
            mq = _merged_quals_clean(q1, rcq, sh)
            s, t = read_order_ee([q + 33 for q in mq]), strided_ee([q + 33 for q in mq])
            if s != t:
                break
        else:
            raise AssertionError("no candidate separates the two sums at length %d" % n)
        p = shifted(rng, F, R, sh, q1, rcq)
        for side, maxee, why in (("at", s, "ok"), ("below", math.nextafter(s, -math.inf), "maxee")):
            disagree = (t <= maxee) != (s <= maxee)
            out.append(pack([p], {"maxee": maxee},
                            [{"edge": "ee_%s" % side, "reason": why, "n": n, "ee": s, "strided": t,
                              "disagree": disagree}]))
    return out


# ---- thresholds -------------------------------------------------------------------------------------------------------

def _with_mismatches(rng, F, R, sh, at, q_mis=10):
    """shifted pair with R1 changed at the given forward positions (inside the overlap), R1 quality q_mis there"""
    r1, q1, r2, q2 = shifted(rng, F, R, sh)
    r1 = bytearray(r1)
    for p in at:
        r1[p] = other(r1[p])[0]
        q1[p] = q_mis
    return bytes(r1), q1, r2, q2


def maxdiffs(d=6):
    rng = np.random.default_rng(11)
    F = R = 150
    sh = 50                                                 # overlap 100: positions 50 .. 149
    p = _with_mismatches(rng, F, R, sh, [55 + 14 * k for k in range(d)])
    return [pack([p], {"maxdiffs": d}, [{"edge": "maxdiffs_at", "reason": "ok", "diffs": d}]),
            pack([p], {"maxdiffs": d - 1}, [{"edge": "maxdiffs_over", "reason": "maxdiffs", "diffs": d}])]


def minovlen(ovs=(12, 31, 32, 33)):
    rng = np.random.default_rng(12)
    out = []
    for ov in ovs:
        F = R = 80
        p = shifted(rng, F, R, F - ov)
        out.append(pack([p], {"minovlen": ov}, [{"edge": "minovlen_at", "reason": "ok", "i": ov}]))
        out.append(pack([p], {"minovlen": ov + 1}, [{"edge": "minovlen_over", "reason": "minovlen", "i": ov}]))
    return out


def maxdiffpct(d=3, i=70):
    rng = np.random.default_rng(13)
    F = R = 90
    sh = F - i
    p = _with_mismatches(rng, F, R, sh, [sh + 10 + 20 * k for k in range(d)])
    pct = 100.0 * d / i
    return [pack([p], {"maxdiffpct": pct}, [{"edge": "maxdiffpct_at", "reason": "ok", "diffs": d, "i": i}]),
            pack([p], {"maxdiffpct": math.nextafter(pct, -math.inf)},
                 [{"edge": "maxdiffpct_below", "reason": "maxdiffpct", "diffs": d, "i": i}])]


# overlap patterns: runs of matches ('M') between low-quality mismatches ('x'); runs of four make no 5-mer
KMER_PATTERNS = (
    ("run7", "MMMMMMMx", 3, "nokmers"),
    ("run8", "MMMMMMMMx", 4, "ok"),
    ("run6_run6", "MMMMMMxMMMMMMx", 4, "ok"),
    ("run6_NN_run6", "MMMMMMNMMMMMMx", 4, "ok"),
    ("run6_NN_run5", "MMMMMMNMMMMMx", 3, "nokmers"),
    ("run8_NN_inside", "MMMMNMMMMx", 0, "nokmers"),
)


def kmers():
    """best diagonal with exactly 3 / exactly 4 matching 5-mers: a planted run (at the start of the overlap, and across
    forward position 32 where the planes change word) followed by runs of four matches"""
    rng = np.random.default_rng(14)
    pairs, expect = [], []
    for name, head, cnt, why in KMER_PATTERNS:
        for left in (20, 27):                             # the overlap starts at forward position 20 / 27
            pat = head + "MMMMx" * 8
            pairs.append(overlap_pair(rng, pat, left=left))
            expect.append({"edge": "kmers_%d" % cnt, "reason": why, "cnt": cnt, "i": len(pat), "name": name})
    return [pack(pairs, {"maxee": 100.0}, expect)]


def stagger():
    """fragment of F - 1, F and F + 1 bases under reads of F: diagonal F + 1 (staggered), F, F - 1"""
    rng = np.random.default_rng(15)
    F = R = 60
    ps = [shifted(rng, F, R, sh) for sh in (-1, 0, 1)]
    out = []
    for st in (0, 1):
        exp = [{"edge": "stagger_frag_%s" % n, "reason": "staggered" if (n == "F-1" and not st) else "ok", "i": F - sh}
               for n, sh in (("F-1", -1), ("F", 0), ("F+1", 1))]
        out.append(pack(ps, {"allow_stagger": st}, exp))
    return out


def _score(q1s, q2s, eqs):
    """the diagonal's score and drop replayed from the 3' end (lists in forward order)"""
    score = high = dropmax = 0.0
    for qa, qb, e in zip(q1s[::-1], q2s[::-1], eqs[::-1]):
        if e:
            score += G.MATCH[qa][qb]
            high = max(high, score)
        else:
            score += G.MISM[qa][qb]
            if score < high - dropmax:
                dropmax = high - score
    return score, dropmax


def score_edge(ov=10, width=0.05):
    """an error-free overlap of ov bases whose qualities put the score inside [16, 16 + width) (merges) and inside
    (16 - width, 16) (fails minscore)"""
    rng = np.random.default_rng(16)
    found = {}
    for _ in range(20000):
        qa = [int(x) for x in rng.integers(2, 41, ov)]
        qb = [int(x) for x in rng.integers(2, 41, ov)]
        s, _ = _score(qa, qb, [True] * ov)
        side = "above" if 16.0 <= s < 16.0 + width else "below" if 16.0 - width < s < 16.0 else None
        if side and side not in found:
            found[side] = (qa, qb, s)
        if len(found) == 2:
            break
    pairs, expect = [], []
    for side in ("above", "below"):
        qa, qb, s = found[side]
        F = R = 40
        sh = F - ov
        pairs.append(shifted(rng, F, R, sh, [Q40] * sh + qa, qb + [Q40] * (R - ov)))
        expect.append({"edge": "score_%s" % side, "reason": "ok" if side == "above" else "minscore", "score": s})
    return [pack(pairs, {"maxee": 100.0}, expect)]


def drop_edge(width=0.05):
    """a clean overlap scored from its 3' end: `a` matches, two adjacent mismatches whose qualities put the drop inside
    [16, 16 + width) (the diagonal scores 0: minscore) or (16 - width, 16) (merges), then 30 matches.  a = 10 keeps
    the drop in the first 32-element chunk of the replay, a = 31 puts the second mismatch at element 32 (the drop
    reaches the window only in the next chunk), a = 40 puts both in the second chunk."""
    rng = np.random.default_rng(17)
    pairs, expect = [], []
    for a in (10, 31, 40):
        found = {}
        b = 30
        ov = a + 2 + b
        for _ in range(50000):
            qm = [int(x) for x in rng.integers(2, 41, 4)]
            q1s = [Q40] * b + [qm[0], qm[1]] + [Q40] * a
            q2s = [Q40] * b + [qm[2], qm[3]] + [Q40] * a
            eqs = [True] * b + [False, False] + [True] * a
            s, d = _score(q1s, q2s, eqs)
            side = "above" if 16.0 <= d < 16.0 + width else "below" if 16.0 - width < d < 16.0 else None
            if side and side not in found:
                found[side] = (q1s, q2s, d)
            if len(found) == 2:
                break
        for side in ("above", "below"):
            q1s, q2s, d = found[side]
            F = R = ov + 20
            sh = F - ov
            r1, q1, r2, q2 = shifted(rng, F, R, sh, [Q40] * sh + q1s, q2s + [Q40] * (R - ov))
            r1 = bytearray(r1)
            for p in (sh + b, sh + b + 1):
                r1[p] = other(r1[p])[0]
            pairs.append((bytes(r1), q1, r2, q2))
            expect.append({"edge": "drop_%s" % side, "reason": "minscore" if side == "above" else "ok", "drop": d,
                           "first_mismatch_element": a})
    return [pack(pairs, {"maxee": 100.0}, expect)]


# ---- precedence -------------------------------------------------------------------------------------------------------

def precedence():
    """pairs that break two or three rules at once; each is its own case (the options differ).  The expected reason is
    the first broken rule in the order repeat, staggered, maxdiffs, maxdiffpct, nokmers, minscore, minovlen, maxee."""
    rng = np.random.default_rng(18)
    out = []

    def add(p, params, why, n_rules):
        out.append(pack([p], params, [{"edge": "precedence", "reason": why, "n_rules": n_rules}]))

    # staggered + maxdiffs + maxdiffpct: fragment one base shorter than the reads, six mismatches
    p = _with_mismatches(rng, 60, 60, -1, [5, 15, 25, 35, 45, 55])
    add(p, {"maxdiffs": 3, "maxdiffpct": 5.0}, "staggered", 3)
    add(p, {"maxdiffs": 3, "maxdiffpct": 5.0, "allow_stagger": 1}, "maxdiffs", 2)
    # maxdiffs + maxdiffpct + minovlen
    p = _with_mismatches(rng, 60, 60, 20, [22, 28, 34, 40, 46, 52])
    add(p, {"maxdiffs": 5, "maxdiffpct": 10.0, "minovlen": 50}, "maxdiffs", 3)
    # maxdiffpct + minovlen + maxee
    add(p, {"maxdiffpct": 10.0, "minovlen": 50, "maxee": 1e-3}, "maxdiffpct", 3)
    # minscore + minovlen: eight Q40 matches score 15.998 bits
    p = shifted(rng, 30, 30, 22)
    add(p, {}, "minscore", 2)
    # minovlen + maxee
    p = shifted(rng, 40, 40, 28)
    add(p, {"minovlen": 13, "maxee": 1e-4}, "minovlen", 2)
    # repeat + maxdiffs: a tandem repeat (several diagonals score >= 16 bits) with a mismatch on every one
    unit = rnd(rng, 20)
    frag = bytearray(unit * 8)
    frag[70] = other(frag[70])[0]
    r1, rcb = bytes(frag[:120]), bytes(unit * 8)[40:]
    add(pair(r1, [Q40] * 120, rcb, [Q40] * 120), {"maxdiffs": 0}, "repeat", 2)
    # nokmers + minovlen: unrelated reads (best_i stays 0)
    add((rnd(rng, 50), [Q40] * 50, rnd(rng, 50), [Q40] * 50), {}, "nokmers", 2)
    return out


# ---- options ----------------------------------------------------------------------------------------------------------

def plain_pairs(seed, n=48, ascii=33, params=None):
    """ordinary pairs (2 x 100 off 110-190 bp fragments, a few errors, Q20-Q40) for the option cases"""
    rng = np.random.default_rng(seed)
    pairs = []
    for k in range(n):
        L = int(rng.integers(110, 190))
        F = R = 100
        q1 = [int(x) for x in rng.integers(20, 41, F)]
        rcq = [int(x) for x in rng.integers(20, 41, R)]
        r1, q1, r2, q2 = shifted(rng, F, R, L - R, q1, rcq)
        r1 = bytearray(r1)
        for p in rng.integers(0, F, 2):
            r1[p] = other(r1[p])[0]
        pairs.append((bytes(r1), q1, r2, q2))
    return pack(pairs, params, [{"edge": "plain"} for _ in pairs], ascii=ascii)


def ascii64_sequence():
    """the same pairs in Phred+33 under the defaults, in Phred+64 under ascii = 64, then Phred+33 again: one context
    running them in this order has to rebuild its tables at each step"""
    return [plain_pairs(21), plain_pairs(21, ascii=64), plain_pairs(21)]


def qmax_cases(qmax=41):
    """qmax below 93: a quality exactly at qmax is accepted, one above it stops the call"""
    rng = np.random.default_rng(22)
    at = shifted(rng, 80, 80, 30, [qmax] * 80, [Q40] * 80)
    over = shifted(rng, 80, 80, 30, [Q40] * 79 + [qmax + 1], [Q40] * 80)
    return [pack([at], {"qmax": qmax, "maxee": 100.0}, [{"edge": "qmax_at", "reason": "ok"}]),
            pack([at, over], {"qmax": qmax, "maxee": 100.0},
                 [{"edge": "qmax_at", "reason": "ok"}, {"edge": "qmax_over", "reason": "badqual"}])]


def qout_cases(qmaxout=35, qminout=3):
    """qmaxout / qminout clamp the posterior qualities: agreeing Q40 bases (posterior Q85) come out at qmaxout, a Q2 / Q2
    disagreement (posterior Q2) at qminout"""
    rng = np.random.default_rng(23)
    pairs = [overlap_pair(rng, "MMMMMMMMMMxMMMMMMMMMMxMMMMMMMM"), overlap_pair(rng, "MMMMMMMMMMMMxMMMMMMMMMM")]
    return [pack(pairs, {"qmaxout": qmaxout, "qminout": qminout, "maxee": 100.0},
                 [{"edge": "qout", "reason": "ok", "qmaxout": qmaxout, "qminout": qminout} for _ in pairs])]


# ---- geometry ---------------------------------------------------------------------------------------------------------

def length_grid(stag=1):
    """F, R in LENS in all combinations, each on the diagonals whose shift is 0, +-1, +-31, +-32, +-33, 63, 64, 65 (mod 32:
    0, 1, 31) where they overlap, with a sequencing error now and then"""
    rng = np.random.default_rng(31)
    pairs, expect = [], []
    for F in LENS:
        for R in LENS:
            shs = [sh for sh in (-33, -32, -31, -1, 0, 1, 31, 32, 33, 63, 64, 65) if 1 <= F - sh <= F + R - 1]
            for sh in shs or [0]:
                q1 = [int(x) for x in rng.integers(25, 41, F)]
                rcq = [int(x) for x in rng.integers(25, 41, R)]
                r1, q1, r2, q2 = shifted(rng, F, R, sh, q1, rcq)
                if F > 20 and rng.random() < 0.3:
                    r1 = bytearray(r1)
                    r1[int(rng.integers(0, F))] = ord("G")
                    r1 = bytes(r1)
                pairs.append((r1, q1, r2, q2))
                expect.append({"edge": "grid", "F": F, "R": R, "sh": sh})
    return pack(pairs, {"allow_stagger": stag}, expect)


def low_complexity():
    """poly-A and period-2 reads: every diagonal of a group of 32 is a candidate"""
    pairs, expect = [], []
    for n in (31, 32, 33, 64, 65, 97, 250):
        for unit in (b"A", b"AC", b"AG"):
            frag = (unit * (n + 16))[:n + 16]
            pairs.append(pair(frag[:n], [Q40] * n, frag[16:16 + n], [30] * n))
            expect.append({"edge": "low_complexity", "n": n})
    return pack(pairs, {}, expect)


def limit_equal(seed=41):
    """F = R = the largest length the staging accepts, overlap 150, a few errors; and the same four bases longer"""
    rng = np.random.default_rng(seed)
    L = largest_equal_len()
    r1, q1, r2, q2 = shifted(rng, L, L, L - 150)
    r1 = bytearray(r1)
    for p in (L - 140, L - 77, L - 20):
        r1[p] = other(r1[p])[0]
        q1[p] = 20
    ok = pack([(bytes(r1), q1, r2, q2)], {}, [{"edge": "limit_equal", "reason": "ok", "F": L, "R": L}])
    over = pack([shifted(rng, L + 4, L + 4, L - 146)], {}, [{"edge": "limit_over", "F": L + 4, "R": L + 4}])
    return ok, over


def limit_unequal(R=40, seed=42):
    """R1 as long as the staging allows next to an R2 of R bases, overlapping at R1's 3' end"""
    rng = np.random.default_rng(seed)
    F = largest_f_for(R)
    return pack([shifted(rng, F, R, F - 30)], {"maxee": 100.0},
                [{"edge": "limit_unequal", "reason": "ok", "F": F, "R": R}])


def reuse_mix(nwarps=B200_WARPS, rounds=4, seed=43):
    """More pairs than resident warps, so that every warp merges a pair in its shared-memory slice after a longer one.
    Pair 0 is as long as the staging allows (one CTA per SM: warp w takes pairs w, w + nwarps, ...); the other pairs of
    even rounds are long (150-300 bases), those of odd rounds short (0-90 bases).  Every second long pair has an R2 of
    T only (its reverse complement fills the A plane), and every second short pair puts 40 A behind 30 random A / T
    bases against an R2 of 20 random C / G: no base of R1 matches its reverse complement, so the pair has no 5-mer hit
    (nokmers), while a stale word of the rc A plane behind the R2 would show as hits against the 40 A."""
    rng = np.random.default_rng(seed)
    L = largest_equal_len()
    pairs, expect = [], []
    for rd in range(rounds):
        for w in range(nwarps):
            if rd == 0 and w == 0:
                pairs.append(shifted(rng, L, L, L - 200))
                kind = "limit"
            elif rd % 2 == 0:
                F, R = int(rng.integers(150, 301)), int(rng.integers(150, 301))
                if w % 2:
                    pairs.append((rnd(rng, F), [Q40] * F, b"T" * R, [Q40] * R))
                    kind = "long_polyT"
                else:
                    pairs.append(shifted(rng, F, R, int(rng.integers(F // 3, F - 20))))
                    kind = "long"
            else:
                if w % 2:
                    pairs.append((rnd(rng, 30, b"AT") + b"A" * 40, [Q40] * 70, rnd(rng, 20, b"CG"), [Q40] * 20))
                    kind = "short_probe"
                else:
                    F, R = int(rng.integers(0, 91)), int(rng.integers(0, 91))
                    sh = int(rng.integers(-R // 2, F)) if F else 0
                    pairs.append(shifted(rng, F, R, sh) if F and R else (rnd(rng, F), [Q40] * F, rnd(rng, R), [Q40] * R))
                    kind = "short"
            expect.append({"edge": "reuse", "kind": kind})
    return pack(pairs, {"allow_stagger": 1}, expect)


# ---- consensus --------------------------------------------------------------------------------------------------------

CONSENSUS_BRANCHES = ("n_r1", "n_r2", "n_both", "equal", "equal_iupac", "tie", "r1_better", "r2_better")


def consensus():
    """overlaps with an N in R1, in R2 and in both, equal IUPAC symbols, disagreements with R1 better, R2 better and
    equal qualities, next to ordinary agreeing bases"""
    rng = np.random.default_rng(51)
    pairs = []
    for k in range(6):
        F = R = 90
        sh = 30
        r1, q1, r2, q2 = shifted(rng, F, R, sh, [int(x) for x in rng.integers(10, 41, F)],
                                 [int(x) for x in rng.integers(10, 41, R)])
        a, rcb, rcq = bytearray(r1), bytearray(revcomp(r2)), q2[::-1]
        # forward position p pairs with rc position p - sh; positions chosen 6 apart inside the overlap
        edits = [("n_r1", 40), ("n_r2", 46), ("n_both", 52), ("iupac", 58), ("tie", 64), ("r1_better", 70),
                 ("r2_better", 76), ("tie", 82 + k)]
        for what, p in edits:
            r = p - sh
            if what.startswith("n_"):
                if what != "n_r2":
                    a[p] = ord("N")
                if what != "n_r1":
                    rcb[r] = ord("N")
                q1[p], rcq[r] = 10, 10
            elif what == "iupac":
                a[p] = rcb[r] = ord("RYKMSW"[k])
            else:
                a[p] = other(rcb[r])[0]
                q1[p], rcq[r] = {"tie": (25, 25), "r1_better": (35, 15), "r2_better": (15, 35)}[what]
        pairs.append(pair(bytes(a), q1, bytes(rcb), rcq))
    return pack(pairs, {"maxee": 100.0}, [{"edge": "consensus", "reason": "ok"} for _ in pairs])


def all_cases():
    """every case that runs as one ordinary call, by family"""
    ok, _ = limit_equal()
    return {
        "ee_band": ee_band(),
        "maxdiffs": maxdiffs(), "minovlen": minovlen(), "maxdiffpct": maxdiffpct(), "kmers": kmers(),
        "stagger": stagger(), "score": score_edge(), "drop": drop_edge(),
        "precedence": precedence(),
        "options": ascii64_sequence() + qmax_cases()[:1] + qout_cases(),
        "geometry": [length_grid(1), length_grid(0), low_complexity(), ok, limit_unequal()],
        "consensus": [consensus()],
    }
