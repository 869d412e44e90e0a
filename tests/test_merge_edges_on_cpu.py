"""The edge workloads of tests/merge_edge_cases.py, on the CPU: the C oracle (oracle/ora_merge.c) and the independent
Python statement (tests/golden/make_merge_golden.py) agree on every pair of every case, and every pair lands on the
edge it was built for -- both sides of each threshold, the first of several broken rules, the expected-error band
where the strided sum merge_kernel takes first and the read-order sum disagree about maxee, every consensus branch.
tests/test_gpu_merge_edges.py holds the device to the same cases."""
import math

import numpy as np
import pytest

import merge_edge_cases as E

G = E.G


def oracle_run(oracle, case):
    kw = dict(case.params)
    st = kw.pop("allow_stagger", 0)
    return oracle.merge_pairs(case.fs, case.fq, case.fo, case.rs, case.rq, case.ro,
                              oracle.merge_params(allow_stagger=st, **kw))


def agree(oracle, case):
    """the oracle and the Python statement give the same reason, length, bases and qualities for every pair; returns
    the Python statement's (merged, reason, info) per pair"""
    ml, why, oseq, oqual = oracle_run(oracle, case)
    ref = E.reference(case)
    for i, (merged, r, info) in enumerate(ref):
        assert E.REASONS[why[i]] == r, (i, case.expect[i], r)
        if merged is None or r != "ok":
            assert ml[i] == 0
            continue
        s = int(case.fo[i] + case.ro[i])
        assert ml[i] == len(merged[0])
        assert oseq[s:s + ml[i]].tobytes() == merged[0] and oqual[s:s + ml[i]].tobytes() == merged[1]
    for e, (_, r, _) in zip(case.expect, ref):
        if "reason" in e:
            assert r == e["reason"], e
    return ref


CASES = E.all_cases()


@pytest.mark.parametrize("family", sorted(CASES))
def test_oracle_and_python_statement_agree(oracle, family):
    for case in CASES[family]:
        agree(oracle, case)


def test_ee_band(oracle):
    cases = E.ee_band()
    lengths = set()
    for case in cases:
        (merged, why, info), = agree(oracle, case)
        e, maxee = case.expect[0], case.params["maxee"]
        quals = list(info["merged"][1])
        assert len(quals) == e["n"] and info["ee"] == E.read_order_ee(quals) == e["ee"]
        assert E.strided_ee(quals) == e["strided"]
        # the kernel's strided sum lies inside the replay band, and read order decides
        assert E.in_band(e["strided"], maxee)
        assert (why == "ok") == (e["ee"] <= maxee)
        if e["disagree"]:
            assert (e["strided"] <= maxee) != (e["ee"] <= maxee)
            lengths.add(e["n"])
        assert maxee == e["ee"] if e["edge"] == "ee_at" else maxee == math.nextafter(e["ee"], -math.inf)
    # at every length, including the longest merged read the staging allows, one case needs the replay
    assert lengths == {c.expect[0]["n"] for c in cases}
    assert max(lengths) == 2 * E.largest_equal_len() - 20


def test_thresholds_on_both_sides(oracle):
    seen = set()
    for case in E.maxdiffs() + E.minovlen() + E.maxdiffpct():
        (_, why, info), = agree(oracle, case)
        e = case.expect[0]
        if "diffs" in e:
            assert info["best_diffs"] == e["diffs"]
        if "i" in e:
            assert info["best_i"] == e["i"]
        if e["edge"].startswith("maxdiffs"):
            assert case.params["maxdiffs"] == e["diffs"] - (e["edge"] == "maxdiffs_over")
        if e["edge"].startswith("minovlen"):
            assert case.params["minovlen"] == e["i"] + (e["edge"] == "minovlen_over")
        if e["edge"] == "maxdiffpct_at":
            assert 100.0 * e["diffs"] / e["i"] == case.params["maxdiffpct"]
        if e["edge"] == "maxdiffpct_below":
            assert case.params["maxdiffpct"] == math.nextafter(100.0 * e["diffs"] / e["i"], -math.inf)
        seen.add(e["edge"])
    assert seen == {"maxdiffs_at", "maxdiffs_over", "minovlen_at", "minovlen_over", "maxdiffpct_at", "maxdiffpct_below"}


def test_kmer_threshold(oracle):
    case, = E.kmers()
    counts = set()
    for (r1, q1, r2, q2), e, (_, why, info) in zip(E.records(case), case.expect, agree(oracle, case)):
        rc = r2.translate(E._COMP)[::-1]
        k = G.kmer_counts(r1, rc)
        assert k[e["i"]] == e["cnt"], e                    # the planted diagonal
        if why == "nokmers":
            assert k.max() < 4
        else:
            assert info["best_i"] == e["i"] and info["diags"][e["i"]][0] == 4
        counts.add(e["cnt"])
    assert {3, 4} <= counts


def test_stagger_edges(oracle):
    got = {}
    for case in E.stagger():
        for e, (_, why, info) in zip(case.expect, agree(oracle, case)):
            assert info["best_i"] == e["i"] and info["best_i"] - info["F"] == {"stagger_frag_F-1": 1, "stagger_frag_F": 0,
                                                                               "stagger_frag_F+1": -1}[e["edge"]]
            got[(e["edge"], case.params["allow_stagger"])] = why
    assert got == {("stagger_frag_F-1", 0): "staggered", ("stagger_frag_F", 0): "ok", ("stagger_frag_F+1", 0): "ok",
                   ("stagger_frag_F-1", 1): "ok", ("stagger_frag_F", 1): "ok", ("stagger_frag_F+1", 1): "ok"}


def test_score_and_drop_windows(oracle):
    case, = E.score_edge()
    sides = set()
    for e, (_, why, info) in zip(case.expect, agree(oracle, case)):
        s = info["best_score"]
        assert s == e["score"] and abs(s - 16.0) < 0.05 and (s >= 16.0) == (e["edge"] == "score_above")
        sides.add(e["edge"])
    assert sides == {"score_above", "score_below"}
    case, = E.drop_edge()
    seen = set()
    for (r1, _, _, _), e, (_, why, info) in zip(E.records(case), case.expect, agree(oracle, case)):
        i = len(r1) - 20                                     # the planted overlap
        cnt, score, drop, diffs = info["diags"][i]
        assert drop == e["drop"] and abs(drop - 16.0) < 0.05 and (drop >= 16.0) == (e["edge"] == "drop_above")
        if drop < 16.0:
            assert info["best_i"] == i and score >= 16.0
        seen.add((e["edge"], e["first_mismatch_element"] // 32, (e["first_mismatch_element"] + 1) // 32))
    # a drop inside the first 32-element chunk, one that reaches 16 bits only at the first element of the second,
    # one entirely inside the second; each on both sides of 16 bits
    assert seen == {(s, a, b) for s in ("drop_above", "drop_below") for a, b in ((0, 0), (0, 1), (1, 1))}


def test_precedence(oracle):
    reasons = set()
    for case in E.precedence():
        (_, why, info), = agree(oracle, case)
        broken = E.failing_rules(info, case.params)
        assert len(broken) >= max(2, case.expect[0]["n_rules"]) and broken[0] == why, broken
        reasons.add(why)
    assert reasons == {"repeat", "staggered", "maxdiffs", "maxdiffpct", "nokmers", "minscore", "minovlen"}


def test_options(oracle):
    a33, a64, _ = E.ascii64_sequence()
    r33, r64 = agree(oracle, a33), agree(oracle, a64)
    assert a64.params["ascii"] == 64 and np.array_equal(a64.fq, a33.fq + 31)
    assert sum(w == "ok" for _, w, _ in r33) > 20
    for (m33, w33, _), (m64, w64, _) in zip(r33, r64):
        assert w33 == w64
        if m33 and w33 == "ok":
            assert m64[0] == m33[0] and np.array_equal(np.frombuffer(m64[1], np.uint8), np.frombuffer(m33[1], np.uint8) + 31)
    at, both = E.qmax_cases()
    (_, why, _), = agree(oracle, at)
    assert why == "ok" and at.fq.max() == 33 + at.params["qmax"] < 33 + 93
    with pytest.raises(ValueError):
        oracle_run(oracle, both)
    assert [w for _, w, _ in E.reference(both)] == ["ok", "badqual"]
    assert both.fq.max() == 33 + both.params["qmax"] + 1
    case, = E.qout_cases()
    for e, (merged, why, info) in zip(case.expect, agree(oracle, case)):
        q = np.frombuffer(merged[1], np.uint8) - 33
        sh = info["F"] - info["best_i"]
        ov = q[sh:sh + info["best_i"]]
        assert ov.max() == e["qmaxout"] and ov.min() == e["qminout"]
        # without the clamps the same overlap has posteriors above qmaxout and below qminout
        r1, q1, r2, q2 = E.records(case)[case.expect.index(e)]
        m0, _ = G.merge_pair(r1, q1, r2, q2, maxee=100.0)
        q0 = np.frombuffer(m0[1], np.uint8)[sh:sh + info["best_i"]] - 33
        assert q0.max() > e["qmaxout"] and q0.min() < e["qminout"]


def test_geometry(oracle):
    grid = E.length_grid(1)
    combos = {(e["F"], e["R"]) for e in grid.expect}
    assert combos == {(f, r) for f in E.LENS for r in E.LENS}
    assert {e["sh"] % 32 for e in grid.expect} == {0, 1, 31}
    lc = E.low_complexity()
    full_groups = 0
    for (r1, _, r2, _), (_, why, info) in zip(E.records(lc), agree(oracle, lc)):
        k = G.kmer_counts(r1, r2.translate(E._COMP)[::-1])
        full_groups += any((k[g:g + 32] >= 4).all() for g in range(1, len(k) - 31, 32))
    assert full_groups >= 4                         # poly-A of 64 bases and more
    L = E.largest_equal_len()
    assert E.staging_bytes(L, L) <= E.SMEM_LIMIT < E.staging_bytes(L + 1, L + 1)
    assert E.staging_bytes(L + 4, L + 4) > E.SMEM_LIMIT
    ok, over = E.limit_equal()
    assert ok.expect[0]["F"] == L and over.expect[0]["F"] == L + 4
    un = E.limit_unequal()
    F, R = un.expect[0]["F"], un.expect[0]["R"]
    assert E.staging_bytes(F, R) <= E.SMEM_LIMIT < E.staging_bytes(F + 1, R) and F > 100 * R


def test_reuse_after_longer_pairs(oracle):
    nw = 64                                         # the layout at any resident-warp count; the device test uses its own
    case = E.reuse_mix(nwarps=nw)
    fl, rl = np.diff(case.fo), np.diff(case.ro)
    L = E.largest_equal_len()
    assert fl[0] == rl[0] == L and len(fl) == 4 * nw
    for w in range(nw):
        for k in (0, 2):
            assert fl[k * nw + w] + rl[k * nw + w] > fl[(k + 1) * nw + w] + rl[(k + 1) * nw + w]
            if w % 2:                               # rc of R2 all A, then the stale-word probe
                assert case.expect[k * nw + w]["kind"] == "long_polyT"
                assert case.expect[(k + 1) * nw + w]["kind"] == "short_probe"
    ref = agree(oracle, case)
    probes = [w for (_, w, _), e in zip(ref, case.expect) if e["kind"] == "short_probe"]
    assert probes.count("nokmers") == len(probes)


def test_consensus_branches(oracle):
    case = E.consensus()
    seen = set()
    for _, why, info in agree(oracle, case):
        assert why == "ok"
        seen |= set(info["branch"])
    assert seen == set(E.CONSENSUS_BRANCHES)


def test_tables_have_no_half_way_quality():
    """Python rounds half to even, C half away from zero: no posterior quality of the tables may sit on a half"""
    for px in G.P:
        for py in G.P:
            for p in (px * py / 3.0 / (1.0 - px - py + 4.0 * px * py / 3.0),
                      px * (1.0 - py / 3.0) / (px + py - 4.0 * px * py / 3.0)):
                v = -10.0 * math.log10(p)
                assert v - math.floor(v) != 0.5


def test_tables_equal_the_oracle(oracle):
    match, mism, same, diff, q2p = oracle.merge_tables(oracle.merge_params(ascii=64, qmaxout=35, qminout=3))
    s, d = G.tables(64, 35, 3)
    assert np.array_equal(q2p, G.P) and np.array_equal(match, G.MATCH) and np.array_equal(mism, G.MISM)
    assert np.array_equal(same, s) and np.array_equal(diff, d)
