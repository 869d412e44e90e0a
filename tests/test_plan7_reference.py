"""The HMM stage against an independent float64 statement of hmmsearch (tests/plan7_ref.py, written from SURVEY.md
Appendix A.1-A.5).  The oracle and the kernels follow each other operation for operation, so their own parity tests
cannot see a formulation mistake they share; these tests can.

CPU half: reference vs the oracle.  GPU half: reference vs itsx_search_seqs / itsx_run, long targets included.

Bars: MSV pass counts equal (integer arithmetic).  Bias / Forward pass counts, the reported pair set, envelope
coordinates and printed 0.1-bit scores may differ only where the float64 value lies within a stated distance of the
threshold it was compared with (a near-tie that fp32 rounding may decide either way); those pairs are counted,
listed in the failure message and must stay few.  envsc within 2e-3 nats (scaled with Ld above 1 000),
domcorrection within 2e-3 nats, bit scores within 0.01 bit, lnP within lambda x 0.01.

domcorrection is NOT clamped at 0, neither here nor in the oracle / kernels.  Whether HMMER's rescore_isolated_domain
applies ESL_MAX(0, ...) could not be settled without its source, and SURVEY A.5 states domcorrection as the plain sum
of n2sc over the envelope.  About 40 % of the fixture's domains have a negative sum, so the choice is visible in
domcorrection itself; its effect on a domain's bit score is at most log2(1 + 1/256) = 0.0056 bit.
"""
import math
import os

import numpy as np
import pytest

import plan7_ref as R
from conftest import HMM_DIR

BIG_DOME = 1e300
NEAR_P = 1e-3          # ln P distance from F1 / F3 below which a filter decision is a near-tie
NEAR_T = 0.01          # bits from T
NEAR_RT = 1e-5         # posterior distance from rt1 / rt2 / rt3
NEAR_PRINT = 0.005     # bits from a %.1f rounding edge


# ---------------------------------------------------------------------------------------------------------------
# workloads: (hmm files, prefixes, list of ASCII targets)
def _uniques(fixture_reads, oracle):
    b, seq, off, _ = fixture_reads
    rep, _, _ = oracle.derep(seq, off)
    return [seq[off[i]:off[i + 1]].tobytes() for i in np.flatnonzero(rep == np.arange(len(rep)))]


def _acgt(rng, n):
    return np.frombuffer(b"ACGT", np.uint8)[rng.integers(4, size=n)].tobytes()


def _iupac(rng, s, rate):
    a = bytearray(s)
    for q in np.flatnonzero(rng.random(len(a)) < rate):
        a[q] = int(rng.choice(list(b"NRYMKSWHBVDn")))
    return bytes(a)


def wl_fixture(fixture_reads, oracle):
    return ["M.hmm"], ["3_", "4_"], _uniques(fixture_reads, oracle)


def wl_taxa(fixture_reads, oracle):
    u = _uniques(fixture_reads, oracle)
    rng = np.random.default_rng(11)
    t = u[:24] + [s for s in u if b"N" in s]
    t += [_iupac(rng, u[0], 0.02), u[1].lower(), _iupac(rng, u[2], 0.1).lower()]
    files = sorted(f for f in os.listdir(HMM_DIR) if f.endswith(".hmm") and os.path.getsize(os.path.join(HMM_DIR, f)))
    return files, ["1_", "3_", "4_"], t


def wl_synth(n=120):
    import synth
    seq, off, which, cfg = synth.make_config("c2_small", scale=0.05)
    t = sorted({seq[off[i]:off[i + 1]].tobytes() for i in range(len(off) - 1)})[:n]
    return [cfg["hmm_file"]], [cfg["left_prefix"], cfg["right_prefix"]], t


def wl_lengths(fixture_reads, oracle):
    u = _uniques(fixture_reads, oracle)
    rng = np.random.default_rng(5)
    t = []
    for L in (0, 1, 10, 11, 12, 24, 25, 26, 44, 45, 46, 47, 90):
        t.append(_acgt(rng, L))
        t.append(u[3][80:80 + L])           # the ITS2 start of the fixture is at 84..128
        t.append(u[5][280:280 + L])         # ... its end at 282..326
    return ["M.hmm", "G.hmm"], ["1_", "3_", "4_"], t


def wl_long(lengths=(1000, 2500, 5000, 10000)):
    import synth
    seq, off, which, cfg = synth.make_config("c2_small", scale=0.05)
    rng = np.random.default_rng(17)
    amp = [seq[off[i]:off[i + 1]].tobytes() for i in range(6)]
    t = []
    for q, L in enumerate(lengths):
        core = amp[q % 6] if q % 2 else amp[q % 6] + _acgt(rng, 300) + amp[(q + 1) % 6]
        if q == 1:
            core = _iupac(rng, core, 0.05)
        a = int(rng.integers(0, L - len(core)))
        s = _acgt(rng, a) + core + _acgt(rng, L - len(core) - a)
        t.append(_iupac(rng, s, 0.05) if q == 1 else s)
    return [cfg["hmm_file"]], [cfg["left_prefix"], cfg["right_prefix"]], t


# ---------------------------------------------------------------------------------------------------------------
def _profiles(files, prefixes):
    out = []
    for f in files:
        out += R.parse_hmm(os.path.join(HMM_DIR, f), prefixes)
    return out


def _concat(targets):
    off = np.zeros(len(targets) + 1, np.int64)
    off[1:] = np.cumsum([len(t) for t in targets])
    return np.frombuffer(b"".join(targets), np.uint8).copy(), off


def run_reference(profs, targets, impl_rows=None):
    """Reference results per (profile, target).  impl_rows: the rows of the implementation under test, whose
    cluster envelopes stand in for the stochastic-traceback resolver (which is not restated) inside flagged
    regions; None rescoring a flagged region as one envelope (resolve_multidomain = 0)."""
    seqs = [R.digitize(t) for t in targets]
    md = None
    if impl_rows is not None:
        by = {}
        for r in impl_rows:
            if r["is_multidomain"]:
                by.setdefault((int(r["prof"]), int(r["seq"])), []).append((int(r["ienv"]), int(r["jenv"])))
    out = {}
    for pi, p in enumerate(profs):
        if impl_rows is not None:
            def md(r, i, j, pi=pi):
                envs = [e for e in by.get((pi, r), []) if i <= e[0] and e[1] <= j]
                return envs or None
        for r, d in enumerate(R.search_profile(p, seqs, md_envelopes=md)):
            out[(pi, r)] = d
    return out


def _edge(bits):
    x = bits * 10.0
    return abs(x - math.floor(x) - 0.5) < NEAR_PRINT * 10.0


def compare(profs, targets, ref, impl, label):
    """impl: dict(n_past_msv, n_past_bias, n_past_fwd, rows, positions or None, resolved).  Returns a report."""
    npairs = len(ref)
    n_msv = sum(d["pass_msv"] for d in ref.values())
    assert impl["n_past_msv"] == n_msv, (label, impl["n_past_msv"], n_msv)
    for stage, key in (("bias", "margin_bias"), ("fwd", "margin_fwd")):
        n = sum(d.get("pass_" + stage, False) for d in ref.values())
        near = sum(1 for d in ref.values() if d.get(key, math.inf) < NEAR_P)
        assert abs(impl["n_past_" + stage] - n) <= near, (label, stage, impl["n_past_" + stage], n, near)
    rows = impl["rows"]
    irows = {}
    for r in rows:
        irows.setdefault((int(r["prof"]), int(r["seq"])), []).append(r)
    ref_rep = {k for k, d in ref.items() if d.get("reported")}
    resolved = impl["resolved"]

    def md_pair(k):
        return resolved and any(m for (_, _, m) in ref[k].get("regions", []))

    def near_pair(k):
        d = ref[k]
        return (d.get("margin_T", math.inf) < NEAR_T or d.get("margin_fwd", math.inf) < NEAR_P
                or d.get("margin_bias", math.inf) < NEAR_P or d.get("margin_rt", math.inf) < NEAR_RT or md_pair(k))

    diff = ref_rep ^ set(irows)
    bad = [k for k in diff if not near_pair(k)]
    assert not bad, (label, "reported pair sets differ", [(profs[k[0]].name, k[1], ref[k].get("seq_score"))
                                                          for k in bad[:10]])
    excused = sorted(diff)
    worst = dict(envsc=0.0, dc=0.0, bits=0.0, seq=0.0, lnP=0.0)
    ref_rows = []
    for k in sorted(ref_rep & set(irows)):
        d, ir = ref[k], sorted(irows[k], key=lambda r: int(r["ienv"]))
        L = d["L"]
        rd = sorted(d["doms"], key=lambda x: x["ienv"])
        if [(x["ienv"], x["jenv"]) for x in rd] != [(int(r["ienv"]), int(r["jenv"])) for r in ir]:
            assert d["margin_rt"] < NEAR_RT or md_pair(k), (label, profs[k[0]].name, k[1], "envelopes",
                                                             [(x["ienv"], x["jenv"]) for x in rd],
                                                             [(int(r["ienv"]), int(r["jenv"])) for r in ir])
            excused.append(k)
            continue
        lam, tau = profs[k[0]].lam, profs[k[0]].tau
        for x, r in zip(rd, ir):
            assert bool(r["is_multidomain"]) == x["is_multidomain"], (label, k)
            Ld = x["jenv"] - x["ienv"] + 1
            e = abs(float(r["envsc"]) - x["envsc"])
            assert e <= 2e-3 * max(1.0, Ld / 1000.0), (label, profs[k[0]].name, k[1], "envsc", e, Ld)
            worst["envsc"] = max(worst["envsc"], e)
            if not (x["is_multidomain"] and resolved):
                e = abs(float(r["domcorrection"]) - x["domcorrection"])
                assert e <= 2e-3, (label, profs[k[0]].name, k[1], "domcorrection", e)
                worst["dc"] = max(worst["dc"], e)
                e = abs(float(r["bitscore"]) - x["bits"])
                assert e <= 0.01, (label, profs[k[0]].name, k[1], "bits", e)
                worst["bits"] = max(worst["bits"], e)
                e = abs(float(r["lnP"]) - x["lnP"])
                assert e <= lam * 0.01, (label, k, "lnP", e)
                worst["lnP"] = max(worst["lnP"], e)
                if not _edge(x["bits"]):
                    s10 = impl["score10"]
                    assert s10(float(r["bitscore"])) == s10(x["bits"]), (label, k, "printed score", x["bits"])
            own = R.exp_logsurv(float(r["bitscore"]), tau, lam)
            assert abs(float(r["lnP"]) - own) <= 1e-6 * max(1.0, abs(own)) + 1e-5 * lam, (label, k, "lnP vs bits")
        if "seq_score" in ir[0].dtype.names and not md_pair(k):
            e = abs(float(ir[0]["seq_score"]) - d["seq_score"])
            assert e <= 0.01, (label, profs[k[0]].name, k[1], "seq_score", e)
            worst["seq"] = max(worst["seq"], e)
        for x in rd:
            ref_rows.append((k, x, d))
    assert len(excused) <= max(2, 0.005 * npairs), (label, "too many near-tie pairs", excused)
    return dict(excused=len(excused), worst=worst, ref_rows=ref_rows)


def ref_as_rows(oracle, ref_rows):
    rows = np.zeros(len(ref_rows), dtype=oracle.DOM_DTYPE)
    for q, ((pi, r), x, d) in enumerate(ref_rows):
        rows[q]["seq"], rows[q]["prof"] = r, pi
        rows[q]["ienv"], rows[q]["jenv"] = x["ienv"], x["jenv"]
        rows[q]["envsc"], rows[q]["domcorrection"], rows[q]["bitscore"] = x["envsc"], x["domcorrection"], x["bits"]
        rows[q]["lnP"], rows[q]["is_multidomain"], rows[q]["is_reported"] = x["lnP"], x["is_multidomain"], 1
    return rows


def check_positions(oracle, profs, targets, cmp, side, pos, label):
    """ItsPosition on the reference's rows == the implementation's positions, except targets holding a row whose
    float64 score is within NEAR_PRINT of a %.1f rounding edge."""
    rows = ref_as_rows(oracle, cmp["ref_rows"])
    seqlen = np.array([len(t) for t in targets], np.int32)
    rpos = oracle.itspos(rows, side, seqlen)
    skip = {k[1] for k, x, d in cmp["ref_rows"] if _edge(x["bits"])}
    keep = np.array([i not in skip for i in range(len(targets))])
    for f in ("start", "stop", "tlen", "left_score10", "right_score10"):
        assert np.array_equal(rpos[f][keep], pos[f][keep]), (label, f, np.flatnonzero(rpos[f] != pos[f])[:10])


# ---------------------------------------------------------------------------------------------------------------
# CPU half: reference vs oracle
def _oracle_impl(oracle, files, prefixes, targets, resolve):
    db = oracle.ProfileDB([os.path.join(HMM_DIR, f) for f in files], prefixes)
    seq, off = _concat(targets)
    prm = oracle.default_params(0, resolve)
    prm.domE = BIG_DOME
    rows, nrep, st = db.search(oracle.digitize(seq.tobytes()), off, prm)
    # seq_score per reported pair: pair_run on the same target
    ss = {}
    for k in {(int(r["prof"]), int(r["seq"])) for r in rows}:
        pr, _ = db.pair_run(k[0], oracle.digitize(targets[k[1]]), prm)
        ss[k] = pr.seq_score
    dt = np.dtype(rows.dtype.descr + [("seq_score", "<f4")])
    rows2 = np.zeros(len(rows), dt)
    for n in rows.dtype.names:
        rows2[n] = rows[n]
    rows2["seq_score"] = [ss[(int(r["prof"]), int(r["seq"]))] for r in rows]
    return db, dict(n_past_msv=st.n_past_msv, n_past_bias=st.n_past_bias, n_past_fwd=st.n_past_fwd, rows=rows2,
                    resolved=bool(resolve), score10=oracle.score10)


CPU_CASES = {
    "fixture_its2": (wl_fixture, 1),
    "taxa_iupac": (wl_taxa, 1),
    "synth_resolve0": (lambda f, o: wl_synth(), 0),
    "synth_resolve1": (lambda f, o: wl_synth(), 1),
    "lengths": (wl_lengths, 1),
    "long": (lambda f, o: wl_long((1000, 2500, 5000)), 1),
}


@pytest.mark.parametrize("case", sorted(CPU_CASES))
def test_reference_vs_oracle(case, oracle, fixture_reads):
    make, resolve = CPU_CASES[case]
    files, prefixes, targets = make(fixture_reads, oracle)
    profs = _profiles(files, prefixes)
    db, impl = _oracle_impl(oracle, files, prefixes, targets, resolve)
    assert db.names == [p.name for p in profs]
    ref = run_reference(profs, targets, impl["rows"] if resolve else None)
    rep = compare(profs, targets, ref, impl, case)
    assert sum(d.get("reported", False) for d in ref.values()) > (0 if case == "lengths" else 5)
    print(case, rep["excused"], rep["worst"])


def test_null2_direct_equals_shortcut(fixture_reads, oracle):
    """HMMER's null2 (posteriors of M, I, N, C, J averaged over the envelope) == the shortcut
    1 + sum_k pbar(M_k)(odds_k[x] - 1) that the oracle and kernels evaluate (DESIGN.md section 2), to 1e-10."""
    files, prefixes, targets = wl_fixture(fixture_reads, oracle)
    seqs = [R.digitize(t) for t in targets]
    res = []
    for p in _profiles(files, ["3_"])[::10]:
        items = [(s, 1, len(s)) for s in seqs[:2]] + [(seqs[0], 100, 110), (seqs[1], 5, 5)]
        for d, s in zip(R.search_profile(p, seqs), seqs):
            items += [(s, x["ienv"], x["jenv"]) for x in d.get("doms", [])]
        res += R.rescore_envelopes(p, items)
    assert len(res) > 50
    for e in res:
        assert np.max(np.abs(e["null2"] / e["null2_short"] - 1.0)) < 1e-10
        assert e["rowdev"] < 1e-10                       # every residue is emitted by exactly one state
        assert abs(e["bwd_minus_fwd"]) < 1e-9


def test_reference_known_answers():
    """The reference itself: Forward == Backward in float64, the L = 0 target is never a hit, and a concatemer of
    each copy of the consensus is the envelope of a reported domain."""
    p = R.parse_hmm(os.path.join(HMM_DIR, "M.hmm"), ["3_"])[0]
    rng = np.random.default_rng(3)
    seqs = [rng.integers(0, 15, n).astype(np.uint8) for n in (1, 2, 45, 300)]
    fw = R.forward_batch(p, seqs, [len(s) for s in seqs], True)
    bw = R.backward_batch(p, fw, True)
    assert np.max(np.abs(fw["sc"] - bw["sc"])) < 1e-10
    assert R.search_profile(p, [np.zeros(0, np.uint8)])[0]["pass_fwd"] is False
    cons = np.argmax(p.mat[1:], axis=1).astype(np.uint8)
    s = np.concatenate([rng.integers(0, 4, 40).astype(np.uint8), cons, rng.integers(0, 4, 80).astype(np.uint8), cons,
                        rng.integers(0, 4, 40).astype(np.uint8)])
    d = R.search_profile(p, [s])[0]
    envs = [(x["ienv"], x["jenv"]) for x in d["doms"]]
    assert d["reported"] and (41, 85) in envs and (166, 210) in envs, envs


# ---------------------------------------------------------------------------------------------------------------
# GPU half: reference vs itsx_search_seqs / itsx_run
def _gpu_impl(gpu_ctx, files, prefixes, targets, resolve, domE=BIG_DOME, sides=None):
    from itsxpress_b200 import _lib
    gpu_ctx.load_profiles([os.path.join(HMM_DIR, f) for f in files], prefixes)
    side = gpu_ctx.set_sides_by_prefix(*(sides or prefixes[-2:]))
    seq, off = _concat(targets)
    prm = _lib.default_params()
    prm.resolve_multidomain = resolve
    prm.keep_rows = 1
    prm.domE = domE
    gpu_ctx.search_seqs(seq, off, prm)
    st = gpu_ctx.search_stats()
    from oracle import oracle as O
    return side, dict(n_past_msv=st.n_past_msv, n_past_bias=st.n_past_bias, n_past_fwd=st.n_past_fwd,
                      rows=gpu_ctx.hits(), resolved=bool(resolve), score10=O.score10,
                      positions=gpu_ctx.positions(len(targets)))


GPU_CASES = dict(CPU_CASES, long=(lambda f, o: wl_long(), 1))


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(GPU_CASES))
def test_reference_vs_gpu(case, gpu_ctx, oracle, fixture_reads):
    make, resolve = GPU_CASES[case]
    files, prefixes, targets = make(fixture_reads, oracle)
    profs = _profiles(files, prefixes)
    sides = ("3_", "4_") if "3_" in prefixes else (prefixes[0], prefixes[-1])
    side, impl = _gpu_impl(gpu_ctx, files, prefixes, targets, resolve, sides=sides)
    assert gpu_ctx.names == [p.name for p in profs]
    ref = run_reference(profs, targets, impl["rows"] if resolve else None)
    rep = compare(profs, targets, ref, impl, case)
    if not resolve or case in ("fixture_its2", "taxa_iupac", "lengths", "long"):
        check_positions(oracle, profs, targets, rep, side, impl["positions"], case)
    print(case, "excused", rep["excused"], "longest", max(len(t) for t in targets), rep["worst"])


@pytest.mark.gpu
def test_reference_vs_gpu_default_dome(gpu_ctx, oracle, fixture_reads):
    """The default domE: every printed row is one of the reference's domains, with its score."""
    files, prefixes, targets = wl_fixture(fixture_reads, oracle)
    profs = _profiles(files, prefixes)
    side, impl = _gpu_impl(gpu_ctx, files, prefixes, targets, 1, domE=oracle.default_params().domE,
                           sides=("3_", "4_"))
    ref = run_reference(profs, targets, impl["rows"])
    by = {}
    for k, d in ref.items():
        for x in d.get("doms", []):
            by[(k[0], k[1], x["ienv"], x["jenv"])] = x
    rows = impl["rows"]
    assert len(rows) > 1000
    for r in rows:
        x = by[(int(r["prof"]), int(r["seq"]), int(r["ienv"]), int(r["jenv"]))]
        assert abs(float(r["bitscore"]) - x["bits"]) <= 0.01


@pytest.mark.gpu
def test_long_read_among_short_whole_path(gpu_ctx, oracle):
    """One 10 kb read among ~1 000 reads of 250 bp through the whole path (itsx_run): the scratch of the Forward /
    Backward and envelope stages is sized by the longest read, so this read must neither run the GPU out of memory
    nor change the other reads; its ItsPosition equals the reference's."""
    import synth
    seq, off, which, cfg = synth.make_config("c2_small", scale=0.05)
    n = 1000
    reads = [seq[off[i]:off[i + 1]].tobytes() for i in range(n)]
    rng = np.random.default_rng(23)
    amp = reads[0]
    long = _acgt(rng, 4000) + amp + _acgt(rng, 10000 - 4000 - len(amp))
    reads.insert(500, long)
    s, o = _concat(reads)
    files, prefixes = [cfg["hmm_file"]], [cfg["left_prefix"], cfg["right_prefix"]]
    gpu_ctx.load_profiles([os.path.join(HMM_DIR, f) for f in files], prefixes)
    side = gpu_ctx.set_sides_by_prefix(*prefixes)
    out, st = gpu_ctx.run(s, o)
    assert st.n_reads == n + 1
    # the short reads: the same bounds as without the long read
    s2, o2 = _concat(reads[:500] + reads[501:])
    out2, _ = gpu_ctx.run(s2, o2)
    for f in ("keep", "lo", "hi"):
        a = np.delete(out[f], 500)
        assert np.array_equal(a, out2[f]), f
    # the long read against the reference
    profs = _profiles(files, prefixes)
    ref = run_reference(profs, [long])
    rows = []
    for (pi, r), d in ref.items():
        if d.get("reported"):
            rows += [((pi, r), x, d) for x in d["doms"]]
    rpos = oracle.itspos(ref_as_rows(oracle, rows), side, np.array([len(long)], np.int32))
    assert rpos["start"][0] >= 0 and rpos["stop"][0] > rpos["start"][0]
    keep, lo, hi = oracle.trim_bounds(np.array([0, len(long)], np.int64), np.zeros(1, np.int32), rpos["start"],
                                      rpos["stop"], rpos["tlen"])
    assert (out["keep"][500], out["lo"][500], out["hi"][500]) == (keep[0], lo[0], hi[0])


@pytest.mark.gpu
def test_concatemer_beyond_maxdom_fails_cleanly(gpu_ctx, oracle):
    """A hit with more than ITSX_MAXDOM (8) envelopes: the search stops with ITSX_ELIMIT and says why (pinned
    behaviour; a concatemer read fails the whole sample)."""
    from itsxpress_b200 import _lib
    p = R.parse_hmm(os.path.join(HMM_DIR, "M.hmm"), ["3_"])[0]
    rng = np.random.default_rng(9)
    cons = "".join("ACGT"[i] for i in np.argmax(p.mat[1:], axis=1)).encode()
    read = b"".join(_acgt(rng, 60) + cons for _ in range(10)) + _acgt(rng, 60)
    d = R.search_profile(p, [R.digitize(read)])[0]
    assert len(d["doms"]) > 8
    gpu_ctx.load_profiles([os.path.join(HMM_DIR, "M.hmm")], [p.name])
    gpu_ctx.set_sides_by_prefix("3_", "4_")
    s, o = _concat([read])
    with pytest.raises(_lib.ItsxError, match="ITSX_MAXDOM"):
        gpu_ctx.search_seqs(s, o, _lib.default_params())
