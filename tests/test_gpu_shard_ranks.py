"""The sharded sample (csrc/shard.cu driven by distributed.run_sharded) at 2 to 64 ranks on one GPU.

Every rank is a thread with its own LOCAL and OWNER context (tests/shard_cases.py) and runs the real run_sharded with
the GPU engine; the exchanges go through ThreadComm, which keeps a copy of what each rank sent.  Every case is held to
(a) derep_ref, a plain dereplication: global representative, strand, class count, Σ n_owned; (b) the recorded
exchanges: split sizes = the plan, every local unique once, buckets and arrivals in ascending global index, records and
bases = the reads, one owner per class, answers = the class's representative and strand; (c) the one-GPU path on the
concatenated sample: keep / lo / hi and the per-profile reported-hit counts of itsx_run, the re-expanded slices of
itsx_run_trim with gather=True, their counts with gather="device"."""
import os
import sys

import numpy as np
import pytest

from conftest import HMM_DIR, ROOT

sys.path.insert(0, os.path.join(ROOT, "tests"))

import shard_cases as S  # noqa: E402

pytestmark = pytest.mark.gpu

M_HMM = [os.path.join(HMM_DIR, "M.hmm")]


@pytest.fixture(scope="module", autouse=True)
def _pool(gpu_ctx):
    """Up to 129 contexts share the GPU here, and a context keeps the scratch of its largest search until it is
    destroyed: the contexts earlier modules leave behind (the session's, the pipeline's shared one) are re-created
    empty first."""
    import gc
    import torch
    from itsxpress_b200 import SeqSample
    gc.collect()                       # contexts nobody references any more are destroyed now, not at exit
    gpu_ctx.close()
    gpu_ctx.__init__(gpu_ctx.device)
    if SeqSample._CTX is not None:
        SeqSample.reset_sessions()
        SeqSample._CTX.close()
        SeqSample._CTX = None
        SeqSample._GENERATION += 1
    torch.cuda.empty_cache()
    free, total = torch.cuda.mem_get_info(0)
    print("device memory free before the sharded cases: %.1f of %.1f GB" % (free / 2 ** 30, total / 2 ** 30))
    yield S.POOL
    S.POOL.close()


def _quals(reads, seed=3):
    rng = np.random.default_rng(seed)
    return [rng.integers(35, 74, len(r), dtype=np.uint8).tobytes() for r in reads]


def _params(keep_rows=0, domz_upper=0, domE=None):
    from itsxpress_b200 import _lib
    prm = _lib.default_params()
    prm.keep_rows, prm.domz_upper = keep_rows, domz_upper
    if domE is not None:
        prm.domE = domE
    return prm


def check_case(G, reads, quals, paths, prefixes, params=None, gathers=(False, True, "device")):
    """(a), (b) and (c) for one sample on G ranks; returns the gather=False run (outs, world, blocks)."""
    seq, off, qual = S.pack(reads, quals)
    ctxs = S.POOL.ranks(G)
    single = S.POOL.single
    S.load_profiles(ctxs[1] + [single], paths, prefixes)
    ref = S.derep_ref(reads)
    want, st = single.run(seq, off, params)
    want = {k: v.copy() for k, v in want.items()}
    nrep = single.nreported().astype(np.int64)
    assert st.n_unique == ref[2] and np.array_equal(want["rep"], ref[0])
    wt, st2 = single.run_trim(seq, qual, off, params)
    wt = {k: v.copy() for k, v in wt.items()}
    first = None
    for gather in gathers:
        outs, world, blocks = S.run_ranks(G, ctxs, seq, off, qual=qual, params=params, gather=gather,
                                          want_rep=gather is False)
        for o in outs:
            assert o["n_unique_global"] == ref[2] and np.array_equal(o["nreported"], nrep)
        assert sum(o["n_owned"] for o in outs) == ref[2]
        S.check_exchange(world, blocks, reads, ref)
        ki, oo = wt["kept_index"], wt["out_off"]
        for o, (lo, hi) in zip(outs, blocks):
            a, b = np.searchsorted(ki, lo), np.searchsorted(ki, hi)
            if gather is False:
                for k in ("keep", "lo", "hi"):
                    assert np.array_equal(o[k], want[k][lo:hi]), (k, lo, hi)
            elif gather is True:
                assert np.array_equal(o["kept_index"] + lo, ki[a:b]), (lo, hi)
                assert np.array_equal(o["out_off"], oo[a:b + 1] - oo[a]), (lo, hi)
                assert np.array_equal(o["out_seq"], wt["out_seq"][oo[a]:oo[b]]), (lo, hi)
                assert np.array_equal(o["out_qual"], wt["out_qual"][oo[a]:oo[b]]), (lo, hi)
            else:
                assert o["n_kept"] == b - a and o["out_bytes"] == oo[b] - oo[a], (lo, hi)
        if gather is False:
            S.check_derep(outs, blocks, reads, ref)
            first = (outs, world, blocks)
    assert st2.n_kept == int(want["keep"].sum())
    return first


@pytest.fixture(scope="module")
def fixture_case(fixture_reads):
    b, seq, off, qual = fixture_reads
    return S.fixture_case(seq, off, qual)


# A search context sizes its scratch for a whole GPU (Forward/Backward and envelope slabs for every resident warp: about
# 30-40 GB per context at 250-441 bp) and only shrinks it when the device is full, so the long-read cases stop at three
# owners (plus the one-GPU context); short-read cases go to 64 ranks.
@pytest.mark.parametrize("G", [1, 2, 3])
def test_fixture(fixture_case, G):
    reads, quals = fixture_case
    outs, world, blocks = check_case(G, reads, quals, M_HMM, ["3_", "4_"])
    assert sum(int(o["keep"].sum()) for o in outs) > 50
    assert sum(int(o["strand"].sum()) for o in outs) >= 7


_SYNTH = {}


def _synthetic(name, scale):
    if (name, scale) not in _SYNTH:
        import synth
        seq, off, which, cfg = synth.make_config(name, scale=scale)
        reads, quals = S.spread_revcomp_copies(seq, off, synth.make_quals(9, off))
        _SYNTH.clear()
        _SYNTH[(name, scale)] = reads, quals, [os.path.join(synth.HMM_DIR, f) for f in cfg["search_files"]], \
            [cfg["left_prefix"], cfg["right_prefix"]]
    return _SYNTH[(name, scale)]


@pytest.mark.parametrize("name,scale", [("c2_small", 1.0), ("c4s", 0.05)])
@pytest.mark.parametrize("G", [2, 3])
def test_synthetic(name, scale, G):
    reads, quals, paths, pre = _synthetic(name, scale)
    n = len(reads)
    for keep_rows in (1, 2):
        outs, _, _ = check_case(G, reads, quals, paths, pre, params=_params(keep_rows, n))
        assert sum(int(o["keep"].sum()) for o in outs) > 0.5 * n
        assert sum(int(o["strand"].sum()) for o in outs) >= 50


@pytest.mark.parametrize("kind,G", [("main", 2), ("main", 3), ("main", 7), ("main", 64), ("twenty", 64), ("five", 8)])
def test_degenerate(kind, G):
    reads = S.degenerate_reads(kind)
    outs, world, blocks = check_case(G, reads, _quals(reads), M_HMM, ["3_", "4_"])
    if kind == "main":
        assert sum(int(o["strand"].sum()) for o in outs) >= 10
    if G > len(reads):
        assert sum(1 for lo, hi in blocks if hi == lo) == G - len(reads)


@pytest.mark.parametrize("G", [1, 2])
def test_only_empty_reads(G):
    """A read set whose reads are all empty (no bases: nothing to pack) on one GPU and sharded."""
    reads = S.degenerate_reads("empty")
    seq, off = S.pack(reads)
    rep, strand, nu = S.POOL.single.derep(seq, off)
    assert nu == 1 and np.array_equal(rep, np.zeros(len(reads))) and not strand.any()
    rep, strand, nu = S.POOL.single.derep(seq[:0], off[:3])          # two empty reads
    assert nu == 1 and list(rep) == [0, 0]
    outs, _, _ = check_case(G, reads, reads, M_HMM, ["3_", "4_"])
    assert sum(int(o["keep"].sum()) for o in outs) == 0


@pytest.mark.parametrize("G", [3, 5])
def test_key_collisions(G):
    """64-bit keys cut to 6 bits on every rank: owners resolve classes through collide_kernel, the first arrival (the
    smallest global index) must still be the representative."""
    reads = S.rand_reads(np.random.default_rng(7), 1500, 30, 60)
    local, owner = S.POOL.ranks(G)
    try:
        for c in local + owner:
            c.set_key_bits(6)
        check_case(G, reads, _quals(reads), M_HMM, ["3_", "4_"], gathers=(False,))
        assert sum(c.derep_stats().n_collided for c in owner) > 0
        assert sum(c.derep_stats().n_collided for c in local) > 0
    finally:
        for c in local + owner:
            c.set_key_bits(64)


def test_world_out_of_range_leaves_the_context_usable(fixture_case):
    from itsxpress_b200 import _lib
    from itsxpress_b200.distributed import GpuEngine
    reads, quals = fixture_case
    seq, off = S.pack(reads)
    local, owner = S.POOL.ranks(2)
    eng = GpuEngine(local[0], owner[0])
    eng.local_derep(seq, off)
    for G in (65, 0):
        with pytest.raises(_lib.ItsxError) as e:
            eng.plan(G)
        assert e.value.code == -3
    check_case(2, reads, quals, M_HMM, ["3_", "4_"], gathers=(False,))


# ---- domZ: the compact row mode of a sharded owner -------------------------------------------------------------------
def _winners(rows, side, printed):
    """ItsPosition's pick per (sequence, side) among the printed rows (table order, strict > on the printed 0.1-bit
    score: the first row wins) -> {(seq, side): (score10, ienv, jenv)}."""
    r = rows[printed]
    sd = side[r["prof"]]
    ok = sd >= 0
    r, sd, idx = r[ok], sd[ok], np.flatnonzero(ok)
    s10 = np.rint(r["bitscore"].astype(np.float64) * 10.0).astype(np.int64)
    order = np.lexsort((idx, -s10, sd, r["seq"]))
    key = r["seq"][order].astype(np.int64) * 2 + sd[order]
    firsts = order[np.concatenate([[True], key[1:] != key[:-1]])] if len(order) else order
    return {(int(r["seq"][i]), int(sd[i])): (int(s10[i]), int(r["ienv"][i]), int(r["jenv"][i])) for i in firsts}


def _band_winners(rows, side, domZ, n_bound, domE):
    """(seq, side) pairs whose pick changes when rows with P x n_bound <= domE count as printed although
    P x domZ > domE (what an owner that bounds domZ by its own class count n_bound does in the compact row mode)."""
    P = np.exp(rows["lnP"])
    printed = P * domZ[rows["prof"]] <= domE
    wrong = printed | (P * n_bound <= domE)
    a, b = _winners(rows, side, printed), _winners(rows, side, wrong)
    return sum(1 for k, v in b.items() if a.get(k) != v)


def _all_rows(single, seq, off):
    """The one-GPU keep_rows = 1 table with every row of every reported hit (domE never excludes one), and domZ."""
    single.run(seq, off, _params(keep_rows=1, domE=1e300))
    return single.hits(), single.nreported().astype(np.float64)


def test_domz_trap_with_explicit_params():
    """keep_rows = 2, domz_upper = 0, four owners of c2_small: domE is chosen so that at least 20 (seq, side) picks
    change if an owner bounds domZ by its own class count.  The sharded run must still equal the one-GPU run."""
    reads, quals, paths, pre = _synthetic("c2_small", 1.0)
    seq, off = S.pack(reads)
    G = 4
    S.POOL.close()                     # four owners and the one-GPU context: nothing else may hold search scratch
    ctxs = S.POOL.ranks(G)
    single = S.POOL.single
    S.load_profiles(ctxs[1] + [single], paths, pre)
    side = single.set_sides_by_prefix(*pre)
    rows, domZ = _all_rows(single, seq, off)
    outs, world, blocks = S.run_ranks(G, ctxs, seq, off, params=_params(keep_rows=1))
    owner = S.check_exchange(world, blocks, reads)
    n_owned = np.array([o["n_owned"] for o in outs])
    # every row's own owner: the class of search-set sequence u is the one whose first read is first[u]
    first = np.flatnonzero(S.derep_ref(reads)[0] == np.arange(len(reads)))
    n_bound = n_owned[np.array([owner[int(first[u])] for u in rows["seq"]])]
    P = np.exp(rows["lnP"])
    cand = np.unique(P * n_bound)
    cand = cand[(cand > 0) & np.isfinite(cand)]
    best = max((_band_winners(rows, side, domZ, n_bound, e), e) for e in np.quantile(cand, np.linspace(0.02, 0.6, 30)))
    nwin, domE = best
    print("domz trap: domE=%.4g, %d picks change, n_owned=%s, domZ max=%d" % (domE, nwin, list(n_owned), domZ.max()))
    assert nwin >= 20
    band = (P * n_bound <= domE) & (P * domZ[rows["prof"]] > domE)
    assert band.sum() >= 20
    check_case(G, reads, quals, paths, pre, params=_params(keep_rows=2, domE=domE), gathers=(False, "device"))


def test_domz_trap_default_params_above_200k_classes_per_owner():
    """params=None on two owners of more than 200 000 classes each (the compact row mode by default): the sharded run
    equals the one-GPU run.  How many picks the default domE puts in the band is printed."""
    import synth
    from itsxpress_b200.distributed import GpuEngine
    seq, off, which, cfg = synth.make_config("c4s", scale=1.2)
    paths = [os.path.join(synth.HMM_DIR, f) for f in cfg["search_files"]]
    pre = [cfg["left_prefix"], cfg["right_prefix"]]
    G = 2
    S.POOL.close()
    local, owner = S.POOL.ranks(G)
    single = S.POOL.single
    S.load_profiles(owner + [single], paths, pre)
    want, st = single.run(seq, off)
    want = {k: v.copy() for k, v in want.items()}
    import torch
    outs, world, blocks = S.run_world(G, seq, off, lambda r: GpuEngine(local[r], owner[r]),
                                      device=torch.device("cuda", 0))
    n_owned = [o["n_owned"] for o in outs]
    assert min(n_owned) > 200_000 and sum(n_owned) == st.n_unique
    for o, (lo, hi) in zip(outs, blocks):
        for k in ("rep", "keep", "lo", "hi"):
            assert np.array_equal(o[k], want[k][lo:hi]), (k, lo, hi)
    side = single.set_sides_by_prefix(*pre)
    rows, domZ = _all_rows(single, seq, off)
    rep = want["rep"]
    first = np.flatnonzero(rep == np.arange(len(rep)))
    owner_of = {}
    for src, (lo, hi) in enumerate(blocks):
        g, _ = S._records(world.sent["records"][src][0])
        dst = np.repeat(np.arange(G), world.sent["records"][src][1])
        owner_of.update(zip(g.tolist(), dst.tolist()))
    n_bound = np.array(n_owned)[np.array([owner_of[int(first[u])] for u in rows["seq"]])]
    print("domz trap, default params: %d picks in the band, n_owned=%s" %
          (_band_winners(rows, side, domZ, n_bound, 10.0), n_owned))
