"""The host driver of the search (csrc/search.cu, search_stage1 / search_stage2): state carried from one chunk of stage 1
to the next, and the side streams and timers a context shares between the search and the paired-end merge."""
import os

import numpy as np
import pytest

from conftest import HMM_DIR, TD

pytestmark = pytest.mark.gpu

POS_KEYS = ("start", "stop", "tlen", "left_score10", "left_from", "left_to", "right_score10", "right_from", "right_to")


def _fixture_uniques(gpu_ctx, seq, off):
    rep, _, nu = gpu_ctx.derep(seq, off)
    idx = np.flatnonzero(rep == np.arange(len(rep)))
    assert len(idx) == nu
    parts = [seq[off[i]:off[i + 1]] for i in idx]
    uoff = np.zeros(nu + 1, np.int64)
    uoff[1:] = np.cumsum([len(p) for p in parts])
    return np.concatenate(parts), uoff


def _stage1_counts(ctx):
    st = ctx.search_stats()
    return dict(msv=st.n_past_msv, bias=st.n_past_bias, fwd=st.n_past_fwd, hits=st.n_hits_reported,
                domains=st.n_domains), ctx.nreported().copy()


@pytest.mark.parametrize("keep_rows", [1, 2])
def test_stage1_over_several_chunks(gpu_ctx, fixture_reads, keep_rows):
    """The fixture's uniques searched alone (one chunk), then tiled so that stage 1 runs at least three chunks
    (a chunk holds min(2^22, max(1024, 2^27 / P)) sequences): every stage-1 count is the single run's times the number
    of copies, and with the single run's reported-hit counts (domZ) every copy gets the single run's positions.  This
    holds only if the domain rows, the compact-row counter, the envelope total and the per-profile bounds carry over
    correctly from one chunk to the next."""
    from itsxpress_b200 import _lib
    _, seq, off, _ = fixture_reads
    useq, uoff = _fixture_uniques(gpu_ctx, seq, off)
    nu = len(uoff) - 1
    files = sorted(f for f in os.listdir(HMM_DIR) if f.endswith(".hmm"))
    P = gpu_ctx.load_profiles([os.path.join(HMM_DIR, f) for f in files], ["1_", "4_"])
    gpu_ctx.set_sides_by_prefix("1_", "4_")
    prm = _lib.default_params()
    prm.keep_rows = keep_rows

    gpu_ctx.search_seqs_stage1(useq, uoff, prm)
    one, one_nrep = _stage1_counts(gpu_ctx)
    assert one["domains"] > 0 and one_nrep.sum() > 0
    gpu_ctx.search_stage2()
    one_pos = {k: v.copy() for k, v in gpu_ctx.positions(nu).items()}
    assert (one_pos["tlen"] > 0).any()

    copies = (2 * 2**27 // P) // nu + 1
    n_seq = copies * nu
    assert n_seq * P > 2 * 2**27
    tseq = np.tile(useq, copies)
    toff = np.concatenate([np.arange(copies, dtype=np.int64).repeat(nu) * uoff[-1] + np.tile(uoff[:-1], copies),
                           [copies * uoff[-1]]])
    gpu_ctx.search_seqs_stage1(tseq, toff, prm)
    many, many_nrep = _stage1_counts(gpu_ctx)
    assert gpu_ctx.search_stats().n_seq == n_seq
    assert many == {k: copies * v for k, v in one.items()}
    assert np.array_equal(many_nrep, copies * one_nrep)

    gpu_ctx.nreported_set(one_nrep)
    gpu_ctx.search_stage2()
    pos = gpu_ctx.positions(n_seq)
    for k in POS_KEYS:
        assert np.array_equal(pos[k].reshape(copies, nu), np.broadcast_to(one_pos[k], (copies, nu))), k


def test_search_then_merge_on_a_fresh_context(fixture_reads):
    """A search before the first merge on a context: merge still times its kernel, and the context stays usable."""
    from itsxpress_b200 import _lib
    from itsxpress_b200.fastq import read_fastq
    _, seq, off, _ = fixture_reads
    ctx = _lib.Context(0)
    try:
        ctx.load_profiles([os.path.join(HMM_DIR, "M.hmm")], ["3_", "4_"])
        useq, uoff = _fixture_uniques(ctx, seq, off)
        ctx.search_seqs(useq, uoff)
        assert ctx.search_stats().n_domains > 0

        b1 = read_fastq(os.path.join(TD, "4774-1-MSITS3_R1.fastq"))
        b2 = read_fastq(os.path.join(TD, "4774-1-MSITS3_R2.fastq"))
        fs, fo = b1.seq_concat()
        rs, ro = b2.seq_concat()
        ml, *_ = ctx.merge_pairs(fs, b1.qual_concat()[0], fo, rs, b2.qual_concat()[0], ro)
        assert (ml > 0).any()
        assert ctx.merge_stats().ms_kernel > 0

        _, _, nu = ctx.derep(seq, off)
        ctx.search()
        st = ctx.search_stats()
        assert st.n_seq == nu and st.n_domains > 0
    finally:
        ctx.close()
