"""itsx_cluster with per_sample = 1 on the B200: several samples resident (itsx_reads_set_samples) are clustered each on
its own in one call.  Against tests/cluster_ref.c run on every sample alone: centroid row, strand, ed, unique of row and
the read -> row map, on planted samples (shared templates at other abundances, a cross-sample neighbour that a leaked
edge would capture, an empty and a one-class sample), with the default and an interleaved order; domZ and positions
per sample equal clustering and searching each sample alone; the flag without sample ids changes nothing; and the
QIIME 2 actions at cluster_id = 0.995 write the same bytes batched as in the per-sample loop."""
import os

import numpy as np
import pytest

import cluster_cases as K
import cluster_samples_cases as S
from conftest import HMM_DIR
from itsxpress_b200 import SeqSample
from itsxpress_b200 import _lib

pytestmark = pytest.mark.gpu


def resident(ctx, seq, off, sample, n_samples):
    ctx.reads_upload(seq, off)
    ctx.set_samples(sample, n_samples)
    nu = ctx.derep_resident(build_search_set=False)
    first, _ = ctx.derep_clusters(nu)
    _, _, class_uid = ctx.derep_map(len(off) - 1)
    return nu, first, class_uid


@pytest.mark.parametrize("given_order", [False, True])
@pytest.mark.parametrize("X", [0.9, 0.97, 0.99, 0.995])
def test_per_sample_equals_reference_on_each_sample(gpu_ctx, X, given_order):
    D = int(_lib.cluster_dtable(X, 250)[250])
    samples = S.planted_samples(11, D)
    seq, off, sample = S.pack_samples(samples)
    nu, first, class_uid = resident(gpu_ctx, seq, off, sample, len(samples))
    order = S.interleaved_order(np.random.default_rng(12), first, sample) if given_order else None
    nc = gpu_ctx.cluster(X, order, per_sample=True)
    got = gpu_ctx.cluster_fetch(nu, nc)
    want = S.per_sample_reference(seq, off, first, class_uid, sample, X, order)
    assert nc == want[0]
    for g, w, name in zip(got, want[1:], ("centroid row", "strand", "ed", "unique of row")):
        assert np.array_equal(g, w), name
    _, _, uid = gpu_ctx.derep_map(len(sample))
    assert np.array_equal(uid, got[0][class_uid])
    assert np.array_equal(gpu_ctx.derep_clusters(nu)[0], first)
    # the cross-sample neighbour (sample 4, within D of sample 0's most abundant class) stays a centroid of its own
    x = len(sample) - len(samples[4]) + 3
    assert got[3][got[0][class_uid[x]]] == class_uid[x]
    st = gpu_ctx.cluster_stats()
    assert 0 < nc < nu and st.n_accepted > 0


def test_key_collisions_between_samples_are_dropped(gpu_ctx):
    """With 6-bit segment keys every lookup also hits classes of other samples (the sample seed no longer separates
    them): only the sample check of the lookups keeps candidates inside a sample, and the result is still each sample's
    own -- the cross-sample neighbour, whose segments now hit the class it is close to, stays a centroid."""
    X = 0.99
    D = int(_lib.cluster_dtable(X, 250)[250])
    samples = S.planted_samples(15, D)
    seq, off, sample = S.pack_samples(samples)
    nu, first, class_uid = resident(gpu_ctx, seq, off, sample, len(samples))
    nc = gpu_ctx.cluster(X, per_sample=True)
    full = gpu_ctx.cluster_stats().n_candidates
    gpu_ctx.cluster_set_key_bits(6)
    try:
        nc = gpu_ctx.cluster(X, per_sample=True)
        got = gpu_ctx.cluster_fetch(nu, nc)
        st = gpu_ctx.cluster_stats()
    finally:
        gpu_ctx.cluster_set_key_bits(64)
    assert st.n_candidates > 10 * full                     # the short keys do collide
    want = S.per_sample_reference(seq, off, first, class_uid, sample, X)
    assert nc == want[0]
    for g, w, name in zip(got, want[1:], ("centroid row", "strand", "ed", "unique of row")):
        assert np.array_equal(g, w), name
    x = len(sample) - len(samples[4]) + 3
    assert got[3][got[0][class_uid[x]]] == class_uid[x]


def test_per_sample_domz_and_positions_equal_each_sample_alone(gpu_ctx):
    from itsxpress_b200 import fastq as fq
    b = fq.read_fastq(K.MERGED)
    rs, ro = b.seq_concat()
    reads = [rs[ro[i]:ro[i + 1]].tobytes() for i in range(b.n)]
    rng = np.random.default_rng(13)
    samples = [reads, [reads[i] for i in rng.choice(b.n, 150)], [], [reads[i] for i in rng.choice(b.n, 40)]]
    gpu_ctx.load_profiles([os.path.join(HMM_DIR, "M.hmm")], ["3_", "4_"])
    gpu_ctx.set_sides_by_prefix("3_", "4_")
    X, names = 0.99, ("start", "stop", "tlen", "left_score10", "right_score10")
    alone = []
    for s in samples:
        if not s:
            alone.append(None)
            continue
        seq, off = K.pack(s)
        gpu_ctx.derep(seq, off)
        nc = gpu_ctx.cluster(X)
        gpu_ctx.search()
        alone.append((gpu_ctx.nreported().copy(), gpu_ctx.positions(nc)))
    seq, off, sample = S.pack_samples(samples)
    nu, first, _ = resident(gpu_ctx, seq, off, sample, len(samples))
    nc = gpu_ctx.cluster(X, per_sample=True)
    uor = gpu_ctx.cluster_fetch(nu, nc)[3]
    gpu_ctx.search()
    nrep = gpu_ctx.nreported(len(samples))
    pos = gpu_ctx.positions(nc)
    row_sample = sample[first[uor]]
    assert nc < nu
    for k, a in enumerate(alone):
        rows = np.flatnonzero(row_sample == k)
        if a is None:
            assert len(rows) == 0 and not nrep[k].any()
            continue
        assert np.array_equal(nrep[k], a[0]), k
        for n in names:
            assert np.array_equal(pos[n][rows], a[1][n]), (k, n)
    assert len({tuple(a[0]) for a in alone if a is not None}) > 1          # the samples' domZ differ


def test_per_sample_without_sample_ids_is_the_plain_call(gpu_ctx):
    seq, off = K.pack(K.planted(14, D=2))
    res = []
    for per_sample in (False, True):
        _, _, nu = gpu_ctx.derep(seq, off)
        nc = gpu_ctx.cluster(0.99, per_sample=per_sample)
        res.append(gpu_ctx.cluster_fetch(nu, nc))
    assert all(np.array_equal(a, b) for a, b in zip(*res))


@pytest.fixture()
def live(gpu_ctx, monkeypatch):
    monkeypatch.setattr(SeqSample, "get_context", lambda: gpu_ctx)
    SeqSample.reset_sessions()
    yield gpu_ctx
    SeqSample.reset_sessions()


def test_q2_batches_equal_the_per_sample_loop(live, tmp_path, monkeypatch):
    S.check_q2_batches_equal_loop(live, tmp_path, monkeypatch)
