"""itsx_cluster on the B200 against the brute-force CPU reference (tests/cluster_ref.c): for every unique, the centroid
row, strand and ed are equal, on planted workloads (variants at D and D+1 edits, edits in the first and last segment,
reverse complements, N / IUPAC / lower case, length differences at the D(L) boundary, ties, chains), at several identities,
with the default and a given order; long reads at 0.99 and ITSX_ELIMIT above the band cap; the remap of the search set and
the read -> row map; and the command line end to end."""
import numpy as np
import pytest

import cluster_cases as K
import cluster_ref as R
from itsxpress_b200 import SeqSample
from itsxpress_b200 import _lib

pytestmark = pytest.mark.gpu


def gpu_vs_ref(ctx, reads, X, order=None):
    seq, off = K.pack(reads)
    rep, _, nu = ctx.derep(seq, off)
    first, _ = ctx.derep_clusters(nu)
    _, _, class_uid = ctx.derep_map(len(reads))
    nc = ctx.cluster(X, order)
    got = ctx.cluster_fetch(nu, nc)
    want = R.cluster(seq, off, first, R.default_order(rep) if order is None else order, X)
    assert nc == want[0]
    for g, w, name in zip(got, want[1:], ("centroid row", "strand", "ed", "unique of row")):
        assert np.array_equal(g, w), name
    # the read -> row map is the centroid row of the read's class; the exact classes stay what the derep returned
    _, _, uid = ctx.derep_map(len(reads))
    assert np.array_equal(uid, got[0][class_uid])
    assert np.array_equal(ctx.derep_clusters(nu)[0], first)
    return nu, nc, ctx.cluster_stats()


@pytest.mark.parametrize("X", [0.99, 0.995])
@pytest.mark.parametrize("seed", [1, 2])
def test_planted_equals_reference(gpu_ctx, X, seed):
    D = int(_lib.cluster_dtable(X, 250)[250])
    nu, nc, st = gpu_vs_ref(gpu_ctx, K.planted(seed, D=D), X)
    assert 0 < nc < nu and st.n_accepted > 0 and st.n_verified <= st.n_candidates


def test_given_order_equals_reference(gpu_ctx):
    reads = K.planted(3)
    seq, off = K.pack(reads)
    _, _, nu = gpu_ctx.derep(seq, off)
    order = np.random.default_rng(3).permutation(nu).astype(np.int32)
    gpu_vs_ref(gpu_ctx, reads, 0.995, order)


def test_d_zero_gives_the_derep_classes(gpu_ctx):
    nu, nc, st = gpu_vs_ref(gpu_ctx, K.planted(4), 0.9999)
    assert nc == nu and st.n_accepted == 0


def test_empty_one_class_and_no_neighbours(gpu_ctx):
    assert gpu_vs_ref(gpu_ctx, [], 0.99)[:2] == (0, 0)
    assert gpu_vs_ref(gpu_ctx, [b"ACGT" * 60] * 3, 0.99)[:2] == (1, 1)
    rng = np.random.default_rng(5)
    reads = [bytes(rng.choice(list(b"ACGT"), 250).tolist()) for _ in range(50)]
    assert gpu_vs_ref(gpu_ctx, reads, 0.99)[:2] == (50, 50)


def test_long_reads_and_the_band_cap(gpu_ctx):
    gpu_vs_ref(gpu_ctx, K.long_reads(6, [2000, 3500, 6000]), 0.99)
    seq, off = K.pack(K.long_reads(7, [6600]))
    gpu_ctx.derep(seq, off)
    with pytest.raises(_lib.ItsxError) as e:
        gpu_ctx.cluster(0.99)
    assert e.value.code == -6


def test_samples_are_refused(gpu_ctx):
    reads = K.planted(8)
    seq, off = K.pack(reads)
    gpu_ctx.reads_upload(seq, off)
    gpu_ctx.set_samples(np.zeros(len(reads), np.int32), 1)
    gpu_ctx.derep_resident(build_search_set=False)
    with pytest.raises(_lib.ItsxError) as e:
        gpu_ctx.cluster(0.99)
    assert e.value.code == -3


def test_two_runs_are_identical(gpu_ctx):
    reads = K.planted(9, ntemplates=40)
    seq, off = K.pack(reads)
    res = []
    for _ in range(2):
        _, _, nu = gpu_ctx.derep(seq, off)
        nc = gpu_ctx.cluster(0.99)
        res.append(gpu_ctx.cluster_fetch(nu, nc))
    assert all(np.array_equal(a, b) for a, b in zip(*res))


@pytest.fixture()
def live(gpu_ctx, monkeypatch):
    monkeypatch.setattr(SeqSample, "get_context", lambda: gpu_ctx)
    SeqSample.reset_sessions()
    yield gpu_ctx
    SeqSample.reset_sessions()


def test_cluster_cli(live, tmp_path):
    K.check_cluster_cli(tmp_path)


def test_no_accepted_pairs_equals_exact(live, tmp_path):
    K.check_no_accepted_pairs_equals_exact(tmp_path)
    (tmp_path / "p").mkdir()
    K.check_no_accepted_pairs_equals_exact(tmp_path / "p", paired=True)


def test_paired_cluster_cli(live, tmp_path):
    K.check_paired_cluster_cli(tmp_path)
