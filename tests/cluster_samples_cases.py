"""Per-sample clustering (itsx_cluster with per_sample = 1): the reference result built from tests/cluster_ref.c run on
each sample alone, planted multi-sample workloads, and the QIIME 2 check that batched passes at cluster_id < 1 write the
bytes of the per-sample loop.  Shared by tests/test_gpu_cluster_samples.py (on the device) and
tests/test_cluster_samples_on_oracle.py (CPU reference standing in for it)."""
import os

import numpy as np

import cluster_cases as K
import cluster_ref as R

from itsxpress_b200 import fastq as fq


def per_sample_reference(seq, off, first, uid, sample, cluster_id, order=None):
    """(n_centroids, centroid_row_of_unique, strand_of_unique, ed_of_unique, unique_of_row) of per-sample clustering:
    R.cluster on each sample's classes alone, taken in ``order`` restricted to the sample (None: the sample's own
    default order), mapped back to batch unique indices; centroid rows follow ``order`` (None: the batch's default order)
    across samples.  first / uid: the batch derep (unique -> first read, read -> unique); sample: per read."""
    first = np.asarray(first, np.int64)
    uid = np.asarray(uid, np.int64)
    sample = np.asarray(sample)
    nu = len(first)
    rep = first[uid] if len(uid) else uid
    glob = R.default_order(rep) if order is None else np.asarray(order, np.int64)
    cent, strand, ed = np.empty(nu, np.int64), np.empty(nu, np.uint8), np.empty(nu, np.int32)
    of_unique = sample[first] if nu else np.zeros(0, np.int32)
    for k in np.unique(of_unique):
        us = np.flatnonzero(of_unique == k)                 # the sample's classes, in first-occurrence order
        if order is None:
            reads = np.flatnonzero(sample == k)
            local = R.default_order(np.searchsorted(reads, rep[reads]))
        else:
            local = np.searchsorted(us, glob[np.isin(glob, us)])
        _, crow_k, strand_k, ed_k, uor_k = R.cluster(seq, off, first[us], local, cluster_id)
        cent[us] = us[uor_k[crow_k]]
        strand[us], ed[us] = strand_k, ed_k
    rank = np.empty(nu, np.int64)
    rank[glob] = np.arange(nu)
    uor = np.unique(cent)
    uor = uor[np.argsort(rank[uor])]
    row = np.empty(nu, np.int64)
    row[uor] = np.arange(len(uor))
    return len(uor), row[cent].astype(np.int32), strand, ed, uor.astype(np.int32)


def planted_samples(seed, D):
    """Five samples: a planted workload (K.planted); the same templates at other abundances; an empty sample; a sample
    of one class; and a read within D edits of the most abundant class of sample 0 that only a leaked cross-sample edge
    could pull into that class (on its own it is a centroid, among unrelated reads)."""
    rng = np.random.default_rng(seed)
    a = K.planted(seed, D=D)
    uniq = list(dict.fromkeys(a))
    b = [r for r in uniq if rng.random() < 0.6 for _ in range(int(rng.integers(1, 5)))]
    b = [b[i] for i in rng.permutation(len(b))]
    top = max(uniq, key=a.count)
    assert a.count(top) >= 2
    x = K.edit(rng, top, D)
    while x in uniq:
        x = K.edit(rng, top, D)
    e = [bytes(rng.choice(list(b"ACGT"), 250).tolist()) for _ in range(6)]
    e.insert(3, x)
    return [a, b, [], [uniq[1]] * 3, e]


def pack_samples(samples):
    """reads of all samples (one after the other) and the sample id of every read"""
    reads = [r for s in samples for r in s]
    sample = np.repeat(np.arange(len(samples), dtype=np.int32), [len(s) for s in samples])
    seq, off = K.pack(reads)
    return seq, off, sample


def interleaved_order(rng, first, sample):
    """a random order of every sample's classes, the samples interleaved at random"""
    of_unique = sample[first]
    per = {k: list(rng.permutation(np.flatnonzero(of_unique == k))) for k in np.unique(of_unique)}
    slots = rng.permutation(np.concatenate([np.full(len(v), k) for k, v in per.items()])) if per else []
    return np.array([per[k].pop(0) for k in slots], np.int32)


# ---- QIIME 2 actions at cluster_id < 1: batched passes == the per-sample loop ----------------------------------------
SIZES = [30, 17, 25, 0, 12, 28, 9, 22, 15, 30, 20, 11, 26, 18, 24, 14, 19]


def make_artifact(root):
    from test_gpu_merge import _make_artifact
    return _make_artifact(root, SIZES, seed=5)


def make_single_artifact(root, seed=5):
    """A single-end per-sample directory of len(SIZES) samples drawn from the merged fixture reads (overlapping subsets,
    so the same sequences occur in several samples), one of them empty."""
    import gzip
    b = fq.read_fastq(K.MERGED)
    rng = np.random.default_rng(seed)
    os.makedirs(root)
    lines = ["sample-id,filename,direction"]
    for k, n in enumerate(SIZES):
        pick = np.sort(rng.choice(b.n, size=n, replace=False)) if n else np.zeros(0, np.int64)
        fn = "S%d_%d_L001_R1_001.fastq.gz" % (k, k)
        with gzip.open(os.path.join(root, fn), "wb", compresslevel=1) as f:
            f.write(fq.format_records(b, pick, np.zeros(len(pick), np.int32), b.s_len[pick].astype(np.int32)))
        lines.append("S%d,%s,forward" % (k, fn))
    with open(os.path.join(root, "MANIFEST"), "w") as f:
        f.write("\n".join(lines) + "\n")
    return root


def _spy(monkeypatch, ctx, name, log):
    orig = getattr(ctx, name)

    def f(*a, **kw):
        out = orig(*a, **kw)
        log.append((name, kw.get("per_sample", False), out))
        return out
    monkeypatch.setattr(ctx, name, f)


def check_q2_batches_equal_loop(ctx, tmp_path, monkeypatch, cluster_id=0.995):
    """trim_single (merged reads as single-end samples), trim_pair and trim_pair_output_unmerged (read pairs) at
    ``cluster_id`` with BATCH_READS = 0 (the per-sample loop),
    4 000 000 (one pass) and a budget that gives several multi-sample passes: the same files and MANIFEST; the batched
    runs upload once per pass and cluster each pass per sample, and some classes do merge."""
    from itsxpress_b200 import q2_itsxpress as q2
    arts = {False: make_single_artifact(str(tmp_path / "in1")), True: make_artifact(str(tmp_path / "in2"))}
    log = []
    for name in ("reads_upload", "derep_resident", "cluster"):
        _spy(monkeypatch, ctx, name, log)
    actions = (("single", q2.trim_single, False), ("pair", q2.trim_pair, True),
               ("pair-unmerged", q2.trim_pair_output_unmerged, True))
    for action, fn, paired_in in actions:
        art = arts[paired_in]
        rows = list(q2.PerSampleDir(art).manifest.view(None).itertuples())
        small = _several_passes_budget(q2, rows, paired_in)
        groups = q2._batches(rows, paired_in, small)
        outs = []
        for budget, npass in ((0, 0), (4_000_000, 1), (small, len(groups))):
            monkeypatch.setattr(q2, "BATCH_READS", budget)
            del log[:]
            outs.append(str(fn(q2.PerSampleDir(art), region="ITS2", taxa="M", cluster_id=cluster_id)))
            assert sum(1 for e in log if e[0] == "reads_upload") == npass, (action, budget)
            batched = [e for e in log if e[0] == "cluster"]
            if npass:
                assert len(batched) == npass and all(e[1] for e in batched), (action, budget)
                nu = sum(e[2] for e in log if e[0] == "derep_resident")
                assert sum(e[2] for e in batched) < nu, (action, budget)       # classes did merge
        ref = outs[0]
        names = sorted(f for f in os.listdir(ref) if f.endswith(".gz"))
        assert len(names) == len(SIZES) * (2 if action == "pair-unmerged" else 1)
        total = 0
        for got in outs[1:]:
            assert sorted(f for f in os.listdir(got) if f.endswith(".gz")) == names
            for n in names:
                want = fq._open_bytes(os.path.join(ref, n))
                assert fq._open_bytes(os.path.join(got, n)) == want, (action, n)
                total += len(want)
            assert open(os.path.join(got, "MANIFEST")).read() == open(os.path.join(ref, "MANIFEST")).read()
        assert total > 100_000, action


def _several_passes_budget(q2, rows, paired_in):
    """the smallest BATCH_READS (in steps of ~25 %) at which q2._batches puts every sample into a pass of several
    samples, and there are at least two passes"""
    b = 8
    while b < 1 << 30:
        groups = q2._batches(rows, paired_in, b)
        if len(groups) >= 2 and all(len(g) > 1 for g in groups):
            return b
        b = b * 5 // 4 + 1
    raise AssertionError("no budget gives several multi-sample passes")
