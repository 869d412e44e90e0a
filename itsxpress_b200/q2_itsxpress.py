"""QIIME 2 driver with the reference's action signatures (itsxpress/q2_itsxpress.py: trim_single :120,
trim_pair :156, trim_pair_output_unmerged :194, main :232-364) on top of the GPU path.

Per sample (derep clusters, Z and domZ are per sample upstream, :273-296): check the FASTQs, [merge pairs],
dereplicate (or, with cluster_id < 1, cluster the dereplicated classes on the GPU: SeqSample.cluster), build the
runtime profile set, search, ItsPosition, Dedup, write gzipped output named after the input file into a Casava-1.8
single-lane-per-sample directory.  Small samples share one device pass (_process_batch) at any cluster_id; with
cluster_id < 1 each sample of the pass is clustered on its own, in the order SeqSample.cluster uses.  trim_ccs, and
below 100 % identity ITSX_CLUSTER=vsearch and ITSX_STREAM=1, keep every sample in the per-sample loop (_can_batch).

``per_sample_sequences`` is duck-typed exactly as upstream uses it: ``.manifest.view(pd.DataFrame)`` must give
a frame indexed by sample id with columns ``forward`` [, ``reverse``].  When q2_types is installed the real
directory formats are used; otherwise `CasavaDir` / `PerSampleDir` below read and write the same on-disk
layout (``MANIFEST``, ``metadata.yml``, ``<sample>_<n>_L001_R<d>_001.fastq.gz``).
"""
import logging
import math
import os
import pathlib
import shutil
import tempfile

import pandas as pd

from . import fastq as fq
from . import main as itsxpress

try:  # pragma: no cover - only with QIIME 2 installed
    from q2_types.per_sample_sequences import CasavaOneEightSingleLanePerSampleDirFmt
except ModuleNotFoundError:
    CasavaOneEightSingleLanePerSampleDirFmt = None

default_cluster_id = 1.0


class _Manifest:
    def __init__(self, frame):
        self._frame = frame

    def view(self, kind):
        return self._frame


class PerSampleDir:
    """A SingleLanePerSample{Single,Paired}EndFastqDirFmt directory on disk (data/MANIFEST layout)."""

    def __init__(self, path):
        self.path = str(path)
        man = pd.read_csv(os.path.join(self.path, "MANIFEST"), comment="#")
        rows = {}
        for sid, fn, direction in zip(man["sample-id"], man["filename"], man["direction"]):
            rows.setdefault(sid, {})[direction] = os.path.join(self.path, fn)
        cols = ["forward", "reverse"] if any("reverse" in v for v in rows.values()) else ["forward"]
        frame = pd.DataFrame([[v.get(c) for c in cols] for v in rows.values()], index=list(rows), columns=cols)
        frame.index.name = "sample-id"
        self.manifest = _Manifest(frame)

    def __str__(self):
        return self.path


class CasavaDir:
    """Stand-in for CasavaOneEightSingleLanePerSampleDirFmt(): str() is a fresh directory to write into."""

    def __init__(self, path=None):
        self.path = path if path is not None else tempfile.mkdtemp(prefix="q2-CasavaOneEightSingleLanePerSampleDirFmt-")

    def __str__(self):
        return self.path

    def write_manifest(self):
        """MANIFEST + metadata.yml for the files present (what QIIME 2 derives when it imports the directory)."""
        lines = ["sample-id,filename,direction"]
        for fn in sorted(os.listdir(self.path)):
            if fn.endswith(".fastq.gz"):
                stem = fn.rsplit("_", 4)
                direction = "reverse" if "_R2_" in fn else "forward"
                lines.append("%s,%s,%s" % (stem[0], fn, direction))
        with open(os.path.join(self.path, "MANIFEST"), "w") as f:
            f.write("\n".join(lines) + "\n")
        with open(os.path.join(self.path, "metadata.yml"), "w") as f:
            f.write("{phred-offset: 33}\n")


def _set_fastqs_and_check(fastq, fastq2, tempdir, sample_id, single_end, reversed_primers, allow_staggered_reads,
                          threads):
    try:
        itsxpress._check_fastqs(fastq=fastq, fastq2=fastq2)
        paired_end = itsxpress._is_paired(fastq=fastq, fastq2=fastq2, single_end=single_end)
    except (NotADirectoryError, FileNotFoundError):
        raise ValueError("There is a problem with the fastq file(s) you selected")
    if paired_end:
        sobj = itsxpress.SeqSamplePairedNotInterleaved(fastq=fastq, fastq2=fastq2, tempdir=tempdir,
                                                       reversed_primers=reversed_primers)
        sobj._merge_reads(threads=threads, stagger=allow_staggered_reads)
        return sobj
    return itsxpress.SeqSampleNotPaired(fastq=fastq, tempdir=tempdir)


_TAXA_LETTERS = {"A": "Alveolata", "B": "Bryophyta", "C": "Bacillariophyta", "D": "Amoebozoa", "E": "Euglenozoa",
                 "F": "Fungi", "G": "Chlorophyta", "H": "Rhodophyta", "I": "Phaeophyceae", "L": "Marchantiophyta",
                 "M": "Metazoa", "O": "Oomycota", "P": "Haptophyceae", "Q": "Raphidophyceae", "R": "Rhizaria",
                 "S": "Synurophyceae", "T": "Tracheophyta", "U": "Eustigmatophyceae", "Y": "Parabasalia",
                 "ALL": "All"}


def _taxa_prefix_to_taxa(taxa_prefix):
    """Plugin letter -> taxon name (q2_itsxpress.py:86-117).  'R' gives 'Rhizaria' without the blank that
    definitions.taxa_dict carries, so -- as upstream -- it resolves to no profile file."""
    return _TAXA_LETTERS[taxa_prefix]


def trim_single(per_sample_sequences, region, taxa="F", threads=1, cluster_id=default_cluster_id, trim_ccs=False):
    return main(per_sample_sequences=per_sample_sequences, threads=threads, taxa=taxa, region=region,
                paired_in=False, paired_out=False, reversed_primers=False, allow_staggered_reads=False,
                cluster_id=cluster_id, trim_ccs=trim_ccs)


def trim_pair(per_sample_sequences, region, taxa="F", threads=1, reversed_primers=False, allow_staggered_reads=True,
              cluster_id=default_cluster_id):
    return main(per_sample_sequences=per_sample_sequences, threads=threads, taxa=taxa, region=region, paired_in=True,
                paired_out=False, reversed_primers=reversed_primers, allow_staggered_reads=allow_staggered_reads,
                cluster_id=cluster_id, trim_ccs=False)


def trim_pair_output_unmerged(per_sample_sequences, region, taxa="F", threads=1, reversed_primers=False,
                              allow_staggered_reads=True, cluster_id=default_cluster_id):
    return main(per_sample_sequences=per_sample_sequences, threads=threads, taxa=taxa, region=region, paired_in=True,
                paired_out=True, reversed_primers=reversed_primers, allow_staggered_reads=allow_staggered_reads,
                cluster_id=cluster_id, trim_ccs=False)


def _process_sample(sample, results, tempdir, threads, taxa, region, paired_in, paired_out, reversed_primers,
                    allow_staggered_reads, cluster_id, trim_ccs):
    """One sample of the artifact, start to finish (the body of the reference's loop, q2_itsxpress.py:273-333)."""
    sobj = _set_fastqs_and_check(fastq=sample.forward, fastq2=sample.reverse if paired_in else None,
                                 tempdir=tempdir, sample_id=sample.Index, single_end=not paired_in,
                                 reversed_primers=reversed_primers, allow_staggered_reads=allow_staggered_reads,
                                 threads=threads)
    if trim_ccs:
        sobj.orient_reads(threads=threads)
    if math.isclose(cluster_id, 1, rel_tol=1e-05):
        sobj.deduplicate(threads=threads)
    else:
        sobj.cluster(threads=threads, cluster_id=cluster_id)
    try:
        hmmfile = itsxpress.create_runtime_hmm(taxa, region, tempdir)
        sobj._search(hmmfile=hmmfile, threads=threads)
    except (ModuleNotFoundError, FileNotFoundError, NotADirectoryError):
        raise ValueError("the profile search could not run: libitsx_b200 or a profile file is missing")
    its_pos = itsxpress.ItsPosition(domtable=sobj.dom_file, region=region)
    dedup_obj = itsxpress.Dedup(uc_file=sobj.uc_file, rep_file=sobj.rep_file, seq_file=sobj.seq_file,
                                fastq=sobj.r1, fastq2=sobj.fastq2)
    out_fwd = os.path.join(str(results), pathlib.Path(sample.forward).name)
    if paired_out:
        out_rev = os.path.join(str(results), pathlib.Path(sample.reverse).name)
        dedup_obj.create_paired_trimmed_seqs(out_fwd, out_rev, gzipped=True, zstd_file=False, itspos=its_pos,
                                             wri_file=True, trim_ccs=trim_ccs)
    else:
        dedup_obj.create_trimmed_seqs(out_fwd, gzipped=True, zstd_file=False, itspos=its_pos, wri_file=True,
                                      tempdir=sobj.tempdir, trim_ccs=trim_ccs)


# ---- several samples in one device pass (SURVEY 8f row 3) ---------------------------------------------------------
# The reference runs vsearch and hmmsearch once PER SAMPLE (q2_itsxpress.py:273-296), so classes never span samples and
# domZ is per sample.  libitsx_b200 keeps exactly that while batching: the sample id is part of the derep key and of the
# class test, reported hits are counted per (sample, profile) (itsx_reads_set_samples), and with cluster_id < 1 every
# sample is clustered on its own (itsx_cluster per_sample).  One pass then carries the merged reads of as many samples
# as fit BATCH_READS; an artifact of many small samples costs one chain of launches instead of one per sample.  Outputs
# are byte-identical to the per-sample loop (tests/test_gpu_merge.py, tests/test_gpu_cluster_samples.py).
BATCH_READS = int(os.environ.get("ITSX_Q2_BATCH_READS", "4000000"))      # 0 = the per-sample loop


def _batches(rows, paired_in, budget):
    """Consecutive samples grouped so that a group's reads (estimated from the input size) fit `budget`.  A sample that
    alone takes more than an eighth of the budget is a group of its own: it fills the device without company and goes
    through the per-sample path, which overlaps reading the next sample's files with the GPU work."""
    groups, cur, est = [], [], 0
    for s in rows:
        try:
            size = os.path.getsize(s.forward)
        except OSError:
            size = 0
        # ~250-byte records per read; gzip shrinks amplicon FASTQ ~4-5x
        reads = size // (60 if str(s.forward).endswith((".gz", ".zst")) else 250) + 1
        if reads > budget // 8:
            if cur:
                groups.append(cur)
            groups.append([s])
            cur, est = [], 0
            continue
        if cur and est + reads > budget:
            groups.append(cur)
            cur, est = [], 0
        cur.append(s)
        est += reads
    if cur:
        groups.append(cur)
    return groups


def _cluster_batch(ctx, items, starts, nu, cluster_id):
    """Every sample of the resident batch clustered on its own at ``cluster_id`` in one itsx_cluster call.  A sample's
    classes are taken in the order SeqSample.cluster gives them (host.cluster_order over the sample's reads and labels;
    merged records keep R1's title, so a merged read's label is its R1 id), the samples' orders one after the other.
    Returns the centroid count; the search set and the read -> row map are the centroids' afterwards."""
    import numpy as np
    from . import host
    first, _ = ctx.derep_clusters(nu)
    rep = ctx.derep_map(int(starts[-1]))[0]
    order = [np.zeros(0, np.int64)]
    for k, it in enumerate(items):
        a, b = int(starts[k]), int(starts[k + 1])
        if a < b:
            ids = it["b1"].ids()
            labels = [ids[i] for i in it["idx"].tolist()]
            order.append(np.searchsorted(first, host.cluster_order(rep[a:b] - a, labels) + a))
    nc = ctx.cluster(cluster_id, np.concatenate(order).astype(np.int32), per_sample=True)
    st = ctx.cluster_stats()
    logging.info("GPU clustering of %d samples at %.4g identity, each on its own: %d unique sequences -> %d centroids (%d "
                 "candidate pairs, %d distinct, %d accepted, %d rounds), %.2f ms on device" %
                 (len(items), cluster_id, nu, nc, st.n_candidates, st.n_verified, st.n_accepted, st.n_rounds, st.ms_total))
    return nc


def _process_batch(rows, results, tempdir, threads, taxa, region, paired_in, paired_out, reversed_primers,
                   allow_staggered_reads, cluster_id):
    """The samples `rows` through ONE derep [+ per-sample clustering] + search pass; per sample the files the sequential
    loop writes."""
    import numpy as np
    from . import _lib
    from .SeqSample import get_context
    from .definitions import REGION_PREFIXES, maxmismatches, vsearch_fastq_qmax
    ctx = get_context()
    items = []
    # every file of the batch is read / inflated / scanned on the read-ahead threads while the loop below merges the
    # samples one after the other (the batch holds all of them in memory anyway)
    fq.prefetch([f for sample in rows for f in (sample.forward, sample.reverse if paired_in else None)])
    for sample in rows:
        sobj_check = (sample.forward, sample.reverse if paired_in else None)
        try:
            itsxpress._check_fastqs(fastq=sobj_check[0], fastq2=sobj_check[1])
        except (NotADirectoryError, FileNotFoundError):
            raise ValueError("There is a problem with the fastq file(s) you selected")
        if paired_in:
            r1, r2 = (sample.reverse, sample.forward) if reversed_primers else (sample.forward, sample.reverse)
            b1, b2 = fq.read_fastq_many([r1, r2])
            if b1.n != b2.n:
                raise ValueError("More %s reads than %s reads" % (("forward", "reverse") if b1.n > b2.n else
                                                                  ("reverse", "forward")))
            fseq, foff = b1.seq_concat()
            fqual, _ = b1.qual_concat()
            rseq, roff = b2.seq_concat()
            rqual, _ = b2.qual_concat()
            prm = _lib.merge_params(allow_stagger=allow_staggered_reads, maxdiffs=maxmismatches, maxee=2.0,
                                    qmax=vsearch_fastq_qmax)
            _, _, idx, off, seq, qual = ctx.merge_pairs(fseq, fqual, foff, rseq, rqual, roff, prm)
            items.append(dict(sample=sample, b1=b1, b2=b2, idx=idx, off=off, seq=seq, qual=qual,
                              raw1=(fseq, fqual, foff), raw2=(rseq, rqual, roff)))
        else:
            b = fq.read_fastq(sample.forward)
            seq, off = b.seq_concat()
            qual, _ = b.qual_concat()
            items.append(dict(sample=sample, b1=b, idx=np.arange(b.n, dtype=np.int32), off=off, seq=seq, qual=qual))
    counts = np.array([len(it["off"]) - 1 for it in items], np.int64)
    starts = np.concatenate([[0], np.cumsum(counts)])
    seq_all = np.concatenate([it["seq"] for it in items]) if len(items) else np.zeros(0, np.uint8)
    base = np.concatenate([[0], np.cumsum([int(it["off"][-1]) for it in items])])
    off_all = np.concatenate([[0]] + [it["off"][1:] + base[k] for k, it in enumerate(items)]).astype(np.int64)
    sample_of_read = np.repeat(np.arange(len(items), dtype=np.int32), counts)
    try:
        hmmfile = itsxpress.create_runtime_hmm(taxa, region, tempdir)
        if ctx.load_profiles([hmmfile], None) == 0:
            raise FileNotFoundError(hmmfile)
    except (ModuleNotFoundError, FileNotFoundError, NotADirectoryError):
        raise ValueError("the profile search could not run: libitsx_b200 or a profile file is missing")
    ctx.set_sides_by_prefix(*REGION_PREFIXES[region])
    n_all = len(off_all) - 1
    ctx.reads_upload(seq_all, off_all)
    ctx.set_samples(sample_of_read, max(len(items), 1))
    nrow = nu = ctx.derep_resident()
    if not math.isclose(cluster_id, 1, rel_tol=1e-05):
        nrow = _cluster_batch(ctx, items, starts, nu, cluster_id)
    ctx.search()
    if not paired_out:
        # merged / single-end output: the re-expansion of the whole batch in one go, split by sample afterwards
        ctx.quals_upload(np.concatenate([it["qual"] for it in items]) if len(items) else np.zeros(0, np.uint8))
        ctx.trim_gather_resident(0)
        ki, oo, os_, oq = ctx.run_fetch()
        for k, it in enumerate(items):
            a, b = np.searchsorted(ki, starts[k]), np.searchsorted(ki, starts[k + 1])
            kept_local = ki[a:b] - starts[k]
            text = fq.format_gathered(it["b1"], it["idx"][kept_local], oo[a:b + 1] - oo[a], os_[oo[a]:oo[b]],
                                      oq[oo[a]:oo[b]], as_array=True)
            out_fwd = os.path.join(str(results), pathlib.Path(it["sample"].forward).name)
            fq.write_compressed(out_fwd, text, gzipped=True, zstd_file=False, n_records=len(kept_local))
        return
    # unmerged output: R1 [start:stop], R2 [tlen-stop : tlen-start] of every pair whose merged read was kept
    _, _, uid = ctx.derep_map(n_all)
    pos = ctx.positions(nrow)
    start, stop, tlen = pos["start"].copy(), pos["stop"].copy(), pos["tlen"].copy()
    for k, it in enumerate(items):
        b1, b2 = it["b1"], it["b2"]
        uid_pair = np.full(b1.n, -1, np.int32)
        uid_pair[it["idx"]] = uid[starts[k]:starts[k + 1]]
        outs = []
        for mode, b, raw in ((2, b1, it["raw1"]), (1, b2, it["raw2"])):
            ctx.trim_set_map(uid_pair, nrow)
            ctx.positions_set(start, stop, tlen)
            kk, oo, os_, oq = ctx.trim_gather(b.n, mode=mode, seq=raw[0], qual=raw[1], off=raw[2])
            outs.append((fq.format_gathered(b, kk, oo, os_, oq, as_array=True), len(kk)))
        # as upstream (q2_itsxpress.py:311-323): the trimmed r1 goes under the forward file's name, r2 under the reverse's
        fq.write_compressed(os.path.join(str(results), pathlib.Path(it["sample"].forward).name), outs[0][0],
                            gzipped=True, zstd_file=False, n_records=outs[0][1])
        fq.write_compressed(os.path.join(str(results), pathlib.Path(it["sample"].reverse).name), outs[1][0],
                            gzipped=True, zstd_file=False, n_records=outs[1][1])


READ_AHEAD_BYTES = int(os.environ.get("ITSX_READ_AHEAD_BYTES", str(2 << 30)))


def _can_batch(cluster_id, trim_ccs):
    """Whether samples may share device passes: not with trim_ccs (orientation runs per sample).  Below 100 % identity
    also not when ITSX_CLUSTER=vsearch shells out to vsearch, which clusters one sample per call, nor when ITSX_STREAM=1
    streams every sample: SeqSample.cluster then has no labels and orders ties by first occurrence, not by label as a
    batched pass does, so the two could pick different centroids."""
    if not math.isclose(cluster_id, 1, rel_tol=1e-05) and (os.environ.get("ITSX_CLUSTER", "gpu") == "vsearch" or
                                                            os.environ.get("ITSX_STREAM", "auto") == "1"):
        return False
    return BATCH_READS > 0 and not trim_ccs


def _run_rows(rows, results, tempdir, threads, taxa, region, paired_in, paired_out, reversed_primers,
              allow_staggered_reads, cluster_id, trim_ccs, process):
    """The samples `rows` in order: small ones batched into shared device passes, large ones one at a time with the next
    sample's files read ahead.  Returns the sample ids done."""
    done = []
    batch = _can_batch(cluster_id, trim_ccs) and process is _process_sample      # (a caller-supplied per-sample hook is kept)
    groups = _batches(rows, paired_in, BATCH_READS) if batch else [[r] for r in rows]
    flat = [g for g in groups]
    for gi, group in enumerate(flat):
        if len(group) > 1:
            _process_batch(group, results, tempdir, threads, taxa, region, paired_in, paired_out, reversed_primers,
                           allow_staggered_reads, cluster_id)
        else:
            # read the next samples' files while this one is on the GPU (fq.READ_AHEAD of them, within ~2 GB of files)
            ahead_bytes = 0
            for gj in range(gi + 1, min(gi + 1 + fq.READ_AHEAD, len(flat))):
                if len(flat[gj]) != 1:
                    break
                nxt = flat[gj][0]
                files = [nxt.forward, nxt.reverse if paired_in else None]
                ahead_bytes += sum(os.path.getsize(f) for f in files if f and os.path.exists(f))
                if gj > gi + 1 and ahead_bytes > READ_AHEAD_BYTES:
                    break
                fq.prefetch(files)
            process(group[0], results, tempdir, threads, taxa, region, paired_in, paired_out, reversed_primers,
                    allow_staggered_reads, cluster_id, trim_ccs)
        done += [smp.Index for smp in group]
    return done


def main(per_sample_sequences, threads, taxa, region, paired_in, paired_out, reversed_primers, allow_staggered_reads,
         cluster_id, trim_ccs=False):
    taxa = _taxa_prefix_to_taxa(taxa)
    samples = per_sample_sequences.manifest.view(pd.DataFrame)
    try:
        tempdir = tempfile.mkdtemp(prefix="itsxpress_")
    except Exception:
        raise ValueError("Could not create temporary directory")
    results = CasavaOneEightSingleLanePerSampleDirFmt() if CasavaOneEightSingleLanePerSampleDirFmt else CasavaDir()
    rows = list(samples.itertuples())
    try:
        _run_rows(rows, results, tempdir, threads, taxa, region, paired_in, paired_out, reversed_primers,
                  allow_staggered_reads, cluster_id, trim_ccs, _process_sample)
    finally:
        fq.drop_prefetched()
    if trim_ccs:
        print("\n" + "=" * 80 + "\nPacBio CCS trimming complete.\n\nCAUTION: data contain fake sequence at the ends "
              "needed for DADA2\n\nqiime dada2 denoise-ccs --p-front GACAGGTACAAGAAGGA --p-adapter ACTGGAGACTGGGTTAA\n"
              + "*" * 80 + "\n")
    if isinstance(results, CasavaDir):
        results.write_manifest()
    shutil.rmtree(tempdir)
    return results


def deal_samples(sizes, world):
    """Whole samples dealt to `world` ranks, largest first onto the least-loaded rank (derep, Z and domZ are per
    sample upstream, q2_itsxpress.py:273-296, so samples are independent units: SURVEY 8e).  Returns the owner rank of
    every sample; deterministic, so every rank computes the same deal without talking to the others."""
    load = [0] * world
    owner = [0] * len(sizes)
    for i in sorted(range(len(sizes)), key=lambda k: (-int(sizes[k]), k)):
        r = min(range(world), key=lambda q: (load[q], q))
        owner[i] = r
        load[r] += int(sizes[i])
    return owner


def main_sharded(per_sample_sequences, outdir, region, taxa="F", threads=1, paired_in=True, paired_out=True,
                 reversed_primers=False, allow_staggered_reads=True, cluster_id=default_cluster_id, trim_ccs=False,
                 rank=None, world=None, barrier=None, process=None):
    """The samples of one artifact over the GPUs of a box: one process per GPU (``torchrun``; RANK / WORLD_SIZE /
    LOCAL_RANK from the environment), every rank runs the per-sample pipeline of ``main`` on the samples dealt to it
    and writes their files into the shared directory ``outdir``; there is no data-path collective.  ``barrier`` (default:
    ``torch.distributed.barrier`` when a process group is up) separates the work from rank 0 writing MANIFEST and
    metadata.yml.  Returns (CasavaDir over outdir, sample ids this rank processed)."""
    rank = int(os.environ.get("RANK", "0")) if rank is None else rank
    world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else world
    taxa = _taxa_prefix_to_taxa(taxa)
    samples = per_sample_sequences.manifest.view(pd.DataFrame)
    rows = list(samples.itertuples())
    sizes = [os.path.getsize(s.forward) + (os.path.getsize(s.reverse) if paired_in else 0) for s in rows]
    owner = deal_samples(sizes, world)
    os.makedirs(outdir, exist_ok=True)
    results = CasavaDir(outdir)
    tempdir = tempfile.mkdtemp(prefix="itsxpress_r%d_" % rank)
    process = process or _process_sample
    mine = []
    todo = [sample for sample, o in zip(rows, owner) if o == rank]
    try:
        mine += _run_rows(todo, results, tempdir, threads, taxa, region, paired_in, paired_out, reversed_primers,
                          allow_staggered_reads, cluster_id, trim_ccs, process)
    finally:
        fq.drop_prefetched()
        shutil.rmtree(tempdir, ignore_errors=True)
    if barrier is None and world > 1:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            barrier = dist.barrier
    if barrier is not None:
        barrier()
    if rank == 0:
        results.write_manifest()
    if barrier is not None:
        barrier()
    return results, mine


def cli(argv=None):
    """Shell entry for a whole per-sample directory (the `data/` of a QIIME 2 artifact), one process per GPU:

        torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 -m itsxpress_b200.q2_itsxpress \\
            --in ARTIFACT/data --out OUTDIR --region ITS2 --taxa F --mode pair-unmerged

    --mode single | pair | pair-unmerged = the plugin actions trim-single / trim-pair / trim-pair-output-unmerged
    (q2_itsxpress.py:119-230).  With one process it is the plain action writing into OUTDIR."""
    import argparse
    ap = argparse.ArgumentParser(prog="python -m itsxpress_b200.q2_itsxpress", description=cli.__doc__,
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--in", dest="src", required=True, help="per-sample directory with MANIFEST")
    ap.add_argument("--out", required=True, help="output directory (shared by all ranks)")
    ap.add_argument("--region", required=True, choices=["ITS1", "ITS2", "ALL"])
    ap.add_argument("--taxa", default="F", choices=sorted(_TAXA_LETTERS))
    ap.add_argument("--mode", default="pair-unmerged", choices=["single", "pair", "pair-unmerged"])
    ap.add_argument("--threads", type=int, default=1)
    ap.add_argument("--reversed-primers", action="store_true")
    ap.add_argument("--no-staggered", action="store_true", help="do not merge staggered pairs")
    a = ap.parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        if not dist.is_initialized():
            dist.init_process_group("gloo")      # barriers only; every rank computes on the GPU LOCAL_RANK names
    try:
        res, mine = main_sharded(PerSampleDir(a.src), a.out, region=a.region, taxa=a.taxa, threads=a.threads,
                                 paired_in=a.mode != "single", paired_out=a.mode == "pair-unmerged",
                                 reversed_primers=a.reversed_primers, allow_staggered_reads=not a.no_staggered)
    finally:
        if dist is not None and dist.is_initialized():
            dist.destroy_process_group()
    print("rank %s: %d sample(s) -> %s" % (os.environ.get("RANK", "0"), len(mine), str(res)))
    return 0


if __name__ == "__main__":
    import sys
    sys.exit(cli())
