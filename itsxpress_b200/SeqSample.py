"""Per-sample pipeline objects with the reference's names, arguments and error behaviour
(itsxpress/SeqSample.py: SeqSample :18, SeqSampleNotPaired :228, SeqSamplePairedNotInterleaved :244,
ItsPosition :368, Dedup :501) -- but ``deduplicate`` and ``_search`` run on the B200 through
libitsx_b200 instead of shelling out to vsearch / hmmsearch, ItsPosition's arg-max runs on the device,
and the per-read filter / slice / re-expansion of ``create_*trimmed_seqs`` is ``itsx_trim_*``.

Stage hand-off stays what it is upstream: paths to ``uc.txt``, ``rep.fa`` and ``domtbl.txt`` in the temp
directory, so ``ItsPosition(path, region)`` and ``Dedup(uc, rep, seq, ...)`` also work on files written by
the real tools (that is how the reference's tests build them, tests/test_main_pytest.py:32-35,49-53).
Objects created from files that a live GPU session just wrote additionally see that session's arrays and
skip the text round trip.  There is no CPU implementation of the kernels here: without libitsx_b200 and a
B200 these classes raise.
"""
import logging
import os
import shutil
import subprocess

import numpy as np

from . import _lib
from . import fastq as fq
from . import host
from .definitions import ROOT_DIR, REGION_PREFIXES, maxmismatches, vsearch_fastq_qmax

logger = logging.getLogger(__name__)

CCS_FWD = b"GACAGGTACAAGAAGGA"      # synthetic primers of --trim-ccs (SeqSample.py:601-603)
CCS_REV = b"TTAACCCAGTCTCCAGT"

# uc.txt / rep.fa / domtbl.txt are the reference's inter-stage interface and are always written for samples up to
# this many reads (and whenever --keeptemp / ITSX_TEMP_FILES=always asks for them).  Above it, in "auto" mode, the
# text files would dominate the run (a 1 M-read sample has ~16 M domtbl rows), so one-line placeholders are left in
# their place and ItsPosition / Dedup take the arrays of the live GPU session.
TEMP_FILE_POLICY = os.environ.get("ITSX_TEMP_FILES", "auto")      # auto | always | never
TEMP_FILE_AUTO_MAX_READS = 200_000
_PLACEHOLDER = "# itsxpress-b200: not materialised for a large sample; rerun with --keeptemp or ITSX_TEMP_FILES=always\n"

# A single-end / merged input larger than this is STREAMED: parsed chunk by chunk into the device (itsx_reads_begin /
# append / end) and trimmed chunk by chunk on the way out, so neither the text nor its parsed arrays ever sit whole in
# host memory (BASELINE configs[3] is 70 GB of FASTQ text; upstream streams through Biopython, SeqSample.py:742-752,
# 908-949).  ITSX_STREAM=1 forces it, ITSX_STREAM=0 disables it.
STREAM_MIN_BYTES = int(os.environ.get("ITSX_STREAM_MIN_BYTES", str(4 << 30)))


def _stream_wanted(path):
    mode = os.environ.get("ITSX_STREAM", "auto")
    if mode == "1":
        return True
    if mode == "0":
        return False
    try:
        size = os.path.getsize(path)
    except OSError:
        return False
    return size * (4 if path.endswith((".gz", ".zst")) else 1) > STREAM_MIN_BYTES


_CTX = None
_GENERATION = 0           # bumped whenever the shared context's resident sample / search changes
_SESSIONS = {}            # abspath of uc.txt / rep.fa / domtbl.txt  ->  _Session that wrote it


def get_context():
    """The process-wide GPU context (one per process; device = LOCAL_RANK under torchrun, else 0)."""
    global _CTX
    if _CTX is None:
        _CTX = _lib.Context(int(os.environ.get("ITSX_DEVICE", os.environ.get("LOCAL_RANK", "0"))))
    return _CTX


class _Session:
    """What one sample leaves behind on the host after deduplicate() / _search()."""

    def __init__(self):
        self.batch = None          # FastqBatch of seq_file
        self.files = True          # uc.txt / rep.fa / domtbl.txt were written in full
        self.rep = None            # int32[n]  index of the representative read
        self.uid = None            # int32[n]  dense unique id, first-occurrence order
        self.first = None          # int32[U]  read index of every unique
        self.n_unique = 0
        self.derep_gen = -1        # _GENERATION at which the context held this sample's reads
        self.search_gen = -1       # ... and this sample's search results
        self.names = None
        self.nseq = 0
        self.seq_path = None
        self.seq_ids = None
        # paired input merged by _merge_reads in this process: record k of seq_file is pair pair_index[k] of the
        # R1 / R2 files (their paths and parsed batches are kept for create_paired_trimmed_seqs)
        self.pair_index = None
        self.pair_files = None     # (abspath R1, abspath R2)
        self.pair_batches = None   # (FastqBatch R1, FastqBatch R2)
        self.sides_prefix = None   # (left, right) name prefixes the search already selected boundaries for
        self.streamed = False      # the reads went to the device chunk by chunk; no FastqBatch is held
        self.n_reads = 0
        self.chunk_bytes = None    # chunking of the streamed pass (the output pass repeats it)

    def ensure_seq_ids(self):
        if self.seq_ids is None and self.batch is not None and self.first is not None:
            ids = self.ids
            self.seq_ids = [ids[i] for i in self.first.tolist()]
        return self.seq_ids

    @property
    def ids(self):
        """Record ids (first token of the title); materialised on first use."""
        return self.batch.ids() if self.batch is not None else None


def _external(tool, argv, what):
    """Run one of the reference's external steps that are outside the GPU path (merge, orient, cluster)."""
    try:
        p = subprocess.run(argv, stderr=subprocess.PIPE)
        logging.info(p.stderr.decode("utf-8"))
        p.check_returncode()
    except subprocess.CalledProcessError as e:
        logging.exception("Could not perform %s with %s. Error from %s was:\n %s" % (what, tool, tool,
                                                                                     p.stderr.decode("utf-8")))
        raise e
    except FileNotFoundError as f:
        logging.error("%s was not found, make sure %s is installed and executable" % (tool, tool))
        raise f


class SeqSample:
    """Base class: one sample on its way from FASTQ to trimmed FASTQ (reference SeqSample.py:18-225)."""

    def __init__(self, fastq, tempdir):
        self.tempdir = tempdir
        self.fastq = fastq
        self.uc_file = None
        self.rep_file = None
        self.dom_file = None
        self.seq_file = None
        self.r1 = None
        self.fastq2 = None
        self._session = None
        self._merged = None            # (seq.fq path, FastqBatch, bases, offsets) left by _merge_reads for deduplicate
        self.materialize = None        # True / False overrides TEMP_FILE_POLICY (main.py sets it for --keeptemp)

    def _want_files(self, n_reads):
        if self.materialize is not None:
            return bool(self.materialize)
        if TEMP_FILE_POLICY == "always":
            return True
        if TEMP_FILE_POLICY == "never":
            return False
        return n_reads <= TEMP_FILE_AUTO_MAX_READS

    # -- steps outside the named hot path: still the external tool, exactly as upstream ------------------
    def orient_reads(self, threads=1):
        """vsearch --orient against the universal reference (SeqSample.py:48-91); needs vsearch."""
        oriented = os.path.join(self.tempdir, "oriented.fq")
        _external("Vsearch", ["vsearch", "--orient", self.fastq, "--db",
                              os.path.join(ROOT_DIR, "universal_orient_ref_clean.fasta.gz"),
                              "--fastqout", oriented, "--threads", str(threads)], "read orientation")
        self.fastq = self.seq_file = self.r1 = oriented

    def cluster(self, threads, cluster_id=0.995):
        """Greedy clustering of the reads at ``cluster_id`` identity on the GPU; writes ``uc.txt`` and ``rep.fa`` in the
        layout of `vsearch --cluster_size --strand both` (replaces SeqSample.py:133-176).

        The exact derep runs first (in memory or streamed) and its classes are clustered (``itsx_cluster``): classes are
        taken by abundance descending, then by label as ``host.cluster_order`` sorts them (first occurrence for a
        streamed input); a class becomes a centroid unless an earlier centroid is within ``cluster_id`` identity (edit
        distance over the longer length, both strands), else it joins the closest such centroid, the earliest on a tie.
        The search then runs on the centroids only, and every read is trimmed with its centroid's positions.
        Deliberate differences from vsearch (DESIGN.md §6): abundance comes from the exact derep (vsearch, given raw
        reads without --sizein, sees abundance 1 everywhere and sorts by label); the search is exhaustive (no
        --maxaccepts / --maxrejects k-mer heuristics); terminal gaps count (vsearch's default --iddef 2 ignores them,
        so a truncated read would join a longer centroid at 100 % and be cut at coordinates that are not its own).
        The H rows of uc.txt carry '*' in the CIGAR column.  ``threads`` is accepted for the reference's signature.
        ITSX_CLUSTER=vsearch runs the vsearch command of the reference instead."""
        if os.environ.get("ITSX_CLUSTER", "gpu") == "vsearch":
            self.uc_file = os.path.join(self.tempdir, "uc.txt")
            self.rep_file = os.path.join(self.tempdir, "rep.fa")
            _external("Vsearch", ["vsearch", "--cluster_size", self.seq_file, "--centroids", self.rep_file, "--uc",
                                  self.uc_file, "--strand", "both", "--id", str(cluster_id), "--threads",
                                  str(threads)], "clustering")
            return
        self.deduplicate(threads)
        try:
            s = self._session
            ctx = get_context()
            ids = None
            if s.streamed:
                order = None
            else:
                ids = s.ids
                order = np.searchsorted(s.first, host.cluster_order(s.rep, ids)).astype(np.int32)
            nu = s.n_unique
            nc = ctx.cluster(cluster_id, order)
            crow, cstrand, ced, unique_of_row = ctx.cluster_fetch(nu, nc)
            if not s.streamed:
                cls = s.uid                                  # read -> exact class
                cfirst = s.first[unique_of_row]              # centroid row -> its first read
                s.uid = crow[cls] if len(cls) else cls
                s.first = cfirst
                s.rep = cfirst[s.uid] if len(cls) else s.rep
                if s.files:
                    batch = s.batch
                    dstrand = ctx.derep_map(batch.n)[1]
                    strand = dstrand ^ cstrand[cls]
                    L = batch.s_len.astype(np.int64)
                    Lc = np.maximum(L, L[s.rep])
                    ident = np.where(Lc > 0, 100.0 * (Lc - ced[cls]) / np.maximum(Lc, 1), 100.0)
                    with open(self.rep_file, "wb") as f:
                        f.write(host.write_rep_fasta(batch, cfirst.astype(np.int64), ids))
                    with open(self.uc_file, "wb") as f:
                        f.write(host.write_uc_py(s.rep, strand, ids, batch.s_len, cfirst, identity=ident))
            s.n_unique = nc
            s.seq_ids = None
            st = ctx.cluster_stats()
            logging.info("GPU clustering at %.4g identity: %d unique sequences -> %d centroids (%d candidate pairs, %d "
                         "distinct, %d accepted, %d rounds), %.2f ms on device" %
                         (cluster_id, nu, nc, st.n_candidates, st.n_verified, st.n_accepted, st.n_rounds, st.ms_total))
        except Exception as e:
            logging.exception("Could not perform clustering on the GPU.")
            raise e

    # -- the hot path ---------------------------------------------------------------------------------------
    def deduplicate(self, threads=1):
        """Exact full-length dereplication over both strands on the GPU; writes ``uc.txt`` and ``rep.fa`` in
        vsearch's formats (replaces `vsearch --fastx_uniques`, SeqSample.py:93-131).  ``threads`` is accepted
        and unused, as upstream (it is never passed to vsearch, :106-116)."""
        global _GENERATION
        try:
            self.uc_file = os.path.join(self.tempdir, "uc.txt")
            self.rep_file = os.path.join(self.tempdir, "rep.fa")
            merged = getattr(self, "_merged", None)
            self._merged = None
            if merged is None and _stream_wanted(self.seq_file):
                return self._deduplicate_streamed()
            if merged is not None and merged[0] == os.path.abspath(self.seq_file):
                batch, seq, off = merged[1:4]          # records _merge_reads just wrote to seq_file
            else:
                batch = fq.read_fastq(self.seq_file)
                seq, off = batch.seq_concat()
            ctx = get_context()
            rep, strand, nu = ctx.derep(seq, off)
            _GENERATION += 1
            first, _ = ctx.derep_clusters(nu)
            s = _Session()
            s.batch, s.rep, s.first, s.n_unique = batch, rep, first, nu
            s.uid = np.searchsorted(first, rep).astype(np.int32) if nu else np.zeros(0, np.int32)
            s.derep_gen = _GENERATION
            s.seq_path = os.path.abspath(self.seq_file)
            if merged is not None and merged[0] == s.seq_path:
                s.pair_index, s.pair_files, s.pair_batches = merged[4], merged[5], merged[6]
            s.files = self._want_files(batch.n)
            if s.files:
                ids = s.ids
                order = host.cluster_order(rep, ids)
                with open(self.rep_file, "wb") as f:
                    f.write(host.write_rep_fasta(batch, order, ids))
                with open(self.uc_file, "wb") as f:
                    f.write(host.write_uc(rep, strand, ids, batch.s_len, order, batch=batch))
            else:
                logging.info("uc.txt and rep.fa are one-line placeholders for this sample (%d reads > %d); Dedup takes "
                             "the read -> representative map from the GPU session. Use --keeptemp or "
                             "ITSX_TEMP_FILES=always for the full files." % (batch.n, TEMP_FILE_AUTO_MAX_READS))
                for path in (self.rep_file, self.uc_file):
                    with open(path, "w") as f:
                        f.write(_PLACEHOLDER)
            st = ctx.derep_stats()
            logging.info("GPU dereplication: %d reads, %d unique sequences, %.2f ms on device" %
                         (batch.n, nu, st.ms_total))
            self._session = s
            _SESSIONS[os.path.abspath(self.uc_file)] = s
            _SESSIONS[os.path.abspath(self.rep_file)] = s
        except FileNotFoundError as f:
            logging.error("The sequence file %s could not be found." % self.seq_file)
            raise f
        except Exception as e:
            logging.exception("Could not perform dereplication on the GPU.")
            raise e

    def _deduplicate_streamed(self):
        """deduplicate() for a file that is not held in host memory: chunks of whole records are parsed (native scanner,
        next block read / inflated on a background thread) and appended to the device-resident read set; uc.txt and
        rep.fa are placeholders (the session carries the map)."""
        global _GENERATION
        ctx = get_context()
        size = os.path.getsize(self.seq_file)
        est_bases = (size * (4 if self.seq_file.endswith((".gz", ".zst")) else 1)) // 2
        ctx.reads_begin(est_bases // 200, est_bases)
        n = 0
        for chunk in fq.stream_fastq(self.seq_file):
            seq, off = chunk.seq_concat()
            qual, _ = chunk.qual_concat()
            ctx.reads_append(seq, qual, off)
            n += chunk.n
        n_dev, _ = ctx.reads_end()
        assert n_dev == n
        nu = ctx.derep_resident(build_search_set=True)
        _GENERATION += 1
        s = _Session()
        s.streamed, s.n_reads, s.n_unique, s.chunk_bytes = True, n, nu, fq.STREAM_CHUNK_BYTES
        s.derep_gen = _GENERATION
        s.seq_path = os.path.abspath(self.seq_file)
        s.files = False
        s.rep = True               # (marks the session as holding the read -> representative map, on the device)
        logging.info("uc.txt and rep.fa are one-line placeholders: %s was streamed to the GPU in chunks (%d reads); "
                     "Dedup takes the read -> representative map from the GPU session." % (self.seq_file, n))
        for path in (self.rep_file, self.uc_file):
            with open(path, "w") as f:
                f.write(_PLACEHOLDER)
        fq.note_count(self.seq_file, n)
        st = ctx.derep_stats()
        logging.info("GPU dereplication: %d reads, %d unique sequences, %.2f ms on device" % (n, nu, st.ms_total))
        self._session = s
        _SESSIONS[os.path.abspath(self.uc_file)] = s
        _SESSIONS[os.path.abspath(self.rep_file)] = s

    def _search(self, hmmfile, threads):
        """Profile-HMM search of every representative against every profile of ``hmmfile`` on the GPU with
        hmmsearch's thresholds ``-T 10 --F1 1e-6 --F2 1e-6 --F3 1e-6``; writes ``domtbl.txt``
        (replaces SeqSample.py:178-225)."""
        global _GENERATION
        try:
            self.dom_file = os.path.join(self.tempdir, "domtbl.txt")
            if not os.path.exists(hmmfile):
                raise FileNotFoundError(hmmfile)
            ctx = get_context()
            nprof = ctx.load_profiles([hmmfile], None)
            if nprof == 0:
                # upstream: hmmsearch stops with a non-zero status on an HMM file without profiles (a taxon whose
                # file is not shipped, or the QIIME 2 letter that misses its taxa_dict key, main.py:197,214-215),
                # check_returncode() raises and the CLI exits 1 (SeqSample.py:211-225) -- never an empty output
                raise subprocess.CalledProcessError(
                    1, ["itsx_search", "--domtblout", self.dom_file, "-T", "10", "--F1", "1e-6", "--F2", "1e-6",
                        "--F3", "1e-6", hmmfile, str(self.rep_file)],
                    stderr=("Error: no profile in HMM file %s (no profile matches the requested --taxa / --region, "
                            "or the taxon's file is missing from ITSx_db/HMMs)" % hmmfile).encode("utf-8"))
            s = self._session
            resident = (s is not None and s.derep_gen == _GENERATION and
                        os.path.abspath(self.rep_file) in _SESSIONS and _SESSIONS[os.path.abspath(self.rep_file)] is s)
            # Which profiles mark the left and which the right boundary is ItsPosition's business (it is told the region);
            # but a runtime HMM file holds exactly the two name prefixes of its region (main.py:200-208: ITS2 3_/4_,
            # ITS1 1_/2_, ALL 1_/4_), so they are read off the profile names here.  Knowing the sides during the search
            # is what lets a large sample run in the compact row mode (itsx_search_params.keep_rows); a file with any
            # other mix of prefixes is searched with every row kept and the sides set later.
            pre = sorted({nm[:2] for nm in ctx.names})
            sides_known = len(pre) == 2 and all(len(q) == 2 and q[0] in "1234" and q[1] == "_" for q in pre)
            prm = _lib.default_params()
            if resident:
                n_est = s.n_reads if s.streamed else s.batch.n
                nseq = s.n_unique
            else:
                seq_ids, seq, off = _read_fasta(self.rep_file)
                n_est = nseq = len(seq_ids)
            want_table = not getattr(s, "streamed", False) and (not resident or self._want_files(n_est))
            if sides_known:
                ctx.set_sides_by_prefix(pre[0], pre[1])
                prm.keep_rows = 1 if want_table else int(os.environ.get("ITSX_KEEP_ROWS", "0"))
            else:
                ctx.set_sides(np.full(len(ctx.names), -1, np.int8))
                prm.keep_rows = 1
            if resident:
                # representatives are already on the device, in first-occurrence order
                ctx.search(prm)
                seq_ids = None
            else:
                s = _Session()
                ctx.search_seqs(seq, off, prm)
                self._session = s
            s.sides_prefix = (pre[0], pre[1]) if sides_known else None
            _GENERATION += 1
            s.search_gen = _GENERATION
            if resident:
                s.derep_gen = _GENERATION
            s.names, s.nseq = list(ctx.names), nseq
            # a search that was not fed from a resident derep session (rep.fa written by vsearch --cluster_size, or
            # by another process) has no device-side hand-off to ItsPosition / Dedup: its table is always written
            if want_table:
                if seq_ids is None:
                    ids = s.ids
                    seq_ids = [ids[i] for i in s.first.tolist()]
                s.seq_ids = seq_ids
                rows = ctx.hits()
                M = [ctx.profile_M(p) for p in range(len(ctx.names))]
                with open(self.dom_file, "wb") as f:
                    f.write(host.write_domtbl(rows, seq_ids, ctx.names, M, nseq, ctx.nreported()))
                nrows = len(rows)
            else:
                s.files = False
                logging.info("domtbl.txt is a one-line placeholder for this sample (%d sequences > %d); ItsPosition "
                             "takes the positions from the GPU session. Use --keeptemp or ITSX_TEMP_FILES=always for "
                             "the full table." % (nseq, TEMP_FILE_AUTO_MAX_READS))
                with open(self.dom_file, "w") as f:
                    f.write(_PLACEHOLDER)
                nrows = ctx.search_stats().n_domains_reported
            st = ctx.search_stats()
            logging.info("GPU hmmsearch: %d sequences x %d profiles, %d domain rows, %.1f ms on device" %
                         (nseq, len(ctx.names), nrows, st.ms_total))
            _SESSIONS[os.path.abspath(self.dom_file)] = s
        except FileNotFoundError as f:
            logging.error("A file needed by the profile search was not found: %s" % f)
            raise f
        except Exception as e:
            logging.exception("Could not perform ITS identification on the GPU.")
            raise e


class SeqSampleNotPaired(SeqSample):
    """Single-end (or already merged) reads (reference SeqSample.py:228-241)."""

    def __init__(self, fastq, tempdir):
        SeqSample.__init__(self, fastq, tempdir)
        self.seq_file = self.fastq
        self.r1 = self.fastq
        self.fastq2 = None


class SeqSamplePairedNotInterleaved(SeqSample):
    """Paired reads in two files (reference SeqSample.py:244-365)."""

    def __init__(self, fastq, tempdir, fastq2, reversed_primers=False):
        SeqSample.__init__(self, fastq, tempdir)
        if reversed_primers:
            self.r1, self.fastq2 = fastq2, fastq
        else:
            self.r1, self.fastq2 = fastq, fastq2

    def _merge_reads(self, threads, stagger):
        """Merge the read pairs on the GPU and write ``<tempdir>/seq.fq`` (replaces the
        `vsearch --fastq_mergepairs R1 --reverse R2 --fastqout seq.fq --fastq_maxdiffs 40 --fastq_maxee 2
        [--fastq_allowmergestagger] --fastq_qmax 93` process of SeqSample.py:266-365; ``itsx_merge_pairs``,
        csrc/merge.cu).  Records keep R1's title and follow input order, as vsearch writes them.  ``threads`` is
        accepted for the reference's signature.  Inputs may be plain, .gz or .zst (vsearch reads .gz itself; the
        reference unpacks .zst first, :287-306).

        Raises ``subprocess.CalledProcessError`` where the vsearch process would have exited non-zero (files with
        different record counts, a quality value above --fastq_qmax, malformed FASTQ) and ``FileNotFoundError``
        for a missing input, after logging, like the reference (:351-365)."""
        seq_file = os.path.join(self.tempdir, "seq.fq")
        if not os.path.exists(self.tempdir):
            logging.info("Expected %s to exist, but it does not. Creating it now." % self.tempdir)
            os.makedirs(self.tempdir)
        if self.r1 is None or self.fastq2 is None:
            raise ValueError("Both r1 and fastq2 paths must be defined to merge reads.")
        argv = ["itsx_merge_pairs", self.r1, "--reverse", self.fastq2, "--fastqout", seq_file, "--fastq_maxdiffs",
                str(maxmismatches), "--fastq_maxee", str(2), "--threads", str(threads)]
        if stagger:
            argv.append("--fastq_allowmergestagger")
        argv += ["--fastq_qmax", str(vsearch_fastq_qmax)]
        self.seq_file = seq_file
        try:
            try:
                b1, b2 = fq.read_fastq_many([self.r1, self.fastq2])
                if b1.n != b2.n:
                    raise ValueError("More %s reads than %s reads" % (("forward", "reverse") if b1.n > b2.n
                                                                      else ("reverse", "forward")))
                fseq, foff = b1.seq_concat()
                fqual, _ = b1.qual_concat()
                rseq, roff = b2.seq_concat()
                rqual, _ = b2.qual_concat()
                prm = _lib.merge_params(allow_stagger=stagger, maxdiffs=maxmismatches, maxee=2.0,
                                        qmax=vsearch_fastq_qmax)
                ctx = get_context()
                mlen, reason, idx, out_off, out_seq, out_qual = ctx.merge_pairs(fseq, fqual, foff, rseq, rqual, roff,
                                                                               prm)
            except FileNotFoundError:
                raise
            except (ValueError, _lib.ItsxError) as e:
                raise subprocess.CalledProcessError(1, argv, stderr=str(e).encode("utf-8")) from e
            data = fq.format_gathered(b1, idx, out_off, out_seq, out_qual, as_array=True)
            with open(seq_file, "wb") as f:
                f.write(data)
            # deduplicate() takes the merged records from here instead of reading seq.fq back and scanning it again
            self._merged = (os.path.abspath(seq_file), fq.batch_of_gathered(data, b1, idx, out_off), out_seq, out_off,
                            idx, (os.path.abspath(self.r1), os.path.abspath(self.fastq2)), (b1, b2))
            st = ctx.merge_stats()
            why = ", ".join("%s %d" % (_lib.MERGE_REASONS[r], st.by_reason[r])
                            for r in range(1, len(_lib.MERGE_REASONS)) if st.by_reason[r])
            logging.info("Merged %d of %d pairs on the GPU (%.2f ms)%s" % (st.n_merged, st.n_pairs, st.ms_kernel,
                                                                         "; not merged: " + why if why else ""))
        except subprocess.CalledProcessError as e:
            logging.exception("Could not perform read merging. Error was: \n  {}".format(e.stderr.decode("utf-8")))
            raise e
        except FileNotFoundError as f:
            logging.error("Could not perform read merging: %s" % f)
            raise f


def _read_fasta(path):
    """(labels, bases uint8, off int64) of a FASTA file (the `rep.fa` hmmsearch would be given)."""
    labels, parts = [], []
    cur = None
    with open(path, "rb") as f:
        for line in f:
            line = line.rstrip()
            if line.startswith(b">"):
                sp = line[1:].split(None, 1)
                labels.append(sp[0].decode("ascii", "replace") if sp else "")
                cur = []
                parts.append(cur)
            elif cur is not None and line:
                cur.append(line)
    seqs = [b"".join(p) for p in parts]
    off = np.zeros(len(seqs) + 1, np.int64)
    off[1:] = np.cumsum([len(x) for x in seqs])
    return labels, np.frombuffer(b"".join(seqs), np.uint8), off


class ItsPosition:
    """ITS boundary positions per representative sequence (reference SeqSample.py:368-498).

    ``ddict`` has the reference's shape ``{seq: {"left": {score, from_pos, to_pos}, "right": {...}, "tlen": n}}``.
    When ``domtable`` was written by a live GPU search the per-sequence winners are taken straight from the
    device (``itsx_positions``: arg-max of the printed 0.1-bit score per side, first row wins ties) and
    ``ddict`` is only materialised if somebody looks at it.
    """

    def __init__(self, domtable, region):
        self.domtable = domtable
        self._ddict = None
        if region in REGION_PREFIXES:
            self.leftprefix, self.rightprefix = REGION_PREFIXES[region]
        self.region = region
        self._dev = None              # dict of int32 arrays from itsx_positions, per searched sequence
        self._session = None
        s = _SESSIONS.get(os.path.abspath(domtable)) if isinstance(domtable, str) else None
        if s is not None and s.search_gen == _GENERATION and hasattr(self, "leftprefix"):
            ctx = get_context()
            if getattr(s, "sides_prefix", None) != (self.leftprefix, self.rightprefix):
                # the search ran without (or with other) sides: apply this region's and redo the selection
                ctx.set_sides_by_prefix(self.leftprefix, self.rightprefix)
                ctx.search_stage2()
                s.sides_prefix = (self.leftprefix, self.rightprefix)
            self._dev = ctx.positions(s.nseq)
            self._session = s
        else:
            self.parse()

    @property
    def ddict(self):
        if self._ddict is None:
            self._ddict = {}
            self.parse()
        return self._ddict

    @ddict.setter
    def ddict(self, value):
        self._ddict = value

    def _score(self, sequence, stype, score, from_pos, to_pos, tlen):
        """Keep the highest score per side; strict '>' so the first row wins ties (SeqSample.py:400-429)."""
        entry = self._ddict[sequence]
        best = entry.get(stype)
        if best is None:
            entry[stype] = {"score": score, "to_pos": to_pos, "from_pos": from_pos}
            entry["tlen"] = tlen
        elif score > best["score"]:
            best["score"], best["to_pos"], best["from_pos"] = score, to_pos, from_pos

    def parse(self):
        """Read the domain table: columns 0 (target), 2 (tlen), 3 (profile), 13 (domain score), 19/20
        (env from/to) -- SeqSample.py:431-461."""
        if self._ddict is None:
            self._ddict = {}
        try:
            with open(self.domtable, "r") as f:
                for line in f:
                    if line.startswith("#"):
                        continue
                    ll = line.split()
                    sequence, hmmprofile = ll[0], ll[3]
                    score, from_pos, to_pos, tlen = float(ll[13]), int(ll[19]), int(ll[20]), int(ll[2])
                    if sequence not in self._ddict:
                        self._ddict[sequence] = {}
                    if hmmprofile.startswith(self.leftprefix):
                        self._score(sequence, "left", score, from_pos, to_pos, tlen)
                    elif hmmprofile.startswith(self.rightprefix):
                        self._score(sequence, "right", score, from_pos, to_pos, tlen)
        except Exception as e:
            logging.error("Exception occurred when parsing HMMSearch results")
            raise e

    def get_position(self, sequence):
        """(start, stop, tlen): start = left.to_pos, stop = right.from_pos - 1, 0-based; None when a side is
        missing; KeyError when the sequence has no row at all (SeqSample.py:463-498)."""
        try:
            entry = self.ddict[sequence]
            start = int(entry["left"]["to_pos"]) if "left" in entry else None
            stop = int(entry["right"]["from_pos"]) - 1 if "right" in entry else None
            tlen = int(entry["tlen"]) if "tlen" in entry else None
            return (start, stop, tlen)
        except KeyError:
            logging.debug("No ITS stop or start sites were identified for sequence {}, skipping.".format(sequence))
            raise KeyError


class Dedup:
    """Read -> representative map plus the trim / re-expansion step (reference SeqSample.py:501-949)."""

    def __init__(self, uc_file, rep_file, seq_file, fastq=None, fastq2=None):
        self._matchdict = None
        self._matchdict_set = False
        self.uc_file = uc_file
        self.rep_file = rep_file
        self.seq_file = seq_file
        self.fastq = fastq
        self.fastq2 = fastq2
        s = _SESSIONS.get(os.path.abspath(uc_file)) if isinstance(uc_file, str) else None
        self._session = s if (s is not None and s.rep is not None) else None
        if self._session is None:
            self.parse()
            if not self._matchdict and _is_placeholder(uc_file):
                logging.warning("uc file %s is a placeholder (large sample, temp files not materialised)" % uc_file)

    @property
    def matchdict(self):
        if self._matchdict is None and not self._matchdict_set:
            self.parse()
        return self._matchdict

    @matchdict.setter
    def matchdict(self, value):
        self._matchdict = value
        self._matchdict_set = True
        self._session = None          # a hand-made map overrides the session's arrays

    def parse(self):
        """uc.txt: 'S' rows map a read to itself, 'H' rows to column 10; 'C' rows and the strand column are
        ignored (SeqSample.py:542-562)."""
        try:
            md = {}
            with open(self.uc_file, "r") as f:
                for line in f:
                    ll = line.split()
                    if ll[0] == "S":
                        md[ll[8]] = ll[8]
                    elif ll[0] == "H":
                        md[ll[8]] = ll[9]
            self._matchdict = md
        except Exception as e:
            logging.exception("Could not parse the Vsearch '.uc' file.")
            raise e

    # ---- record-at-a-time API (duck-typed itspos; what the reference's unit tests drive) ---------------------
    def _position_of(self, rec_id, itspos):
        """(start, stop, tlen) of a read's representative, or None when the read must be dropped."""
        md = self.matchdict
        if md is None or rec_id not in md:
            return None
        try:
            start, stop, tlen = itspos.get_position(md[rec_id])
        except KeyError:
            return None
        if start is None or stop is None or not start < stop:
            return None
        return start, stop, tlen

    @staticmethod
    def _stitch(record):
        q = record.letter_annotations.get("phred_quality")
        quals = [93] * len(CCS_FWD) + (list(q) if q is not None else [93] * len(record)) + [93] * len(CCS_REV)
        return fq.Record(CCS_FWD.decode() + str(record.seq) + CCS_REV.decode(), id=record.id, name=record.name,
                         description=record.description, quals=quals)

    @staticmethod
    def _report_empty(records, label=""):
        empty = [r.id for r in records if str(r.seq) == ""]
        if empty:
            print("Total number of sequences that are empty%s: " % label, len(empty))
            print("Sequence IDs: ")
            print(empty)

    def _get_trimmed_seq_generator(self, seqgen, itspos, wri_file, trim_ccs=False):
        """Generator of trimmed records in input order; reads without both boundaries (or with
        start >= stop) are skipped; start == 0 is a valid coordinate (SeqSample.py:792-884)."""
        if self.matchdict is None:
            raise ValueError("matchdict must be parsed before calling sequence generators.")

        def trimmed():
            for record in seqgen:
                pos = self._position_of(record.id, itspos)
                if pos is None:
                    continue
                out = record[pos[0]:pos[1]]
                yield self._stitch(out) if trim_ccs else out

        if wri_file:
            return trimmed()
        done = list(trimmed())
        self._report_empty(done)
        return iter(done)

    def _get_paired_seq_generator(self, zipseqgen, itspos, wri_file, trim_ccs=False):
        """Two generators (forward, reverse) of trimmed records; R1 -> [start:stop] (or [start:] when
        stop > tlen), R2 -> [tlen-stop : tlen-start] (SeqSample.py:564-711)."""
        if self.matchdict is None:
            raise ValueError("matchdict must be parsed before calling sequence generators.")

        def pairs():
            for rec1, rec2 in zipseqgen:
                pos = self._position_of(rec1.id, itspos)
                if pos is None:
                    continue
                start, stop, tlen = pos
                if tlen is None:
                    raise ValueError("Could not retrieve valid positions for sequence %s" % rec1.id)
                r2start, r2end = tlen - stop, tlen - start
                a = rec1[start:] if stop > tlen else rec1[start:stop]
                b = rec2[r2start:] if r2end > tlen else rec2[r2start:r2end]
                if trim_ccs:
                    a, b = self._stitch(a), self._stitch(b)
                yield a, b

        if wri_file:
            from itertools import tee
            g1, g2 = tee(pairs(), 2)
            return (a for a, _ in g1), (b for _, b in g2)
        done = list(pairs())
        self._report_empty([a for a, _ in done], " Split A")
        self._report_empty([b for _, b in done], " Split B")
        return (a for a, _ in done), (b for _, b in done)

    # ---- bulk API: whole files through the GPU ---------------------------------------------------------------------
    def _unique_table(self, batch, ids, itspos):
        """uid[read] (dense unique index or -1) and the (start, stop, tlen) table per unique for the reads of
        ``batch``.  Fast path: arrays of the live session; general path: matchdict + itspos.get_position (any
        duck-typed object), evaluated once per distinct representative."""
        s = self._session
        if (s is not None and isinstance(itspos, ItsPosition) and itspos._dev is not None and
                itspos._session is s and s.batch is not None):
            dev = itspos._dev
            if batch is s.batch:
                uid = s.uid
            elif s.pair_batches is not None and batch is s.pair_batches[0]:
                # R1 of the pairs this sample was merged from: merged record k came from pair pair_index[k] (same id,
                # vsearch keeps R1's title), pairs that did not merge are absent from the map (SeqSample.py:591-598)
                uid = np.full(batch.n, -1, np.int32)
                uid[s.pair_index] = s.uid
            else:
                if ids is None:
                    ids = batch.ids()
                where = {k: i for i, k in enumerate(s.ids)}
                uid = np.fromiter((s.uid[where[k]] if k in where else -1 for k in ids), np.int32, len(ids))
            return uid, dev["start"], dev["stop"], dev["tlen"], s.n_unique
        if s is not None and not s.files and not self._matchdict_set:
            raise RuntimeError("the temp files of this sample were not materialised and the GPU session that holds "
                               "its arrays is no longer live; rerun with --keeptemp or ITSX_TEMP_FILES=always")
        if ids is None:
            ids = batch.ids()
        md = self.matchdict or {}
        index, start, stop, tlen = {}, [], [], []
        uid = np.full(len(ids), -1, np.int32)
        for i, rid in enumerate(ids):
            repid = md.get(rid)
            if repid is None:
                continue
            u = index.get(repid)
            if u is None:
                u = index[repid] = len(start)
                try:
                    a, b, c = itspos.get_position(repid)
                except KeyError:
                    a = b = c = None
                start.append(-1 if a is None else a)
                stop.append(-1 if b is None else b)
                tlen.append(-1 if c is None else c)
            uid[i] = u
        return (uid, np.asarray(start, np.int32), np.asarray(stop, np.int32), np.asarray(tlen, np.int32),
                len(start))

    def _trim_file(self, batch, ids, itspos, mode, trim_ccs, table=None):
        """FASTQ text of ``batch`` trimmed on the GPU (mode 0 single, 2 paired R1, 1 paired R2)."""
        global _GENERATION
        uid, start, stop, tlen, nu = table if table is not None else self._unique_table(batch, ids, itspos)
        if mode != 0 and np.any((tlen < 0) & (start >= 0) & (stop >= 0) & (start < stop)):
            raise ValueError("Could not retrieve valid positions for a kept sequence (tlen is missing)")
        ctx = get_context()
        seq, off = batch.seq_concat()
        qual, _ = batch.qual_concat()
        ctx.trim_set_map(uid, nu)
        ctx.positions_set(start, stop, tlen)
        _GENERATION += 1                      # the context no longer holds any session's derep map
        ki, oo, os_, oq = ctx.trim_gather(batch.n, mode=mode, seq=seq, qual=qual, off=off)
        pre = (CCS_FWD, b"~" * len(CCS_FWD)) if trim_ccs else None
        suf = (CCS_REV, b"~" * len(CCS_REV)) if trim_ccs else None
        n_empty = int(np.count_nonzero(np.diff(oo) == 0))
        return fq.format_gathered(batch, ki, oo, os_, oq, prefix=pre, suffix=suf, as_array=True), ki, n_empty

    def create_trimmed_seqs(self, outfile, gzipped, zstd_file, itspos, wri_file, tempdir, trim_ccs=False):
        """Write the reads of ``seq_file`` trimmed to the selected region, input order, plain / gz / zst
        (SeqSample.py:886-949)."""
        ss = self._session
        if (ss is not None and ss.streamed and os.path.abspath(self.seq_file) == ss.seq_path and
                isinstance(itspos, ItsPosition) and itspos._session is ss and not trim_ccs):
            return self._create_trimmed_seqs_streamed(outfile, gzipped, zstd_file, wri_file)
        if self._session is not None and self._session.batch is not None and \
                os.path.abspath(self.seq_file) == self._session.seq_path:
            batch, ids = self._session.batch, None
        else:
            batch, ids = fq.read_fastq(self.seq_file), None
        text, ki, n_empty = self._trim_file(batch, ids, itspos, 0, trim_ccs)
        if not wri_file:
            if n_empty and not trim_ccs:
                print("Total number of sequences that are empty: ", n_empty)
            return
        fq.write_compressed(outfile, text, gzipped=gzipped, zstd_file=zstd_file, n_records=len(ki))

    def _create_trimmed_seqs_streamed(self, outfile, gzipped, zstd_file, wri_file):
        """create_trimmed_seqs for a streamed session: the input is read a second time in the same chunks (only the titles
        are needed from it); every chunk's kept slices come back from the device (itsx_trim_gather_range) and are
        appended to the output."""
        ss = self._session
        if ss.derep_gen != _GENERATION:
            raise RuntimeError("the GPU session that holds this streamed sample is no longer live")
        ctx = get_context()
        writer = fq.ChunkWriter(outfile, gzipped=gzipped, zstd_file=zstd_file) if wri_file else None
        first = n_empty = 0
        try:
            for chunk in fq.stream_fastq(self.seq_file, ss.chunk_bytes):
                nb = int(chunk.s_len.sum())
                ki, oo, os_, oq = ctx.trim_gather_range(first, chunk.n, nb)
                n_empty += int(np.count_nonzero(np.diff(oo) == 0))
                if writer is not None:
                    writer.write(fq.format_gathered(chunk, ki, oo, os_, oq, as_array=True), len(ki))
                first += chunk.n
        finally:
            if writer is not None:
                writer.close()
        if first != ss.n_reads:
            raise RuntimeError("the input changed between the two passes over %s" % self.seq_file)
        if not wri_file and n_empty:
            print("Total number of sequences that are empty: ", n_empty)

    def create_paired_trimmed_seqs(self, outfile1, outfile2, gzipped, zstd_file, itspos, wri_file, trim_ccs=False):
        """Write R1 and R2 trimmed but unmerged (for DADA2), input order (SeqSample.py:713-790)."""
        if self.fastq is None or self.fastq2 is None:
            raise ValueError("Both fastq and fastq2 paths must be defined to create paired trimmed sequences.")
        f1, f2 = self.fastq, self.fastq2
        plain = (".fastq", ".fq")
        if not ((f1.endswith(".gz") and f2.endswith(".gz")) or (f1.endswith(".zst") and f2.endswith(".zst")) or
                (f1.endswith(plain) and f2.endswith(plain))):
            raise ValueError("Fastq and Fastq2 files should both be gzipped (.gz), zstd compressed (.zst) or both "
                             "be uncompressed. Mixed input is not accepted.")
        ps = self._session
        if ps is not None and ps.pair_batches is not None and ps.pair_files == (os.path.abspath(f1), os.path.abspath(f2)):
            b1, b2 = ps.pair_batches            # parsed by _merge_reads a moment ago; equal record counts
            ids1 = None                         # ... and the read -> unique map follows from the merge itself
        else:
            b1, b2 = fq.read_fastq_many([f1, f2])
            n = min(b1.n, b2.n)                 # zip() semantics
            if b1.n != n:
                b1 = _head(b1, n)
            if b2.n != n:
                b2 = _head(b2, n)
            ids1 = b1.ids()                     # the filter is keyed on R1's id (SeqSample.py:591)
        table = self._unique_table(b1, ids1, itspos)                    # both files are keyed on R1's ids
        t1, k1, e1 = self._trim_file(b1, ids1, itspos, 2, trim_ccs, table)
        t2, k2, e2 = self._trim_file(b2, ids1, itspos, 1, trim_ccs, table)
        if not wri_file:
            if (e1 or e2) and not trim_ccs:
                print("Total number of sequences that are empty Split A: ", e1)
                print("Total number of sequences that are empty Split B: ", e2)
            return
        fq.write_compressed(outfile1, t1, gzipped=gzipped, zstd_file=zstd_file, n_records=len(k1))
        fq.write_compressed(outfile2, t2, gzipped=gzipped, zstd_file=zstd_file, n_records=len(k2))


def _is_placeholder(path):
    try:
        with open(path) as f:
            return f.readline().startswith("# itsxpress-b200: not materialised")
    except Exception:
        return False


def _head(batch, n):
    return fq.FastqBatch(batch.buf, batch.t_off[:n], batch.t_len[:n], batch.s_off[:n], batch.s_len[:n],
                         batch.q_off[:n])


def reset_sessions():
    """Forget every live session (tests; long-running drivers between samples)."""
    _SESSIONS.clear()


__all__ = ["SeqSample", "SeqSampleNotPaired", "SeqSamplePairedNotInterleaved", "ItsPosition", "Dedup",
           "get_context", "reset_sessions", "shutil"]
