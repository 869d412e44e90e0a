#!/usr/bin/env python
"""``itsxpress`` command line -- same flags, defaults, log lines, output-suffix rules and exit status as the
reference's itsxpress/main.py (parser :74-170, workflow :486-654), driving the B200 path in SeqSample.py.

Stage order is the reference's: [merge pairs] -> dereplicate -> build the runtime profile set -> search ->
ItsPosition -> Dedup -> write trimmed reads -> count reads.  Pair merging runs on the GPU as well
(SeqSample._merge_reads -> itsx_merge_pairs), and so does clustering at --cluster_id < 1 (SeqSample.cluster ->
itsx_cluster: the exact derep's classes clustered greedily, DESIGN.md section 6; ITSX_CLUSTER=vsearch runs vsearch
--cluster_size instead).  --trim-ccs orientation still needs vsearch and fails the way the reference fails when vsearch
is absent.
"""
import argparse
import contextlib
import gzip
import logging
import math
import os
import shutil
import sys
import tempfile
import time

from . import __version__
from . import fastq as fq
from .definitions import ROOT_DIR, REGION_PREFIXES, taxa_choices, taxa_dict
from .SeqSample import Dedup, ItsPosition, SeqSampleNotPaired, SeqSamplePairedNotInterleaved


def restricted_float(x):
    x = float(x)
    if not 0.99 <= x <= 1.0:
        raise argparse.ArgumentTypeError("%r not in range [0.99, 1.0]" % (x,))
    return x


# (flags, keyword arguments) of every option, in the reference's order (main.py:82-169)
_OPTIONS = (
    (("--fastq", "-f"), dict(type=str, required=True,
                             help="A .fastq, .fq, .fastq.gz or .fq.gz file. Interleaved or not.")),
    (("--single_end", "-s"), dict(action="store_true", default=False,
                                  help="A flag to specify that the FASTQ file is single-ended (not paired). "
                                       "Default is false.")),
    (("--fastq2", "-f2"), dict(type=str, default=None,
                               help="A .fastq, .fq, .fastq.gz or .fq.gz file. representing read 2 (optional)")),
    (("--outfile", "-o"), dict(type=str, required=True,
                               help="the trimmed Fastq file, if it ends in 'gz' it will be gzipped")),
    (("--outfile2", "-o2"), dict(type=str, default=None,
                                 help="the trimmed read 2 Fastq file, if it ends in 'gz' it will be gzipped. If "
                                      "provided, reads will be returned unmerged.")),
    (("--tempdir",), dict(default=None, help="The temp file directory")),
    (("--allow_staggered_reads",), dict(default=True,
                                        help="Allow merging of staggered reads with --fastq_allowmergestagger for "
                                             "Vsearch --fastq_mergepairs. See Vsearch documentation. (Optional) "
                                             "Default is true.")),
    (("--keeptemp",), dict(action="store_true", help="Should intermediate files be kept?")),
    (("--region",), dict(choices=["ITS2", "ITS1", "ALL"], required=True, help="")),
    (("--taxa",), dict(choices=taxa_choices, default="Fungi", help="The taxonomic group sequenced.")),
    (("--cluster_id",), dict(type=restricted_float, default=1.0,
                             help="The percent identity for clustering reads range [0.99-1.0], set to 1 for exact "
                                  "dereplication.")),
    (("--reversed_primers", "-rp"), dict(action="store_true",
                                         help="Primers are in reverse orientation as in Taylor et al. 2016, "
                                              "DOI:10.1128/AEM.02576-16. If selected ITSxpress returns trimmed "
                                              "reads flipped to the forward orientation")),
    (("--trim-ccs",), dict(dest="trim_ccs", action="store_true", default=False,
                           help="Stitch fake forward and reverse complement of fake reverse primer for DADA2 "
                                "denoise-ccs on PacBio reads.")),
    (("--log",), dict(default="ITSxpress.log", help="Log file")),
    (("--threads",), dict(type=int, default=1, help="Number of processor threads to use.")),
)


def myparser():
    parser = argparse.ArgumentParser(
        description="ITSxpress: A python module to rapidly trim ITS amplicon sequences from Fastq files.")
    for flags, kw in _OPTIONS:
        parser.add_argument(*flags, **kw)
    parser.add_argument("--version", "-v", action="version", version="ITSxpress version: " + __version__)
    return parser


_RUNTIME_HMM_CACHE = {}


def create_runtime_hmm(taxa, region, tempdir):
    """Write ``<tempdir>/runtime_selected.hmm`` holding only the profiles whose NAME starts with the region's
    two prefixes, taken from the taxon's file (or every taxon file in ``taxa_dict`` order for "All"); missing
    files are skipped silently -- reference main.py:176-231."""
    hmm_dir = os.path.join(ROOT_DIR, "ITSx_db", "HMMs")
    if taxa in ("All", "all.hmm"):
        files = [f for t, f in taxa_dict.items() if t != "All" and f != "all.hmm"]
    else:
        files = [taxa_dict.get(taxa, taxa)]
    prefixes = REGION_PREFIXES.get(region, ("1_", "2_", "3_", "4_"))
    target = os.path.join(tempdir, "runtime_selected.hmm")
    # a multi-sample driver asks for the same selection once per sample (q2_itsxpress.py:273-296): the text is kept,
    # keyed by the files it came from (path, size, mtime)
    present = [os.path.join(hmm_dir, name) for name in files if os.path.exists(os.path.join(hmm_dir, name))]
    key = (tuple(prefixes), tuple((p, os.path.getsize(p), os.stat(p).st_mtime_ns) for p in present))
    text = _RUNTIME_HMM_CACHE.get(key)
    if text is None:
        parts = []
        for path in present:
            with open(path, "r") as src:
                block, wanted = [], False
                for line in src:
                    block.append(line)
                    if line.startswith("NAME  ") and line[6:].strip().startswith(prefixes):
                        wanted = True
                    if line.strip() == "//":
                        if wanted:
                            parts.extend(block)
                        block, wanted = [], False
        text = "".join(parts)
        _RUNTIME_HMM_CACHE.clear()              # one selection at a time is all a run uses
        _RUNTIME_HMM_CACHE[key] = text
    with open(target, "w") as out:
        out.write(text)
    return target


def _is_paired(fastq, fastq2, single_end):
    if fastq and fastq2:
        return True
    if single_end:
        return False
    if fastq and not fastq2:
        logging.info("Only one fastq file provided. Assuming single-end.")
        return False
    logging.error("ITSxpress requires either a single-end file or two paired-end files. If this is a single-end "
                  "file, please use the --single_end flag.")
    raise AssertionError


def _logger_setup(logfile):
    try:
        logging.basicConfig(level=logging.DEBUG, format="%(asctime)s %(name)-12s %(levelname)-8s %(message)s",
                            datefmt="%m-%d %H:%M", filename=logfile, filemode="w")
        root = logging.getLogger("")
        if not any(getattr(h, "_itsxpress_console", False) for h in root.handlers):
            # (one console handler per process: main() may run several times in one -- tests, the bench, drivers)
            console = logging.StreamHandler()
            console.setLevel(logging.INFO)
            console.setFormatter(logging.Formatter("%(asctime)s: %(levelname)-8s %(message)s"))
            console._itsxpress_console = True
            root.addHandler(console)
    except Exception as e:
        print("An error occurred setting up logging")
        raise e


@contextlib.contextmanager
def read_file(filename, mode="r"):
    """Open a plain, .gz or .zst file as text (main.py:295-330)."""
    handle = None
    try:
        if filename.endswith(".gz"):
            handle = gzip.open(filename, mode + "t")
        elif filename.endswith(".zst"):
            import io
            from . import _zstd
            with open(filename, "rb") as f:
                handle = io.StringIO(_zstd.decompress(f.read()).decode())
        else:
            handle = open(filename, mode)
        yield handle
    except FileNotFoundError as f:
        logging.error("The input file {} could not be found.".format(filename))
        raise f
    except Exception as g:
        logging.error("There appears to be an issue reading the input file {}.".format(filename))
        raise g
    finally:
        if handle is not None:
            handle.close()


def _names_look_paired(id1, id2):
    """BBTools' test for 'these two consecutive records are mates' (main.py:346-386)."""
    if len(id1) != len(id2):
        return False
    s1, s2 = id1.find(" "), id2.find(" ")
    if s1 == s2 and s1 > 0 and len(id1) >= s1 + 3:
        if id1[s1 + 1:s1 + 3] == "1:" and id2[s2 + 1:s2 + 3] == "2:":
            return id1[:s1] == id2[:s1]
    l1, l2 = id1.rfind("/"), id2.rfind("/")
    if l1 == l2 and l1 > 0 and len(id1) >= l1 + 2:
        if id1[l1 + 1] == "1" and id2[l2 + 1] == "2":
            return id1[:l1] == id2[:l1] and id1[l1 + 2:] == id2[l2 + 2:]
    return id1 == id2


def _check_fastqs(fastq, fastq2=None):
    """Validate the first records of the input(s) (ValueError on malformed FASTQ) and warn when a file looks
    interleaved (main.py:333-414)."""
    for path in (fastq, fastq2):
        if not path:
            continue
        if path.endswith(".zst"):
            # only the first frame's first block is decoded (read_file would inflate the whole file for eight lines)
            from . import _zstd
            try:
                text = b""
                with open(path, "rb") as f:
                    for part in _zstd.decompress_stream(f, 1 << 16):
                        text += part
                        if text.count(b"\n") >= 8:
                            break
            except FileNotFoundError as f:
                logging.error("The input file {} could not be found.".format(path))
                raise f
            except Exception as g:
                logging.error("There appears to be an issue reading the input file {}.".format(path))
                raise g
            head = text.decode().splitlines(keepends=True)[:8]
        else:
            with read_file(path) as handle:
                head = []
                for i, line in enumerate(handle):
                    head.append(line)
                    if i >= 7:
                        break
        if not head:
            continue
        if not head[0].startswith("@"):
            raise ValueError("Records in Fastq files should start with '@' character")
        # fewer than 8 lines: the file ends here, so a partial second record is an error (as in Biopython)
        recs = list(fq.iter_records("".join(head).encode()))
        if len(recs) == 2 and _names_look_paired(recs[0].id, recs[1].id):
            logging.warning("The file {} may be interleaved, which is not supported. Please verify your input file "
                            "manually.".format(path))


def _check_total_reads(file, file2=None):
    """Log the number of reads (= every fourth line, main.py:417-438), counted on raw newline bytes."""
    for path in (file, file2):
        if not path:
            continue
        known = fq.cached_count(path)      # a file this run has just scanned or written (size + mtime unchanged)
        if known is not None:
            logging.info("Total number of reads in file {} is {}.".format(path, known))
            continue
        try:
            if path.endswith(".gz"):
                fh = gzip.open(path, "rb")
            elif path.endswith(".zst"):
                import io
                from . import _zstd
                with open(path, "rb") as f:
                    fh = io.BytesIO(_zstd.decompress(f.read()))
            else:
                fh = open(path, "rb")
        except FileNotFoundError as f:
            logging.error("The input file {} could not be found.".format(path))
            raise f
        lines, last = 0, b"\n"
        with fh:
            while True:
                chunk = fh.read(1 << 24)
                if not chunk:
                    break
                lines += chunk.count(b"\n")
                last = chunk[-1:]
        if last != b"\n":
            lines += 1
        logging.info("Total number of reads in file {} is {}.".format(path, (lines + 3) // 4))


def create_temp_directory(tempdir_arg=None):
    """mkdtemp(prefix='itsxpress_') under the user's directory or the default location; None on failure."""
    try:
        if tempdir_arg:
            if os.path.isfile(tempdir_arg):
                logging.error(f"A file with the same name '{tempdir_arg}' already exists. Cannot create directory.")
                return None
            if not os.path.exists(tempdir_arg):
                os.makedirs(tempdir_arg)
                logging.info(f"Directory '{tempdir_arg}' has been created.")
            else:
                logging.info(f"Directory '{tempdir_arg}' already exists.")
            temp_dir = tempfile.mkdtemp(prefix="itsxpress_", dir=tempdir_arg)
            logging.info(f"Temporary directory '{temp_dir}' has been created at the user-defined location.")
        else:
            temp_dir = tempfile.mkdtemp(prefix="itsxpress_")
            logging.info(f"Temporary directory '{temp_dir}' has been created at the default location.")
        return temp_dir
    except Exception as e:
        logging.error(f"Failed to create temporary directory: {e}")
        return None


def _suffix_flags(*paths):
    """(gzipped, zstd_file) from the LAST suffix of every output; mixed suffixes -> plain (main.py:556-624)."""
    last = {p.split(".")[-1] for p in paths}
    if last == {"gz"}:
        return True, False
    if last == {"zst"}:
        return False, True
    return False, False


def main(args=None):
    t0 = time.time()
    parser = myparser()
    if not args:
        args = parser.parse_args()
    _logger_setup(args.log)
    session_tempdir = None
    try:
        if args.trim_ccs:
            args.single_end = True
        logging.info("Starting ITSxpress version  {}".format(__version__))
        logging.info("Verifying the input sequences.")
        _check_fastqs(args.fastq, args.fastq2)
        paired_end = _is_paired(args.fastq, args.fastq2, args.single_end)
        session_tempdir = create_temp_directory(tempdir_arg=args.tempdir)
        if session_tempdir is None:
            raise ValueError("Failed to create temporary directory")
        if paired_end:
            logging.info("Sequences are paired-end in two files. They will be merged on the GPU (vsearch --fastq_mergepairs semantics).")
            sobj = SeqSamplePairedNotInterleaved(fastq=args.fastq, fastq2=args.fastq2, tempdir=session_tempdir,
                                                 reversed_primers=args.reversed_primers)
            sobj._merge_reads(threads=str(args.threads), stagger=args.allow_staggered_reads)
        else:
            logging.info("Sequences are assumed to be single-end.")
            sobj = SeqSampleNotPaired(fastq=args.fastq, tempdir=session_tempdir)
        if args.keeptemp:
            sobj.materialize = True        # --keeptemp: leave complete uc.txt / rep.fa / domtbl.txt behind
        if args.trim_ccs:
            logging.info("Orients PacBio reads using Vsearch --orient against the universal reference database.")
            sobj.orient_reads(threads=str(args.threads))
        logging.info("Unique sequences are being written to a temporary FASTA file (GPU dereplication).")
        if math.isclose(args.cluster_id, 1, rel_tol=1e-05):
            sobj.deduplicate(threads=str(args.threads))
        else:
            sobj.cluster(threads=str(args.threads), cluster_id=args.cluster_id)
        logging.info("Searching for ITS start and stop sites with the GPU profile-HMM cascade.")
        hmmfile = create_runtime_hmm(args.taxa, args.region, session_tempdir)
        sobj._search(hmmfile=hmmfile, threads=str(args.threads))
        logging.info("Parsing HMM results.")
        its_pos = ItsPosition(domtable=sobj.dom_file, region=args.region)
        dedup_obj = Dedup(uc_file=sobj.uc_file, rep_file=sobj.rep_file, seq_file=sobj.seq_file, fastq=sobj.r1,
                          fastq2=sobj.fastq2)
        if args.outfile2:
            gz, zs = _suffix_flags(args.outfile, args.outfile2)
            dedup_obj.create_paired_trimmed_seqs(args.outfile, args.outfile2, gzipped=gz, zstd_file=zs,
                                                 itspos=its_pos, wri_file=True, trim_ccs=args.trim_ccs)
        else:
            gz, zs = _suffix_flags(args.outfile)
            dedup_obj.create_trimmed_seqs(args.outfile, gzipped=gz, zstd_file=zs, itspos=its_pos, wri_file=True,
                                          tempdir=sobj.tempdir, trim_ccs=args.trim_ccs)
        logging.info("Counting reads after trimming.")
        _check_total_reads(args.fastq, args.fastq2 if args.fastq2 else None)
        _check_total_reads(args.outfile, args.outfile2 if args.outfile2 else None)
        logging.info("ITSxpress ran in {}".format(time.strftime("%H:%M:%S", time.gmtime(time.time() - t0))))
    except Exception as e:
        logging.error("ITSxpress terminated with errors. See the log file for details.")
        logging.error(e)
        raise SystemExit(1)
    finally:
        if session_tempdir is not None and not args.keeptemp:
            shutil.rmtree(session_tempdir, ignore_errors=True)


if __name__ == "__main__":
    main()
