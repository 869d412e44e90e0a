"""Planted clustering workloads and the command-line checks shared by tests/test_gpu_cluster.py (on the device) and
tests/test_cluster_on_oracle.py (CPU reference standing in for it)."""
import os

import numpy as np

from conftest import TD

from itsxpress_b200 import SeqSample
from itsxpress_b200 import fastq as fq
from itsxpress_b200 import main as cli

MERGED = os.path.join(TD, "4774-1-MSITS3_merged.fastq")
COMP = bytes.maketrans(b"ACGT", b"TGCA")


def rc(s):
    return s.translate(COMP)[::-1]


def pack(reads):
    off = np.zeros(len(reads) + 1, np.int64)
    off[1:] = np.cumsum([len(r) for r in reads])
    return np.frombuffer(b"".join(reads), np.uint8).copy(), off


def edit(rng, s, k, where=None):
    """s with k random edits (substitution / insertion / deletion); where = (lo, hi) confines their positions"""
    s = bytearray(s)
    for _ in range(k):
        lo, hi = where if where else (0, len(s))
        p = int(rng.integers(lo, max(lo + 1, min(hi, len(s)))))
        op = int(rng.integers(3))
        if op == 0:
            s[p] = b"ACGT"[(b"ACGT".index(s[p]) + 1 + int(rng.integers(3))) % 4] if s[p] in b"ACGT" else ord("A")
        elif op == 1:
            s.insert(p, b"ACGT"[int(rng.integers(4))])
        elif len(s) > 1:
            del s[p]
    return bytes(s)


def planted(seed, L=250, ntemplates=12, D=1):
    """templates with variants at exactly D and D+1 edits (edits in the first and last segment too), reverse
    complements, lower case / N / IUPAC reads, length changes at the D(L) boundary, chains, and identity ties"""
    rng = np.random.default_rng(seed)
    reads = []
    for t in range(ntemplates):
        T = bytes(rng.choice(list(b"ACGT"), L).tolist())
        reads += [T] * int(rng.integers(1, 6))
        for k in (D, D + 1, D, D + 1):
            reads.append(edit(rng, T, k))
        reads.append(edit(rng, T, D, (0, L // (D + 2))))           # first segment
        reads.append(edit(rng, T, D, (L - L // (D + 2), L)))       # last segment
        reads.append(rc(edit(rng, T, D)))                           # reverse strand
        reads.append(T[:L - D])                                     # length difference D (accepted)
        reads.append(T[:L - D - 1])                                 # length difference D + 1 (rejected)
        reads.append(T + T[:D])                                     # longer by D
        x = bytearray(edit(rng, T, D))
        x[int(rng.integers(L - 1))] = ord("N")
        reads.append(bytes(x).lower())                              # lower case with an N
        y = bytearray(T)
        y[int(rng.integers(L))] = ord("R")
        reads.append(bytes(y))                                      # IUPAC symbol
        a = edit(rng, T, D)                                         # chain T - a - b where only order decides
        reads += [a, edit(rng, a, D)]
        b2 = bytearray(T)                                           # tie: one substitution from two centroids
        p = int(rng.integers(L))
        b2[p] = b"ACGT"[(b"ACGT".index(b2[p]) + 1) % 4]
        reads.append(bytes(b2))
    reads.append(b"")                                               # an empty read
    reads.append(bytes(rng.choice(list(b"ACGT"), 77).tolist()))    # a class without neighbours
    perm = rng.permutation(len(reads))
    return [reads[i] for i in perm]


def long_reads(seed, lengths, X=0.99):
    rng = np.random.default_rng(seed)
    reads = []
    for L in lengths:
        T = bytes(rng.choice(list(b"ACGT"), L).tolist())
        D = int(L * (1 - X))
        reads += [T, T, edit(rng, T, D), edit(rng, T, D + 1), rc(edit(rng, T, D // 2)), edit(rng, T, D, (0, L // (D + 1)))]
    return reads


def run_cli(tmp, fastq, outname, *extra, fastq2=None):
    out = os.path.join(str(tmp), outname)
    argv = ["--fastq", fastq, "--outfile", out, "--region", "ITS2", "--taxa", "Metazoa",
            "--log", os.path.join(str(tmp), "log.txt"), "--tempdir", str(tmp)]
    argv += ["--fastq2", fastq2] if fastq2 else ["--single_end"]
    cli.main(args=cli.myparser().parse_args(argv + list(extra)))
    return out


def _tempdir(tmp):
    d = [os.path.join(str(tmp), x) for x in os.listdir(str(tmp)) if os.path.isdir(os.path.join(str(tmp), x))]
    assert len(d) == 1, d
    return d[0]


def check_cluster_cli(tmp_path):
    """--cluster_id 0.995 --keeptemp single-end: uc.txt has the --cluster_size layout, and every kept read is its
    centroid's slice (centroid from uc.txt, positions from domtbl.txt, both parsed from the files: Dedup built from the
    written uc.txt gives what the live session gave)"""
    run = tmp_path / "a"
    run.mkdir()
    out = run_cli(run, MERGED, "out.fq", "--cluster_id", "0.995", "--keeptemp")
    tdir = _tempdir(run)
    rows = [ln.split("\t") for ln in open(os.path.join(tdir, "uc.txt")).read().splitlines()]
    kinds = [r[0] for r in rows]
    assert kinds == sorted(kinds, key=lambda k: k == "C")       # every C row after every S / H row
    b = fq.read_fastq(MERGED)
    assert sum(k in "SH" for k in kinds) == b.n
    md = {r[8]: (r[8] if r[0] == "S" else r[9]) for r in rows if r[0] in "SH"}
    cents = [r[8] for r in rows if r[0] == "S"]
    assert [ln[1:].split()[0] for ln in open(os.path.join(tdir, "rep.fa")) if ln.startswith(">")] == cents
    SeqSample.reset_sessions()
    pos = SeqSample.ItsPosition(os.path.join(tdir, "domtbl.txt"), "ITS2")
    got = fq.read_fastq(out)
    want = []
    ids = b.ids()
    seq, off = b.seq_concat()
    for i, rid in enumerate(ids):
        try:
            start, stop, _ = pos.get_position(md[rid])
        except KeyError:
            continue
        if start is None or stop is None or not start < stop:
            continue
        want.append((rid, seq[off[i]:off[i + 1]].tobytes()[start:stop]))
    gs, go = got.seq_concat()
    assert [(rid, gs[go[k]:go[k + 1]].tobytes()) for k, rid in enumerate(got.ids())] == want
    assert len(want) > 100
    # Dedup from the written uc.txt (no live session) trims the same way
    SeqSample.reset_sessions()
    d = SeqSample.Dedup(os.path.join(tdir, "uc.txt"), os.path.join(tdir, "rep.fa"), MERGED)
    out2 = os.path.join(str(run), "out2.fq")
    d.create_trimmed_seqs(out2, gzipped=False, zstd_file=False, itspos=pos, wri_file=True, tempdir=tdir)
    assert open(out2, "rb").read() == open(out, "rb").read()


def check_no_accepted_pairs_equals_exact(tmp_path, paired=False):
    """at an identity where no two classes are accepted (D(L) = 0 below 1 kb at 0.999) the output is the exact path's"""
    kw = {}
    r1 = MERGED
    if paired:
        r1, kw["fastq2"] = os.path.join(TD, "4774-1-MSITS3_R1.fastq"), os.path.join(TD, "4774-1-MSITS3_R2.fastq")
    outs = []
    for cid in ("1", "0.999"):
        run = tmp_path / ("c" + cid)
        run.mkdir()
        o = run_cli(run, r1, "out.fq", "--cluster_id", cid, **kw)
        outs.append(open(o, "rb").read())
    assert outs[0] == outs[1] and len(outs[0]) > 0


def check_paired_cluster_cli(tmp_path):
    """paired input at 0.995, merged output and unmerged (R1 / R2) output"""
    r1, r2 = os.path.join(TD, "4774-1-MSITS3_R1.fastq"), os.path.join(TD, "4774-1-MSITS3_R2.fastq")
    run = tmp_path / "m"
    run.mkdir()
    o = run_cli(run, r1, "out.fq", "--cluster_id", "0.995", fastq2=r2)
    assert fq.read_fastq(o).n > 100
    run = tmp_path / "u"
    run.mkdir()
    o1 = run_cli(run, r1, "out1.fq", "--cluster_id", "0.995", "--outfile2", os.path.join(str(run), "out2.fq"), fastq2=r2)
    a, b = fq.read_fastq(o1), fq.read_fastq(os.path.join(str(run), "out2.fq"))
    assert a.n == b.n > 100 and a.ids() == b.ids()
