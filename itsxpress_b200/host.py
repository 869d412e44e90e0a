"""Host-side emitters of the inter-stage files the reference keeps in its temp dir.

The reference hands results from stage to stage as FILES written by the external tools
(`uc.txt`, `rep.fa` from vsearch, `domtbl.txt` from hmmsearch; itsxpress/SeqSample.py:104-105,190 and
`--keeptemp`, itsxpress/main.py:125-128).  The GPU path produces arrays; these functions render the
arrays in the tools' formats so that ``Dedup(uc_file, ...)`` / ``ItsPosition(domtable, ...)`` keep working
from paths exactly as the reference's tests construct them (tests/test_main_pytest.py:32-35,49-53).
Formats: SURVEY.md Appendix B (vsearch) and HMMER's --domtblout (22 fields + description).
"""
import numpy as np


def cluster_order(rep_index, ids):
    """Representative read indices in vsearch's cluster order: abundance descending, then label ascending
    (byte-wise, like strcmp) -- SURVEY.md Appendix B, verified against tests/test_data/ex_tmpdir/uc.txt."""
    rep_index = np.asarray(rep_index)
    n = len(rep_index)
    ab = np.bincount(rep_index, minlength=n)
    first = np.flatnonzero(rep_index == np.arange(n))
    labels = [ids[i].encode() if isinstance(ids[i], str) else bytes(ids[i]) for i in first.tolist()]
    order = sorted(range(len(first)), key=lambda k: (-int(ab[first[k]]), labels[k]))
    return first[np.asarray(order, dtype=np.int64)] if len(order) else first


def _ascii_labels(batch):
    """the batch's labels (offset, length) if every label byte is ASCII (the native emitters copy bytes, the Python ones
    encode the decoded ids), else None"""
    lab_off, lab_len = batch.labels()
    if batch.n:
        from .fastq import _gather
        packed, _ = _gather(batch.buf, lab_off, lab_len)
        if packed.size and int(packed.max()) > 127:
            return None
    return lab_off, lab_len


def _vp(a):
    import ctypes
    return a.ctypes.data_as(ctypes.c_void_p)


def write_rep_fasta(batch, order, ids, width=80):
    """rep.fa as `vsearch --fastaout`: '>label' then the sequence as stored, wrapped at 80 columns (native formatter;
    ``write_rep_fasta_py`` is the reference of the format)."""
    from . import _lib
    lab = _ascii_labels(batch)
    order = np.ascontiguousarray(order, dtype=np.int64)
    if lab is None:
        return write_rep_fasta_py(batch, order, ids, width)
    s_off = np.ascontiguousarray(batch.s_off, dtype=np.int64)
    s_len = np.ascontiguousarray(batch.s_len, dtype=np.int64)
    buf = np.ascontiguousarray(batch.buf)
    L = s_len[order] if len(order) else np.zeros(0, np.int64)
    cap = int((L + L // width + 4).sum() + lab[1][order].sum()) + 64 if len(order) else 64
    dst = np.empty(cap, np.uint8)
    n = _lib.lib().itsx_repfa_format(_vp(buf), _vp(s_off), _vp(s_len), _vp(lab[0]), _vp(lab[1]), _vp(order), len(order),
                                     int(width), _vp(dst), cap)
    if n < 0:
        return write_rep_fasta_py(batch, order, ids, width)
    return dst[:n].tobytes()


def write_rep_fasta_py(batch, order, ids, width=80):
    """rep.fa as `vsearch --fastaout`: '>label' then the sequence as stored, wrapped at 80 columns."""
    out = []
    for i in np.asarray(order).tolist():
        s = batch.buf[int(batch.s_off[i]):int(batch.s_off[i]) + int(batch.s_len[i])].tobytes()
        out.append(b">" + ids[i].encode() + b"\n")
        for j in range(0, len(s), width):
            out.append(s[j:j + width] + b"\n")
    return b"".join(out)


def write_uc(rep_index, strand, ids, lengths, order, batch=None):
    """uc.txt as `vsearch --uc` for --fastx_uniques: per cluster an S row then its H rows in input order, then one C row
    per cluster; 10 tab-separated columns.  With the ``batch`` the ids come from, the native formatter writes it
    (``write_uc_py`` is the reference of the format: 4 us per read)."""
    lab = _ascii_labels(batch) if batch is not None else None
    if lab is None:
        return write_uc_py(rep_index, strand, ids, lengths, order)
    from . import _lib
    rep = np.ascontiguousarray(rep_index, dtype=np.int32)
    st = None if strand is None else np.ascontiguousarray(strand, dtype=np.uint8)
    ln = np.ascontiguousarray(lengths, dtype=np.int64)
    order = np.ascontiguousarray(order, dtype=np.int64)
    buf = np.ascontiguousarray(batch.buf)
    n = len(rep)
    maxlab = int(lab[1].max()) if n else 0
    cap = n * (2 * maxlab + 64) + 2 * len(order) * (maxlab + 64) + 64
    dst = np.empty(cap, np.uint8)
    got = _lib.lib().itsx_uc_format(_vp(rep), None if st is None else _vp(st), _vp(ln), n, _vp(order), len(order), _vp(buf),
                                    _vp(lab[0]), _vp(lab[1]), _vp(dst), cap)
    if got < 0:
        return write_uc_py(rep_index, strand, ids, lengths, order)
    return dst[:got].tobytes()


def write_uc_py(rep_index, strand, ids, lengths, order, identity=None):
    """uc.txt as `vsearch --uc` for --fastx_uniques: per cluster an S row then its H rows in input order,
    then one C row per cluster; 10 tab-separated columns.  ``identity`` (percent per read) fills the H rows' identity
    column, as --cluster_size writes it; without it every H row is 100.0."""
    rep_index = np.asarray(rep_index)
    n = len(rep_index)
    order = np.asarray(order).tolist()
    cl_of_rep = {r: c for c, r in enumerate(order)}
    members = [[] for _ in order]
    for i in range(n):
        r = int(rep_index[i])
        if r != i:
            members[cl_of_rep[r]].append(i)
    lines = []
    for c, r in enumerate(order):
        lines.append("S\t%d\t%d\t*\t*\t*\t*\t*\t%s\t*\n" % (c, int(lengths[r]), ids[r]))
        for i in members[c]:
            lines.append("H\t%d\t%d\t%.1f\t%s\t0\t0\t*\t%s\t%s\n" %
                         (c, int(lengths[i]), 100.0 if identity is None else float(identity[i]),
                          "-" if strand is not None and strand[i] else "+", ids[i], ids[r]))
    for c, r in enumerate(order):
        lines.append("C\t%d\t%d\t*\t*\t*\t*\t*\t%s\t*\n" % (c, 1 + len(members[c]), ids[r]))
    return "".join(lines).encode()


DOMTBL_HEADER = (
    "#                                                                            --- full sequence --- "
    "-------------- this domain -------------   hmm coord   ali coord   env coord\n"
    "# target name        accession   tlen query name           accession   qlen   E-value  score  bias   #  of"
    "  c-Evalue  i-Evalue  score  bias  from    to  from    to  from    to  acc description of target\n"
    "#------------------- ---------- ----- -------------------- ---------- ----- --------- ------ ----- --- ---"
    " --------- --------- ------ ----- ----- ----- ----- ----- ----- ----- ---- ---------------------\n")


def _g2(x):
    """C printf('%9.2g') for E-values."""
    return "%9.2g" % x


DOMTBL_FOOTER = "#\n# Program:         itsxpress-b200 (hmmsearch-compatible table)\n# [ok]\n"


def _labels(names):
    """byte strings back to back + int64 offsets, or None if a label is not ASCII (padding is per character)"""
    try:
        enc = [n.encode("ascii") for n in names]
    except UnicodeEncodeError:
        return None
    off = np.zeros(len(enc) + 1, np.int64)
    np.cumsum([len(e) for e in enc], out=off[1:])
    return np.frombuffer(b"".join(enc) + b"\0", np.uint8), off, max([len(e) for e in enc], default=0)


def write_domtbl(rows, seq_ids, prof_names, prof_M, nseq_total, nreported):
    """domtbl.txt in hmmsearch's --domtblout layout: the native formatter (csrc/fastq_host.cpp, all host threads; the
    Python loop below costs 25 us per row -- 6 s for a sample of 20 000 reads, a minute at 200 000), byte-identical to
    ``write_domtbl_py``, which stays as the reference of the format and for labels that are not ASCII."""
    from . import _lib
    rows = np.ascontiguousarray(rows)
    sl, pl = _labels(seq_ids), _labels(prof_names)
    if sl is None or pl is None or rows.dtype != _lib.ROW_DTYPE:
        return write_domtbl_py(rows, seq_ids, prof_names, prof_M, nseq_total, nreported)
    M = np.ascontiguousarray(prof_M, dtype=np.int32)
    nrep = np.ascontiguousarray(nreported, dtype=np.int32)
    cap = len(rows) * (max(sl[2], 20) + max(pl[2], 20) + 320) + 64
    head, foot = DOMTBL_HEADER.encode(), DOMTBL_FOOTER.encode()
    dst = np.empty(len(head) + cap + len(foot), np.uint8)          # header, rows and footer in place: one copy out
    dst[:len(head)] = np.frombuffer(head, np.uint8)
    body = dst[len(head):]
    n = _lib.lib().itsx_domtbl_format(_vp(rows), len(rows), _vp(sl[0]), _vp(sl[1]), _vp(pl[0]), _vp(pl[1]), _vp(M), _vp(nrep),
                                      float(nseq_total), _vp(body), cap)
    if n < 0:
        return write_domtbl_py(rows, seq_ids, prof_names, prof_M, nseq_total, nreported)
    body[n:n + len(foot)] = np.frombuffer(foot, np.uint8)
    return dst[:len(head) + n + len(foot)].tobytes()


def write_domtbl_py(rows, seq_ids, prof_names, prof_M, nseq_total, nreported):
    """domtbl.txt rows in hmmsearch's --domtblout layout (whitespace separated, 22 fields + description).

    The six fields ItsPosition reads (SeqSample.py:445-450: target name, tlen, query name, domain score,
    env from, env to) carry the computed values; E-values and the full-sequence score are computed as HMMER
    does (Z = number of targets, domZ = hits reported for the profile).  Alignment-derived columns
    (bias, hmm/ali coordinates, acc) are not needed for trimming and are not computed on the device:
    ali = env, hmm = 1..M, bias and acc are printed as 0 -- stated in DESIGN.md.
    """
    out = [DOMTBL_HEADER]
    if len(rows):
        # number of reported domains per (profile, sequence) hit, in row order
        key = rows["prof"].astype(np.int64) * (int(rows["seq"].max()) + 1) + rows["seq"]
        _, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
        ndom_of = cnt[inv]
        k_in_hit = np.zeros(len(rows), np.int64)
        seen = {}
        for t, k in enumerate(key.tolist()):
            seen[k] = seen.get(k, 0) + 1
            k_in_hit[t] = seen[k]
    for t in range(len(rows)):
        r = rows[t]
        p = int(r["prof"])
        Z = float(nseq_total)
        domZ = float(nreported[p])
        ev = np.exp(float(r["seq_lnP"])) * Z
        cev = np.exp(float(r["lnP"])) * domZ
        iev = np.exp(float(r["lnP"])) * Z
        out.append("%-20s %-10s %5d %-20s %-10s %5d %s %6.1f %5.1f %3d %3d %s %s %6.1f %5.1f %5d %5d %5d %5d %5d %5d %4.2f %s\n" % (
            seq_ids[int(r["seq"])], "-", int(r["tlen"]), prof_names[p], "-", int(prof_M[p]),
            _g2(ev), float(r["seq_score"]), 0.0, int(k_in_hit[t]), int(ndom_of[t]),
            _g2(cev), _g2(iev), float(r["bitscore"]), 0.0,
            1, int(prof_M[p]), int(r["ienv"]), int(r["jenv"]), int(r["ienv"]), int(r["jenv"]), 0.0, "-"))
    out.append(DOMTBL_FOOTER)
    return "".join(out).encode()
