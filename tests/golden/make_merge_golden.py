"""Golden vectors for the paired-end merge (SURVEY 8f row 2): an independent, definition-level pure-Python statement
of `vsearch --fastq_mergepairs --fastq_maxdiffs 40 --fastq_maxee 2 [--fastq_allowmergestagger] --fastq_qmax 93`
(SeqSample.py:314-349), run on the reference's own paired fixtures, written to tests/golden/c1_merge.tsv:

    file  stagger  pair  reason  merged_len  crc32(bases)  crc32(qualities)

It shares no code with oracle/ora_merge.c (k-mers counted by their definition on every diagonal, byte loops for the scores and the merged read) and
exists so that the C oracle and the CUDA kernel are checked against something that is not themselves.  vsearch
itself is not installed anywhere this project builds, so these are vectors of the RESTATED algorithm ("parity
unpinned" against a real vsearch run; see oracle/ora_merge.c for what the reference's fixtures do pin).

Usage (repo root):  python tests/golden/make_merge_golden.py
"""
import gzip
import math
import os
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TD = os.path.join(HERE, "..", "test_data")
REASONS = ("ok", "repeat", "staggered", "maxdiffs", "maxdiffpct", "nokmers", "minscore", "minovlen", "maxee")


def q_to_p(x):
    return 0.75 if x < 2 else 10.0 ** (-x / 10.0)


def q_from_p(p, ascii=33, qmaxout=41, qminout=0):
    return ascii + max(qminout, min(qmaxout, int(round(-10.0 * math.log10(p)))))


def tables(ascii=33, qmaxout=41, qminout=0):
    """posterior qualities (as characters) of agreeing / disagreeing bases for every pair of quality values"""
    same = [[q_from_p(px * py / 3.0 / (1.0 - px - py + 4.0 * px * py / 3.0), ascii, qmaxout, qminout) for py in P]
            for px in P]
    diff = [[q_from_p(px * (1.0 - py / 3.0) / (px + py - 4.0 * px * py / 3.0), ascii, qmaxout, qminout) for py in P]
            for px in P]
    return same, diff


P = [q_to_p(x) for x in range(94)]
SAME, DIFF = tables()
MATCH = [[math.log2((1.0 - px - py + px * py * 4.0 / 3.0) / 0.25) for py in P] for px in P]
MISM = [[math.log2(((px + py) / 3.0 - px * py * 4.0 / 9.0) / 0.25) for py in P] for px in P]
COMP = {ord(a): ord(b) for a, b in zip("ACGTURYSWKMBDHVN", "TGCAAYRSWMKVHDBN")}
PLAIN = np.frombuffer(b"ACGTU", np.uint8)


def read_fq(path):
    op = gzip.open if path.endswith(".gz") else open
    out = []
    with op(path, "rb") as f:
        while True:
            h = f.readline().rstrip(b"\r\n")
            if not h:
                break
            s = f.readline().rstrip(b"\r\n")
            f.readline()
            q = f.readline().rstrip(b"\r\n")
            out.append((h[1:], s, q))
    return out


def kmer_counts(fs, rc):
    """per diagonal i (index i of the result), the 5-mers that match exactly on it and hold no ambiguous symbol, by
    definition: e[p, r] says forward position p and rc position r hold the same plain base, and a 5-mer starts at
    (p, r) when e holds there and at the four next positions of the diagonal, which is i = F - p + r"""
    F, R = len(fs), len(rc)
    a, b = np.frombuffer(fs, np.uint8), np.frombuffer(rc, np.uint8)
    e = (a[:, None] == b[None, :]) & np.isin(a, PLAIN)[:, None]
    if F < 5 or R < 5:
        return np.zeros(F + R, np.int64)
    k = e[:F - 4, :R - 4].copy()
    for j in range(1, 5):
        k &= e[j:F - 4 + j, j:R - 4 + j]
    p, r = np.nonzero(k)
    return np.bincount(F - p + r, minlength=F + R)


def merge_pair(fs, fq, rs, rq, stagger=False, maxdiffs=40, maxee=2.0, minovlen=10, maxdiffpct=100.0, ascii=33,
               qmax=93, qmaxout=41, qminout=0, info=None):
    """(merged bases, merged qualities) or None, and the reason.  ``info`` (a dict) receives what decided: every
    candidate diagonal's 5-mer count / score / drop / mismatches, the hit count, the best diagonal, and the merged read
    of the best diagonal with its read-order expected errors even when a rule rejects the pair."""
    if any(not 0 <= c - ascii <= qmax for c in fq + rq):
        return None, "badqual"
    same, diff = (SAME, DIFF) if (ascii, qmaxout, qminout) == (33, 41, 0) else tables(ascii, qmaxout, qminout)
    fs = fs.upper()
    F, R = len(fs), len(rs)
    rc = bytes(COMP.get(c, ord("N")) for c in rs.upper()[::-1])
    rcq = rq[::-1]
    best_score, best_i, best_diffs, hits, kmers = 0.0, 0, 0, 0, 0
    diags = {}
    counts = kmer_counts(fs, rc)
    for i in range(1, F + R):
        sh = F - i
        p0, p1 = max(0, sh), min(F, sh + R)
        cnt = int(counts[i])
        if cnt < 4:
            continue
        kmers = 1
        score = high = dropmax = 0.0
        diffs = 0
        for p in range(p1 - 1, p0 - 1, -1):
            qa, qb = fq[p] - ascii, rcq[p - sh] - ascii
            if fs[p] == rc[p - sh]:
                score += MATCH[qa][qb]
                high = max(high, score)
            else:
                score += MISM[qa][qb]
                diffs += 1
                if score < high - dropmax:
                    dropmax = high - score
                if dropmax >= 16.0:          # scores 0 whatever follows
                    break
        diags[i] = (cnt, score, dropmax, diffs)
        if dropmax >= 16.0:
            score = 0.0
        if score >= 16.0:
            hits += 1
        if score > best_score:
            best_score, best_i, best_diffs = score, i, diffs
    if info is not None:
        info.update(diags=diags, hits=hits, kmers=kmers, best_i=best_i, best_score=best_score, best_diffs=best_diffs,
                    F=F, R=R)
    merged = None
    if best_i:
        sh = F - best_i
        ms, mq, ee = bytearray(), bytearray(), 0.0
        branch = {}
        for m in range(max(sh, 0) + min(F - max(sh, 0), R - max(-sh, 0)) + (R - max(-sh, 0) - min(F - max(sh, 0), R - max(-sh, 0)))):
            r = m - sh
            if m < sh:
                s, q = fs[m], fq[m]
            elif m < F and r < R:
                a, b, qa, qb = fs[m], rc[r], fq[m] - ascii, rcq[r] - ascii
                if b == ord("N"):
                    s, q, k = a, fq[m], "n_r2" if a != ord("N") else "n_both"
                elif a == ord("N"):
                    s, q, k = b, rcq[r], "n_r1"
                elif a == b:
                    s, q, k = a, same[qa][qb], "equal" if a in PLAIN else "equal_iupac"
                elif qa > qb:
                    s, q, k = a, diff[qa][qb], "r1_better"
                else:
                    s, q, k = b, diff[qb][qa], "tie" if qa == qb else "r2_better"
                branch[k] = branch.get(k, 0) + 1
            else:
                s, q = rc[r], rcq[r]
            ms.append(s)
            mq.append(q)
            ee += P[q - ascii]
        merged = (bytes(ms), bytes(mq))
        if info is not None:
            info.update(merged=merged, ee=ee, branch=branch)
    if hits > 1:
        return None, "repeat"
    if not stagger and best_i > F:
        return None, "staggered"
    if best_diffs > maxdiffs:
        return None, "maxdiffs"
    if best_i and 100.0 * best_diffs / best_i > maxdiffpct:
        return None, "maxdiffpct"
    if not kmers:
        return None, "nokmers"
    if best_score < 16.0:
        return None, "minscore"
    if best_i < minovlen:
        return None, "minovlen"
    if ee <= maxee:
        return merged, "ok"
    return None, "maxee"


def main():
    rows = []
    for name, r1, r2 in (("4774-1-MSITS3", "4774-1-MSITS3_R1.fastq", "4774-1-MSITS3_R2.fastq"),
                         ("high_qual_scores", "high_qual_scores_R1.fastq.gz", "high_qual_scores_R2.fastq.gz")):
        a, b = read_fq(os.path.join(TD, r1)), read_fq(os.path.join(TD, r2))
        assert len(a) == len(b)
        for stagger in (0, 1):
            for i, ((_, s1, q1), (_, s2, q2)) in enumerate(zip(a, b)):
                res, why = merge_pair(s1, q1, s2, q2, stagger=bool(stagger))
                if res:
                    rows.append((name, stagger, i, why, len(res[0]), zlib.crc32(res[0]), zlib.crc32(res[1])))
                else:
                    rows.append((name, stagger, i, why, 0, 0, 0))
    with open(os.path.join(HERE, "c1_merge.tsv"), "w") as f:
        f.write("# file\tstagger\tpair\treason\tmerged_len\tcrc32_bases\tcrc32_quals\n")
        for r in rows:
            f.write("\t".join(str(x) for x in r) + "\n")
    print(len(rows), "rows")


if __name__ == "__main__":
    main()
