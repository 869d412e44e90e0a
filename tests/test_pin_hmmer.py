"""Pins of the HMM stage that arm themselves.

DESIGN.md section 2 calls the HMM cascade "parity unpinned": no HMMER binary, no `F.hmm` and no `domtbl.txt` fixture exist
in this image (they are listed in the reference's .MISSING_LARGE_BLOBS), so the oracle's restatement of hmmsearch
(oracle/ora_hmm.c) -- and through tests/test_gpu_parity.py the kernels -- are held only to HMMER-free known answers.  The
moment one of the missing pieces is reachable these tests stop skipping:

  * `hmmsearch` on PATH: the reference's own command line (itsxpress/SeqSample.py:191-209: --domtblout -T 10 --F1/2/3 1e-6)
    runs on the reference's `rep.fa` fixture with the runtime profile file create_runtime_hmm writes for a taxon file that
    IS shipped, and every row ItsPosition would read (SeqSample.py:445-450: target, tlen, query, domain score, env from,
    env to) is compared with the oracle's;
  * the reference's `tests/test_data/ex_tmpdir/domtbl.txt` together with `F.hmm`: the same comparison against the rows
    a real hmmsearch wrote (tests/test_main_pytest.py:36-46 quotes three of them: 52.2 / 59.1 / 34.0 bits, env 84..128,
    282..326, 327..370).

What always runs is the plumbing: the parser and the comparison are exercised on a domain table written from the oracle's
own rows in hmmsearch's column layout, intact and perturbed.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import HMM_DIR, TD

REP_FA = os.path.join(TD, "ex_tmpdir", "rep.fa")


def read_fasta(path):
    ids, seqs, cur = [], [], []
    with open(path) as f:
        for line in f:
            line = line.rstrip("\n")
            if line.startswith(">"):
                if ids:
                    seqs.append("".join(cur))
                ids.append(line[1:].split()[0])
                cur = []
            elif line:
                cur.append(line)
    if ids:
        seqs.append("".join(cur))
    return ids, seqs


def parse_domtbl(path):
    """The six fields ItsPosition reads off a --domtblout line (SeqSample.py:445-450), file order."""
    rows = []
    with open(path) as f:
        for line in f:
            if line.startswith("#") or not line.strip():
                continue
            ll = line.split()
            rows.append((ll[0], int(ll[2]), ll[3], float(ll[13]), int(ll[19]), int(ll[20])))
    return rows


def oracle_rows(oracle, hmm_paths, prefixes, ids, seqs):
    """The same six fields from the oracle's reported rows, hmmsearch order; plus the flag 'came out of a multidomain region'
    (the one place where this implementation's tracebacks are not draw-for-draw HMMER's, DESIGN.md section 2)."""
    db = oracle.ProfileDB(hmm_paths, prefixes)
    text = "".join(seqs).encode()
    off = np.zeros(len(seqs) + 1, np.int64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    rows, _, _ = db.search(oracle.digitize(text), off, oracle.default_params(0, 1))
    out, multi = [], []
    for r in rows:
        if not r["is_reported"]:
            continue
        s = int(r["seq"])
        out.append((ids[s], len(seqs[s]), db.names[int(r["prof"])], oracle.score10(float(r["bitscore"])) / 10.0,
                    int(r["ienv"]), int(r["jenv"])))
        multi.append(bool(r["is_multidomain"]))
    return out, multi


def compare(ref, got, got_multi=None, score_tol=0.1001):
    """Rows matched per (target, query) hit in the order they were printed.  Returns counts of what differs."""
    from collections import defaultdict
    a, b = defaultdict(list), defaultdict(list)
    for r in ref:
        a[(r[0], r[2])].append(r)
    for i, r in enumerate(got):
        b[(r[0], r[2])].append((r, bool(got_multi[i]) if got_multi is not None else False))
    res = {"ref_rows": len(ref), "got_rows": len(got), "hits_missing": 0, "hits_extra": 0, "ndom_differs": 0, "tlen_differs": 0,
           "score_differs": 0, "env_differs": 0, "env_differs_multidomain": 0, "max_score_diff": 0.0}
    for k in a:
        if k not in b:
            res["hits_missing"] += 1
            continue
        da, db_ = sorted(a[k], key=lambda r: r[4]), sorted(b[k], key=lambda t: t[0][4])
        if len(da) != len(db_):
            res["ndom_differs"] += 1
            continue
        for ra, (rb, is_multi) in zip(da, db_):
            res["tlen_differs"] += ra[1] != rb[1]
            d = abs(ra[3] - rb[3])
            res["max_score_diff"] = max(res["max_score_diff"], d)
            res["score_differs"] += d > score_tol
            if (ra[4], ra[5]) != (rb[4], rb[5]):
                res["env_differs_multidomain" if is_multi else "env_differs"] += 1
    res["hits_extra"] = sum(1 for k in b if k not in a)
    return res


def write_domtbl_like_hmmsearch(path, rows):
    """--domtblout's 22 whitespace-separated columns + description, values only where ItsPosition reads them."""
    with open(path, "w") as f:
        f.write("#                                                                            --- full sequence --- -------------- this domain -------------   hmm coord   ali coord   env coord\n")
        f.write("# target name        accession   tlen query name           accession   qlen   E-value  score  bias   #  of  c-Evalue  i-Evalue  score  bias  from    to  from    to  from    to  acc description of target\n")
        for t, tlen, q, score, e0, e1 in rows:
            f.write("%-20s %-10s %5d %-20s %-10s %5d %9.2g %6.1f %5.1f %3d %3d %9.2g %9.2g %6.1f %5.1f %5d %5d %5d %5d %5d %5d %4.2f %s\n" %
                    (t, "-", tlen, q, "-", 45, 1e-9, score, 0.0, 1, 1, 1e-9, 1e-9, score, 0.0, 1, 45, e0, e1, e0, e1, 0.9, "-"))
        f.write("#\n# Program:         hmmsearch\n# [ok]\n")


def assert_pinned(res):
    """The bar of BASELINE.json's north_star: the same hits, the same printed scores, the same envelopes -- envelope
    differences tolerated (and counted) only for rows out of multidomain regions."""
    assert res["hits_missing"] == 0 and res["hits_extra"] == 0 and res["ndom_differs"] == 0, res
    assert res["tlen_differs"] == 0 and res["score_differs"] == 0 and res["env_differs"] == 0, res


def test_comparison_plumbing_on_the_oracles_own_table(oracle, tmp_path):
    ids, seqs = read_fasta(REP_FA)
    assert len(ids) == 137                                   # tests/test_main_pytest.py:49-65
    rows, multi = oracle_rows(oracle, [os.path.join(HMM_DIR, "M.hmm")], ["3_", "4_"], ids[:40], seqs[:40])
    assert len(rows) > 40
    path = str(tmp_path / "domtbl.txt")
    write_domtbl_like_hmmsearch(path, rows)
    back = parse_domtbl(path)
    assert back == rows
    res = compare(back, rows, multi)
    assert_pinned(res)
    assert res["ref_rows"] == res["got_rows"] == len(rows) and res["max_score_diff"] == 0.0
    # perturbations are seen: an envelope end, a score, a missing hit
    bent = list(rows)
    k = next(i for i, m in enumerate(multi) if not m)
    bent[k] = bent[k][:5] + (bent[k][5] + 1,)
    assert compare(bent, rows, multi)["env_differs"] == 1
    bent = list(rows)
    bent[k] = bent[k][:3] + (bent[k][3] + 0.3,) + bent[k][4:]
    assert compare(bent, rows, multi)["score_differs"] == 1
    dropped = [r for r in rows if (r[0], r[2]) != (rows[0][0], rows[0][2])]
    res = compare(rows, dropped, None)
    assert res["hits_missing"] == 1 and compare(dropped, rows, multi)["hits_extra"] == 1
    with pytest.raises(AssertionError):
        assert_pinned(res)


@pytest.mark.skipif(shutil.which("hmmsearch") is None, reason="no HMMER binary in this image (DESIGN.md section 2: parity unpinned)")
def test_oracle_against_a_live_hmmsearch(oracle, tmp_path):
    from itsxpress_b200 import main as cli
    ids, seqs = read_fasta(REP_FA)
    for taxa, tfile in (("Metazoa", "M.hmm"), ("Alveolata", "A.hmm")):
        if not os.path.exists(os.path.join(HMM_DIR, tfile)):
            continue
        tmp = str(tmp_path / taxa)
        os.makedirs(tmp)
        hmmfile = cli.create_runtime_hmm(taxa=taxa, region="ITS2", tempdir=tmp)
        dom = os.path.join(tmp, "domtbl.txt")
        subprocess.run(["hmmsearch", "--domtblout", dom, "-T", "10", "--cpu", "1", "--tformat", "fasta", "--F1", "1e-6",
                        "--F2", "1e-6", "--F3", "1e-6", hmmfile, REP_FA], check=True, stdout=subprocess.DEVNULL)
        rows, multi = oracle_rows(oracle, [os.path.join(HMM_DIR, tfile)], ["3_", "4_"], ids, seqs)
        res = compare(parse_domtbl(dom), rows, multi)
        print(taxa, res)
        assert_pinned(res)


DOMTBL_FIXTURE = os.path.join(TD, "ex_tmpdir", "domtbl.txt")
F_HMM = os.path.join(HMM_DIR, "F.hmm")


@pytest.mark.skipif(not (os.path.exists(DOMTBL_FIXTURE) and os.path.exists(F_HMM)),
                    reason="the reference's domtbl.txt fixture and F.hmm are not in tests/test_data and ITSx_db "
                           "(the reference ships neither)")
def test_oracle_against_the_references_domtbl_fixture(oracle):
    ids, seqs = read_fasta(REP_FA)
    ref = parse_domtbl(DOMTBL_FIXTURE)
    # the three rows the reference's own test quotes (tests/test_main_pytest.py:36-46)
    assert any(r[3] == 52.2 and (r[4], r[5]) == (84, 128) for r in ref)
    queries = {r[2] for r in ref}
    prefixes = sorted({q[:2] for q in queries})              # the profile classes the fixture was searched with
    rows, multi = oracle_rows(oracle, [F_HMM], prefixes, ids, seqs)
    res = compare(ref, rows, multi)
    print(res)
    assert_pinned(res)
