#!/usr/bin/env python
"""Cost of itsx_cluster on an amplicon-like sample, and the search time it saves.

Workload (seeded): configs[1]'s shape, 1 M reads of 250 bp, drawn from random templates with Zipf abundances, with
Illumina-like substitutions (per base) and rare single-base indels, tuned to about 30 % unique sequences.  bench.py's
synthetic configs have independent random spacers, so clustering finds nothing there; this workload is what the option
is for: sequencing-error variants of far fewer true sequences.

Prints one JSON line: ms per clustering stage, candidate / distinct / accepted pair counts, centroids at 0.995 and 0.99,
and the search time (ITS2 profiles of M.hmm) over the centroids against the search time over all uniques.  With --check
it also verifies that two runs are identical, that every member is within D of its centroid and no two centroids accept
each other (CPU reference on the centroids), and that a --check-n-unique subsample equals the CPU reference.
    python tools/cluster_rate.py [--reads N] [--check] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def make_reads(n, L=250, ntemplates=4000, sub=0.0014, indel=0.02, seed=11):
    rng = np.random.default_rng(seed)
    tmpl = rng.integers(0, 4, (ntemplates, L), dtype=np.uint8)
    w = 1.0 / np.arange(1, ntemplates + 1) ** 1.1
    t = rng.choice(ntemplates, n, p=w / w.sum())
    r = tmpl[t]
    m = rng.random((n, L)) < sub
    r[m] = (r[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) % 4
    acgt = np.frombuffer(b"ACGT", np.uint8)
    r = acgt[r]
    reads = [row.tobytes() for row in r]
    for i in np.flatnonzero(rng.random(n) < indel):
        p = int(rng.integers(1, L - 1))
        s = reads[i]
        reads[i] = s[:p] + s[p + 1:] if rng.random() < 0.5 else s[:p] + b"ACGT"[int(rng.integers(4)):][:1] + s[p:]
    off = np.zeros(n + 1, np.int64)
    off[1:] = np.cumsum([len(x) for x in reads])
    return np.frombuffer(b"".join(reads), np.uint8).copy(), off


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--check-n-unique", type=int, default=20_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from itsxpress_b200 import _lib
    seq, off = make_reads(a.reads)
    ctx = _lib.Context(0)
    hmm = os.path.join(ROOT, "itsxpress_b200", "ITSx_db", "HMMs", "M.hmm")
    ctx.load_profiles([hmm], ["3_", "4_"])
    ctx.set_sides_by_prefix("3_", "4_")
    prm = _lib.default_params()
    out = {"reads": a.reads, "bp": 250}
    _, _, nu = ctx.derep(seq, off)
    out["uniques"] = nu
    ctx.search(prm)                         # warm-up of the search shapes
    ctx.derep(seq, off)
    ctx.search(prm)
    out["search_ms_uniques"] = ctx.search_stats().ms_total
    for X in (0.995, 0.99):
        ctx.derep(seq, off)
        ctx.cluster(X)                      # warm-up
        ctx.derep(seq, off)
        t0 = time.perf_counter()
        nc = ctx.cluster(X)
        wall = (time.perf_counter() - t0) * 1e3
        st = ctx.cluster_stats().asdict()
        ctx.search(prm)
        rec = dict(st, centroids=nc, wall_ms=wall, search_ms_centroids=ctx.search_stats().ms_total)
        rec["search_ms_saved"] = out["search_ms_uniques"] - rec["search_ms_centroids"]
        rec["cluster_over_saved"] = st["ms_total"] / rec["search_ms_saved"] if rec["search_ms_saved"] > 0 else None
        out["id_%g" % X] = rec
    if a.check:
        import cluster_ref as R
        X = 0.995
        _, _, nu = ctx.derep(seq, off)
        first, _ = ctx.derep_clusters(nu)
        runs = []
        for _ in range(2):
            ctx.derep(seq, off)
            nc = ctx.cluster(X)
            runs.append(ctx.cluster_fetch(nu, nc))
        chk = {"two_runs_identical": all(np.array_equal(x, y) for x, y in zip(*runs))}
        crow, strand, ed, uor = runs[0]
        lens = off[first + 1] - off[first]
        D = _lib.cluster_dtable(X, int(lens.max()))
        cl = uor[crow]
        chk["members_within_D"] = bool(np.all(ed <= D[np.maximum(lens, lens[cl])]))
        # centroids among themselves: the reference makes every one a centroid again
        cf = first[uor]
        nc2 = R.cluster(seq, off, cf, np.arange(len(cf), dtype=np.int32), X)[0]
        chk["centroids_pairwise_rejected"] = nc2 == len(cf)
        # subsample: the reads of the first classes (first occurrence order) until check_n_unique classes
        rep, _, _ = ctx.derep(seq, off)
        cls = np.searchsorted(first, rep)
        keep = np.flatnonzero(cls < a.check_n_unique)
        sub = [seq[off[i]:off[i + 1]].tobytes() for i in keep]
        s2 = np.frombuffer(b"".join(sub), np.uint8).copy()
        o2 = np.zeros(len(sub) + 1, np.int64)
        o2[1:] = np.cumsum([len(x) for x in sub])
        rep2, _, nu2 = ctx.derep(s2, o2)
        f2, _ = ctx.derep_clusters(nu2)
        nc = ctx.cluster(X)
        g = ctx.cluster_fetch(nu2, nc)
        t0 = time.perf_counter()
        w = R.cluster(s2, o2, f2, R.default_order(rep2), X)
        chk["subsample_uniques"] = nu2
        chk["subsample_ref_s"] = time.perf_counter() - t0
        chk["subsample_equals_reference"] = nc == w[0] and all(np.array_equal(x, y) for x, y in zip(g, w[1:]))
        out["check"] = chk
    import subprocess
    try:
        out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                    capture_output=True, text=True).stdout.strip()
    except OSError:
        out["gpu"] = None
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
