#!/usr/bin/env python
"""The QIIME 2 action trim_single at cluster_id = 0.995 on an artifact of many small samples: the per-sample loop
(ITSX_Q2_BATCH_READS = 0) against the default batched pass, in which each sample is clustered on its own.

Workload (seeded): --samples single-end samples of --reads reads each, written as a per-sample directory of .fastq.gz.
True sequences are --templates variants (2 % substitutions) of the 227 merged ITS2 amplicons of the test fixture (330 to
441 bp), so the search has domains to find; each sample draws its reads from a random quarter of them with Zipf
abundances, and every read carries Illumina-like substitutions (0.14 % per base) and, for 2 % of reads, one indel.
Samples therefore share most of their sequences, and each sample's error variants cluster at 0.995.

Timed: the wall time of trim_single per artifact, loop and batched alternated (--repeats each, after one warm-up of
both on a small artifact), with the device time of derep, clustering and search summed over the calls of each run.  The
runs must write identical files and MANIFESTs.  Prints one JSON line with the card's name and power limit.
    python tools/cluster_batch_rate.py [--samples 128] [--reads 25000] [--repeats 2] [--out FILE]"""
import argparse
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ACGT = np.frombuffer(b"ACGT", np.uint8)


def templates(n, seed):
    from itsxpress_b200 import fastq as fq
    b = fq.read_fastq(os.path.join(ROOT, "tests", "test_data", "4774-1-MSITS3_merged.fastq"))
    seq, off = b.seq_concat()
    rng = np.random.default_rng(seed)
    out = []
    for t in range(n):
        i = t % b.n
        s = seq[off[i]:off[i + 1]].copy()
        if t >= b.n:
            m = rng.random(len(s)) < 0.02
            s[m] = ACGT[(np.searchsorted(ACGT, s[m]) + rng.integers(1, 4, int(m.sum()))) % 4]
        out.append(s)
    return out


def write_artifact(root, nsamples, nreads, ntemplates, seed=7):
    tmpl = templates(ntemplates, seed)
    tlen = np.array([len(t) for t in tmpl])
    mat = np.zeros((ntemplates, int(tlen.max())), np.uint8)
    for t, s in enumerate(tmpl):
        mat[t, :len(s)] = s
    rng = np.random.default_rng(seed + 1)
    os.makedirs(root)
    lines = ["sample-id,filename,direction"]
    for k in range(nsamples):
        pool = rng.choice(ntemplates, max(1, ntemplates // 4), replace=False)
        w = 1.0 / np.arange(1, len(pool) + 1) ** 1.1
        pick = pool[rng.choice(len(pool), nreads, p=w / w.sum())]
        r = mat[pick]
        m = rng.random(r.shape) < 0.0014
        r[m] = ACGT[(np.searchsorted(ACGT, r[m]) + rng.integers(1, 4, int(m.sum()))) % 4]
        indel = rng.random(nreads) < 0.02
        recs = []
        for i, t in enumerate(pick.tolist()):
            x = r[i, :tlen[t]].tobytes()
            if indel[i]:
                p = int(rng.integers(1, len(x) - 1))
                x = x[:p] + x[p + 1:] if rng.random() < 0.5 else x[:p] + b"ACGT"[int(rng.integers(4)):][:1] + x[p:]
            recs.append(b"@s%d_r%d\n%s\n+\n%s\n" % (k, i, x, b"I" * len(x)))
        fn = "S%d_%d_L001_R1_001.fastq.gz" % (k, k)
        with gzip.open(os.path.join(root, fn), "wb", compresslevel=1) as f:
            f.write(b"".join(recs))
        lines.append("S%d,%s,forward" % (k, fn))
    with open(os.path.join(root, "MANIFEST"), "w") as f:
        f.write("\n".join(lines) + "\n")
    return root


class StageTimes:
    """device ms of derep, clustering and search, summed over the calls made through the shared context"""

    def __init__(self, ctx):
        self.ms = {"derep": 0.0, "cluster": 0.0, "search": 0.0}
        for name, stats, key in (("derep", "derep_stats", "derep"), ("derep_resident", "derep_stats", "derep"),
                                 ("cluster", "cluster_stats", "cluster"), ("search", "search_stats", "search")):
            self._wrap(ctx, name, getattr(ctx, stats), key)

    def _wrap(self, ctx, name, stats, key):
        orig = getattr(ctx, name)

        def f(*a, **kw):
            out = orig(*a, **kw)
            self.ms[key] += float(stats().ms_total)
            return out
        setattr(ctx, name, f)

    def take(self):
        out = dict(self.ms)
        for k in self.ms:
            self.ms[k] = 0.0
        return out


def run(q2, art, budget, times):
    q2.BATCH_READS = budget
    times.take()
    t0 = time.perf_counter()
    res = q2.trim_single(q2.PerSampleDir(art), region="ITS2", taxa="M", cluster_id=0.995)
    wall = time.perf_counter() - t0
    return str(res), dict(wall_s=wall, **{"device_ms_" + k: v for k, v in times.take().items()})


def files_of(d):
    from itsxpress_b200 import fastq as fq
    names = sorted(f for f in os.listdir(d) if f.endswith(".gz"))
    return {n: fq._open_bytes(os.path.join(d, n)) for n in names}, open(os.path.join(d, "MANIFEST")).read()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=128)
    ap.add_argument("--reads", type=int, default=25_000)
    ap.add_argument("--templates", type=int, default=2000)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from itsxpress_b200 import SeqSample
    from itsxpress_b200 import q2_itsxpress as q2
    default_budget = q2.BATCH_READS
    assert default_budget > 0
    work = tempfile.mkdtemp(prefix="cluster_batch_rate_")
    try:
        t0 = time.perf_counter()
        art = write_artifact(os.path.join(work, "in"), a.samples, a.reads, a.templates)
        small = write_artifact(os.path.join(work, "warm"), 3, 500, 200, seed=3)
        out = {"samples": a.samples, "reads_per_sample": a.reads, "templates": a.templates, "cluster_id": 0.995,
               "batch_reads": default_budget, "gen_s": time.perf_counter() - t0}
        times = StageTimes(SeqSample.get_context())
        for budget in (0, default_budget):               # module loads, search shapes
            run(q2, small, budget, times)
        runs = {"loop": [], "batched": []}
        ref = None
        for _ in range(a.repeats):
            for mode, budget in (("loop", 0), ("batched", default_budget)):
                d, rec = run(q2, art, budget, times)
                got = files_of(d)
                shutil.rmtree(d, ignore_errors=True)
                if ref is None:
                    ref = got
                assert got == ref, "%s output differs from the first run" % mode
                runs[mode].append(rec)
        out["runs"] = runs
        out["output_bytes"] = sum(len(v) for v in ref[0].values())
        out["outputs_identical"] = True
        for mode, recs in runs.items():
            out[mode + "_wall_s_min"] = min(r["wall_s"] for r in recs)
        out["speedup_wall"] = out["loop_wall_s_min"] / out["batched_wall_s_min"]
    finally:
        shutil.rmtree(work, ignore_errors=True)
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


if __name__ == "__main__":
    main()
