"""world_size-2 gloo test (CPU) of the sharded driver: results must equal the single-process pipeline on the
concatenated input -- global first-occurrence representatives, strands, keep / lo / hi for every read."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tests"))


def _free_port():
    """A port nobody holds right now, for the gloo rendezvous of the ranks a test starts."""
    import socket
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def _single(O, eng, seq, off):
    rep, strand, nu = O.derep(seq, off)
    idx = np.flatnonzero(rep == np.arange(len(rep)))
    parts = [seq[off[i]:off[i + 1]] for i in idx]
    uoff = np.zeros(len(idx) + 1, np.int64)
    uoff[1:] = np.cumsum([len(p) for p in parts])
    rows, nrep, st = eng.db.search(O.digitize(np.concatenate(parts).tobytes()), uoff)
    pos = O.itspos(rows, eng.side, np.diff(uoff).astype(np.int32))
    n = len(rep)
    s = np.full(n, -1, np.int32); e = s.copy(); t = s.copy()
    s[idx] = pos["start"]; e[idx] = pos["stop"]; t[idx] = pos["tlen"]
    keep, lo, hi = O.trim_bounds(off, rep, s, e, t, mode=0)
    return rep, strand, keep, lo, hi, nu, nrep


@pytest.mark.parametrize("world", [1, 2, 3])
def test_run_sharded_equals_single(tmp_path, world):
    import dist_worker as W
    port = _free_port()
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   OMP_NUM_THREADS="2")
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "dist_worker.py"), str(tmp_path)],
                                      env=env))
    for p in procs:
        assert p.wait(timeout=600) == 0
    seq, off = W.dataset()
    O, eng = W.engine()
    rep, strand, keep, lo, hi, nu, nrep = _single(O, eng, seq, off)
    assert keep.sum() > 50 and strand.sum() >= 2
    got = [np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)) for r in range(world)]
    assert int(got[0]["blo"]) == 0 and int(got[-1]["bhi"]) == len(off) - 1
    for k, want in (("rep", rep), ("strand", strand), ("keep", keep), ("lo", lo), ("hi", hi)):
        assert np.array_equal(np.concatenate([g[k] for g in got]), want), k
    for g in got:
        assert int(g["n_unique_global"]) == nu
        assert np.array_equal(g["nreported"], nrep)
    assert sum(int(g["n_owned"]) for g in got) == nu


def test_block_range_partitions():
    from itsxpress_b200.distributed import block_range
    for n in (0, 1, 7, 100):
        for w in (1, 2, 3, 8):
            blocks = [block_range(n, r, w) for r in range(w)]
            assert blocks[0][0] == 0 and blocks[-1][1] == n
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(w - 1))
            assert max(b - a for a, b in blocks) - min(b - a for a, b in blocks) <= 1


@pytest.mark.parametrize("world", [1, 2, 3])
def test_q2_samples_dealt_to_ranks(tmp_path, world):
    """q2_itsxpress.main_sharded over gloo: every sample of a 7-sample paired artifact is processed by exactly one
    rank, the loads are balanced by input size, all outputs land in the shared directory and rank 0's MANIFEST lists
    them all (SURVEY 8e: whole samples shard across GPUs with no data-path collective)."""
    import gzip
    from itsxpress_b200 import q2_itsxpress as q2
    src = tmp_path / "in"
    src.mkdir()
    lines = ["sample-id,filename,direction"]
    sizes = {}
    rng = np.random.default_rng(5)
    for k, n in enumerate([900, 50, 400, 420, 30, 880, 10]):
        sid = "S%d" % k
        for d, tag in (("forward", "R1"), ("reverse", "R2")):
            fn = "%s_%d_L001_%s_001.fastq.gz" % (sid, k, tag)
            with gzip.open(str(src / fn), "wb", compresslevel=1) as f:
                f.write(bytes(rng.integers(65, 90, n * 50, dtype=np.uint8)))
            lines.append("%s,%s,%s" % (sid, fn, d))
            sizes[sid] = sizes.get(sid, 0) + os.path.getsize(str(src / fn))
    (src / "MANIFEST").write_text("\n".join(lines) + "\n")
    out = tmp_path / "out"
    port = _free_port()
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "dist_q2_worker.py"), str(src),
                                       str(out)], env=env))
    for p in procs:
        assert p.wait(timeout=300) == 0
    mine = [open(str(out / ("rank%d.txt" % r))).read().split() for r in range(world)]
    assert sorted(sum(mine, [])) == sorted(sizes)                       # each sample exactly once
    loads = [sum(sizes[s] for s in m) for m in mine]
    assert max(loads) <= sum(loads) / world + max(sizes.values())       # greedy bound: within one sample of the mean
    man = open(str(out / "MANIFEST")).read().splitlines()
    assert man[0] == "sample-id,filename,direction" and len(man) == 1 + 14
    assert sorted(l.split(",")[1] for l in man[1:]) == sorted(l.split(",")[1] for l in lines[1:])
    assert q2.deal_samples([5, 5, 5, 5], 2) == [0, 1, 0, 1] and q2.deal_samples([], 4) == []


def test_q2_main_sharded_two_ranks_real_pipeline_on_the_oracle(tmp_path, oracle, monkeypatch):
    """The same over gloo with the REAL per-sample / batched pipeline on every rank (the CPU oracle stands in for each
    rank's device, tests/oracle_context.py): the files two ranks write into the shared directory are, byte for byte, the
    files one process writes -- samples of 17..60 pairs that share sequences, one of them empty."""
    from itsxpress_b200 import SeqSample
    from itsxpress_b200 import fastq as fq
    from itsxpress_b200 import q2_itsxpress as q2
    from oracle_context import OracleContext
    from test_gpu_merge import _make_artifact
    art = _make_artifact(str(tmp_path / "in"), [60, 17, 40, 0, 25])
    out = tmp_path / "out"
    port = _free_port()
    world = 2
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "dist_q2_worker.py"), art, str(out), "oracle"],
                                      env=env))
    for p in procs:
        assert p.wait(timeout=600) == 0
    mine = [open(str(out / ("rank%d.txt" % r))).read().split() for r in range(world)]
    assert sorted(sum(mine, [])) == ["S0", "S1", "S2", "S3", "S4"] and all(mine)
    ctx = OracleContext(oracle)
    monkeypatch.setattr(SeqSample, "get_context", lambda: ctx)
    monkeypatch.setattr(fq, "GZIP_BACKEND", "host")
    SeqSample.reset_sessions()
    ref = q2.trim_pair_output_unmerged(q2.PerSampleDir(art), region="ITS2", taxa="M")
    names = sorted(f for f in os.listdir(str(ref)) if f.endswith(".gz"))
    assert len(names) == 10 and sorted(f for f in os.listdir(str(out)) if f.endswith(".gz")) == names
    total = 0
    for n in names:
        want = fq._open_bytes(os.path.join(str(ref), n))
        assert fq._open_bytes(os.path.join(str(out), n)) == want, n
        total += len(want)
    assert total > 20_000
    assert open(str(out / "MANIFEST")).read() == open(os.path.join(str(ref), "MANIFEST")).read()
    SeqSample.reset_sessions()
