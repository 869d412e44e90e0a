"""The in-process sharded harness (tests/shard_cases.py) proved on the CPU: derep_ref against the oracle's
dereplication (itself pinned to vsearch's uc.txt), and G ranks as threads running the real run_sharded with the
oracle-backed engine against one process and against the same world run as gloo processes."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tests"))

import shard_cases as S  # noqa: E402


def _check_ref(oracle, reads):
    seq, off = S.pack(reads)
    rep, strand, nu = S.derep_ref(reads)
    orep, ostrand, onu = oracle.derep(seq, off)
    assert nu == onu
    assert np.array_equal(rep, orep)
    assert np.array_equal(strand, ostrand)
    return rep, strand, nu


def test_derep_ref_equals_oracle_on_the_fixture(oracle, fixture_reads):
    b, seq, off, qual = fixture_reads
    assert _check_ref(oracle, S.unpack(seq, off))[2] == 137
    reads, _ = S.fixture_case(seq, off, qual)
    rep, strand, _ = _check_ref(oracle, reads)
    assert strand.sum() >= 7 and np.any(rep[227:] < 227)


@pytest.mark.parametrize("seed,n,lo,hi", [(1, 4000, 1, 40), (2, 3000, 200, 300), (3, 3000, 15, 17), (4, 2000, 0, 70)])
def test_derep_ref_equals_oracle_on_random_reads(oracle, seed, n, lo, hi):
    reads = S.rand_reads(np.random.default_rng(seed), n, lo, hi)
    rep, strand, nu = _check_ref(oracle, reads)
    assert strand.sum() > 0 and nu < n
    assert any(r != r.upper() for r in reads) and any(set(r.upper()) - set(b"ACGTU") for r in reads)


@pytest.mark.parametrize("kind", ["main", "twenty", "five", "empty"])
def test_derep_ref_equals_oracle_on_degenerate_reads(oracle, kind):
    reads = S.degenerate_reads(kind)
    rep, strand, nu = _check_ref(oracle, reads)
    if kind == "main":
        assert strand.sum() >= 10 and b"" in reads


class _Serialised:
    """Every call into the wrapped object holds one lock: the oracle builds its tables lazily, unguarded."""

    def __init__(self, obj, lock):
        self._obj, self._lock = obj, lock

    def __getattr__(self, name):
        a = getattr(self._obj, name)
        if not callable(a) or isinstance(a, type):
            return a

        def call(*args, **kw):
            with self._lock:
                return a(*args, **kw)
        return call


def _oracle_world(G, seq, off):
    import dist_worker as W
    O, eng = W.engine()
    lock = threading.Lock()
    O_s, db_s = _Serialised(O, lock), _Serialised(eng.db, lock)
    return S.run_world(G, seq, off, lambda r: W.OracleEngine(O_s, db_s, eng.side))


@pytest.fixture(scope="module")
def oracle_single():
    import dist_worker as W
    from test_distributed import _single
    seq, off = W.dataset()
    O, eng = W.engine()
    return seq, off, _single(O, eng, seq, off)


@pytest.mark.parametrize("G", [1, 2, 3, 5, 8])
def test_thread_ranks_on_the_oracle_equal_one_process(oracle_single, G):
    seq, off, (rep, strand, keep, lo, hi, nu, nrep) = oracle_single
    outs, world, blocks = _oracle_world(G, seq, off)
    for k, want in (("rep", rep), ("strand", strand), ("keep", keep), ("lo", lo), ("hi", hi)):
        assert np.array_equal(np.concatenate([o[k] for o in outs]), want), k
    for o in outs:
        assert o["n_unique_global"] == nu and np.array_equal(o["nreported"], nrep)
    reads = S.unpack(seq, off)
    ref = S.derep_ref(reads)
    S.check_derep(outs, blocks, reads, ref)
    owner = S.check_exchange(world, blocks, reads, ref)
    assert len(owner) == nu and (G == 1 or len(set(owner.values())) == G)
    assert keep.sum() > 50 and strand.sum() >= 2


def test_thread_ranks_equal_the_gloo_world_of_three(oracle_single, tmp_path):
    """The same world as three gloo processes (tests/dist_worker.py) and as three threads: every rank's every output."""
    from test_distributed import _free_port
    seq, off, _ = oracle_single
    port = _free_port()
    procs = []
    for r in range(3):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="3", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   OMP_NUM_THREADS="2")
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "dist_worker.py"), str(tmp_path)],
                                      env=env))
    for p in procs:
        assert p.wait(timeout=600) == 0
    outs, _, blocks = _oracle_world(3, seq, off)
    for r, (o, (lo, hi)) in enumerate(zip(outs, blocks)):
        g = np.load(os.path.join(str(tmp_path), "rank%d.npz" % r))
        assert (int(g["blo"]), int(g["bhi"])) == (lo, hi)
        for k, v in o.items():
            assert np.array_equal(np.asarray(v), g[k]), (r, k)


def test_a_failing_rank_stops_the_others():
    """A rank that raises aborts the barrier the others wait on; its exception, not BrokenBarrierError, comes back."""
    def fn(r, world):
        if r == 2:
            raise ValueError("rank 2 fails")
        return world.gather(r, r)

    with pytest.raises(ValueError, match="rank 2 fails"):
        S.run_threads(4, fn, timeout=60)
    assert S.run_threads(3, lambda r, w: w.gather(r, r * r))[0] == [[0, 1, 4]] * 3
