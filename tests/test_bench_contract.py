"""bench.py contract (no GPU needed): the CPU-reference arm prints exactly ONE JSON line on stdout with the keys the
driver reads, and `--impl reference` under a multi-rank launch prints it on rank 0 only.  On the GPU: --dump-outputs
writes the same arrays from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = ["--impl", "reference", "--scale", "0.01", "--steps", "1", "--warmup", "0"]


def _run(env_extra=None, args=REFERENCE, rc=0):
    env = dict(os.environ)
    env.update(env_extra or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=env,
                       cwd=ROOT, timeout=600)
    assert p.returncode == rc, p.stderr[-2000:]
    return p.stdout


def test_reference_arm_prints_one_json_line():
    out = _run()
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "reads/s" and d["unit"] == "reads/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == os.cpu_count()
    assert d["e2e"] == {"value": d["value"], "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_are_silent():
    out = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert out.strip() == ""


def test_bad_arguments_are_refused(tmp_path):
    assert _run(args=REFERENCE[:-4] + ["--steps", "0"], rc=2) == ""
    assert _run(args=REFERENCE + ["--dump-outputs", str(tmp_path / "d")], rc=2) == ""
    assert not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_repeat_from_run_to_run(tmp_path):
    args = ["--scale", "0.01", "--steps", "2", "--warmup", "0", "--no-cli", "--no-cpu-baseline", "--dump-outputs"]
    dumps = []
    for k in range(2):
        d = json.loads(_run(args=args + [str(tmp_path / str(k))]))
        assert d["steps"] == 2
        names = sorted(os.listdir(str(tmp_path / str(k))))
        dumps.append({n: np.load(str(tmp_path / str(k) / n)) for n in names})
    a, b = dumps
    assert sorted(a) == sorted(b) == sorted("%s_%s.npy" % (leg, k) for leg in ("resident", "e2e")
                                          for k in ("kept_index", "out_off", "out_seq", "out_qual", "counts"))
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for n in a:
        assert a[n].dtype in (np.float32, np.float64) and np.array_equal(a[n], b[n]), n
    r = d["result"]
    for leg in ("resident", "e2e"):
        n_reads, n_unique, n_kept, out_bytes = a[leg + "_counts.npy"]
        assert (n_unique, n_kept, out_bytes) == (r["n_unique"], r["n_kept"], r["out_bytes"]) and n_reads > n_unique
        assert 0 < n_kept == len(a[leg + "_kept_index.npy"]) and a[leg + "_out_off.npy"][-1] == out_bytes
    for k in ("kept_index", "out_off", "out_seq", "out_qual"):
        assert np.array_equal(a["resident_%s.npy" % k], a["e2e_%s.npy" % k]), k
