"""itsx_merge_pairs on the B200 at the edges of the merge (tests/merge_edge_cases.py), against the C oracle: the
expected-error band around maxee where only the read-order replay decides, every threshold on both sides, pairs that
break several rules, options the command line never passes (Phred+64, qmax, qmaxout / qminout, maxdiffpct) and the
tables they key, read lengths around the 32-bit plane words, the longest reads the shared-memory staging takes and
one step beyond, warps reusing their slice after a longer pair, and every consensus branch.  Reasons, lengths, packed
bases and qualities and the per-reason counts must equal the oracle's (_compare of tests/test_gpu_merge.py); what
each case is built to hit is proven on the CPU by tests/test_merge_edges_on_cpu.py."""
import numpy as np
import pytest

import merge_edge_cases as E
from itsxpress_b200 import _lib
from test_gpu_merge import _compare

pytestmark = pytest.mark.gpu


def run(oracle, ctx, case):
    kw = dict(case.params)
    st = kw.pop("allow_stagger", 0)
    ml, why, *_ = _compare(oracle, ctx, case.fs, case.fq, case.fo, case.rs, case.rq, case.ro, st, **kw)
    for e, w in zip(case.expect, why):
        if "reason" in e:
            assert _lib.MERGE_REASONS[w] == e["reason"], e
    return ml, why


@pytest.mark.parametrize("family", ["ee_band", "maxdiffs", "minovlen", "maxdiffpct", "kmers", "stagger", "score", "drop",
                                    "precedence", "consensus"])
def test_edges(oracle, gpu_ctx, family):
    for case in E.all_cases()[family]:
        run(oracle, gpu_ctx, case)


def test_options_on_one_context(oracle, gpu_ctx):
    """defaults, Phred+64, defaults again, qmax = 41, qmaxout / qminout, defaults: the context rebuilds its tables at
    every change of the options"""
    a33, a64, _ = E.ascii64_sequence()
    _, w33 = run(oracle, gpu_ctx, a33)
    _, w64 = run(oracle, gpu_ctx, a64)
    assert np.array_equal(w33, w64)
    run(oracle, gpu_ctx, a33)
    at, over = E.qmax_cases()
    run(oracle, gpu_ctx, at)
    with pytest.raises(_lib.ItsxError) as e:
        gpu_ctx.merge_pairs(over.fs, over.fq, over.fo, over.rs, over.rq, over.ro,
                            _lib.merge_params(**over.params))
    assert e.value.code == -7 and "qmax" in str(e.value)
    qout, = E.qout_cases()
    run(oracle, gpu_ctx, qout)
    run(oracle, gpu_ctx, a33)


def test_length_grid_and_low_complexity(oracle, gpu_ctx):
    for case in (E.length_grid(1), E.length_grid(0), E.low_complexity()):
        run(oracle, gpu_ctx, case)


def test_staging_limit(oracle, gpu_ctx):
    ok, over = E.limit_equal()
    run(oracle, gpu_ctx, ok)
    run(oracle, gpu_ctx, E.limit_unequal())
    with pytest.raises(_lib.ItsxError) as e:
        gpu_ctx.merge_pairs(over.fs, over.fq, over.fo, over.rs, over.rq, over.ro)
    assert e.value.code == -6 and "shared-memory staging" in str(e.value)
    # the context merges an ordinary batch afterwards
    ml, _ = run(oracle, gpu_ctx, E.plain_pairs(61))
    assert (ml > 0).sum() > 20


def test_reuse_after_longer_pairs(oracle, gpu_ctx):
    """more pairs than resident warps at one CTA per SM: every warp merges short pairs in its slice after long ones"""
    import torch
    nwarps = torch.cuda.get_device_properties(0).multi_processor_count * E.MG_WARPS
    case = E.reuse_mix(nwarps=nwarps)
    assert E.staging_bytes(int(np.diff(case.fo).max()), int(np.diff(case.ro).max())) > E.SMEM_LIMIT // 2
    _, why = run(oracle, gpu_ctx, case)
    probe = np.array([e["kind"] == "short_probe" for e in case.expect])
    assert (why[probe] == _lib.MERGE_REASONS.index("nokmers")).all()
