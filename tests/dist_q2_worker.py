"""Worker for the world_size-2 gloo test of q2_itsxpress.main_sharded (CPU, no GPU): the deal of samples to ranks,
the shared output directory and the MANIFEST written after the barrier are the product's; the per-sample pipeline is
replaced by a stub that copies the forward (and reverse) file, since the real one needs a B200 -- or, with a third
argument "oracle", it is the real pipeline with the CPU oracle standing in for every rank's device (tests/oracle_context.py)."""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def stub(sample, results, tempdir, threads, taxa, region, paired_in, paired_out, *rest):
    shutil.copy(sample.forward, os.path.join(str(results), os.path.basename(sample.forward)))
    if paired_out:
        shutil.copy(sample.reverse, os.path.join(str(results), os.path.basename(sample.reverse)))


def main():
    src, out = sys.argv[1], sys.argv[2]
    engine = sys.argv[3] if len(sys.argv) > 3 else "stub"
    if engine == "oracle":
        os.environ["ITSX_GZIP"] = "host"        # no device on any rank: zlib writes the .gz output (read at import)
    import torch.distributed as dist
    from itsxpress_b200 import q2_itsxpress as q2
    dist.init_process_group("gloo")
    if engine == "oracle":
        # the REAL per-sample / batched pipeline of every rank, with the CPU oracle standing in for its device
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from itsxpress_b200 import SeqSample
        from oracle import oracle as O
        from oracle_context import OracleContext
        O.lib()
        ctx = OracleContext(O)
        SeqSample.get_context = lambda: ctx
        res, mine = q2.main_sharded(q2.PerSampleDir(src), out, region="ITS2", taxa="M", paired_in=True, paired_out=True)
    else:
        res, mine = q2.main_sharded(q2.PerSampleDir(src), out, region="ITS2", taxa="M", process=stub)
    with open(os.path.join(out, "rank%d.txt" % dist.get_rank()), "w") as f:
        f.write("\n".join(mine))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
