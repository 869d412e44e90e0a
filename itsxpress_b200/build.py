"""Build libitsx_b200.so in-tree with nvcc for sm_100a (no JIT, no torch extension machinery).

Usage: python -m itsxpress_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libitsx_b200.so")
SOURCES = ["api.cu", "derep.cu", "cluster.cu", "search.cu", "trim.cu", "shard.cu", "merge.cu", "deflate.cu", "hmmfile.cpp", "fastq_host.cpp", "inflate_host.cpp"]
HEADERS = [os.path.join(CSRC, "itsx_internal.h"), os.path.join(CSRC, "deflate_core.h"), os.path.join(HERE, "..", "include", "itsx_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-fmad=false",
         "-Xcompiler", "-fPIC,-O3,-ffp-contract=off", "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def _stale(out, deps):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    objs, procs = [], []
    for src in SOURCES:
        sp = os.path.join(CSRC, src)
        obj = os.path.join(objdir, src.rsplit(".", 1)[0] + ".o")
        objs.append(obj)
        if force or _stale(obj, [sp] + HEADERS):
            cmd = [NVCC] + FLAGS + ["-x", "cu", "-c", sp, "-o", obj]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        with open(os.path.join(objdir, src + ".log"), "w") as f:
            f.write(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on " + src)
    if force or procs or _stale(LIB, objs):
        subprocess.check_call([NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lpthread"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
