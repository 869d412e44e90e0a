#!/usr/bin/env python
"""Build an experimental variant of libitsx_b200.so: one source recompiled with extra -D flags, the other objects reused.

  python tools/build_variant.py NAME -DFB_DECODE_PF=8 ...   ->  tools/variants/NAME.so   (search.cu)
  python tools/build_variant.py NAME --source merge.cu ...    (another source of itsxpress_b200/csrc)
  python tools/build_variant.py NAME --source /tmp/m1/merge.cu    (an edited copy, e.g. a mutant: it replaces the
                                                                   source of the same name; includes resolve in csrc)

Run a bench or the tests against it with ITSX_B200_LIB=tools/variants/NAME.so (experiments only; the product
loads itsxpress_b200/libitsx_b200.so).
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from itsxpress_b200 import build as B  # noqa: E402


def main():
    name, args = sys.argv[1], sys.argv[2:]
    src = os.path.join(B.CSRC, "search.cu")
    if "--source" in args:
        k = args.index("--source")
        src = args[k + 1]
        args = args[:k] + args[k + 2:]
        if os.sep not in src:
            src = os.path.join(B.CSRC, src)
    base = os.path.basename(src)
    if base not in B.SOURCES:
        raise SystemExit("--source must be (a copy of) one of " + ", ".join(B.SOURCES))
    defs = args
    B.build()
    vdir = os.path.join(ROOT, "tools", "variants")
    os.makedirs(vdir, exist_ok=True)
    obj = os.path.join(vdir, name + "." + base.rsplit(".", 1)[0] + ".o")
    cmd = [B.NVCC] + B.FLAGS + defs + ["-I", B.CSRC, "-x", "cu", "-c", os.path.abspath(src), "-o", obj]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    open(os.path.join(vdir, name + ".log"), "w").write(out.stdout)
    if out.returncode:
        sys.stderr.write(out.stdout)
        raise SystemExit(1)
    objs = [os.path.join(B.CSRC, "build", s.rsplit(".", 1)[0] + ".o") for s in B.SOURCES if s != base] + [obj]
    lib = os.path.join(vdir, name + ".so")
    subprocess.check_call([B.NVCC, "-shared", "-o", lib] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lpthread"])
    for line in out.stdout.splitlines():
        if "fb_kernel" in line or "env_kernel" in line or "mdclust" in line:
            print(line[:60])
    print(lib)


if __name__ == "__main__":
    main()
