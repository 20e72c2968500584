"""Build libss_b200.so in-tree with nvcc for sm_100a (no torch extension machinery: the
library is a plain C-ABI shared object, loaded with ctypes)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libss_b200.so")
SOURCES = ["capi.cu", "kde.cu", "kde_fp64.cu", "mpc_host.cu", "mpc_simt.cu", "mpc_score.cu", "mpc_tc.cu", "mpc_tc_quad.cu", "mpc_fp64.cu", "plan_geom.cu", "value_net.cu", "peer.cu", "dyn_train.cu", "mt19937.cu", "py_random.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"] + os.environ.get("SS_NVCC_EXTRA", "").split()


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + \
           [os.path.join(HERE, "..", "include", "ss_b200.h")]
    return any(os.path.getmtime(p) > t for p in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link libss_b200.so next to this file."""
    if not force and not needs_build():
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [_nvcc()] + [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + \
              ["-Xptxas", "-v" if verbose else "-O3", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out.decode())
        if p.returncode:
            raise RuntimeError("nvcc failed on %s" % src)
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-lcudart"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
