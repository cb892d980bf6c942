"""Build libnpbnn_b200.so (hand-written sm_100a CUDA + C ABI) in-tree with nvcc.

    python -m npbnn_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libnpbnn_b200.so")
SOURCES = ["bnn_forward.cu", "bnn_sparse.cu", "bnn_mcmc.cu", "bnn_chainloop.cu", "bnn_pred_lp.cu", "bnn_capi.cu"]
HEADERS = ["bnn_common.cuh", "bnn_kernels.h", "bnn_mh_body.cuh", "bnn_generic_body.cuh", os.path.join("..", "..", "include", "npbnn_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = _nvcc()
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode:
                raise RuntimeError("nvcc failed on %s" % src)
            with open(o + ".ptxas.log", "w") as f:
                f.write(r.stdout + r.stderr)
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
