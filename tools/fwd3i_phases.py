"""Per-phase clocks of k_fwd3i (int8 first layer) at the config-4 shape: builds a copy of the library whose forward
translation unit is compiled with BNN_FWD3I_PHASES (clock64 stamps, bnn_forward.cu) into a temporary directory, scores
32 weight sets on 1M rows a few times and prints, per (128-row block, weight set) pair, the average clocks of each
phase of a compute warp and of the MMA thread, as one JSON line.  Needs the library built (python -m npbnn_b200.build).

    python tools/fwd3i_phases.py [--rows 1000000] [--sets 32] [--reps 5]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PHASES = {0: "compute: wait for the accumulators (tfull)", 1: "compute: drain + recombine (+ pending softmax epilogue)",
          2: "compute: wait for the layers-2/3 weights", 3: "compute: layers 2/3 (FP64 DMMA + activations)",
          4: "compute: whole pair", 6: "mma thread: wait for drained accumulators and operands",
          7: "mma thread: issue 42 MMAs + commit"}


def build_instrumented(tmp):
    from npbnn_b200 import build as b
    b.build()
    nvcc = b._nvcc()
    obj = os.path.join(tmp, "bnn_forward_phases.o")
    subprocess.run([nvcc] + b.NVCC_FLAGS + ["-DBNN_FWD3I_PHASES", "-c", os.path.join(b.CSRC, "bnn_forward.cu"), "-o", obj],
                   check=True, capture_output=True)
    objs = [obj] + [os.path.join(b.CSRC, s.replace(".cu", ".o")) for s in b.SOURCES if s != "bnn_forward.cu"]
    lib = os.path.join(tmp, "libnpbnn_b200_phases.so")
    subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs, check=True)
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--sets", type=int, default=32)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        lib_path = build_instrumented(tmp)
        from npbnn_b200 import _lib as L
        L.LIB_PATH = lib_path
        from npbnn_b200.engine import Engine, NetShape
        from npbnn_b200 import workloads as wl
        x, labels = wl.c4_data(args.rows, seed=3)
        sets = wl.c4_init_weights(args.sets)
        eng = Engine(NetShape(64, list(wl.C4_SHAPES), act="swish", lik=L.LIK_CATEGORICAL))
        eng.set_data(x, labels.astype(np.int64))
        h = ctypes.CDLL(lib_path)
        buf = (ctypes.c_ulonglong * 16)()
        eng.forward_lik(sets)                                   # warm-up
        eng.synchronize()
        assert h.bnn_fwd3i_phase_clocks(buf, 1) == 0
        for _ in range(args.reps):
            eng.forward_lik(sets)
        eng.synchronize()
        assert h.bnn_fwd3i_phase_clocks(buf, 0) == 0
        kernel = eng.last_kernel
        eng.close()
    v = list(buf)
    pairs_c, pairs_m = max(v[8], 1), max(v[9], 1)
    out = {"kernel": kernel, "rows": args.rows, "sets": args.sets, "reps": args.reps,
           "clk_per_pair": {PHASES[i]: round(v[i] / (pairs_c if i < 6 else pairs_m), 1) for i in PHASES}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
