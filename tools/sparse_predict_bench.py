#!/usr/bin/env python
"""Posterior prediction of the BASELINE config 3 network (create_mask [120, 80] tanh, 40 features, 5 classes) on the
block-sparse prediction kernel against the dense kernels (option sparse=0), same engine call, same inputs.

    python tools/sparse_predict_bench.py [OUT.json]     (default profiles/r03_sparse_predict.json)

Cells: the config 3 network at rows 10,000 / 200,000 x posterior samples 100 / 1,000, and two block networks at 200,000
x 1,000 whose dense evaluation is the specialised k_fwd3 kernel (family A), one of them with a cover near the
program builder's limit (a quarter of the dense work).  Each cell times one bnn_predict call (mean and votes)
with the features and samples already on the device, host clock around the call and a device synchronise: the
sparse column includes the device check that the samples are zero outside the pattern.  Warm-up call, then the median
of 5.  Rates: row-samples/s, and GFLOP/s on the 1,525 flop per row and sample of the block-sparse network.  The card's
name, power limit and clocks are read in the same run."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import npbnn_b200.api as api
from npbnn_b200 import _lib as L
from npbnn_b200 import predshard
from npbnn_b200.engine import Engine, NetShape, flatten_weights

SPARSE_FLOP = 2 * (120 + 240 + 80 * 5) + 5           # per row and sample, the block sparsity exploited (tools/bench_configs.py)


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm,clocks.mem"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60)
        return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]))
    except Exception as e:           # the numbers below still stand; say that the card was not read
        return {"error": repr(e)}


def block_net(f, groups, n1, n2, per, k):
    """`groups` blocks of `per` consecutive features -> n1 nodes -> n2 nodes, dense output layer (bias on it only)."""
    shapes = [(groups * n1, f), (groups * n2, groups * n1), (k, groups * n2 + 1)]
    mask = [np.zeros(s) for s in shapes]
    for g in range(groups):
        mask[0][g * n1:(g + 1) * n1, g * per:(g + 1) * per] = 1
        mask[1][g * n2:(g + 1) * n2, g * n1:(g + 1) * n1] = 1
    mask[2][:] = 1
    return shapes, mask


def measure(name, shapes, mask, act, k, cells, flop, s_max, rng, info_rows):
    net = NetShape(shapes[0][1], shapes, act=act, lik=L.LIK_CATEGORICAL)
    f = shapes[0][1]
    n_max = max(n for n, _ in cells)
    sets = np.stack([flatten_weights([rng.normal(0, 0.5, s) * m for s, m in zip(shapes, mask)]) for _ in range(s_max)])
    pattern = predshard.zero_pattern(sets, net)
    x = rng.standard_normal((n_max, f))
    eng = Engine(net)
    dev = eng.device
    xd = torch.as_tensor(x, device=dev)
    wd = torch.as_tensor(sets, device=dev)
    md = torch.empty((n_max, k), dtype=torch.float64, device=dev)
    vd = torch.empty((n_max, k), dtype=torch.float64, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())

    def call(n, S):
        L.check(eng.lib.bnn_predict(eng._h, p(xd), n, p(wd), S, None, None, None, 0, p(md), p(vd), None, eng._stream()))
        torch.cuda.synchronize()

    def timed(n, S, reps=5):
        call(n, S)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            call(n, S)
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))

    for n, S in cells:
        row = {"network": name, "rows": n, "samples": S}
        outs = {}
        for label, sparse in (("dense", 0), ("sparse", 1)):
            eng.set_option("sparse", sparse)
            eng._set_pattern(pattern)
            med, lo, hi = timed(n, S)
            row[label] = {"seconds": med, "min": lo, "max": hi, "kernel": eng.last_kernel,
                          "row_samples_per_s": n * S / med, "gflops_sparse_count": n * S * flop / med / 1e9}
            outs[label] = (md[:n].cpu().numpy().copy(), vd[:n].cpu().numpy().copy())
        row["speedup"] = row["dense"]["seconds"] / row["sparse"]["seconds"]
        (ma, va), (mb, vb) = outs["sparse"], outs["dense"]
        row["max_rel_diff_mean"] = float(np.max(np.abs(ma - mb) / np.maximum(np.abs(mb), 1e-300)))
        row["votes_identical"] = bool(np.array_equal(va, vb))
        info_rows.append(row)
        print(json.dumps(row), flush=True)
    eng.close()


def sparse_flop(shapes, mask):
    """2 x (multiply-adds of the block cover) + activations of the hidden units, per row and sample."""
    nnz = sum(int(m[:, 1:].sum()) if s[1] == shapes[i - 1][0] + 1 and i else int(m.sum())
              for i, (s, m) in enumerate(zip(shapes, mask)))
    return 2 * nnz + sum(s[0] for s in shapes[:-1])


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r03_sparse_predict.json")
    rng = np.random.default_rng(0)
    info = gpu_info()
    rows = []
    shapes = [(120, 40), (80, 120), (5, 81)]
    idx = [list(range(40)), sum(([g] * 3 for g in range(40)), []), []]
    mask = api.create_mask([np.zeros(s) for s in shapes], idx, [[3] * 40, [2] * 40, []])
    measure("c3 [120, 80] tanh, 40 features, 5 classes", shapes, mask, "tanh", 5,
            [(10_000, 100), (10_000, 1000), (200_000, 100), (200_000, 1000)], SPARSE_FLOP, 1000, rng, rows)
    # block networks whose dense evaluation at 200k rows is the specialised k_fwd3 family A (16 -> 64 -> 32 -> 16 pad)
    fam = [("16 features -> 16 x [4 -> 2] swish, 8 classes (k_fwd3 family A when dense; uniform pairs)",
            block_net(16, 16, 4, 2, 1, 8)),
           ("16 features -> 8 x [2 features -> 8 -> 4] swish, 8 classes (cover 0.19 of dense: near the builder's "
            "limit; general program)", block_net(16, 8, 8, 4, 2, 8))]
    for name, (sh, mk) in fam:
        measure(name, sh, mk, "swish", 8, [(200_000, 1000)], sparse_flop(sh, mk), 1000, rng, rows)
    res = {"what": "bnn_predict (mean + votes) of block-masked networks: block-sparse prediction kernel vs dense kernels",
           "gpu": info, "flop_per_row_sample_sparse_c3": SPARSE_FLOP, "timing": "host clock around call + synchronise, "
           "median of 5 after one warm-up; inputs on the device; the sparse column includes the device check of the "
           "samples against the pattern",
           "cells": rows}
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
