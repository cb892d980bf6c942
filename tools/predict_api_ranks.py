#!/usr/bin/env python
"""BASELINE config 5 shape through the reference-facing Python surface on 1, 2, 4 and 8 GPUs: bn.get_posterior_cat_prob
(BNN_lib.py:352-397) modes 1 / 0 / 2 on 1,000,000 host rows with S = 1,000 posterior samples, return_dense=False, as
tools/predict_api_c5.py times it on one GPU.  With N ranks the same script runs under torchrun and the call is
collective (predshard.predict_ranks): every rank holds the full host features and samples, scores its rows x samples
block and receives the full [N, K] summary.  Per world size it records the wall time of each call (barrier, call,
device synchronise, barrier) and, for mode 1, the time rank 0 spends in the engine call on its own block alone.

    python tools/predict_api_ranks.py OUT.json [S]          (launches one torchrun per world size the machine has GPUs for)"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def worker(part_path, S):
    import numpy as np
    import torch
    import torch.distributed as dist
    import np_bnn as bn
    from npbnn_b200 import api, predshard, workloads as wl
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl")
    rank = dist.get_rank() if world > 1 else 0
    sync = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    n = 1_000_000
    x, _ = wl.c4_data(n, seed=0)
    rng = np.random.default_rng(5)
    base = wl.c4_init_weights(1)[0]
    post = [{"weights": [w + rng.normal(0, 0.05, w.shape) for w in base], "alphas": [0.0]} for _ in range(S)]
    af = bn.ActFun(fun="swish")
    kw = dict(actFun=af, output_act_fun=bn.SoftMax, return_dense=False)
    bn.get_posterior_cat_prob(x[:4096], post[:8], post_summary_mode=1, **kw)
    bn.get_posterior_cat_prob(x, post, post_summary_mode=1, **kw)          # warm-up at the timed shape
    runs = []
    for mode in (1, 0, 2):
        np.random.seed(7)
        sync()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, summ = bn.get_posterior_cat_prob(x, post, post_summary_mode=mode, **kw)
        torch.cuda.synchronize()
        sync()
        dt = time.perf_counter() - t0
        runs.append({"post_summary_mode": mode, "seconds": dt, "row_samples_per_s": n * S / dt,
                     "tflops": n * S * wl.C4_FLOP_PER_ROW / dt / 1e12, "summary_shape": list(np.shape(summ)),
                     "row_sums_ok": bool(np.allclose(np.sum(summ, axis=1), 1.0))})
    grid = predshard.grid_for(n, S, world)
    (a, b), (c, d), _, _, _ = predshard.partition(n, S, world, rank, grid)
    eng = api._predict_engine(post[0]["weights"], 64, af, bn.SoftMax)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.predict(x[a:b], [p["weights"] for p in post[c:d]], mean=True)
    torch.cuda.synchronize()
    block = time.perf_counter() - t0
    if rank == 0:
        json.dump({"world": world, "grid_rows_x_sample_groups": list(grid), "runs": runs,
                   "rank0_block_rows": b - a, "rank0_block_samples": d - c,
                   "rank0_block_engine_call_seconds_mode1": block}, open(part_path, "w"), indent=1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main(out_path, S):
    import torch
    n_gpus = torch.cuda.device_count()
    if n_gpus == 0:
        raise SystemExit("no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"what": __doc__.split("\n\n")[0].replace("\n", " "), "rows": 1_000_000, "samples": S,
           "gpus": smi, "worlds": []}
    me = os.path.abspath(__file__)
    for world in (1, 2, 4, 8):
        if world > n_gpus:
            res["worlds"].append({"world": world, "not measured": "%d GPUs on this machine" % n_gpus})
            continue
        part = out_path + ".w%d" % world
        if world == 1:
            cmd = [sys.executable, me, "--worker", part, str(S)]
        else:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", str(world), "--master-addr",
                   "127.0.0.1", "--master-port", str(38500 + world), me, "--worker", part, str(S)]
        subprocess.run(cmd, check=True, timeout=1800)
        res["worlds"].append(json.load(open(part)))
        os.remove(part)
        print(json.dumps(res["worlds"][-1]), flush=True)
    one = {r["post_summary_mode"]: r["seconds"] for r in res["worlds"][0]["runs"]}
    for w in res["worlds"]:
        for r in w.get("runs", []):
            r["speedup_over_1_gpu"] = one[r["post_summary_mode"]] / r["seconds"]
    json.dump(res, open(out_path, "w"), indent=1)


if __name__ == "__main__":
    if sys.argv[1] == "--worker":
        worker(sys.argv[2], int(sys.argv[3]))
    else:
        main(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 1000)
