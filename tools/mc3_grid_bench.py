#!/usr/bin/env python
"""MC3 with more GPUs than chains: the c4 problem (1,000,000 x 64 rows, [64, 32] swish, 10 classes, bias on the last
layer) with 4 tempered chains (rng="philox", swap every 100 iterations) through bn.MC3, on 1 GPU and on every visible
GPU, where the ranks form the chain blocks x row shards grid of mc3.chain_grid (4 chains on 8 GPUs: 4 x 2).  Reports
chain-steps/s with the card's name and power limit; GPU counts of 2, 4 and 8 that are not visible are "not measured".
Logging is a no-op: this is the rate of the sampler, not of the files.

    python tools/mc3_grid_bench.py OUT.json [--iterations 2000] [--warmup 100]
(runs the 1-GPU leg itself and the N-GPU leg under torch.distributed.run)"""
import argparse, json, os, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import torch.distributed as dist

CHAINS = 4


class _NoLog:
    def log_sample(self, *a):
        pass

    log_weights = log_sample


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def leg(args):
    """One measurement on WORLD_SIZE ranks; rank 0 returns the result."""
    import np_bnn as bn
    from npbnn_b200 import workloads as wl
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl")
    x, y = wl.c4_data(args.rows, seed=0)
    dat = {"data": x, "labels": y.astype(np.int64), "label_dict": np.arange(10), "test_data": [], "test_labels": []}

    def run(n_it):
        np.random.seed(1234)
        bnn = bn.npBNN(dat, n_nodes=[64, 32], use_bias_node=-1, seed=1, actFun=bn.ActFun(fun="swish"))
        m = bn.MC3(bnn, logger=_NoLog(), n_post_samples=10, sampling_f=100, n_iteration=n_it, n_chains=CHAINS,
                   swap_frequency=100, verbose=0, print_f=10 ** 9, rng="philox", swap_seed=77, device=local)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        m.run_mcmc()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return time.perf_counter() - t0, m

    run(args.warmup)
    dt, m = run(args.iterations)
    st = m._group.eng.read_state(weights=False)
    out = {"n_gpus": world, "grid_chain_blocks_x_row_shards": [m.Q, m.R], "iterations": args.iterations,
           "seconds": dt, "chain_steps_per_s": CHAINS * args.iterations / dt,
           "cold_chain_logPost": float(st.logPost[np.flatnonzero(st.temperature == 1)[0]])
           if np.any(st.temperature == 1) else None}
    if world > 1:
        dist.destroy_process_group()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?")
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--iterations", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--leg", action="store_true", help="internal: one measurement (under torch.distributed.run)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mc3_grid_bench needs CUDA GPUs")
    if args.leg:
        res = leg(args)
        if int(os.environ.get("RANK", "0")) == 0:
            print("LEG " + json.dumps(res), flush=True)
        return
    n_vis = torch.cuda.device_count()
    res = {"what": __doc__.split("\n\n")[0].replace("\n", " "), "card_and_power_limit": _card(), "rows": args.rows,
           "chains": CHAINS, "visible_gpus": n_vis, "legs": {}}
    counts = sorted({1, n_vis} | {2, 4, 8})
    for n in counts:
        if n > n_vis:
            res["legs"][str(n)] = "not measured"
            continue
        if n != 1 and n != n_vis:
            res["legs"][str(n)] = "not measured"
            continue
        cmd = [sys.executable, os.path.abspath(__file__), "--leg", "--rows", str(args.rows), "--iterations",
               str(args.iterations), "--warmup", str(args.warmup)]
        if n > 1:
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                   "--master-port", str(36500 + os.getpid() % 2000)] + cmd[1:]
        p = subprocess.run(cmd, capture_output=True, text=True, cwd=tempfile.gettempdir())
        lines = [l for l in p.stdout.splitlines() if l.startswith("LEG ")]
        if p.returncode != 0 or not lines:
            raise SystemExit("leg on %d GPU(s) failed:\n%s\n%s" % (n, p.stdout[-2000:], p.stderr[-4000:]))
        res["legs"][str(n)] = json.loads(lines[-1][4:])
        print(n, res["legs"][str(n)], flush=True)
    print(json.dumps(res), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
