#!/usr/bin/env python
"""MC3 through the reference-facing Python surface (`import np_bnn as bn`) on 1 or N GPUs: the same script as
bnn_runner_MC3.py:17-48 in miniature.  Run once as a plain process and once under torchrun; with device-generated
proposals keyed on the global chain index, broadcast seeds and an explicit swap seed the N-rank run must write the SAME
.log rows as the single-process run (only rank 0 writes).  N_CHAINS (default 8) below the number of ranks runs the
chain blocks x row shards grid of mc3.chain_grid (2 chains on 4 ranks: 2 x 2).

    python tools/mc3_api_multi.py OUTDIR [N_CHAINS]
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/mc3_api_multi.py OUTDIR [N_CHAINS]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import torch.distributed as dist
import np_bnn as bn

outdir = sys.argv[1]
n_chains = int(sys.argv[2]) if len(sys.argv) > 2 else 8
world = int(os.environ.get("WORLD_SIZE", "1"))
if world > 1:
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    dist.init_process_group("nccl")
rank = dist.get_rank() if world > 1 else 0
os.makedirs(outdir, exist_ok=True)
rng = np.random.default_rng(0)
n = 20000
x = rng.standard_normal((n, 64))
w_true = rng.standard_normal((64, 6))
y = np.argmax(x @ w_true + rng.normal(0, 1.0, (n, 6)), 1)
dat = {"data": x[:18000], "labels": y[:18000], "label_dict": np.arange(6), "test_data": x[18000:], "test_labels": y[18000:]}
np.random.seed(1234)
bnn = bn.npBNN(dat, n_nodes=[32, 16], use_bias_node=-1, seed=1, actFun=bn.ActFun(fun="swish"))
logger = bn.postLogger(bnn, filename="mc3_%s_c%d_w%d" % (os.environ.get("MC3_RNG", "philox"), n_chains, world), wdir=outdir)
mc3 = bn.MC3(bnn, logger=logger, n_post_samples=20, sampling_f=50, n_iteration=2000, n_chains=n_chains, swap_frequency=50,
             verbose=0, print_f=10 ** 9, adapt_f=0.3, adapt_fM=0.6, adapt_freq=25, adapt_stop=500, rng=os.environ.get("MC3_RNG", "philox"), swap_seed=77,
             device=int(os.environ.get("LOCAL_RANK", "0")))
t0 = time.perf_counter()
mc3.run_mcmc()
torch.cuda.synchronize()
dt = time.perf_counter() - t0
if rank == 0:
    rows = open(logger._logfile).read().splitlines()
    print("world %d (grid %d x %d): %d iterations x %d chains in %.2f s (%.0f chain-steps/s), %d log rows, last: %s" %
          ((world, mc3.Q, mc3.R, 2000, n_chains, dt, n_chains * 2000 / dt, len(rows), rows[-1][:120])), flush=True)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
