#!/usr/bin/env python
"""MC3 with trainable genReLU slopes (ActFun(trainable=True)) through the reference-facing surface on 1 or N ranks.
Every layout of the same chain count must write the same .log rows and keep the same posterior samples (weights and
`alphas`) in its .pkl: chain blocks on their own ranks (chain sharding) and, with more ranks than chains, the chain
blocks x row shards grid of mc3.chain_grid.  Only rank 0 writes.

    python tools/mc3_trainable_multi.py OUTDIR N_CHAINS
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/mc3_trainable_multi.py OUTDIR N_CHAINS

MC3_RNG=host|philox picks the proposal source (default philox).  Ranks use NCCL when each has a GPU of its own and
gloo when ranks share GPUs (rank r runs on GPU r mod the GPU count)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import np_bnn as bn

outdir = sys.argv[1]
n_chains = int(sys.argv[2])
rng_mode = os.environ.get("MC3_RNG", "philox")
world = int(os.environ.get("WORLD_SIZE", "1"))
device = int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count()
if world > 1:
    torch.cuda.set_device(device)
    dist.init_process_group("nccl" if world <= torch.cuda.device_count() else "gloo")
os.makedirs(outdir, exist_ok=True)
rng = np.random.default_rng(5)
n, f, k = 2400, 12, 4
x = rng.standard_normal((n, f))
y = np.argmax(x @ rng.standard_normal((f, k)) + rng.normal(0, 1.0, (n, k)), 1)
dat = {"data": x[:2000], "labels": y[:2000], "test_data": x[2000:], "test_labels": y[2000:]}
np.random.seed(1234)
# small initial slopes: MC3 builds its chains without init_additional_prob (BNN_mc3.py:61-75), so the first proposals
# carry the whole Exp(10) term of the slopes
af = bn.ActFun(fun="genReLU", prm=np.array([0.02, 0.04]), trainable=True)
bnn = bn.npBNN(dat, n_nodes=[8, 4], use_bias_node=2, seed=1, actFun=af)
logger = bn.postLogger(bnn, filename="mc3t_%s_c%d" % (rng_mode, n_chains), wdir=outdir)
mc3 = bn.MC3(bnn, logger=logger, n_post_samples=50, sampling_f=20, n_iteration=400, n_chains=n_chains, swap_frequency=20,
             verbose=0, print_f=10 ** 9, adapt_f=0.2, adapt_fM=0.6, adapt_freq=10, adapt_stop=100, rng=rng_mode,
             swap_seed=77, device=device)
mc3.run_mcmc()
torch.cuda.synchronize()
if world > 1:
    dist.barrier()
    if dist.get_rank() == 0:
        print("world %d: grid %d x %d" % (world, mc3.Q, mc3.R), flush=True)
    dist.destroy_process_group()
