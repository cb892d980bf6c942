"""MC3 on a chain blocks x row shards rank grid (mc3.chain_grid): the grid choice, the owner of a chain, and the swap
step and rank-0 logging of a 2 x 2 grid over four gloo ranks on CPU tensors."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_chain_grid_table():
    from npbnn_b200 import mc3
    table = {(4, 8): (4, 2), (1, 8): (1, 8), (3, 4): (2, 2), (2, 4): (2, 2), (5, 8): (4, 2), (7, 8): (4, 2),
             (3, 8): (2, 4), (4, 6): (3, 2), (5, 6): (3, 2), (1, 1): (1, 1), (4, 4): (4, 1), (32, 8): (8, 1),
             (5, 2): (2, 1), (8, 3): (3, 1)}
    for (n, world), grid in table.items():
        assert mc3.chain_grid(n, world) == grid, (n, world)
    for n in range(1, 17):
        for world in range(1, 17):
            Q, R = mc3.chain_grid(n, world)
            assert Q * R == world and 1 <= Q <= n
            if world <= n:
                assert (Q, R) == (world, 1)


def _owner_before_grid(chain, n_chains, world):
    from npbnn_b200 import mc3
    for r in range(world):
        start, n = mc3.chain_partition(n_chains, world, r)
        if start <= chain < start + n:
            return r


def test_owner_follows_the_grid():
    from npbnn_b200 import mc3
    # R = 1: the owner of chain sharding over all ranks
    for n, world in ((32, 8), (5, 2), (8, 8), (7, 3)):
        assert [mc3.owner_of(c, n, world) for c in range(n)] == [_owner_before_grid(c, n, world) for c in range(n)]
    # 3 chains on 2 x 2: chains 0, 1 in block 0 (ranks 0, 1), chain 2 in block 1 (ranks 2, 3); the r = 0 rank owns
    assert [mc3.owner_of(c, 3, 4, 2) for c in range(3)] == [0, 0, 2]
    # 4 chains on 4 x 2
    assert [mc3.owner_of(c, 4, 8, 2) for c in range(4)] == [0, 2, 4, 6]
    assert [mc3.owner_of(0, 1, 8, 8)] == [0]


def test_exchange_counts_only_the_first_row_shard():
    """The gather of a 2 x 2 grid: ranks 1 and 3 (r = 1) contribute no chains, so their copies never enter the swap."""
    from npbnn_b200 import mc3
    lp_all = np.array([-10.0, -12.5, -9.25])
    seen = {}

    def gather(local, counts, group):
        seen["counts"] = list(counts)
        return lp_all.copy()

    temps = mc3.default_temperatures(3, 0.8)
    t, _, _, lp = mc3.exchange(torch.tensor(lp_all[:2]), temps, mc3.SwapRNG(7), None, 4, 2, gather=gather)
    assert seen["counts"] == [2, 0, 1, 0] and np.array_equal(lp, lp_all)
    mc3.exchange(torch.tensor(lp_all[:2]), temps, mc3.SwapRNG(7), None, 2, 1, gather=gather)
    assert seen["counts"] == [2, 1]


GRID_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
rank, port, out = int(sys.argv[1]), sys.argv[2], sys.argv[3]
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
dist.init_process_group("gloo", rank=rank, world_size=4)
np.random.seed(100 + rank)                       # deliberately different numpy states on the ranks
import np_bnn as bn
from npbnn_b200 import api, mc3
from tests import golden_data
n = 3
Q, R = mc3.chain_grid(n, 4)
assert (Q, R) == (2, 2)
q, r = divmod(rank, R)
start, cnt = mc3.chain_partition(n, Q, q)
lp_all = np.array([-10.0, -12.5, -9.25])
temps = mc3.default_temperatures(n, 0.8)
rng = mc3.SwapRNG(7)
log = []
for it in range(20):
    lp = lp_all + 0.1 * it * np.arange(n)
    # the r = 1 copy is made different on purpose: it must not enter the swap
    local = torch.tensor(lp[start:start + cnt] + (1000.0 if r else 0.0))
    temps, swapped, pair, got = mc3.exchange(local, temps, rng, None, 4, R)
    log.append((temps.copy(), got.copy(), pair))
np.save(out + "/temps_%%d.npy" %% rank, np.array([l[0] for l in log]))
np.save(out + "/lp_%%d.npy" %% rank, np.array([l[1] for l in log]))
np.save(out + "/pairs_%%d.npy" %% rank, np.array([l[2] for l in log]))

# logging: the cold chain (index 2) lives in block 1 (ranks 2, 3); rank 2's state reaches rank 0, which alone writes
dat = golden_data.synth_class(60, 4, 3, 1, 10)
bnn = bn.npBNN(dat, n_nodes=[4, 3], init_weights=[np.full(s, 0.5) for s in ((4, 5), (3, 5), (3, 3))])
logger = bn.postLogger(bnn, filename="grid", wdir=out)
m = object.__new__(api.MC3)                      # the logging step of MC3.run_mcmc without a device
m.n_chains, m.world, m.rank, m.R, m.logger, m._bnn = n, 4, rank, R, logger, bnn
m.current_temperatures = np.array([0.8, 0.9, 1.0])
cold = None
if q == 1:
    b = api.deepcopy(bnn)
    b._w_layers = [w + (1.0 if r == 0 else 7.0) for w in b._w_layers]
    mc = object.__new__(api.MCMC)
    mc.__dict__.update(_current_iteration=40, _logPost=-12.5, _logLik=-10.0, _logPrior=-2.5, _accuracy=0.75,
                       _test_accuracy=0.5, _label_acc=np.array([0.1, 0.2, 0.3]), _acceptance_rate=0.25, _mcmc_id=2,
                       _n_post_samples=5, _temperature=1.0)
    cold = (b, mc)
m._log_on_rank0(cold)
np.save(out + "/nsamples_%%d.npy" %% rank, np.array([len(logger._post_weight_samples)]))
dist.destroy_process_group()
'''


def test_mc3_grid_2x2_four_ranks_gloo(tmp_path):
    """Four gloo ranks as 2 chain blocks x 2 row shards: every rank reaches the temperatures and swap pairs of a
    single-rank exchange of the same log-posteriors, only the r = 0 copy of a block enters, the cold chain's state
    comes from the r = 0 rank of its block, and only rank 0 writes the .log / .pkl."""
    from npbnn_b200 import mc3
    script = tmp_path / "w.py"
    script.write_text(GRID_WORKER % {"root": ROOT})
    port = str(33500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), port, str(tmp_path)]) for r in range(4)]
    for p in procs:
        assert p.wait(timeout=240) == 0
    t = [np.load(tmp_path / ("temps_%d.npy" % r)) for r in range(4)]
    lp = [np.load(tmp_path / ("lp_%d.npy" % r)) for r in range(4)]
    pairs = [np.load(tmp_path / ("pairs_%d.npy" % r)) for r in range(4)]
    for r in range(1, 4):
        assert np.array_equal(t[r], t[0]) and np.array_equal(lp[r], lp[0]) and np.array_equal(pairs[r], pairs[0])
    n = 3
    lp_all = np.array([-10.0, -12.5, -9.25])
    temps = mc3.default_temperatures(n, 0.8)
    rng = mc3.SwapRNG(7)
    for it in range(20):
        x = lp_all + 0.1 * it * np.arange(n)
        temps, _, pair, got = mc3.exchange(torch.tensor(x), temps, rng)
        assert np.array_equal(got, lp[0][it]) and tuple(pair) == tuple(pairs[0][it])
        assert np.array_equal(temps, t[0][it])
    assert [int(np.load(tmp_path / ("nsamples_%d.npy" % r))[0]) for r in range(4)] == [1, 0, 0, 0]
    rows = open(tmp_path / "grid_l4_3.log").read().strip().split("\n")
    assert len(rows) == 2 and rows[1].split("\t")[0] == "40"
    import pickle
    b, mc, lg = pickle.load(open(tmp_path / "grid_l4_3.pkl", "rb"))
    assert np.all(lg._post_weight_samples[0]["weights"][0] == 1.5)
