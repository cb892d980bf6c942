"""GPU: MC3 on a chain blocks x row shards grid (mc3.chain_grid) and the count likelihoods under row sharding.

A 2 x 2 grid is emulated in one process: four Engines (two chain blocks x two row shards) driven through the
orchestration functions of the package (rowshard.exchange / mh_steps, mc3.exchange) with the all-reduce and the
all-gather done in process, against one unsharded engine holding all the chains."""
import glob
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from npbnn_b200 import _lib as L
from npbnn_b200 import api, mc3, rowshard
from npbnn_b200.engine import Engine, NetShape
from tests.test_gpu_count_lik import KIND, _problem
from tests.test_gpu_parity import _c4_like, rel_close

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ADAPT = dict(adapt_f=0.1, adapt_fM=0.6, adapt_freq=5, adapt_stop=40)


def _sum_over_shards(reds):
    """In-process all-reduce: every shard's [C, n_values] tensor becomes the sum over the block's shards."""
    total = reds[0].clone()
    for t in reds[1:]:
        total += t
    for t in reds:
        t.copy_(total)


def _shards(net, x, y, xt, yt, R, sets, **kw):
    """The R row shards of one chain block, initial state exchanged."""
    out = []
    for r in range(R):
        a, b = rowshard.row_partition(len(x), R, r)
        ta, tb = rowshard.row_partition(len(xt), R, r)
        e = Engine(net)
        e.set_data(x[a:b], y[a:b], xt[ta:tb], yt[ta:tb])
        e.enable_rowshard(len(x), "manual")
        e.chains_init(sets, **kw)
        out.append(e)
    rowshard.exchange(out, _sum_over_shards, 2)
    return out


def _host_draws(eng, chain_ids, n_steps):
    """MC3's host draws for the chains of `eng` (randomize_seed: reseeded per (iteration, global chain)), from the
    engine's own state after the adaptation the device applies first; stops at the next adaptation point."""
    st = eng.read_state(weights=False)
    it = int(st.iteration[0])
    max_n = np.array([r * c for r, c in eng.net.shapes])
    for c in range(eng.n_chains):
        api._mirror_adaptation(st, c, it, ADAPT["adapt_freq"], ADAPT["adapt_stop"], ADAPT["adapt_f"], ADAPT["adapt_fM"],
                               max_n, int(max_n.sum()))
    k = min(n_steps, api._steps_to_adaptation(it, ADAPT["adapt_freq"], ADAPT["adapt_stop"]))
    grp = SimpleNamespace(net=eng.net, n=eng.n_chains, n_act_prm=0, freq_indicator=0.0, use_fi=False)
    inj = api._ChainGroup.draw_steps(grp, [None] * eng.n_chains, st, chain_ids, k,
                                     reseed=lambda cid, i: np.random.default_rng(i + cid), adapt_stop=ADAPT["adapt_stop"])
    return k, inj


@pytest.mark.parametrize("rng", ["philox", "host"])
def test_grid_2x2_matches_unsharded_mc3(rng):
    n_chains, world, Q, R, period, n_periods = 4, 4, 2, 2, 10, 5
    x, labels, sets = _c4_like(3000, n_chains, seed=23)
    xt, lt = x[2600:], labels[2600:]
    x, labels = x[:2600], labels[:2600]
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=L.LIK_CATEGORICAL)
    temps0 = mc3.default_temperatures(n_chains, 0.8)
    full = Engine(net)
    full.set_data(x, labels, xt, lt)
    full.chains_init(sets, temperature=temps0, seed=77, **ADAPT)
    blocks = []
    for q in range(Q):
        start, cnt = mc3.chain_partition(n_chains, Q, q)
        blocks.append((start, cnt, _shards(net, x, labels, xt, lt, R, sets[start:start + cnt],
                                           temperature=temps0[start:start + cnt], seed=77, chain_offset=start, **ADAPT)))
    temps_full = temps0.copy()
    ref_rng = mc3.SwapRNG(5)
    ranks = [SimpleNamespace(q=p // R, r=p % R, temps=temps0.copy(), rng=mc3.SwapRNG(5)) for p in range(world)]
    n_swaps = 0
    for period_i in range(n_periods):
        if rng == "philox":
            full.mh_steps(period)
            for _, _, shards in blocks:
                rowshard.mh_steps(shards, period, None, _sum_over_shards)
        else:
            done = 0
            while done < period:
                k, inj = _host_draws(full, list(range(n_chains)), period - done)
                full.mh_steps(k, inj)
                for start, cnt, shards in blocks:
                    draws = [_host_draws(e, list(range(start, start + cnt)), period - done) for e in shards]
                    assert all(d[0] == k for d in draws)
                    for key in draws[0][1]:
                        assert np.array_equal(draws[0][1][key], draws[1][1][key])     # every rank draws the same
                    rowshard.mh_steps(shards, k, draws[0][1], _sum_over_shards)
                done += k
        # swap: the single-rank exchange and the four ranks' exchanges with an in-process all-gather
        temps_full, swapped, pair, lp_full = mc3.exchange(full.gather(L.F_LOGPOST), temps_full, ref_rng)
        full.set_temperature(temps_full)
        n_swaps += swapped
        locals_ = [blocks[p.q][2][p.r].gather(L.F_LOGPOST) for p in ranks]

        def gather(local, counts, group):
            return np.concatenate([locals_[p][:counts[p]].cpu().numpy() for p in range(world)])

        for p in ranks:
            start, cnt, shards = blocks[p.q]
            p.temps, sw, pr, lp = mc3.exchange(locals_[p.q * R + p.r], p.temps, p.rng, None, world, R, gather=gather)
            assert sw == swapped and pr == pair and rel_close(lp, lp_full, rtol=1e-12)
            assert np.array_equal(p.temps, temps_full), (period_i, p.temps, temps_full)
            shards[p.r].set_temperature(p.temps[start:start + cnt])
        s0 = full.read_state()
        for start, cnt, shards in blocks:
            st = [e.read_state() for e in shards]
            assert np.array_equal(st[0].f64, st[1].f64) and np.array_equal(st[0].i32, st[1].i32)   # ranks bit-identical
            assert np.array_equal(st[0].w, st[1].w)
            sl = slice(start, start + cnt)
            assert np.array_equal(st[0].temperature, s0.temperature[sl])
            assert np.array_equal(st[0].n_accepted, s0.n_accepted[sl]) and np.array_equal(st[0].w, s0.w[sl])
            assert np.array_equal(st[0].update_n, s0.update_n[sl]) and np.array_equal(st[0].i32, s0.i32[sl])
            assert np.all(st[0].iteration == period * (period_i + 1))
            assert rel_close(st[0].logLik, s0.logLik[sl], rtol=1e-12)
            assert rel_close(st[0].logPost, s0.logPost[sl], rtol=1e-12)
    assert n_swaps >= 1 and np.all(s0.n_accepted > 0)
    for _, _, shards in blocks:
        for e in shards:
            e.close()
    full.close()


@pytest.mark.parametrize("mode", ["poisson", "negbin"])
def test_count_likelihood_row_shards_match_unsharded(mode):
    """Two row shards of a count model against the unsharded run: lgamma(k + 1) from each shard's own targets, the
    1 + 3K slots exchanged in order, the MSE sums over all rows."""
    m, sets, _ = _problem(mode, 2600, 12, (16, 8), "swish", 1, seed=31, n_sets=3, n_test=400)
    net = NetShape.from_weights(sets[0], 12, act="swish", lik=KIND[mode])
    kw = dict(temperature=[1.0, 0.9, 0.8], seed=91, **ADAPT)
    full = Engine(net)
    full.set_data(m.x, m.labels, m.x_test, m.labels_test)
    full.chains_init(sets, **kw)
    shards = _shards(net, m.x, m.labels, m.x_test, m.labels_test, 2, sets, **kw)
    s0 = full.read_state()
    for e in shards:
        st = e.read_state()
        assert rel_close(st.logLik, s0.logLik, rtol=1e-12)
        assert rel_close(st.sum_r2, s0.sum_r2, rtol=1e-12) and rel_close(st.sum_r2_test, s0.sum_r2_test, rtol=1e-12)
    T = 30
    full.mh_steps(T)
    rowshard.mh_steps(shards, T, None, _sum_over_shards)
    s0 = full.read_state()
    assert np.all(s0.n_accepted > 0)
    st = [e.read_state() for e in shards]
    assert np.array_equal(st[0].f64, st[1].f64)
    for s in st:
        assert np.array_equal(s.n_accepted, s0.n_accepted) and np.array_equal(s.w, s0.w)
        assert np.array_equal(s.i32, s0.i32)
        assert rel_close(s.logLik, s0.logLik, rtol=1e-12)
        assert rel_close(s.sum_r, s0.sum_r, rtol=1e-12) and rel_close(s.sum_r2, s0.sum_r2, rtol=1e-12)
        assert rel_close(s.sum_r2_test, s0.sum_r2_test, rtol=1e-12)
    for e in shards + [full]:
        e.close()


def test_mcmc_row_shard_accepts_a_count_likelihood(tmp_path):
    """Under a process group (here of one rank) MCMC(row_shard=True) takes a count likelihood; without one it refuses
    the request (tests/test_cpu_count_lik.py)."""
    import torch.distributed as dist
    import np_bnn as bn
    rng = np.random.default_rng(3)
    x = rng.standard_normal((500, 5))
    y = rng.poisson(np.exp(0.3 * x[:, :1])).astype(np.float64)
    dat = {"data": x, "labels": y, "test_data": [], "test_labels": []}
    np.random.seed(4)
    bnn = bn.npBNN(dat, n_nodes=[6, 4], estimation_mode="custom", size_output=2, output_act_fun=bn.RegressTransform)
    with pytest.raises(NotImplementedError):
        bn.MCMC(bnn, likelihood_f=bn.poi_likelihood, row_shard=True, n_iteration=20)
    dist.init_process_group("gloo", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1)
    try:
        m = bn.MCMC(bnn, likelihood_f=bn.poi_likelihood, row_shard=True, n_iteration=20)
        m.run(bnn, 5)
    finally:
        dist.destroy_process_group()
    assert m._current_iteration == 5 and np.isfinite(m._logLik) and m._accuracy_f is bn.poi_acc


def _log_rows(outdir):
    (path,) = glob.glob(os.path.join(outdir, "*.log"))
    return [line.split("\t") for line in open(path).read().strip().split("\n")]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_mc3_grid_over_ranks_writes_the_single_process_log(tmp_path):
    """tools/mc3_api_multi.py under torchrun with more ranks than chains (2 chains on 4 GPUs: 2 x 2; 1 chain on 2 or 3
    GPUs: 1 x 2) writes the .log of the single-process run."""
    n_gpus = 4 if torch.cuda.device_count() >= 4 else 2
    n_chains = n_gpus // 2
    tool = os.path.join(ROOT, "tools", "mc3_api_multi.py")
    env = dict(os.environ, MC3_RNG="philox")
    one, many = str(tmp_path / "one"), str(tmp_path / "many")
    subprocess.run([sys.executable, tool, one, str(n_chains)], check=True, env=env, timeout=900)
    subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", str(n_gpus), "--master-addr",
                    "127.0.0.1", "--master-port", str(35500 + os.getpid() % 2000), tool, many, str(n_chains)],
                   check=True, env=env, timeout=900)
    a, b = _log_rows(one), _log_rows(many)
    assert a[0] == b[0] and len(a) == len(b) > 2
    for ra, rb in zip(a[1:], b[1:]):
        assert ra[0] == rb[0] and ra[-1] == rb[-1]              # iteration and the cold chain's id (swap sequence)
        assert rel_close([float(v) for v in ra[1:-1]], [float(v) for v in rb[1:-1]], rtol=1e-12)
