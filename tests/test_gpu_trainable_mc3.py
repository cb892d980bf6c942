"""GPU: trainable activation slopes (ActFun(trainable=True)) in MC3, and mh_step(additional_prob=) with device-drawn
proposals (bnn_chains_set_additional_prob)."""
import glob
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from npbnn_b200 import _lib as L
from oracle import npbnn_oracle as orc
from tests import _golden as G

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the two network shapes of the syn_trainable_* goldens; small initial slopes, because MC3 builds its chains without
# init_additional_prob (BNN_mc3.py:61-75) and the first proposals then carry the whole Exp(10) term
CASES = {"genReLU": ("syn_trainable_genrelu", [0.02, 0.04]), "tanh": ("syn_trainable_tanh", [0.03, 0.01])}
ADAPT = dict(adapt_freq=5, adapt_f=0.2, adapt_fM=0.6, adapt_stop=40)


def _dat(z):
    return {"data": np.array(z["x"]), "labels": np.array(z["labels"]), "test_data": np.array(z["x_test"]),
            "test_labels": np.array(z["labels_test"])}


def _model(act, seed=7, **kw):
    import npbnn_b200 as bn
    name, alphas = CASES[act]
    z, meta = G.load(name)
    np.random.seed(seed)
    af = bn.ActFun(fun=act, prm=np.array(alphas), trainable=True)
    return bn.npBNN(_dat(z), n_nodes=meta["n_nodes"], actFun=af, use_bias_node=meta["use_bias_node"],
                    prior_f=meta["prior"], p_scale=meta["p_scale"], seed=seed, **kw)


def _ring(st, c):
    """The chain's last accept outcomes, oldest first (MCMC._last_accepted_mem, BNN_env.py:523-529)."""
    i = st.i32[c]
    n, h = int(i[L.I_RING_LEN]), int(i[L.I_RING_HEAD])
    return [int(i[L.I_RING + (h + j) % 100]) for j in range(n)]


def _rel(a, b, tol):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.all(np.abs(a - b) <= tol * np.maximum(np.abs(b), 1.0))


def test_mc3_chain_views_own_their_activation():
    import npbnn_b200 as bn
    bnn = _model("genReLU")
    mc3 = bn.MC3(bnn, logger=None, n_chains=3, swap_frequency=5, n_iteration=10, verbose=0)
    afs = [b._act_fun for b, _ in mc3.singleChainArgs]
    assert len({id(a) for a in afs}) == 3 and all(a is not bnn._act_fun for a in afs)
    assert all(a._trainable and np.array_equal(a._acc_prm, [0.02, 0.04]) for a in afs)
    assert mc3._group.eng.read_state().alpha.shape == (3, 3)
    with pytest.raises(NotImplementedError):
        bn.MCMC(_model("genReLU"), init_additional_prob=-1.0, _group=mc3._group, _slot=0)


def test_one_chain_mc3_is_the_single_chain_sampler(tmp_path):
    """MC3(n_chains=1) against MCMC(randomize_seed=True, mcmc_id=0) with the same adaptation, rng="host": the period
    is drawn in slices by a worker thread (step0 > 0), the single chain step by step."""
    import npbnn_b200 as bn
    period, n_periods = 20, 6
    b1 = _model("genReLU")
    logger = bn.postLogger(b1, filename="one", wdir=str(tmp_path))
    mc3 = bn.MC3(b1, logger=logger, n_chains=1, swap_frequency=period, n_iteration=period * n_periods, verbose=0, **ADAPT)
    mc3.async_pickle = False
    mc3.n_mc3_iteration = 1
    b2 = _model("genReLU")
    mcmc = bn.MCMC(b2, n_iteration=period * n_periods, mcmc_id=0, randomize_seed=True, **ADAPT)
    n_acc = 0
    for p in range(n_periods):
        mc3.run_mcmc()
        for _ in range(period):
            mcmc.mh_step(b2)
        s1, s2 = mc3._group.eng.read_state(), mcmc._group.eng.read_state()
        assert np.array_equal(s1.i32, s2.i32), p                   # accept outcomes, counters, adaptation sizes
        assert np.array_equal(s1.alpha, s2.alpha) and np.array_equal(s1.alpha_prop, s2.alpha_prop), p
        assert np.array_equal(s1.w, s2.w), p
        assert _rel(s1.logPost, s2.logPost, 1e-9) and _rel(s1.logPrior, s2.logPrior, 1e-9), p
        b, m = mc3.singleChainArgs[0]
        assert np.array_equal(b._act_fun._acc_prm, b2._act_fun._acc_prm)
        n_acc = int(s1.n_accepted[0])
    assert n_acc > 0 and not np.array_equal(b2._act_fun._acc_prm, [0.02, 0.04])


class _RecordSwap:
    """A seeded swap generator that records its draws, for the oracle to replay."""

    def __init__(self, seed):
        self._rs = np.random.RandomState(seed)
        self.draws = []

    def pair(self, n):
        j, k = self._rs.choice(range(n), 2, replace=False)
        self.draws.append([int(j), int(k)])
        return int(j), int(k)

    def log_uniform(self):
        v = float(np.log(self._rs.random_sample()))
        self.draws[-1].append(v)
        return v


@pytest.mark.parametrize("act", ["genReLU", "tanh"])
def test_mc3_trainable_matches_oracle(act):
    """Three tempered chains with trainable slopes, rng="host": each chain is the oracle driven with
    default_rng(iteration + chain) at the temperatures of the run, the swaps replayed on the oracle's log-posteriors."""
    import npbnn_b200 as bn
    period, n_periods, n_chains = 10, 6, 3
    bnn = _model(act)
    w0 = [w.copy() for w in bnn._w_layers]
    mc3 = bn.MC3(bnn, logger=None, n_chains=n_chains, swap_frequency=period, n_iteration=period * n_periods, verbose=0,
                 **ADAPT)
    mc3._swap_rng = sw = _RecordSwap(3)
    mc3.n_mc3_iteration = 1
    mc3.run_mcmc = mc3._run_mcmc                        # no logger
    mc3._log_on_rank0 = lambda cold: None
    mc3.logger = type("NoLog", (), {"log_sample": lambda *a: None, "log_weights": lambda *a: None})()
    z, meta = G.load(CASES[act][0])
    chains = []
    for c in range(n_chains):
        m = orc.Model(x=np.array(z["x"]), labels=np.array(z["labels"]), weights=[w.copy() for w in w0], act=act,
                      alphas=np.array(CASES[act][1]), prior=meta["prior"], prior_scale=np.ones(3) * meta["p_scale"],
                      x_test=np.array(z["x_test"]), labels_test=np.array(z["labels_test"]), act_trainable=True)
        s = orc.make_sampler(m, temperature=mc3.temperatures[c], n_iteration=period, **ADAPT)
        chains.append((m, s))
    temps = mc3.temperatures.copy()
    n_swaps = 0
    for p in range(n_periods):
        mc3.run_mcmc()
        for c, (m, s) in enumerate(chains):
            for _ in range(period):
                orc.mh_step(m, s, rs=np.random.default_rng(s.it + c))
        j, k, log_u = sw.draws[p]
        temps, swapped, _ = orc.mc3_swap(np.array([s.logPost for _, s in chains]), temps, j, k, log_u)
        n_swaps += swapped
        assert np.array_equal(mc3.current_temperatures, temps), p
        for c, (m, s) in enumerate(chains):
            s.temperature = temps[c]
        st = mc3._group.eng.read_state()
        for c, (m, s) in enumerate(chains):
            assert _ring(st, c) == s.acc_mem, (p, c)
            assert np.array_equal(st.alpha[c][:2], m.alphas), (p, c)
            for li in range(3):
                assert np.array_equal(st.weights(c)[li], m.weights[li]), (p, c, li)
            assert _rel(st.logLik[c], s.logLik, 1e-9) and _rel(st.logPrior[c], s.logPrior, 1e-9), (p, c)
            b, mm = mc3.singleChainArgs[c]
            assert np.array_equal(b._act_fun._acc_prm, m.alphas) and mm._temperature == temps[c]
    assert n_swaps >= 1
    assert all(sum(s.acc_mem[1:]) > 0 for _, s in chains)
    assert all(not np.array_equal(m.alphas, CASES[act][1]) for m, _ in chains)


@pytest.mark.parametrize("rng", ["host", "philox"])
def test_small_data_chain_loop_matches_launch_sequence(rng):
    """c1-sized trainable MC3 (2,250 + 250 rows, 128 features, [5, 5], bias mode 2): the persistent k_chain_loop
    pre-proposes the slope block of every chain; the launch sequence (option chain_loop = 0) computes the same chains."""
    import npbnn_b200 as bn
    r = np.random.default_rng(11)
    x = r.standard_normal((2500, 128))
    y = np.argmax(x[:, :5] + r.normal(0, 0.5, (2500, 5)), 1)
    dat = {"data": x[:2250], "labels": y[:2250], "test_data": x[2250:], "test_labels": y[2250:]}
    runs = []
    for loop in (1, 0):
        np.random.seed(3)
        bnn = bn.npBNN(dat, n_nodes=[5, 5], use_bias_node=2, seed=5,
                       actFun=bn.ActFun(fun="genReLU", prm=np.array([0.02, 0.03]), trainable=True))
        mc3 = bn.MC3(bnn, logger=None, n_chains=4, swap_frequency=25, n_iteration=100, verbose=0, rng=rng, swap_seed=9,
                     **ADAPT)
        eng = mc3._group.eng
        eng.set_option("chain_loop", 2 if loop else 0)          # 2: wherever it fits
        mc3.logger = type("NoLog", (), {"log_sample": lambda *a: None, "log_weights": lambda *a: None})()
        mc3._run_mcmc()
        kern = eng.lib.bnn_last_kernel(eng._h).decode()
        assert (kern == "k_chain_loop") == bool(loop), kern
        runs.append((eng.read_state(), mc3.current_temperatures.copy()))
        eng.close()
    (a, ta), (b, tb) = runs
    assert np.array_equal(a.f64, b.f64) and np.array_equal(a.i32, b.i32) and np.array_equal(a.w, b.w)
    assert np.array_equal(ta, tb)
    assert np.all(a.n_accepted > 0) and not np.all(a.alpha[:, :2] == [0.02, 0.03])


def _philox_mcmc(seed=7, **options):
    import npbnn_b200 as bn
    z, meta = G.load("syn_swish_cauchy")
    np.random.seed(seed)
    bnn = bn.npBNN(_dat(z), n_nodes=meta["n_nodes"], use_bias_node=meta["use_bias_node"], prior_f=meta["prior"],
                   p_scale=meta["p_scale"], seed=seed, actFun=bn.ActFun(fun=meta["act"]))
    mcmc = bn.MCMC(bnn, n_iteration=1000, rng="philox")
    for k, v in options.items():
        mcmc._group.eng.set_option(k, v)
    return bnn, mcmc


def _check_prior(bnn, mcmc, a, where):
    """After an accepted step: logPrior = calc_prior(accepted weights) + additional_prob (BNN_env.py:481)."""
    lp = bnn.calc_prior()
    assert abs(mcmc._logPrior - (lp + a)) <= 1e-12 * max(1.0, abs(lp)), (where, mcmc._logPrior, lp, a)


def test_additional_prob_with_device_drawn_proposals():
    """rng="philox", one step per call: after every accepted step logPrior = calc_prior(accepted weights) +
    additional_prob, and a new value reaches the next step.  (This data set is small: the steps run in k_chain_loop.)"""
    bnn, mcmc = _philox_mcmc()
    n_acc = 0
    for t, a in enumerate([-0.7] * 15 + [2.5] * 15 + [0.0] * 10):
        mcmc.mh_step(bnn, additional_prob=a)
        assert mcmc._group.eng.read_state(weights=False).f64[0, L.F_ADD_PROB] == a, t
        if mcmc._last_accepted:
            n_acc += 1
            _check_prior(bnn, mcmc, a, t)
    assert n_acc >= 3


def _runtime_calls(fn):
    """Names of the CUDA runtime calls fn() makes, as the profiler records them."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
    return [e.name for e in prof.events()]


# a never-set value (null pointer), the first value (pointer set: the graphs captured without it are dropped), changes
# that only copy into the buffer, and 0
ADD_PROB_SEQ = (None, None, None, -1.25, -1.25, -1.25, 3.0, 3.0, -0.5, 0.0, 0.0)


def test_additional_prob_reaches_graph_replays():
    """The launch sequence (option chain_loop = 0), whose multi-step calls are captured into CUDA graphs and replayed:
    a value set after a capture reaches the replay, and the first value after never-set ones is not lost in graphs
    captured while it was null.  Graph replays and eager launches (option graphs = 0) end in the same chain with the
    same launch count, and the replays are cudaGraphLaunch calls."""
    runs = []
    for graphs in (1, 0):
        bnn, mcmc = _philox_mcmc(chain_loop=0, graphs=graphs)
        eng = mcmc._group.eng
        traced = None
        for i, a in enumerate(ADD_PROB_SEQ):
            def step():
                if a is None:
                    mcmc.run(bnn, 8)
                else:
                    mcmc.run(bnn, 8, additional_prob=a)
                eng.synchronize()
            if i == len(ADD_PROB_SEQ) - 2:          # a replay in the graphs = 1 run
                traced = _runtime_calls(step)
            else:
                step()
            assert eng.last_kernel != "k_chain_loop", eng.last_kernel
            st = eng.read_state(weights=False)
            assert st.f64[0, L.F_ADD_PROB] == (a or 0.0), (graphs, i, a)     # the last proposal's additional_prob
            if mcmc._last_accepted:
                _check_prior(bnn, mcmc, a or 0.0, (graphs, i))
        st = eng.read_state()
        runs.append((st, eng.launch_count, traced))
    (a, na, ca), (b, nb, cb) = runs
    assert np.array_equal(a.f64, b.f64) and np.array_equal(a.i32, b.i32) and np.array_equal(a.w, b.w)
    assert na == nb and int(a.n_accepted[0]) > 0
    assert "cudaGraphLaunch" in ca and "cudaGraphLaunch" not in cb, (sorted(set(ca)), sorted(set(cb)))


@pytest.mark.parametrize("chain_loop", [1, 0])
def test_additional_prob_zero_is_never_set(chain_loop):
    """additional_prob = 0 set after a non-zero value steps the chain that never had one, in the persistent loop and
    through the eager and graph-replayed launch sequence.  (Both runs are of this code; against earlier builds the
    never-set path is the one bench.py's outputs compare.)"""
    ref_b, ref = _philox_mcmc(chain_loop=chain_loop)
    b0, m0 = _philox_mcmc(chain_loop=chain_loop)
    m0._group.eng.set_additional_prob([1.5])
    m0._group.eng.set_additional_prob([0.0])
    for n in (1, 8, 8, 8, 30):
        ref.run(ref_b, n)
        m0.run(b0, n)
    assert (ref._group.eng.last_kernel == "k_chain_loop") == bool(chain_loop)
    a, b = ref._group.eng.read_state(), m0._group.eng.read_state()
    assert np.array_equal(a.i32, b.i32) and np.array_equal(a.f64, b.f64) and np.array_equal(a.w, b.w)
    assert int(a.n_accepted[0]) > 0


def test_additional_prob_entry_point_validates():
    bnn, mcmc = _philox_mcmc()
    eng = mcmc._group.eng
    with pytest.raises(L.NpbnnError):
        eng.set_additional_prob([np.nan])
    eng.set_additional_prob([0.25])
    eng.mh_steps(1)
    assert eng.read_state(weights=False).f64[0, L.F_ADD_PROB] == 0.25
    eng.set_additional_prob(None)                          # back to none
    eng.mh_steps(1)
    assert eng.read_state(weights=False).f64[0, L.F_ADD_PROB] == 0.0


# ---------------------------------------------------------------------------------------------- rank layouts
def _run_tool(outdir, n_chains, world, rng):
    tool = os.path.join(ROOT, "tools", "mc3_trainable_multi.py")
    env = dict(os.environ, MC3_RNG=rng)
    if world == 1:
        cmd = [sys.executable, tool, outdir, str(n_chains)]
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
               "--master-port", str(36500 + (os.getpid() + 7 * world + n_chains) % 2000), tool, outdir, str(n_chains)]
    subprocess.run(cmd, check=True, env=env, timeout=900)
    (log,) = glob.glob(os.path.join(outdir, "*.log"))
    (pkl,) = glob.glob(os.path.join(outdir, "*.pkl"))
    return open(log, "rb").read(), pickle.load(open(pkl, "rb"))[2]._post_weight_samples


# (chains, ranks): chain sharding (4 chains on 2 ranks: 2 x 1) and chain blocks x row shards grids (mc3.chain_grid:
# 4 chains on 8 ranks: 4 x 2, 2 chains on 4 ranks: 2 x 2, one chain on 2 ranks: 1 x 2).  Ranks beyond the GPU count
# share GPUs over gloo; with a GPU per rank the ranks use NCCL.
LAYOUTS = [(4, 2), (4, 8), (2, 4), (1, 2)]


@pytest.mark.parametrize("rng", ["host", "philox"])
def test_rank_layouts_write_the_single_rank_files(rng, tmp_path):
    """Every layout writes the .log and keeps the .pkl posterior samples (weights, alphas) of the one-rank run of the
    same chains.  The logged cold chain is rank 0's own in some rows and, in others, a chain another rank owns and
    sends (MC3._log_on_rank0), both under chain sharding and on a grid: the runs start with the cold temperature on the
    last chain block, and the swaps move it."""
    import warnings
    import torch
    from npbnn_b200 import mc3 as M
    ran, ones = [], {}
    owners_seen = set()
    for n_chains, world in LAYOUTS:
        if n_chains not in ones:
            ones[n_chains] = _run_tool(str(tmp_path / ("one_c%d" % n_chains)), n_chains, 1, rng)
        one = ones[n_chains]
        many = _run_tool(str(tmp_path / ("c%d_w%d" % (n_chains, world))), n_chains, world, rng)
        Q, R = M.chain_grid(n_chains, world)
        rows_a, rows_b = one[0].decode().split("\r\n"), many[0].decode().split("\r\n")
        assert len(rows_a) == len(rows_b) > 10
        if R == 1:
            assert one[0] == many[0], (n_chains, world)           # byte-identical .log
        else:
            # a row shard sums its own rows: logLik / logPost / logPrior agree to the last bits, everything else exactly
            for ra, rb in zip(rows_a[1:], rows_b[1:]):
                fa, fb = ra.split("\t"), rb.split("\t")
                assert fa[0] == fb[0] and fa[4:] == fb[4:], (n_chains, world, ra, rb)
                if fa[1:4] != fb[1:4]:
                    assert _rel([float(v) for v in fa[1:4]], [float(v) for v in fb[1:4]], 1e-12)
        # the last column is the cold chain's mcmc_id: which rank held the chain each logged row came from
        owners = {M.owner_of(int(r.split("\t")[-1]), n_chains, world, R) for r in rows_b[1:] if r}
        owners_seen |= {("sent" if o > 0 else "own", "grid" if R > 1 else "chain-sharded") for o in owners}
        assert len(one[1]) == len(many[1]) > 5
        for sa, sb in zip(one[1], many[1]):
            assert sa["mcmc_it"] == sb["mcmc_it"] and np.array_equal(sa["alphas"], sb["alphas"])
            for wa, wb in zip(sa["weights"], sb["weights"]):
                assert np.array_equal(wa, wb)
        backend = "nccl" if world <= torch.cuda.device_count() else "gloo, %d GPU(s) shared" % torch.cuda.device_count()
        ran.append("%d chains on %d ranks (%d x %d, %s, cold chain from ranks %s)" %
                   (n_chains, world, Q, R, backend, sorted(owners)))
    # rows from rank 0's own cold chain, and from cold chains that another rank sends, under chain sharding and on a grid
    assert {("sent", "chain-sharded"), ("sent", "grid")} <= owners_seen and "own" in {o for o, _ in owners_seen}
    warnings.warn("rank layouts run (rng=%s): %s" % (rng, "; ".join(ran)))
    assert len(ran) == len(LAYOUTS)
