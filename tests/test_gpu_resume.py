"""GPU: resumable samplers.  A run of 2N iterations against the same run split at iteration N, where the second half
runs in a new Python process from the [bnn, mcmc, logger] pickle (load_obj -> raise _n_iterations -> run_mcmc), or from
a pickled MC3: the .log files are byte-identical, the final state rows and weights bit-identical and the posterior sample
lists equal."""
import json
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from npbnn_b200 import _lib as L
from oracle import npbnn_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 60                     # the split point (a sampling point); the full run has 2N iterations
# adaptation every 5 iterations up to 1.5 N, on both sides of the split: an acceptance rate (k / d, d <= 101) is never
# 0.905, so every adaptation point shrinks or widens the proposals
ADAPT = dict(adapt_freq=5, adapt_f=0.905, adapt_fM=0.905, adapt_stop=int(1.5 * N))
RUN = dict(sampling_f=10, print_f=20, n_post_samples=5)

CHILD = r'''
import pickle, sys
sys.path.insert(0, %(root)r)
import numpy as np
import npbnn_b200 as bn
from npbnn_b200.engine import flatten_weights
pkl, out, n_total, np_state = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4]
if np_state != "-":
    with open(np_state, "rb") as f:
        np.random.set_state(pickle.load(f))
bnn, mcmc, logger = bn.load_obj(pkl)
mcmc._n_iterations = n_total
bn.run_mcmc(bnn, mcmc, logger)
with open(out, "wb") as f:
    pickle.dump({"f64": mcmc._chain_state["f64"], "i32": mcmc._chain_state["i32"], "w": flatten_weights(bnn._w_layers),
                 "post": logger._post_weight_samples, "kernel": mcmc._group.eng.last_kernel}, f)
'''

MC3_CHILD = r'''
import pickle, sys
sys.path.insert(0, %(root)r)
import numpy as np
import npbnn_b200 as bn
from npbnn_b200.engine import flatten_weights
pkl, out, n_periods, np_state = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4]
with open(np_state, "rb") as f:
    np.random.set_state(pickle.load(f))
with open(pkl, "rb") as f:
    mc3 = pickle.load(f)
mc3.n_mc3_iteration = n_periods
mc3.run_mcmc()
with open(out, "wb") as f:
    pickle.dump({
        "temps": mc3.current_temperatures,
        "f64": np.stack([m._chain_state["f64"] for _, m in mc3.singleChainArgs]),
        "i32": np.stack([m._chain_state["i32"] for _, m in mc3.singleChainArgs]),
        "w": np.stack([flatten_weights(b._w_layers) for b, _ in mc3.singleChainArgs]),
        "post": mc3.logger._post_weight_samples}, f)
'''


def _child(tmp_path, script, *args):
    path = tmp_path / "child.py"
    path.write_text(script % {"root": ROOT})
    out = tmp_path / "child_out.pkl"
    r = subprocess.run([sys.executable, str(path)] + [str(a) for a in args[:1]] + [str(out)] + [str(a) for a in args[1:]],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    with open(out, "rb") as f:
        return pickle.load(f)


def _same_posterior(a, b):
    assert len(a) == len(b) and len(a) > 0
    for x, y in zip(a, b):
        assert sorted(x) == sorted(y)
        assert x["mcmc_it"] == y["mcmc_it"]
        assert all(np.array_equal(u, v) for u, v in zip(x["weights"], y["weights"]))
        assert np.array_equal(np.asarray(x["alphas"]), np.asarray(y["alphas"]))
        if "error_prm" in x:
            assert np.array_equal(np.asarray(x["error_prm"]), np.asarray(y["error_prm"]))


# ------------------------------------------------------------------------------------------------ models
def _cls_data(n, f, k, seed, n_test=0):
    rs = np.random.default_rng(seed)
    x = rs.standard_normal((n + n_test, f))
    t = rs.normal(0, 1, (k, f))
    y = np.argmax(x @ t.T + rs.normal(0, 0.5, (n + n_test, k)), axis=1)
    return {"data": x[:n], "labels": y[:n], "test_data": x[n:], "test_labels": y[n:]}


def _c1(bn):
    np.random.seed(11)
    return bn.npBNN(_cls_data(2250, 128, 5, 1, n_test=250), n_nodes=[5, 5], actFun=bn.ActFun(fun="tanh"), use_bias_node=2,
                    seed=11)


def _c4(bn):
    from npbnn_b200 import workloads as wl
    x, y = wl.c4_data(40000, seed=2)
    np.random.seed(12)
    return bn.npBNN({"data": x, "labels": y, "test_data": [], "test_labels": []}, n_nodes=[64, 32],
                    actFun=bn.ActFun(fun="swish"), use_bias_node=-1, seed=12)


def _regress(bn):
    rs = np.random.default_rng(3)
    x = rs.standard_normal((600, 6))
    y = np.sin(x[:, :2]) + 0.1 * rs.standard_normal((600, 2))
    np.random.seed(13)
    af = bn.ActFun(fun="genReLU", prm=np.array([0.05, 0.1]), trainable=True)
    return bn.npBNN({"data": x[:500], "labels": y[:500], "test_data": x[500:], "test_labels": y[500:]}, n_nodes=[8, 4],
                    estimation_mode="regression", empirical_error=True, actFun=af, seed=13)


def _hyper(bn):
    np.random.seed(14)
    bnn = bn.npBNN(_cls_data(800, 7, 3, 4), n_nodes=[6, 4], actFun=bn.ActFun(fun="tanh"), use_bias_node=2, hyper_p=1,
                   seed=14)
    bnn.sample_prior_scale()
    return bnn


def _indicators(bn):
    np.random.seed(15)
    return bn.npBNN(_cls_data(800, 9, 3, 5), n_nodes=[6, 5, 4], actFun=bn.ActFun(fun="tanh"), use_bias_node=2,
                    freq_indicator=0.3, feature_indicators=True, seed=15)


def _poisson(bn):
    rs = np.random.default_rng(6)
    x = rs.standard_normal((700, 5))
    y = rs.poisson(np.exp(0.5 + x @ rs.normal(0, 0.4, (1, 5)).T)).astype(np.float64)
    np.random.seed(16)
    return bn.npBNN({"data": x[:600], "labels": y[:600], "test_data": x[600:], "test_labels": y[600:]}, n_nodes=[8, 4],
                    estimation_mode="custom", size_output=1, output_act_fun=bn.RegressTransform, seed=16)


def _masked(bn):
    np.random.seed(17)
    bnn = bn.npBNN(_cls_data(3000, 8, 4, 7), n_nodes=[24, 16], actFun=bn.ActFun(fun="tanh"), use_bias_node=-1, seed=17)
    m = bn.create_mask(bnn._w_layers, indx_input_list=[list(range(8)), sum(([g] * 3 for g in range(8)), []), []],
                       nodes_per_feature_list=[[3] * 8, [2] * 8, []])
    bnn.apply_mask(m)
    return bnn


# name: (model, MCMC keywords, kernel the steps run in (prefix), global numpy draws in the run)
CASES = {
    "c1_host": (_c1, dict(rng="host"), "k_chain_loop", False),
    "c1_philox": (_c1, dict(rng="philox"), "k_chain_loop", False),
    "c4_philox": (_c4, dict(rng="philox"), "k_fwd3", False),
    "regression_genrelu": (_regress, dict(), None, False),
    "hyper_p1": (_hyper, dict(), None, False),
    "indicators_host": (_indicators, dict(), None, True),
    "poisson": (_poisson, dict(likelihood_f="poi_likelihood"), None, False),
    "block_masked": (_masked, dict(), "k_fwd_sparse", False),
}


def _sampler(bn, name, tmp, n_iteration):
    make, kw, _, _ = CASES[name]
    bnn = make(bn)
    kw = dict(kw)
    if "likelihood_f" in kw:
        kw["likelihood_f"] = getattr(bn, kw["likelihood_f"])
    mcmc = bn.MCMC(bnn, n_iteration=n_iteration, **RUN, **ADAPT, **kw)
    os.makedirs(tmp, exist_ok=True)
    logger = bn.postLogger(bnn, filename=os.path.join(str(tmp), "run"))
    return bnn, mcmc, logger


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_split_run_continues_bit_for_bit(tmp_path, name):
    import npbnn_b200 as bn
    from npbnn_b200.engine import flatten_weights
    kernel, global_draws = CASES[name][2], CASES[name][3]
    # the split run: N iterations here, N more in a new process from the pickle
    bnn, mcmc, logger = _sampler(bn, name, tmp_path / "split", 2 * N)
    mcmc._n_iterations = N
    bn.run_mcmc(bnn, mcmc, logger)
    state_at_n = np.array(mcmc._chain_state["f64"])
    np_state = "-"
    if global_draws:
        np_state = tmp_path / "np_state.pkl"
        with open(np_state, "wb") as f:
            pickle.dump(np.random.get_state(), f)
    split = _child(tmp_path, CHILD, logger._pklfile, 2 * N, np_state)
    # the uninterrupted run
    bnn2, mcmc2, logger2 = _sampler(bn, name, tmp_path / "full", 2 * N)
    bn.run_mcmc(bnn2, mcmc2, logger2)
    with open(logger._logfile, "rb") as f1, open(logger2._logfile, "rb") as f2:
        log1, log2 = f1.read(), f2.read()
    assert log1.count(b"\n") == 1 + 2 * N // RUN["sampling_f"]
    assert log1 == log2
    assert np.array_equal(split["f64"], mcmc2._chain_state["f64"])
    assert np.array_equal(split["i32"], mcmc2._chain_state["i32"])
    assert np.array_equal(split["w"], flatten_weights(bnn2._w_layers))
    _same_posterior(split["post"], logger2._post_weight_samples)
    assert int(split["i32"][L.I_ITERATION]) == 2 * N
    if kernel is not None:
        assert split["kernel"].startswith(kernel) and mcmc2._group.eng.last_kernel.startswith(kernel)
    # adaptation fired before and after the split
    assert 0.05 != state_at_n[L.F_UPDATE_F] != split["f64"][L.F_UPDATE_F]


@pytest.mark.gpu
@pytest.mark.parametrize("rng,swap_seed", [("host", None), ("philox", None), ("host", 5)])
def test_pickled_mc3_continues_bit_for_bit(tmp_path, rng, swap_seed):
    """swap_seed=None: swaps from numpy's global generator, whose state the caller restores; swap_seed: a seeded
    SwapRNG, which the pickle carries."""
    import npbnn_b200 as bn
    from npbnn_b200.engine import flatten_weights
    period, P = 10, 4

    def build(tmp, n_periods):
        np.random.seed(21)
        bnn = bn.npBNN(_cls_data(1500, 10, 3, 8), n_nodes=[6, 4], actFun=bn.ActFun(fun="tanh"), use_bias_node=2, seed=21)
        os.makedirs(tmp, exist_ok=True)
        logger = bn.postLogger(bnn, filename=os.path.join(str(tmp), "mc3"))
        mc3 = bn.MC3(bnn, logger, n_chains=4, swap_frequency=period, n_iteration=period * n_periods, verbose=0,
                     sampling_f=period, n_post_samples=5, adapt_freq=5, adapt_f=0.9, adapt_fM=0.95, adapt_stop=60,
                     min_temperature=0.5, rng=rng, swap_seed=swap_seed)
        return mc3

    mc3 = build(tmp_path / "split", 2 * P)
    mc3.n_mc3_iteration = P
    mc3.run_mcmc()
    pkl = tmp_path / "mc3_state.pkl"
    with open(pkl, "wb") as f:
        pickle.dump(mc3, f)
    np_state = tmp_path / "np_state.pkl"
    with open(np_state, "wb") as f:
        pickle.dump(np.random.get_state(), f)
    split = _child(tmp_path, MC3_CHILD, pkl, P, np_state)
    full = build(tmp_path / "full", 2 * P)
    full.run_mcmc()
    with open(mc3.logger._logfile, "rb") as f1, open(full.logger._logfile, "rb") as f2:
        assert f1.read() == f2.read()
    assert np.array_equal(split["temps"], full.current_temperatures)
    st = full._group.eng.read_state()
    assert np.array_equal(split["f64"], st.f64) and np.array_equal(split["i32"], st.i32)
    assert np.array_equal(split["w"], np.stack([flatten_weights(b._w_layers) for b, _ in full.singleChainArgs]))
    assert np.array_equal(split["w"], st.w)
    _same_posterior(split["post"], full.logger._post_weight_samples)
    assert np.all(st.iteration == 2 * P * period)


def _old_pickle(cls, d):
    """An object of `cls` that unpickles to exactly the attribute dict d, as a pickle of an earlier version does."""
    o = cls.__new__(cls)
    o.__dict__.update(d)
    return _Raw(o)


class _Raw:
    """Pickles `o` with its __dict__ as it is, bypassing o.__getstate__."""

    def __init__(self, o):
        self.o = o

    def __reduce__(self):
        return _restore_raw, (type(self.o), self.o.__dict__)


def _restore_raw(cls, d):
    o = cls.__new__(cls)
    o.__setstate__(dict(d))
    return o


@pytest.mark.gpu
def test_refusals_of_pickles_that_cannot_resume(tmp_path):
    import npbnn_b200 as bn
    # a pickle written before samplers carried their state: stepping raises, prediction still reads it
    bnn, mcmc, logger = _sampler(bn, "c1_host", tmp_path / "old", 2 * N)
    mcmc._n_iterations = 20
    bn.run_mcmc(bnn, mcmc, logger)
    b, m, lg = bn.load_obj(logger._pklfile)
    # what MCMC.__getstate__ wrote before samplers carried their state: no state rows, generator or sharding flag
    d = {k: v for k, v in m.__dict__.items() if k not in ("_chain_state", "_rs_state", "_rs", "_device", "_row_sharded")}
    d.update(_rs=None, update_function=None, _n_iterations=40)
    m = pickle.loads(pickle.dumps(_old_pickle(bn.MCMC, d)))
    with pytest.raises(RuntimeError, match="npBNN\\(pickle_file"):
        bn.run_mcmc(b, m, lg)
    with pytest.raises(RuntimeError, match="npBNN\\(pickle_file"):
        m.mh_step(b)
    res = bn.get_posterior_est(logger._pklfile)
    assert res["post_est"].shape[0] == len(lg._post_weight_samples)
    # the cold-chain pickle of an MC3 run: resume the MC3 object instead
    np.random.seed(3)
    b3 = bn.npBNN(_cls_data(400, 5, 3, 9), n_nodes=[4, 3], actFun=bn.ActFun(fun="tanh"), seed=3)
    lg3 = bn.postLogger(b3, filename=str(tmp_path / "mc3"))
    mc3 = bn.MC3(b3, lg3, n_chains=3, swap_frequency=10, n_iteration=20, verbose=0, sampling_f=10)
    mc3.run_mcmc()
    b, m, lg = bn.load_obj(lg3._pklfile)
    m._n_iterations = 100
    with pytest.raises(RuntimeError, match="MC3 object"):
        bn.run_mcmc(b, m, lg)
    # a row-sharded sampler
    b, m, lg = bn.load_obj(logger._pklfile)
    m._row_sharded = True
    with pytest.raises(NotImplementedError, match="row-sharded"):
        m.mh_step(b)


@pytest.mark.gpu
def test_fresh_sampler_from_non_unit_indicators():
    """npBNN._indicators / _feature_indicators set before MCMC.__init__: the chain starts from them (the initial
    logPrior is calc_prior() with the indicator term, the initial logLik that of w0 * ind on the transformed features),
    and the first steps run from there."""
    import npbnn_b200 as bn
    bnn = _indicators(bn)
    rs = np.random.default_rng(30)
    bnn._indicators = rs.integers(0, 2, bnn._w_layers[0].shape).astype(np.float64)
    bnn._feature_indicators = np.array([1, 0, 1, 1, 0, 1, 1, 1, 0])
    mcmc = bn.MCMC(bnn, n_iteration=100, rng="host")
    assert np.array_equal(mcmc._chain_state["ind"], bnn._indicators)
    assert np.array_equal(mcmc._chain_state["fi"], [1, 0, 1, 1, 0, 1, 1, 1, 0])
    assert abs(mcmc._logPrior - bnn.calc_prior()) <= 1e-9 * abs(bnn.calc_prior())
    x = orc.feature_transform(bnn._data, bnn._feature_indicators, bnn._feature_means)
    y = orc.forward(x, bnn._w_layers, "tanh", None, "softmax", indicators=bnn._indicators)
    ll = orc.loglik_categorical(y, bnn._labels)
    assert abs(mcmc._logLik - ll) <= 1e-9 * abs(ll)
    assert mcmc._accuracy == np.mean(np.argmax(y, axis=1) == bnn._labels)
    mcmc.run(bnn, 10)
    assert mcmc._current_iteration == 10


DIST_WORKER = r'''
import json, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch.distributed as dist
import npbnn_b200 as bn
rank, store = int(sys.argv[1]), sys.argv[2]
dist.init_process_group("gloo", store=dist.FileStore(store, 2), rank=rank, world_size=2)
# the states rank 0 pickles: a row-sharded MCMC and an MC3 run on two ranks
m = bn.MCMC.__new__(bn.MCMC)
m.__setstate__({"_group": None, "_rs": None, "_chain_state": {}, "_own_group": True, "_row_sharded": True,
                "_n_iterations": 10, "_current_iteration": 0})
mc3 = bn.MC3.__new__(bn.MC3)
mc3.__dict__.update({"_group": None, "world": 2})
out = []
for step in (lambda: bn.run_mcmc(None, m, None), lambda: m.mh_step(None), mc3.run_mcmc):
    try:
        step()
        out.append("ran")
    except NotImplementedError as e:
        out.append("refused: " + str(e))
print(json.dumps(out))
dist.destroy_process_group()
'''


def test_resuming_over_ranks_is_refused_gloo(tmp_path):
    """Two gloo ranks on CPU: an unpickled row-sharded MCMC and an unpickled two-rank MC3 refuse to continue, before any
    device work, with the reason."""
    script = tmp_path / "w.py"
    script.write_text(DIST_WORKER % {"root": ROOT})
    procs = [subprocess.Popen([sys.executable, str(script), str(r), str(tmp_path / "store")], stdout=subprocess.PIPE,
                              text=True) for r in range(2)]
    try:
        outs = [p.communicate(timeout=240)[0] for p in procs]
    finally:
        for p in procs:          # a rank left waiting for its peer does not outlive the test
            if p.poll() is None:
                p.kill()
                p.wait()
    assert all(p.returncode == 0 for p in procs)
    for o in outs:
        res = json.loads(o.strip().splitlines()[-1])
        assert len(res) == 3 and all(r.startswith("refused: ") and "rank 0" in r for r in res), res


class _EveryPickle(__import__("npbnn_b200").postLogger):
    """postLogger that keeps the bytes of every pickle it writes (the async writer keeps only the newest)."""

    def _save(self, objs):
        _EveryPickle.kept.append((objs[1]._current_iteration, pickle.dumps(objs)))


@pytest.mark.gpu
def test_pipelined_run_resumes_from_an_intermediate_logging_point(tmp_path):
    """rng="philox" with weight and feature indicators through the pipelined run_mcmc, which queues the steps of later
    logging points before it exports one: the pickle written at an intermediate point holds the indicators of that
    point's iteration, and the run resumed from it ends bit-identical to the uninterrupted run; the pipelined run's
    logged samples are those of the synchronous loop."""
    import npbnn_b200 as bn
    from npbnn_b200.engine import flatten_weights

    def build(tmp, cls=bn.postLogger):
        bnn = _indicators(bn)
        mcmc = bn.MCMC(bnn, n_iteration=2 * N, rng="philox", sampling_f=10, print_f=1000, n_post_samples=100, **ADAPT)
        os.makedirs(tmp, exist_ok=True)
        return bnn, mcmc, cls(bnn, filename=os.path.join(str(tmp), "run"))

    _EveryPickle.kept = []
    bnn, mcmc, logger = build(tmp_path / "keep", _EveryPickle)
    bn.run_mcmc(bnn, mcmc, logger, pipeline_depth=4)
    b0, m0, l0 = build(tmp_path / "sync")
    bn.run_mcmc(b0, m0, l0, pipeline_depth=0)
    with open(logger._logfile, "rb") as f1, open(l0._logfile, "rb") as f2:
        assert f1.read() == f2.read()
    _same_posterior(logger._post_weight_samples, l0._post_weight_samples)
    assert np.array_equal(mcmc._chain_state["f64"], m0._chain_state["f64"])
    it, blob = _EveryPickle.kept[2]
    assert it == 30
    b, m, lg = pickle.loads(blob)
    assert np.array_equal(m._chain_state["ind"], b._indicators)
    b1, m1, l1 = build(tmp_path / "resumed")
    bn.run_mcmc(b, m, l1)
    assert np.array_equal(m._chain_state["f64"], mcmc._chain_state["f64"])
    assert np.array_equal(m._chain_state["i32"], mcmc._chain_state["i32"])
    assert np.array_equal(m._chain_state["ind"], mcmc._chain_state["ind"])
    assert np.array_equal(m._chain_state["fi"], mcmc._chain_state["fi"])
    assert np.array_equal(flatten_weights(b._w_layers), flatten_weights(bnn._w_layers))


@pytest.mark.gpu
def test_device_additional_prob_survives_a_resume():
    """mh_step(additional_prob=a) with rng="philox" keeps a as the chain's device value: an unpickled sampler writes it
    back, and stepping on with the same a continues bit for bit."""
    import npbnn_b200 as bn
    from npbnn_b200.engine import flatten_weights
    a = -0.75

    def build():
        bnn = _c1(bn)
        return bnn, bn.MCMC(bnn, n_iteration=100, rng="philox", **ADAPT)

    bnn, mcmc = build()
    mcmc.run(bnn, 30, additional_prob=a)
    b, m = pickle.loads(pickle.dumps([bnn, mcmc]))
    assert m._chain_state["add_prob"] == a
    mcmc.run(bnn, 30, additional_prob=a)
    m.run(b, 30, additional_prob=a)
    assert np.array_equal(m._chain_state["f64"], mcmc._chain_state["f64"])
    assert np.array_equal(m._chain_state["i32"], mcmc._chain_state["i32"])
    assert np.array_equal(flatten_weights(b._w_layers), flatten_weights(bnn._w_layers))
    # the value entered the chain: a run with additional_prob=0 differs
    b2, m2 = build()
    m2.run(b2, 60)
    assert m2._chain_state["f64"][L.F_LOGPRIOR] != mcmc._chain_state["f64"][L.F_LOGPRIOR]
