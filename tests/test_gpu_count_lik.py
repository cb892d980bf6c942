"""GPU: the count likelihoods of estimation_mode="custom" (BNN_LIK_POISSON / NEGBIN / NEGBIN10, BNN_lik.py:5-66) against
the oracle -- scoring on every forward kernel (k_fwd3 families, the generic kernel, the persistent chain loop, the
block-sparse kernels), replayed MH chains, the Python surface (log, pickle, prediction, MC3) and a statistical check
against a known Poisson teacher."""
import csv
import os

import numpy as np
import pytest

from npbnn_b200 import _lib as L
from oracle import npbnn_oracle as orc
from tests import count_oracle as corc
from tests.test_gpu_parity import rel_close

pytestmark = pytest.mark.gpu

ACTS = ["ReLU", "genReLU", "swish", "tanh"]
KIND = {"poisson": L.LIK_POISSON, "negbin": L.LIK_NEGBIN, "negbin10": L.LIK_NEGBIN10}
# output width per mode: Poisson reads column 0 of two, negbin models two label columns (negbin_likelihood2d), negbin10
# one (negbin_likelihood_base10)
WIDTH = {"poisson": 2, "negbin": 4, "negbin10": 2}
PFX = {"ReLU": "relu", "genReLU": "leaky", "swish": "swish", "tanh": "tanh"}


def _shapes(f, hidden, out, bias):
    b1, b2, b3 = int(bias >= 1), int(bias >= 2), int(bias in (3, -1))
    return [(hidden[0], f + b1), (hidden[1], hidden[0] + b2), (out, hidden[1] + b3)]


def _problem(mode, n, f, hidden, act, bias, seed, n_sets=3, n_test=0, mask=None, shapes=None):
    rng = np.random.default_rng(seed)
    shapes = shapes or _shapes(f, hidden, WIDTH[mode], bias)
    out = shapes[-1][0]
    x = rng.standard_normal((n + n_test, f))
    alphas = np.array([0.05, 0.3]) if act == "genReLU" else None
    teacher = [rng.normal(0, 0.3, s) for s in shapes]
    z = orc.forward(x, teacher, act, alphas, "identity")
    n_lab = 1 if mode != "negbin" else out // 2
    lab = rng.poisson(np.exp(np.clip(z[:, :n_lab], -3, 3))).astype(np.float64)
    lab[::13] = 0.0
    # weight scale: outputs stay in a range where the reference's formula is well conditioned (with p -> 1, 1 - p
    # amplifies a one-ulp difference of exp between libraries; the kinds of non-finite value are checked separately)
    sd = 0.3 * min(1.0, np.sqrt(32.0 / f))
    sets = [[rng.normal(0, sd, s) * (1 if mask is None else m) for s, m in zip(shapes, mask or shapes)]
            for _ in range(n_sets)]
    m = corc.CountModel(x=x[:n], labels=lab[:n], weights=[w.copy() for w in sets[0]], act=act, alphas=alphas, mode=mode,
                  x_test=x[n:] if n_test else None, labels_test=lab[n:] if n_test else None, mask=mask)
    return m, sets, alphas


def _engine(m, **opts):
    from npbnn_b200.engine import Engine, NetShape
    eng = Engine(NetShape.from_weights(m.weights, m.x.shape[1], act=m.act, lik=KIND[m.mode]))
    for k, v in opts.items():
        eng.set_option(k, v)
    eng.set_data(m.x, m.labels, m.x_test, m.labels_test)
    return eng


def _alpha_rows(alphas, n):
    return None if alphas is None else np.tile(np.resize(alphas, 3), (n, 1))


def _check_scores(eng, m, sets, alphas, kernel_prefix):
    res = eng.forward_lik(sets, alphas=_alpha_rows(alphas, len(sets)), lik_temp=0.5)     # lik_temp is ignored
    assert eng.last_kernel.startswith(kernel_prefix), eng.last_kernel
    for i, w in enumerate(sets):
        y = orc.forward(m.x, w, m.act, m.alphas, "identity")
        ref = corc.loglik_count(y, m.labels, m.mode)
        assert rel_close(res["loglik"][i], ref), (i, res["loglik"][i], ref)
        sr, sr2 = corc.count_sums(y, m.labels, m.mode)
        scale = np.sqrt(sr2 * len(y))
        assert np.allclose(res["sums"][i][0], sr, rtol=1e-9, atol=1e-12 * np.max(scale))
        assert rel_close(res["sums"][i][1], sr2)
        if m.x_test is not None:
            yt = orc.forward(m.x_test, w, m.act, m.alphas, "identity")
            assert rel_close(res["sums"][i][2], corc.count_sums(yt, m.labels_test, m.mode)[1])
    return res


def test_non_finite_values_have_the_host_formulas_kind():
    """One linear layer on all-zero features: every row's output is the bias, so each weight set is one (z0, z1) pair,
    from underflow to overflow of exp / 10**.  Device log-likelihoods are NaN / -inf exactly where the oracle's are,
    and equal to it at moderate outputs."""
    from npbnn_b200.engine import Engine, NetShape
    zs = [-800.0, -400.0, -40.0, -1.0, 0.0, 1.0, 40.0, 400.0, 800.0]
    pairs = [(a, b) for a in zs for b in zs]
    sets = np.array([[a, 0.0, b, 0.0] for a, b in pairs])          # [2, 1 + 1] layer: bias in column 0
    kinds = set()
    for mode in ("poisson", "negbin", "negbin10"):
        for k in (0.0, 1.0, 37.0, 1e6):
            eng = Engine(NetShape(1, [(2, 2)], act="tanh", lik=KIND[mode]))
            x, lab = np.zeros((40, 1)), np.full((40, 1), k)
            eng.set_data(x, lab)
            got = eng.forward_lik(sets)["loglik"]
            assert eng.last_kernel == "k_fwd_generic"
            for (a, b), g in zip(pairs, got):
                ref = corc.loglik_count(np.tile([[a, b]], (40, 1)), lab, mode)
                if np.isnan(ref) or np.isinf(ref):
                    assert (np.isnan(g) and np.isnan(ref)) or g == ref, (mode, k, a, b, g, ref)
                    kinds.add("nan" if np.isnan(ref) else str(ref))
                elif abs(a) <= 1 and abs(b) <= 1:
                    assert rel_close(g, ref), (mode, k, a, b, g, ref)
                else:
                    assert np.isfinite(g), (mode, k, a, b, g, ref)
            eng.close()
    assert {"nan", "-inf"} <= kinds


def _inj_arrays(inj, nl):
    cap = max(1, sum(len(l[0]) for l in inj.layers if l is not None))
    arr = {"proposed": np.zeros((1, 1, nl), np.int32), "count": np.zeros((1, 1, nl), np.int32),
           "ix": np.zeros((1, 1, cap), np.int32), "iy": np.zeros((1, 1, cap), np.int32),
           "dz": np.zeros((1, 1, cap)), "log_u": np.full((1, 1), inj.log_u)}
    o = 0
    for l, lay in enumerate(inj.layers):
        if lay is None:
            continue
        cnt = len(lay[0])
        arr["proposed"][0, 0, l], arr["count"][0, 0, l] = 1, cnt
        arr["ix"][0, 0, o:o + cnt], arr["iy"][0, 0, o:o + cnt], arr["dz"][0, 0, o:o + cnt] = lay
        o += cnt
    return arr


def _replay(eng, m, w0, alphas, n_steps, kernel, mask=None, seed=2):
    """n_steps injected MH iterations on the device and in the oracle: same decisions, logLik_prop within 1e-9,
    bit-identical final weights."""
    nl = len(w0)
    s = corc.make_sampler(m, n_iteration=1000, update_f=[0.1] * nl, lik_temp=0.5)
    eng.chains_init([w0], update_f=[0.1] * nl, alphas=None if alphas is None else np.resize(alphas, nl), mask=mask,
                    adapt_stop=50, lik_temp=0.5)
    st = eng.read_state()
    assert rel_close(st.logLik[0], s.logLik) and rel_close(st.logPrior[0], s.logPrior)
    rs = np.random.default_rng(seed)
    n_acc = 0
    for it in range(n_steps):
        inj = orc.draw_injection(m, s, rs)
        d = corc.mh_step(m, s, inj)
        eng.mh_steps(1, _inj_arrays(inj, nl))
        assert eng.last_kernel.startswith(kernel), eng.last_kernel
        st = eng.read_state()
        assert st.last_accepted[0] == d["accepted"], it
        assert rel_close(st.logLik_prop[0], d["logLik_prime"]), (it, st.logLik_prop[0], d["logLik_prime"])
        n_acc += d["accepted"]
    for a, b in zip(st.weights(0), m.weights):
        assert np.array_equal(a, b)
    n = m.x.shape[0]
    assert np.isclose(np.sum(st.sum_r2[0]) / (n * eng.K), s.accuracy, rtol=1e-9)
    return n_acc


@pytest.mark.parametrize("act", ACTS)
@pytest.mark.parametrize("mode", ["poisson", "negbin", "negbin10"])
@pytest.mark.parametrize("family", ["A", "B"])
def test_fwd3_families_score_count_likelihoods(family, mode, act):
    """4,099 + 200 test rows (ragged last tile, train / test boundary inside a tile) on the exact-width families,
    then the generic kernel on the same layout."""
    f, hidden = (64, (64, 32)) if family == "A" else (32, (32, 16))
    m, sets, alphas = _problem(mode, 4099, f, hidden, act, bias=-1 if family == "A" else 2, seed=11, n_test=200)
    eng = _engine(m)
    _check_scores(eng, m, sets, alphas, "k_fwd3<%s,%d,%d,%d" % (PFX[act], f, hidden[0], hidden[1]))
    eng.set_option("force_generic", 1)
    _check_scores(eng, m, sets, alphas, "k_fwd_generic")
    eng.close()


@pytest.mark.parametrize("mode", ["poisson", "negbin", "negbin10"])
def test_padded_up_network_and_mh_replay(mode):
    """A smaller three-layer network on 30,011 rows is padded up to family B: scores, then 6 replayed MH steps on
    k_fwd3; then 8 replayed steps of another chain on the generic kernel (force_generic, no chain loop)."""
    m, sets, alphas = _problem(mode, 30_011, 20, (24, 12), "swish", 2, seed=5, n_test=333)
    eng = _engine(m)
    _check_scores(eng, m, sets, alphas, "k_fwd3<swish,32,32,16")
    _replay(eng, m, sets[0], alphas, 6, "k_fwd3<swish,32,32,16")
    eng.close()
    m, sets, alphas = _problem(mode, 4099, 20, (24, 12), "tanh", 2, seed=6, n_test=100)
    eng = _engine(m, force_generic=1, chain_loop=0)
    _replay(eng, m, sets[0], alphas, 8, "k_fwd_generic")
    eng.close()


@pytest.mark.parametrize("mode", ["poisson", "negbin", "negbin10"])
def test_chain_loop_replay(mode):
    """Small data (the reference's example sizes): the MH steps run inside the persistent k_chain_loop."""
    m, sets, alphas = _problem(mode, 400, 6, (5, 5), "tanh", 1, seed=7, n_test=50)
    eng = _engine(m, chain_loop=2)
    _replay(eng, m, sets[0], alphas, 8, "k_chain_loop")
    eng.close()


@pytest.mark.parametrize("mode", ["poisson", "negbin"])
def test_block_masked_count_model(mode):
    """create_mask-style block network: scored at chains_init and stepped on the sparse kernel the dispatcher picks."""
    f, g1, g2 = 12, 3, 2
    shapes = [(f * g1, f), (f * g2, f * g1), (WIDTH[mode], f * g2 + 1)]
    mask = [np.zeros(s) for s in shapes]
    for g in range(f):
        mask[0][g * g1:(g + 1) * g1, g] = 1
        mask[1][g * g2:(g + 1) * g2, g * g1:(g + 1) * g1] = 1
    mask[2][:] = 1
    m, sets, _ = _problem(mode, 3000, f, None, "swish", 0, seed=9, mask=mask, shapes=shapes)
    eng = _engine(m)
    _replay(eng, m, sets[0], None, 8, "k_fwd_sparse", mask=mask)
    eng.close()


# ------------------------------------------------------------------------------------------------ Python surface
def _count_dat(rng, n, n_test, f=5, cols=1):
    x = rng.standard_normal((n + n_test, f))
    w = rng.normal(0, 0.4, (cols, f))
    y = rng.poisson(np.exp(0.5 + x @ w.T)).astype(np.float64)
    return {"data": x[:n], "labels": y[:n], "test_data": x[n:], "test_labels": y[n:]}


@pytest.mark.parametrize("lik", ["negbin_likelihood", "poi_likelihood", "negbin_likelihood2d"])
def test_run_mcmc_log_pickle_and_prediction(tmp_path, lik):
    """The example script of the count models: a seeded run_mcmc (host-drawn proposals) writes a .log whose header is
    log_header's custom branch and whose likelihood / MSE columns follow an oracle replay of the same draws; the
    pickle is read back by get_posterior_est."""
    import npbnn_b200 as bn
    cols = 2 if lik == "negbin_likelihood2d" else 1
    rng = np.random.default_rng(21)
    dat = _count_dat(rng, 500, 80, cols=cols)
    np.random.seed(5)
    out = 1 if lik == "poi_likelihood" else 2 * cols
    bnn = bn.npBNN(dat, n_nodes=[8, 4], estimation_mode="custom", size_output=out, output_act_fun=bn.RegressTransform)
    w0 = [w.copy() for w in bnn._w_layers]
    lf = getattr(bn, lik)
    mcmc = bn.MCMC(bnn, likelihood_f=lf, n_iteration=60, sampling_f=10, print_f=1000, n_post_samples=10)
    logger = bn.postLogger(bnn, filename=str(tmp_path / "cnt"), log_all_weights=0)
    bn.run_mcmc(bnn, mcmc, logger)
    with open(logger._logfile) as fh:
        rows = list(csv.reader(fh, delimiter="\t"))
    assert rows[0] == bn.log_header(bnn) and "MSE" in rows[0] and not any(h.startswith("sig_") for h in rows[0])
    assert len(rows) == 7 and all(len(r) == len(rows[0]) for r in rows[1:])
    mode = {"poi_likelihood": "poisson", "negbin_likelihood": "negbin", "negbin_likelihood2d": "negbin"}[lik]
    m = corc.CountModel(x=dat["data"], labels=dat["labels"], weights=w0, act="ReLU", mode=mode, x_test=dat["test_data"],
                  labels_test=dat["test_labels"])
    s = corc.make_sampler(m, n_iteration=60)
    rs = np.random.default_rng(1234)
    logged = {}
    for it in range(1, 61):
        corc.mh_step(m, s, rs=rs)
        if it % 10 == 0:
            logged[it] = (s.logLik, s.accuracy, s.test_accuracy)
    for r in rows[1:]:
        ll, mse, tmse = logged[int(r[0])]
        assert rel_close(float(r[2]), ll), (r[0], r[2], ll)
        assert np.isclose(float(r[4]), mse, rtol=1e-9) and np.isclose(float(r[5]), tmse, rtol=1e-9)
    for a, b in zip(bnn._w_layers, m.weights):
        assert np.array_equal(a, b)
    assert os.path.exists(logger._pklfile)
    est = bn.get_posterior_est(logger._pklfile)
    post = [p["weights"] for p in logger._post_weight_samples]
    dense, mean = orc.posterior_predict(dat["data"], post, "ReLU", None, "identity", 1)
    assert np.allclose(est["prm_mean"], mean, rtol=1e-10, atol=1e-11)
    assert est["post_est"].shape == (len(post), 500, out)


def test_mc3_with_a_count_likelihood_runs_and_swaps(tmp_path, capsys):
    import npbnn_b200 as bn
    rng = np.random.default_rng(3)
    dat = _count_dat(rng, 300, 0)
    np.random.seed(2)
    bnn = bn.npBNN(dat, n_nodes=[6, 3], estimation_mode="custom", size_output=2, output_act_fun=bn.RegressTransform)
    logger = bn.postLogger(bnn, filename=str(tmp_path / "mc3"))
    mc3 = bn.MC3(bnn, logger, n_chains=4, swap_frequency=10, n_iteration=200, sampling_f=50, print_f=1000,
                 likelihood_f=bn.negbin_likelihood, accuracy_f=bn.negbin_acc, swap_seed=7)
    mc3.run_mcmc()
    assert "SWAPPED" in capsys.readouterr().out
    for b, mc in mc3.singleChainArgs:
        assert mc._current_iteration == 200 and np.isfinite(mc._logLik) and mc._label_acc == []
        y = orc.forward(bnn._data, b._w_layers, "ReLU", None, "identity")
        assert rel_close(mc._logLik, corc.loglik_count(y, bnn._labels, "negbin"))


def test_philox_posterior_tracks_a_poisson_teacher():
    """Statistical sanity on data simulated from a known Poisson teacher network (rng="philox"): a chain started from
    the teacher's weights plus N(0, 0.3) noise moves its posterior-mean rate onto the teacher's -- within 30 % on at
    least 75 % of the rows, and at least halving the mean squared rate error of the start.  A sign or parametrisation
    error in the likelihood (which a replay against a wrong oracle would copy) drives it away instead."""
    import npbnn_b200 as bn
    rng = np.random.default_rng(8)
    n, f = 3000, 4
    x = rng.standard_normal((n, f))
    teacher = [rng.normal(0, 0.6, (6, f + 1)), rng.normal(0, 0.6, (1, 6))]
    rate = np.exp(orc.forward(x, teacher, "tanh", None, "identity")[:, 0])
    y = rng.poisson(rate).astype(np.float64)[:, None]
    w0 = [w + rng.normal(0, 0.3, w.shape) for w in teacher]
    bnn = bn.npBNN({"data": x, "labels": y, "test_data": [], "test_labels": []}, n_nodes=[6], init_weights=w0,
                   estimation_mode="custom", size_output=1, output_act_fun=bn.RegressTransform, actFun=bn.ActFun("tanh"))
    mcmc = bn.MCMC(bnn, likelihood_f=bn.poi_likelihood, n_iteration=4000, rng="philox", adapt_f=0.2, adapt_fM=0.4,
                   adapt_freq=100, adapt_stop=2000)
    post = []
    for _ in range(20):
        mcmc.run(bnn, 200)
        if mcmc._current_iteration > 2000:
            post.append([w.copy() for w in bnn._w_layers])
    est = np.mean([np.exp(orc.forward(x, w, "tanh", None, "identity")[:, 0]) for w in post], axis=0)
    start = np.exp(orc.forward(x, w0, "tanh", None, "identity")[:, 0])
    rel = np.abs(est - rate) / rate
    assert np.mean(rel < 0.3) >= 0.75, np.mean(rel < 0.3)
    assert np.mean((est - rate) ** 2) < 0.5 * np.mean((start - rate) ** 2), (np.mean((est - rate) ** 2),
                                                                             np.mean((start - rate) ** 2))
