"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the reference goldens.

Tolerances: FP64 mode, log-likelihood / log-prior within 1e-9 relative (BASELINE.json north_star);
integer counters, accept decisions and weights bit-exact on injected proposals."""
import numpy as np
import pytest

from oracle import npbnn_oracle as orc
from tests import _golden as G

pytestmark = pytest.mark.gpu

RTOL = 1e-9
L_ADD_PROB = 8      # BNN_F_ADD_PROB (include/npbnn_b200.h)
LIK = {"classification": 0, "regression": 1, "regression-error": 2}


def rel_close(a, b, rtol=RTOL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.allclose(a, b, rtol=rtol, atol=rtol * 1e-3)


def make_engine(m, meta=None):
    from npbnn_b200.engine import Engine, NetShape
    net = NetShape.from_weights(m.weights, m.x.shape[1], act=m.act, lik=LIK[m.mode])
    eng = Engine(net)
    eng.set_data(m.x, m.labels, m.x_test, m.labels_test, inst_w=m.inst_w, class_w=m.class_w)
    return eng


def oracle_score(m, weights, sig=None, lik_temp=1.0):
    y = orc.forward(m.x, weights, m.act, m.alphas, m.out_kind)
    out = {}
    if m.mode == "classification":
        out["loglik"] = orc.loglik_categorical(y, m.labels, m.class_w, m.inst_w, lik_temp)
        nc, ck, tk, hist = orc.class_counters(y, m.labels)
        out["n_correct"], out["class_correct"], out["pred_hist"] = nc, ck, hist
        if m.x_test is not None:
            yt = orc.forward(m.x_test, weights, m.act, m.alphas, m.out_kind)
            out["n_correct_test"] = orc.class_counters(yt, m.labels_test)[0]
    else:
        sr, sr2 = orc.regression_sums(y, m.labels)
        out["sum_r"], out["sum_r2"] = sr, sr2
        if m.mode == "regression":
            s = np.std(y - m.labels, axis=0) if sig == "empirical" else (1.0 if sig is None else sig)
            out["loglik"] = orc.loglik_regression(y, m.labels, s, lik_temp)
        else:
            out["loglik"] = orc.loglik_regression_error(y, m.labels, lik_temp)
        if m.x_test is not None:
            yt = orc.forward(m.x_test, weights, m.act, m.alphas, m.out_kind)
            out["sum_r2_test"] = orc.regression_sums(yt, m.labels_test)[1]
    return out


@pytest.mark.parametrize("name", G.CHAIN_CASES)
def test_forward_lik_matches_oracle(name):
    """bnn_forward_lik on the golden data: initial weights, final weights and random jitter, batched."""
    z, meta = G.load(name)
    m = G.build_model(z, meta)
    nl = G.n_layers(meta)
    rng = np.random.default_rng(3)
    sets = [m.weights, [np.array(z["wN_%d" % i]) for i in range(nl)]]
    for s in range(5):
        sets.append([w + rng.normal(0, 0.3, w.shape) for w in m.weights])
    eng = make_engine(m)
    al = None if m.alphas is None else np.tile(np.resize(m.alphas, nl), (len(sets), 1))
    sig_mode = 1 if meta.get("empirical_error") else 0
    for host in (False, True):
        res = eng.forward_lik(sets, alphas=al, sigma_mode=sig_mode, lik_temp=meta["lik_temp"], host=host)
        for i, w in enumerate(sets):
            ref = oracle_score(m, w, "empirical" if sig_mode else None, meta["lik_temp"])
            assert rel_close(res["loglik"][i], ref["loglik"]), (name, i, res["loglik"][i], ref["loglik"])
            if m.mode == "classification":
                K = eng.K
                c = res["counts"][i]
                assert c[0] == ref["n_correct"]
                assert np.array_equal(c[2:2 + K], ref["class_correct"])
                assert np.array_equal(c[2 + K:2 + 2 * K], ref["pred_hist"])
                if m.x_test is not None:
                    assert c[1] == ref["n_correct_test"]
            else:
                assert rel_close(res["sums"][i][0], ref["sum_r"], 1e-9) or np.allclose(res["sums"][i][0], ref["sum_r"], atol=1e-9)
                assert rel_close(res["sums"][i][1], ref["sum_r2"])
                if m.x_test is not None:
                    assert rel_close(res["sums"][i][2], ref["sum_r2_test"])
    # the -m gpu run must go through the CUDA library, never a fallback
    assert eng.launch_count > 0
    eng.close()


@pytest.mark.parametrize("prior,scale", [(1, 1.0), (2, 0.7), (3, 1.3), (0, 1.0), (1, [0.5, 1.0, 2.0])])
def test_log_prior_matches_oracle(prior, scale):
    z, meta = G.load("syn_swish_cauchy")
    m = G.build_model(z, meta)
    eng = make_engine(m)
    rng = np.random.default_rng(1)
    sets = [[w + rng.normal(0, 0.5, w.shape) for w in m.weights] for _ in range(4)]
    got = eng.log_prior(sets, prior, scale)
    sc = np.broadcast_to(np.asarray(scale, dtype=np.float64), (3,))
    for i, w in enumerate(sets):
        assert rel_close(got[i], orc.log_prior(w, prior, sc)), (prior, i)
    eng.close()


def _init_chains(eng, m, meta, n_chains):
    w0 = [m.weights] * n_chains
    nl = len(m.weights)
    n_it = meta["n_iteration"]
    eng.chains_init(w0, temperature=meta["temperature"], update_f=meta["update_f"][:nl], update_ws=meta["update_ws"][:nl],
                    prior=meta["prior"], prior_scale=meta["p_scale"], w_bound=meta["w_bound"], mask=m.mask,
                    alphas=None if m.alphas is None else np.concatenate([m.alphas, np.zeros(nl)])[:nl],
                    sigma_mode=1 if meta.get("empirical_error") else 0, lik_temp=meta["lik_temp"],
                    adapt_f=meta["adapt_f"], adapt_fM=meta["adapt_fM"], adapt_freq=meta["adapt_freq"],
                    adapt_stop=int(n_it * 0.05), n_act_prm=len(m.alphas) if m.act_trainable else 0,
                    init_additional_prob=meta.get("init_additional_prob", 0.0))


@pytest.mark.parametrize("name", G.CHAIN_CASES)
def test_chain_replay_step_by_step(name):
    """Replay the reference's recorded proposals one MH iteration at a time: proposal log-lik / log-prior
    within 1e-9, identical accept decisions, identical adaptation state, bit-identical weights."""
    z, meta = G.load(name)
    m = G.build_model(z, meta)
    eng = make_engine(m)
    _init_chains(eng, m, meta, 2)
    st = eng.read_state()
    N = m.x.shape[0]
    assert rel_close(st.logLik, float(z["init_logLik"])) and rel_close(st.logPrior, float(z["init_logPrior"]))
    assert np.array_equal(st.update_n[0], z["init_update_n"])
    n_steps = min(int(z["n_steps"]), 60)
    near_tie = 0
    for t in range(n_steps):
        eng.mh_steps(1, G.injection_arrays(z, meta, t, t + 1, 2))
        st = eng.read_state()
        for c in range(2):
            assert rel_close(st.logLik_prop[c], z["steps_logLik_prime"][t]), (t, st.logLik_prop[c], float(z["steps_logLik_prime"][t]))
            # the golden holds calc_prior() alone; the proposal's log-prior adds additional_prob (BNN_env.py:481)
            add = float(st.f64[c, L_ADD_PROB])
            assert rel_close(st.logPrior_prop[c] - add, z["steps_logPrior_prime"][t]), t
            margin = abs((float(z["steps_logLik_prime"][t]) + float(z["steps_logPrior_prime"][t]) + add - float(z["steps_logPost"][t - 1] if t else z["init_logLik"] + z["init_logPrior"])) * meta["temperature"] - float(z["steps_log_u"][t]))
            if margin < 1e-8:
                near_tie += 1       # decision inside the summation-order noise: reported, not asserted
                continue
            assert st.last_accepted[c] == int(z["steps_accepted"][t]), t
            assert rel_close(st.logLik[c], z["steps_logLik"][t]) and rel_close(st.logPost[c], z["steps_logPost"][t])
            assert st.iteration[c] == t + 1
            assert abs(st.acceptance_rate[c] - float(z["steps_acceptance_rate"][t])) < 1e-15
            assert np.array_equal(st.update_n[c], z["steps_update_n"][t]), t
            assert np.allclose(st.update_f[c], z["steps_update_f"][t], rtol=1e-14)
            assert np.allclose(st.update_ws[c], z["steps_update_ws"][t], rtol=1e-14)
            assert np.allclose(st.freq_layer_update[c], z["steps_freq_layer_update"][t], rtol=1e-14)
            if m.act_trainable:
                assert np.allclose(st.alpha[c][:len(m.alphas)], z["steps_act_prm"][t], rtol=1e-14, atol=0), t
            if meta["mode"] == "classification":
                assert st.n_correct[c] / N == float(z["steps_accuracy"][t])
                assert np.array_equal(st.pred_hist[c] / N, z["steps_label_freq"][t])
                if m.x_test is not None:
                    assert st.n_correct_test[c] / m.x_test.shape[0] == float(z["steps_test_accuracy"][t])
            else:
                assert rel_close(np.sum(st.sum_r2[c]) / (N * eng.K), z["steps_accuracy"][t])
                assert rel_close(st.sum_r2[c] / N, z["steps_label_acc"][t])
                if meta["mode"] == "regression":
                    assert rel_close(st.sigma[c], z["steps_error_prm"][t])
    assert near_tie == 0
    eng.close()


@pytest.mark.parametrize("name", G.CHAIN_CASES)
def test_chain_replay_one_launch(name):
    """All recorded iterations in ONE bnn_mh_steps call (no host round trips): final weights bit-identical
    to the reference's, accept count identical."""
    z, meta = G.load(name)
    m = G.build_model(z, meta)
    eng = make_engine(m)
    _init_chains(eng, m, meta, 3)
    T = int(z["n_steps"])
    eng.mh_steps(T, G.injection_arrays(z, meta, 0, T, 3))
    st = eng.read_state()
    for c in range(3):
        assert st.n_accepted[c] == int(np.sum(z["steps_accepted"]))
        for i, w in enumerate(st.weights(c)):
            assert np.array_equal(w, z["wN_%d" % i]), (name, c, i)
        assert rel_close(st.logLik[c], z["steps_logLik"][T - 1])
        assert rel_close(st.logPrior[c], z["steps_logPrior"][T - 1])
    eng.close()


def test_headline_shape_goldens_run_on_the_specialised_kernels():
    """The reference-generated goldens of the two headline network shapes go through the kernels the bench times:
    syn_c4_shape ([64,32] swish, K=10) -> k_fwd3, syn_c3_shape (block-masked [120,80] tanh) -> k_fwd_sparse."""
    z, meta = G.load("syn_c4_shape")
    m = G.build_model(z, meta)
    eng = make_engine(m)
    _init_chains(eng, m, meta, 2)
    eng.mh_steps(2, G.injection_arrays(z, meta, 0, 2, 2))
    eng.synchronize()
    assert eng.last_kernel.startswith("k_fwd3"), eng.last_kernel
    eng.close()
    z, meta = G.load("syn_c3_shape")
    v = G.ChainView(z, 0)
    m = G.build_model(v, meta)
    eng = make_engine(m)
    _init_chains(eng, m, meta, 2)
    eng.mh_steps(2, G.injection_arrays(v, meta, 0, 2, 2))
    eng.synchronize()
    assert eng.last_kernel.startswith("k_fwd_sparse"), eng.last_kernel
    eng.close()


def _c3_golden():
    z, meta = G.load("syn_c3_shape")
    views = [G.ChainView(z, c) for c in range(meta["n_chains"])]
    models = [G.build_model(v, meta) for v in views]
    return z, meta, views, models


def test_c3_shape_eight_chains_step_by_step():
    """BASELINE config 3's network at its real shape (F=40, block-masked [120,80] tanh, K=5, 8 chains batched on one
    GPU), against the reference's own recorded chains (tests/golden/make_golden.py: case_c3_shape): every chain has
    its own initial weights and its own proposal stream; all 8 run in ONE k_fwd_sparse pass per iteration."""
    z, meta, views, models = _c3_golden()
    nc = len(models)
    m0 = models[0]
    eng = make_engine(m0)
    nl = len(m0.weights)
    eng.chains_init([m.weights for m in models], temperature=1.0, update_f=meta["update_f"], update_ws=meta["update_ws"],
                    prior=1, prior_scale=1.0, mask=m0.mask, adapt_stop=int(meta["n_iteration"] * 0.05))
    st = eng.read_state()
    N, Nt = m0.x.shape[0], m0.x_test.shape[0]
    for c, v in enumerate(views):
        assert rel_close(st.logLik[c], float(v["init_logLik"])) and rel_close(st.logPrior[c], float(v["init_logPrior"]))
        assert np.array_equal(st.update_n[c], v["init_update_n"])
        assert st.n_correct[c] / N == float(v["init_accuracy"])
    T = int(views[0]["n_steps"])
    for t in range(T):
        eng.mh_steps(1, G.stack_injections([G.injection_arrays(v, meta, t, t + 1, 1) for v in views]))
        assert eng.last_kernel.startswith("k_fwd_sparse"), eng.last_kernel
        st = eng.read_state()
        for c, v in enumerate(views):
            assert rel_close(st.logLik_prop[c], v["steps_logLik_prime"][t]), (t, c)
            assert rel_close(st.logPrior_prop[c], v["steps_logPrior_prime"][t]), (t, c)
            assert st.last_accepted[c] == int(v["steps_accepted"][t]), (t, c)
            assert rel_close(st.logLik[c], v["steps_logLik"][t]) and rel_close(st.logPost[c], v["steps_logPost"][t])
            assert st.n_correct[c] / N == float(v["steps_accuracy"][t])
            assert st.n_correct_test[c] / Nt == float(v["steps_test_accuracy"][t])
            assert np.array_equal(st.pred_hist[c] / N, v["steps_label_freq"][t])
            assert abs(st.acceptance_rate[c] - float(v["steps_acceptance_rate"][t])) < 1e-15
    for c, v in enumerate(views):
        for i, w in enumerate(st.weights(c)):
            assert np.array_equal(w, v["wN_%d" % i]), (c, i)
            assert np.all(w[m0.mask[i] == 0] == 0)
    eng.close()


def test_c3_shape_eight_chains_one_launch():
    z, meta, views, models = _c3_golden()
    m0 = models[0]
    eng = make_engine(m0)
    eng.chains_init([m.weights for m in models], update_f=meta["update_f"], update_ws=meta["update_ws"], prior=1,
                    prior_scale=1.0, mask=m0.mask, adapt_stop=int(meta["n_iteration"] * 0.05))
    T = int(views[0]["n_steps"])
    eng.mh_steps(T, G.stack_injections([G.injection_arrays(v, meta, 0, T, 1) for v in views]))
    st = eng.read_state()
    assert eng.last_kernel.startswith("k_fwd_sparse"), eng.last_kernel
    for c, v in enumerate(views):
        assert st.n_accepted[c] == int(np.sum(v["steps_accepted"]))
        for i, w in enumerate(st.weights(c)):
            assert np.array_equal(w, v["wN_%d" % i]), (c, i)
        assert rel_close(st.logLik[c], v["steps_logLik"][T - 1]) and rel_close(st.logPrior[c], v["steps_logPrior"][T - 1])
    # the final predictions of chain 0 against the reference's mcmc._y
    y = eng.predict(m0.x, [st.weights(0)], mean=False, dense=True)["dense"][0]
    assert np.allclose(y, views[0]["yN"], rtol=1e-10, atol=1e-300)
    eng.close()


def test_predict_matches_reference_goldens():
    from npbnn_b200.engine import Engine, NetShape
    z, meta = G.load("predict")
    x = z["x"]
    for ci, case in enumerate(meta["cases"]):
        post = [[z["p%d_s%d_w%d" % (ci, j, li)] for li in range(3)] for j in range(meta["S"])]
        net = NetShape.from_weights(post[0], x.shape[1], act=case["act"], lik=0)
        eng = Engine(net)
        al = None if not case["alphas"] else np.tile(np.resize(np.array(case["alphas"]), 3), (meta["S"], 1))
        out = eng.predict(x, post, alphas=al, mean=True, votes=True, dense=True)
        assert np.allclose(out["dense"], z["p%d_dense" % ci], rtol=1e-10, atol=1e-300)
        assert np.allclose(out["mean"], z["p%d_mode1" % ci], rtol=1e-10, atol=1e-300)
        assert np.array_equal(out["votes"], z["p%d_mode0" % ci])
        # PDP grid steps (BNN_pdp.py:63-82): column overwrite fused into the X staging
        for focal in (1, 3):
            feats = z["p%d_pdp%d_feature" % (ci, focal)]
            gold = z["p%d_pdp%d" % (ci, focal)]
            for n in range(feats.shape[0]):
                o = eng.predict(x, post, alphas=al, override=([focal], feats[n, :]), mean=True)
                smean = np.cumsum(o["mean"], axis=1)       # cumsum commutes with the mean over samples
                assert np.allclose(np.mean(smean, axis=0), gold[n, :, 0], rtol=1e-10)
                q = np.quantile(smean, q=(0.025, 0.975), axis=0)
                assert np.allclose(q[0], gold[n, :, 1], rtol=1e-9) and np.allclose(q[1], gold[n, :, 2], rtol=1e-9)
        eng.close()


def _c4_like(n, n_sets, seed=0):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, 64))
    shapes = [(64, 64), (32, 64), (10, 33)]
    teacher = [rng.normal(0, 0.5, s) for s in shapes]
    labels = np.argmax(orc.forward(x, teacher, "swish", None, "softmax"), axis=1)
    sets = [[rng.normal(0, 0.3, s) for s in shapes] for _ in range(n_sets)]
    return x, labels, sets


@pytest.mark.parametrize("n", [16, 1000, 4099])
def test_c4_shape_specialised_kernel(n):
    """BASELINE config 4 shape (64 -> 64 -> 32 -> 10, swish, bias on the last layer) at small N: the
    shape-specialised kernel against the oracle and against the generic kernel."""
    from npbnn_b200.engine import Engine, NetShape
    x, labels, sets = _c4_like(n, 5)
    m = orc.Model(x=x, labels=labels, weights=sets[0], act="swish", mode="classification")
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    eng = Engine(net)
    eng.set_data(x, labels)
    res = eng.forward_lik(sets)
    assert eng.last_kernel.startswith("k_fwd3"), eng.last_kernel
    eng.set_option("force_generic", 1)
    gen = eng.forward_lik(sets)
    assert eng.last_kernel == "k_fwd_generic"
    for i, w in enumerate(sets):
        ref = oracle_score(m, w)
        assert rel_close(res["loglik"][i], ref["loglik"]), (i, res["loglik"][i], ref["loglik"])
        assert rel_close(gen["loglik"][i], ref["loglik"])
        K = 10
        for r in (res, gen):
            c = r["counts"][i]
            assert c[0] == ref["n_correct"]
            assert np.array_equal(c[2:2 + K], ref["class_correct"]) and np.array_equal(c[2 + K:2 + 2 * K], ref["pred_hist"])
    # prediction through the specialised kernel
    eng.set_option("force_generic", 0)
    out = eng.predict(x, sets, mean=True, votes=True, dense=True)
    assert eng.last_kernel.startswith("k_fwd3")
    dense_ref, mean_ref = orc.posterior_predict(x, sets, "swish", None, "softmax", 1)
    _, votes_ref = orc.posterior_predict(x, sets, "swish", None, "softmax", 0)
    assert np.allclose(out["dense"], dense_ref, rtol=1e-10, atol=1e-300)
    assert np.allclose(out["mean"], mean_ref, rtol=1e-10, atol=1e-300)
    assert np.array_equal(out["votes"], votes_ref)
    eng.close()


@pytest.mark.parametrize("n,n_sets", [(50000, 5), (30011, 7), (28416 * 2 + 16 * 29, 3)])
def test_c4_shape_tail_round_split(n, n_sets):
    """k_fwd3 deals the (tile group, weight set) pairs of the last, partially filled round out over the CTAs
    (one or two segments per CTA).  Sizes chosen so that CTAs get two segments, an uneven share and a tail
    behind full rounds (148 SMs x 12 warps x 16 rows = 28,416 rows per full round).  Against the oracle and the
    generic kernel; the decomposition must not change a single bit between two geometries of the same rows."""
    from npbnn_b200.engine import Engine, NetShape
    x, labels, sets = _c4_like(n, n_sets)
    m = orc.Model(x=x, labels=labels, weights=sets[0], act="swish", mode="classification")
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    eng = Engine(net)
    eng.set_data(x, labels)
    res = eng.forward_lik(sets)
    assert eng.last_kernel.startswith("k_fwd3<"), eng.last_kernel
    for i, w in enumerate(sets):
        ref = oracle_score(m, w)
        assert rel_close(res["loglik"][i], ref["loglik"]), (i, res["loglik"][i], ref["loglik"])
        c = res["counts"][i]
        assert c[0] == ref["n_correct"]
        assert np.array_equal(c[2:12], ref["class_correct"]) and np.array_equal(c[12:22], ref["pred_hist"])
    # the same sets scored one at a time (different pair decomposition): identical bits
    for i in (0, n_sets - 1):
        one = eng.forward_lik([sets[i]])
        assert one["loglik"][0] == res["loglik"][i]
        assert np.array_equal(one["counts"][0], res["counts"][i])
    eng.close()


@pytest.mark.parametrize("kind", ["class", "instance"])
@pytest.mark.parametrize("n,n_sets", [(4099, 1), (50000, 5)])
def test_c4_shape_weighted_likelihood(kind, n, n_sets):
    """The weighted-likelihood instantiation of the shape-specialised kernel (class weights, BNN_env.py:97-100, or
    instance weights, BNN_lib.py:103-118) at the config-4 shape: sizes with one and with several weight sets per tile,
    full rounds plus a split tail, so that the epilogue carried across tile boundaries sees the right labels and
    weights.  Against the oracle and the generic kernel."""
    from npbnn_b200.engine import Engine, NetShape
    x, labels, sets = _c4_like(n, n_sets, seed=12)
    rng = np.random.default_rng(1)
    cw = rng.uniform(0.5, 2.0, 10) if kind == "class" else None
    iw = rng.uniform(0.2, 1.8, n) if kind == "instance" else None
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    eng = Engine(net)
    eng.set_data(x, labels, inst_w=iw, class_w=cw)
    res = eng.forward_lik(sets, lik_temp=0.9)
    assert eng.last_kernel.startswith("k_fwd3<"), eng.last_kernel
    eng.set_option("force_generic", 1)
    gen = eng.forward_lik(sets, lik_temp=0.9)
    assert eng.last_kernel == "k_fwd_generic"
    for i, w in enumerate(sets):
        y = orc.forward(x, w, "swish", None, "softmax")
        ref = orc.loglik_categorical(y, labels, cw, iw, 0.9)
        assert rel_close(res["loglik"][i], ref), (i, res["loglik"][i], ref)
        assert rel_close(gen["loglik"][i], ref)
        assert res["counts"][i][0] == orc.class_counters(y, labels)[0]
    eng.close()


def test_c4_shape_train_and_test_rows_in_one_pass():
    """Training rows and test rows are staged back to back and scored in one pass (test rows only feed the test-accuracy
    counter, RunPredictInd on accept, BNN_env.py:511-515).  Config-4 shape with a train / test boundary inside a warp
    tile and several weight sets: log-likelihood over the training rows only, both accuracy counters exact."""
    from npbnn_b200.engine import Engine, NetShape
    x, labels, sets = _c4_like(30_011 + 3_005, 4, seed=14)
    n_tr = 30_011
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    eng = Engine(net)
    eng.set_data(x[:n_tr], labels[:n_tr], x[n_tr:], labels[n_tr:])
    res = eng.forward_lik(sets)
    assert eng.last_kernel.startswith("k_fwd3<"), eng.last_kernel
    for i, w in enumerate(sets):
        y = orc.forward(x, w, "swish", None, "softmax")
        assert rel_close(res["loglik"][i], orc.loglik_categorical(y[:n_tr], labels[:n_tr]))
        assert res["counts"][i][0] == orc.class_counters(y[:n_tr], labels[:n_tr])[0]
        assert res["counts"][i][1] == orc.class_counters(y[n_tr:], labels[n_tr:])[0]
        assert np.array_equal(res["counts"][i][12:22], orc.class_counters(y[:n_tr], labels[:n_tr])[3])
    eng.close()


def test_c4_full_size_properties():
    """BASELINE config 4 at FULL size (1M x 64, 32 weight sets): the oracle cannot score this in seconds, so
    parity is carried by size-independent properties of the likelihood pass --
      * additivity over a row partition (log-likelihood sums to 1e-12 relative, integer counters add exactly),
      * an oracle check on a random 20k-row subset of the same rows,
      * duplicate weight sets give identical bits, two runs give identical bits,
      * invariance under a row permutation (1e-12 relative, counters exactly)."""
    import torch
    from npbnn_b200.engine import Engine, NetShape
    from npbnn_b200 import workloads as wl
    n, C = 1_000_000, 32
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(n, 64, dtype=torch.float64, device="cuda", generator=g)
    rng = np.random.default_rng(3)
    shapes = list(wl.C4_SHAPES)
    teacher = [rng.normal(0, 0.5, s) for s in shapes]
    sets = [[rng.normal(0, 0.2, s) for s in shapes] for _ in range(C - 1)]
    sets.append([a.copy() for a in sets[3]])                      # duplicate of set 3
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    eng = Engine(net)
    lab = torch.as_tensor(eng.predict(x, [teacher], mean=True)["mean"]).argmax(1).to(torch.int32).cuda()
    eng.set_data(x, lab)
    full = eng.forward_lik(sets)
    assert eng.last_kernel.startswith("k_fwd3<"), eng.last_kernel
    assert np.all(np.isfinite(full["loglik"]))
    again = eng.forward_lik(sets)
    assert np.array_equal(full["loglik"], again["loglik"]) and np.array_equal(full["counts"], again["counts"])
    assert full["loglik"][3] == full["loglik"][C - 1] and np.array_equal(full["counts"][3], full["counts"][C - 1])
    assert np.all(full["counts"][:, 2:12].sum(1) == full["counts"][:, 0])         # per-class hits add up to hits
    assert np.all(full["counts"][:, 12:22].sum(1) == n)                           # every row predicted once
    # additivity over an uneven row partition
    cuts = [0, 16, 123_457, 500_000, 999_983, n]
    ll = np.zeros(C)
    cnt = np.zeros_like(full["counts"])
    for a, b in zip(cuts[:-1], cuts[1:]):
        eng.set_data(x[a:b], lab[a:b])
        part = eng.forward_lik(sets)
        ll += part["loglik"]
        cnt += part["counts"]
    assert np.allclose(ll, full["loglik"], rtol=1e-12, atol=0)
    assert np.array_equal(cnt, full["counts"])
    # oracle on a random subset of the same rows
    idx = torch.as_tensor(np.sort(rng.choice(n, 20_000, replace=False))).cuda()
    xs, ys = x[idx], lab[idx]
    eng.set_data(xs, ys)
    sub = eng.forward_lik(sets[:3])
    m = orc.Model(x=xs.cpu().numpy(), labels=ys.cpu().numpy().astype(np.int64), weights=sets[0], act="swish",
                  mode="classification")
    for i in range(3):
        ref = oracle_score(m, sets[i])
        assert rel_close(sub["loglik"][i], ref["loglik"])
        assert sub["counts"][i][0] == ref["n_correct"]
        assert np.array_equal(sub["counts"][i][12:22], ref["pred_hist"])
    # row permutation
    perm = torch.randperm(n, device="cuda", generator=g)
    eng.set_data(x[perm], lab[perm])
    pr = eng.forward_lik(sets)
    assert np.allclose(pr["loglik"], full["loglik"], rtol=1e-12, atol=0)
    assert np.array_equal(pr["counts"], full["counts"])
    eng.close()


def test_c5_full_size_prediction_properties():
    """BASELINE config 5 shape at full row count (1M x 64 rows, 48 posterior samples; the 10k samples of the config are
    the same kernel looped): size-independent properties of the posterior-prediction pass --
      * mean probabilities and vote shares are distributions per row (sum to 1, votes are multiples of 1/S),
      * the mean over all samples is the sample-weighted mean of the means over two disjoint sample batches,
      * a row block predicted alone equals the same rows of the full pass bit for bit,
      * an oracle check on 5,000 random rows."""
    import torch
    from npbnn_b200.engine import Engine, NetShape
    from npbnn_b200 import workloads as wl
    n, S = 1_000_000, 48
    g = torch.Generator(device="cuda").manual_seed(21)
    x = torch.randn(n, 64, dtype=torch.float64, device="cuda", generator=g)
    rng = np.random.default_rng(6)
    shapes = list(wl.C4_SHAPES)
    sets = [[rng.normal(0, 0.25, s) for s in shapes] for _ in range(S)]
    eng = Engine(NetShape.from_weights(sets[0], 64, act="swish", lik=0))
    full = eng.predict(x, sets, mean=True, votes=True)
    assert eng.last_kernel.startswith("k_fwd3<"), eng.last_kernel
    mean, votes = full["mean"], full["votes"]
    assert mean.shape == (n, 10) and np.all(mean >= 0)
    assert np.allclose(mean.sum(1), 1.0, rtol=0, atol=1e-13) and np.allclose(votes.sum(1), 1.0, rtol=0, atol=1e-13)
    assert np.allclose(votes * S, np.round(votes * S), rtol=0, atol=1e-9)
    a = eng.predict(x, sets[:20], mean=True, votes=True)
    b = eng.predict(x, sets[20:], mean=True, votes=True)
    assert np.allclose((20 * a["mean"] + 28 * b["mean"]) / S, mean, rtol=1e-13, atol=1e-16)
    assert np.allclose((20 * a["votes"] + 28 * b["votes"]) / S, votes, rtol=0, atol=1e-13)
    blk = eng.predict(x[300_016:400_016], sets, mean=True, votes=True)
    assert np.array_equal(blk["mean"], mean[300_016:400_016]) and np.array_equal(blk["votes"], votes[300_016:400_016])
    idx = np.sort(rng.choice(n, 5_000, replace=False))
    xs = x[torch.as_tensor(idx).cuda()].cpu().numpy()
    _, mean_ref = orc.posterior_predict(xs, sets, "swish", None, "softmax", 1)
    _, votes_ref = orc.posterior_predict(xs, sets, "swish", None, "softmax", 0)
    assert np.allclose(mean[idx], mean_ref, rtol=1e-10, atol=1e-300)
    assert np.array_equal(votes[idx], votes_ref)
    eng.close()


def test_unknown_options_are_refused():
    """bnn_set_option refuses a name it does not know, including the removed tensor-core first layer ("tensor_l1"),
    and leaves the context usable."""
    from npbnn_b200 import _lib as L
    from npbnn_b200.engine import Engine, NetShape
    x, labels, sets = _c4_like(16, 1)
    eng = Engine(NetShape.from_weights(sets[0], 64, act="swish", lik=0))
    eng.set_data(x, labels)
    for name, value in (("tensor_l1", 1), ("tensor_l1", 0), ("no_such_option", 1)):
        with pytest.raises(L.NpbnnError, match="unknown option " + name):
            eng.set_option(name, value)
    eng.set_option("force_generic", 0)
    assert np.isfinite(eng.forward_lik(sets)["loglik"][0])
    eng.close()


def test_run_is_deterministic():
    """Fixed-order reductions: two identical runs give bit-identical log-likelihoods."""
    from npbnn_b200.engine import Engine, NetShape
    x, labels, sets = _c4_like(20000, 4, seed=5)
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    eng = Engine(net)
    eng.set_data(x, labels)
    a = eng.forward_lik(sets)["loglik"]
    b = eng.forward_lik(sets)["loglik"]
    assert np.array_equal(a, b)
    eng.close()


def test_philox_chains_run_and_agree_with_oracle_state():
    """Free-running (Philox) proposals: the chain's own book-keeping stays consistent -- after T steps
    the stored logLik / logPrior equal the oracle's evaluation of the stored weights."""
    from npbnn_b200.engine import Engine, NetShape
    x, labels, sets = _c4_like(3000, 4, seed=9)
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    eng = Engine(net)
    eng.set_data(x, labels)
    eng.chains_init(sets, temperature=[1.0, 0.95, 0.9, 0.8], seed=42, adapt_f=0.1, adapt_fM=0.6, adapt_freq=10, adapt_stop=100)
    eng.mh_steps(50)
    st = eng.read_state()
    assert np.all(st.iteration == 50)
    assert np.all(st.n_accepted > 0)
    for c in range(4):
        w = st.weights(c)
        m = orc.Model(x=x, labels=labels, weights=w, act="swish", mode="classification")
        ref = oracle_score(m, w)
        assert rel_close(st.logLik[c], ref["loglik"])
        assert rel_close(st.logPrior[c], orc.log_prior(w, 1, np.ones(3)))
        assert st.n_correct[c] == ref["n_correct"]
    eng.close()


@pytest.mark.parametrize("shape", ["small", "c4"])
def test_cuda_graph_replay_matches_eager_launches(shape):
    """bnn_mh_steps without injection replays a captured CUDA graph of the launch sequence from the second call on
    (per n_steps, invalidated by every reconfiguration).  Chains stepped through graphs and chains stepped eagerly
    (option graphs=0) must end in bit-identical states, also across a temperature change and a second chunk length."""
    from npbnn_b200.engine import Engine, NetShape
    rng = np.random.default_rng(4)
    if shape == "c4":
        x, labels, sets = _c4_like(3000, 3, seed=5)
        net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    else:
        x = rng.standard_normal((700, 9))
        labels = rng.integers(0, 4, 700)
        shapes = [(6, 10), (5, 7), (4, 6)]
        sets = [[rng.normal(0, 0.3, s) for s in shapes] for _ in range(3)]
        net = NetShape.from_weights(sets[0], 9, act="tanh", lik=0)
    states = []
    for graphs in (1, 0):
        eng = Engine(net)
        eng.set_data(x, labels)
        eng.chains_init(sets, temperature=[1.0, 0.9, 0.8], seed=77, adapt_f=0.2, adapt_fM=0.6, adapt_freq=5, adapt_stop=40)
        eng.set_option("graphs", graphs)
        for _ in range(4):
            eng.mh_steps(10)                       # eager, capture, replay, replay
        eng.set_temperature([0.8, 1.0, 0.9])
        eng.mh_steps(10)
        for _ in range(3):
            eng.mh_steps(7)
        n_launch = eng.launch_count
        st = eng.read_state()
        states.append((st.f64.copy(), st.i32.copy(), st.w.copy(), n_launch))
        eng.close()
    a, b = states
    assert np.array_equal(a[0], b[0], equal_nan=True) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert np.all(a[1][:, 0] == 71) and a[3] == b[3]


def _random_block_net(rng, f, groups_nodes1, groups_nodes2, k):
    """A create_mask-style block network: feature g -> n1 nodes -> n2 nodes -> dense K outputs (bias on the last layer)."""
    h1, h2 = f * groups_nodes1, f * groups_nodes2
    shapes = [(h1, f), (h2, h1), (k, h2 + 1)]
    mask = [np.zeros(s) for s in shapes]
    for g in range(f):
        mask[0][g * groups_nodes1:(g + 1) * groups_nodes1, g] = 1
        mask[1][g * groups_nodes2:(g + 1) * groups_nodes2, g * groups_nodes1:(g + 1) * groups_nodes1] = 1
    mask[2][:] = 1
    w = [rng.normal(0, 0.4, s) * m for s, m in zip(shapes, mask)]
    return shapes, mask, w


@pytest.mark.parametrize("act", ["tanh", "swish", "ReLU"])
@pytest.mark.parametrize("n", [37, 3000])
def test_block_sparse_kernel_matches_dense_and_oracle(act, n):
    """Masked chains run k_fwd_sparse (dense-block cover of the mask); the same chains with option sparse=0
    run the dense DMMA kernels; both must agree with the oracle at 1e-9 and with each other on every decision."""
    from npbnn_b200.engine import Engine, NetShape
    rng = np.random.default_rng(11)
    f, k = 12, 4
    shapes, mask, w = _random_block_net(rng, f, 3, 2, k)
    x = rng.standard_normal((n, f))
    labels = rng.integers(0, k, n)
    states = []
    for sparse in (1, 0):
        eng = Engine(NetShape(f, shapes, act=act, lik=0))
        eng.set_option("sparse", sparse)
        eng.set_data(x, labels)
        sets = [w, [a + rng.normal(0, 0.2, a.shape) * m for a, m in zip(w, mask)]] if sparse else sets
        eng.chains_init(sets, mask=mask, seed=5)
        assert eng.last_kernel == "k_fwd_generic" if not sparse else eng.last_kernel.startswith("k_fwd_sparse")
        st = eng.read_state()
        for c, ws in enumerate(sets):
            y = orc.forward(x, ws, act, None, "softmax")
            assert rel_close(st.logLik[c], orc.loglik_categorical(y, labels)), (act, n, sparse, c)
            nc, ck, _, hist = orc.class_counters(y, labels)
            assert st.n_correct[c] == nc and np.array_equal(st.class_correct[c], ck) and np.array_equal(st.pred_hist[c], hist)
        eng.mh_steps(25)
        states.append(eng.read_state())
        eng.close()
    a, b = states
    assert np.array_equal(a.n_accepted, b.n_accepted)
    assert np.array_equal(a.w, b.w)                         # identical decisions => bit-identical weights
    assert rel_close(a.logLik, b.logLik)
    for c in range(2):                                      # masked entries stay exactly zero
        for wl_, m in zip(a.weights(c), mask):
            assert np.all(wl_[m == 0] == 0)


def test_block_sparse_falls_back_when_weights_violate_mask():
    from npbnn_b200.engine import Engine, NetShape
    rng = np.random.default_rng(2)
    shapes, mask, w = _random_block_net(rng, 6, 2, 2, 3)
    w[0][0, 5] = 0.3                                        # outside the mask
    x = rng.standard_normal((100, 6))
    labels = rng.integers(0, 3, 100)
    eng = Engine(NetShape(6, shapes, act="tanh", lik=0))
    eng.set_data(x, labels)
    eng.chains_init([w], mask=mask)
    assert eng.last_kernel == "k_fwd_generic"
    st = eng.read_state()
    y = orc.forward(x, w, "tanh", None, "softmax")
    assert rel_close(st.logLik[0], orc.loglik_categorical(y, labels))
    eng.close()


def _mask_net(rng, f, groups1, nodes1, groups2, nodes2, out, out_bias=1):
    """create_mask-style network (oracle block_mask = BNN_lib.py:16-47), weights already masked."""
    h1, h2 = sum(nodes1), (sum(nodes2) if len(groups2) else nodes2)
    shapes = [(h1, f), (h2, h1), (out, h2 + out_bias)]
    mask = [orc.block_mask(shapes[0], groups1, nodes1),
            orc.block_mask(shapes[1], groups2, nodes2 if len(groups2) else []),
            np.ones(shapes[2])]
    w = [rng.normal(0, 0.4, s) * m for s, m in zip(shapes, mask)]
    return shapes, mask, w


@pytest.mark.parametrize("case", ["uneven_blocks", "sparse_then_dense_regression", "regression_head"])
@pytest.mark.parametrize("n,chains", [(40, 3), (1000, 2), (517, 1)])
def test_block_sparse_program_variants(case, n, chains):
    """The dataflow program of k_fwd_sparse on the mask shapes of block_bnns.py:39-81: blocks of unequal size
    (items of > 4 rows are cut), a sparse first layer followed by dense layers, Gaussian likelihoods; odd chain
    counts (chains are evaluated in pairs) and row counts whose last 32-row tile is half empty."""
    from npbnn_b200 import _lib as L
    from npbnn_b200.engine import Engine, NetShape
    rng = np.random.default_rng(17)
    if case == "uneven_blocks":
        f = 28
        groups1 = sum(([4 * r + 0, 4 * r + 1, 4 * r + 1, 4 * r + 2, 4 * r + 3, 4 * r + 3, 4 * r + 3] for r in range(4)), [])
        nodes1 = [3, 6, 5, 2] * 4
        groups2 = sum(([g] * k for g, k in enumerate(nodes1)), [])
        nodes2 = [2, 3, 1, 4] * 4
        shapes, mask, w = _mask_net(rng, f, groups1, nodes1, groups2, nodes2, 3)
        lik, act, out_kind = L.LIK_CATEGORICAL, "tanh", "softmax"
    else:
        f = 30
        head = case == "regression_head"
        shapes, mask, w = _mask_net(rng, f, list(range(f)), [2] * f, [], 4, 4 if head else 2)
        lik = L.LIK_GAUSSIAN_HEAD if head else L.LIK_GAUSSIAN
        act, out_kind = "swish", ("regress-error" if head else "identity")
    x = rng.standard_normal((n, f))
    labels = rng.integers(0, 3, n) if lik == L.LIK_CATEGORICAL else rng.standard_normal((n, 2))
    sets = [[a + rng.normal(0, 0.1, a.shape) * m for a, m in zip(w, mask)] for _ in range(chains)]
    states = []
    for sparse in (1, 0):
        eng = Engine(NetShape(f, shapes, act=act, lik=lik))
        eng.set_option("sparse", sparse)
        eng.set_data(x, labels)
        eng.chains_init(sets, mask=mask, seed=9)
        assert eng.last_kernel == "k_fwd_generic" if not sparse else eng.last_kernel.startswith("k_fwd_sparse")
        st = eng.read_state()
        for c, ws in enumerate(sets):
            y = orc.forward(x, ws, act, None, out_kind)
            if lik == L.LIK_CATEGORICAL:
                assert rel_close(st.logLik[c], orc.loglik_categorical(y, labels)), (case, n, sparse, c)
                nc, ck, _, hist = orc.class_counters(y, labels)
                assert st.n_correct[c] == nc and np.array_equal(st.class_correct[c], ck)
                assert np.array_equal(st.pred_hist[c], hist)
            elif lik == L.LIK_GAUSSIAN:
                assert rel_close(st.logLik[c], orc.loglik_regression(y, labels, 1.0)), (case, n, sparse, c)
                assert rel_close(st.sum_r2[c], orc.regression_sums(y, labels)[1])
            else:
                assert rel_close(st.logLik[c], orc.loglik_regression_error(y, labels)), (case, n, sparse, c)
        eng.mh_steps(20)
        states.append(eng.read_state())
        eng.close()
    a, b = states
    assert np.array_equal(a.n_accepted, b.n_accepted)
    assert np.array_equal(a.w, b.w)
    assert rel_close(a.logLik, b.logLik)


def test_row_sharding_matches_unsharded_chains():
    """Rows split over two "ranks" (two contexts on one GPU, the all-reduce done by hand): the per-chain sums of the
    shards add up to the unsharded partials, so log-likelihoods agree to rounding, counters exactly, and both shards
    take the decisions of the unsharded run (SURVEY.md 8e-2).  A single shard with the identity as all-reduce is
    bit-identical to the ordinary path."""
    from npbnn_b200.engine import Engine, NetShape
    from npbnn_b200 import rowshard
    x, labels, sets = _c4_like(3000, 3, seed=21)
    xt, lt = x[2600:], labels[2600:]
    x, labels = x[:2600], labels[:2600]
    net = NetShape.from_weights(sets[0], 64, act="swish", lik=0)
    kw = dict(temperature=[1.0, 0.9, 0.8], seed=77, adapt_f=0.1, adapt_fM=0.6, adapt_freq=5, adapt_stop=40)
    full = Engine(net)
    full.set_data(x, labels, xt, lt)
    full.chains_init(sets, **kw)
    one = Engine(net)
    one.set_data(x, labels, xt, lt)
    one.enable_rowshard(len(x), lambda t: t)
    one.chains_init(sets, **kw)
    shards = []
    for r in range(2):
        a, b = rowshard.row_partition(len(x), 2, r)
        ta, tb = rowshard.row_partition(len(xt), 2, r)
        e = Engine(net)
        e.set_data(x[a:b], labels[a:b], xt[ta:tb], lt[ta:tb])
        e.enable_rowshard(len(x), "manual")
        e.chains_init(sets, **kw)
        shards.append(e)

    def exchange(accept_mode):
        total = shards[0].rowshard_local() + shards[1].rowshard_local()
        for e in shards:
            e.rowshard_commit(total.clone())
            e.rowshard_update(accept_mode, False)

    exchange(2)
    s0 = full.read_state()
    for e in shards + [one]:
        st = e.read_state()
        assert rel_close(st.logLik, s0.logLik, rtol=1e-12) and np.array_equal(st.n_correct, s0.n_correct)
        assert np.array_equal(st.n_correct_test, s0.n_correct_test)
    T = 30
    full.mh_steps(T)
    one.mh_steps(T)
    for _ in range(T):
        for e in shards:
            e.rowshard_update(0, True)
        exchange(1)
    s0 = full.read_state()
    st1 = one.read_state()
    assert np.array_equal(st1.w, s0.w) and np.array_equal(st1.logLik, s0.logLik) and np.array_equal(st1.i32, s0.i32)
    for e in shards:
        st = e.read_state()
        assert np.array_equal(st.n_accepted, s0.n_accepted) and np.array_equal(st.w, s0.w)
        assert rel_close(st.logLik, s0.logLik, rtol=1e-12) and rel_close(st.logPrior, s0.logPrior, rtol=1e-14)
        assert np.array_equal(st.n_correct, s0.n_correct) and np.array_equal(st.pred_hist, s0.pred_hist)
        assert np.array_equal(st.update_n, s0.update_n) and np.all(st.iteration == T)
    assert np.array_equal(shards[0].read_state().f64, shards[1].read_state().f64)      # ranks stay bit-identical
    for e in shards + [one, full]:
        e.close()


def _chain_loop_cases():
    rng = np.random.default_rng(21)
    cases = {}
    # config-1 shape: [5,5] tanh classifier, X resident in the cluster's shared memory
    x = rng.standard_normal((2500, 128))
    y = rng.integers(0, 5, 2500)
    shp = [(5, 129), (5, 6), (5, 5)]
    cases["c1"] = dict(x=x, y=y, n_test=300, feat=128, act="tanh", lik=0, sets=[[rng.normal(0, 0.2, s) for s in shp] for _ in range(2)],
                       kw=dict(temperature=[1.0, 0.7], adapt_f=0.2, adapt_fM=0.6, adapt_freq=5, adapt_stop=40))
    # config-2 shape: [10,5] ReLU regression with the empirical error, 999 rows
    x = rng.standard_normal((999, 3))
    t = rng.standard_normal((999, 2))
    shp = [(10, 4), (5, 11), (2, 5)]
    cases["c2"] = dict(x=x, y=t, n_test=0, feat=3, act="ReLU", lik=1, sets=[[rng.normal(0, 0.3, s) for s in shp]],
                       kw=dict(sigma_mode=1, prior=1, prior_scale=2.0))
    # wide rows: the tiles of a CTA do not fit in shared memory -> X is streamed from L2 every step
    x = rng.standard_normal((6000, 230))
    y = rng.integers(0, 3, 6000)
    shp = [(8, 231), (7, 9), (3, 8)]
    cases["streamed"] = dict(x=x, y=y, n_test=500, feat=230, act="swish", lik=0,
                             sets=[[rng.normal(0, 0.1, s) for s in shp] for _ in range(3)], kw=dict(w_bound=1.5, prior=2))
    # trainable slopes (genReLU), many chains -> small clusters
    x = rng.standard_normal((700, 9))
    y = rng.integers(0, 4, 700)
    shp = [(6, 10), (5, 7), (4, 6)]
    cases["leaky16"] = dict(x=x, y=y, n_test=0, feat=9, act="genReLU", lik=0,
                            sets=[[rng.normal(0, 0.3, s) for s in shp] for _ in range(16)],
                            kw=dict(alphas=[0.1, 0.2, 0.0], n_act_prm=2, temperature=list(np.linspace(1.0, 0.4, 16))))
    return cases


@pytest.mark.parametrize("case", ["c1", "c2", "streamed", "leaky16"])
def test_chain_loop_matches_launch_sequence(case):
    """Small data sets step inside ONE persistent launch (k_chain_loop: a thread-block cluster per chain, leader CTA =
    update body, all CTAs = forward body, partials / counters through distributed shared memory).  The chains must be
    bit-identical to the per-step launch sequence (option chain_loop=0), for every cluster size, across calls, a
    temperature change and different chunk lengths."""
    from npbnn_b200.engine import Engine, NetShape
    cs = _chain_loop_cases()[case]
    net = NetShape.from_weights(cs["sets"][0], cs["feat"], act=cs["act"], lik=cs["lik"])
    n_chains = len(cs["sets"])
    states = []
    modes = {"c1": ("loop16", "loop4"), "c2": ("loop16", "loop4", "loop1"), "streamed": ("loop16", "loop8"),
             "leaky16": ("loop16", "loop4", "loop1")}[case] + ("sequence",)
    for mode in modes:
        eng = Engine(net)
        n_tr = len(cs["x"]) - cs["n_test"]
        if cs["n_test"]:
            eng.set_data(cs["x"][:n_tr], cs["y"][:n_tr], x_test=cs["x"][n_tr:], y_test=cs["y"][n_tr:])
        else:
            eng.set_data(cs["x"], cs["y"])
        eng.chains_init(cs["sets"], seed=99, **cs["kw"])
        eng.set_option("chain_loop", 0 if mode == "sequence" else 2)        # 2: wherever it fits (1 = where it pays)
        if mode.startswith("loop"):
            eng.set_option("chain_loop_cluster", int(mode[4:]))
        eng.mh_steps(1)
        eng.mh_steps(25)
        assert eng.last_kernel == ("k_fwd_generic" if mode == "sequence" else "k_chain_loop"), eng.last_kernel
        temp = cs["kw"].get("temperature", [1.0] * n_chains)
        eng.set_temperature(list(temp)[::-1])
        eng.mh_steps(13)
        st = eng.read_state()
        states.append((st.f64.copy(), st.i32.copy(), st.w.copy()))
        eng.close()
    ref = states[-1]
    assert np.all(ref[1][:, 0] == 39)
    assert 0 < ref[1][:, 2].sum() < 39 * n_chains         # some proposals accepted, some rejected
    for f64, i32, w in states[:-1]:
        assert np.array_equal(f64, ref[0], equal_nan=True) and np.array_equal(i32, ref[1]) and np.array_equal(w, ref[2])


@pytest.mark.parametrize("seed", range(8))
def test_chain_loop_random_shapes_match_launch_sequence(seed):
    """Randomised differential test of k_chain_loop against the per-step launch sequence: depth 2-4, ragged widths, with
    and without bias columns, categorical / Gaussian / sigma-head likelihoods, class and instance weights, every prior,
    bounded weights, adaptation on, test rows, 1-7 chains, injected-free (device Philox) proposals.  Bit-identical states."""
    from npbnn_b200.engine import Engine, NetShape
    from npbnn_b200 import _lib as L
    rng = np.random.default_rng(1000 + seed)
    depth = int(rng.integers(2, 5))
    f = int(rng.integers(2, 70))
    lik = int(rng.integers(0, 3))
    k = int(rng.integers(2, 9)) if lik == L.LIK_CATEGORICAL else int(rng.integers(1, 4))
    out = k if lik != L.LIK_GAUSSIAN_HEAD else 2 * k
    widths = [int(rng.integers(2, 20)) for _ in range(depth - 1)] + [out]
    shapes, w_in = [], f
    for wdt in widths:
        shapes.append((wdt, w_in + int(rng.integers(0, 2))))
        w_in = wdt
    n, n_test = int(rng.integers(20, 3000)), int(rng.integers(0, 200))
    x = rng.standard_normal((n + n_test, f))
    y = rng.integers(0, k, n + n_test) if lik == L.LIK_CATEGORICAL else rng.standard_normal((n + n_test, k))
    act = ["ReLU", "genReLU", "swish", "tanh"][int(rng.integers(0, 4))]
    n_chains = int(rng.integers(1, 8))
    sets = [[rng.normal(0, 0.3, s) for s in shapes] for _ in range(n_chains)]
    net = NetShape(f, shapes, act=act, lik=lik)
    kw = dict(prior=int(rng.integers(0, 4)), prior_scale=float(rng.uniform(0.5, 3.0)), seed=int(rng.integers(1, 10 ** 6)),
              adapt_f=0.25, adapt_fM=0.5, adapt_freq=int(rng.integers(2, 9)), adapt_stop=30,
              temperature=list(rng.uniform(0.3, 1.0, n_chains)), lik_temp=float(rng.uniform(0.5, 1.0)))
    if rng.integers(0, 2):
        kw["w_bound"] = 1.0
    if act == "genReLU":
        kw.update(alphas=list(rng.uniform(0.0, 0.5, depth)), n_act_prm=int(rng.integers(0, depth + 1)))
    if lik == L.LIK_GAUSSIAN:
        kw["sigma_mode"] = int(rng.integers(0, 2))
    cw = rng.uniform(0.5, 2.0, k) if lik == L.LIK_CATEGORICAL and rng.integers(0, 2) else None
    iw = rng.uniform(0.5, 2.0, n) if lik == L.LIK_CATEGORICAL and rng.integers(0, 2) else None
    states = []
    for loop in (2, 0):
        eng = Engine(net)
        eng.set_data(x[:n], y[:n], x_test=x[n:] if n_test else None, y_test=y[n:] if n_test else None, inst_w=iw, class_w=cw)
        eng.chains_init(sets, **kw)
        eng.set_option("chain_loop", loop)
        eng.mh_steps(17)
        eng.mh_steps(1)
        eng.mh_steps(9)
        kernel = eng.last_kernel
        st = eng.read_state()
        states.append((st.f64.copy(), st.i32.copy(), st.w.copy(), kernel))
        eng.close()
    a, b = states
    assert a[3] == "k_chain_loop" and b[3] == "k_fwd_generic", (a[3], b[3])
    assert np.array_equal(a[0], b[0], equal_nan=True) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert np.all(a[1][:, 0] == 27)


def test_c3_full_size_block_masked_chains():
    """BASELINE config 3 at FULL size (200,000 x 40, create_mask network [120, 80] tanh, 5 classes, 8 chains): the oracle
    scores every chain's initial state on all rows (1e-9, counters exact), and the fused block-pair kernel and the dense
    kernels (option sparse=0) run the same 12 device-generated MH iterations to identical decisions and weights."""
    from npbnn_b200.engine import Engine, NetShape
    import npbnn_b200.api as api
    rng = np.random.default_rng(17)
    n, f, k, C = 200_000, 40, 5, 8
    shapes = [(120, 40), (80, 120), (5, 81)]
    idx = [list(range(40)), sum(([g] * 3 for g in range(40)), []), []]
    mask = api.create_mask([np.zeros(s) for s in shapes], idx, [[3] * 40, [2] * 40, []])
    x = rng.standard_normal((n, f))
    teacher = [rng.normal(0, 1, s) * m for s, m in zip(shapes, mask)]
    h = np.tanh(np.tanh(x @ teacher[0].T) @ teacher[1].T)
    labels = np.argmax(h @ teacher[2][:, 1:].T + teacher[2][:, 0], 1)
    sets = [[rng.normal(0, 0.1, s) * m for s, m in zip(shapes, mask)] for _ in range(C)]
    states = []
    for sparse in (1, 0):
        eng = Engine(NetShape(f, shapes, act="tanh", lik=0))
        eng.set_option("sparse", sparse)
        eng.set_data(x, labels)
        eng.chains_init(sets, mask=mask, seed=23, temperature=list(np.linspace(1.0, 0.5, C)))
        if sparse:
            assert eng.last_kernel == "k_fwd_sparse<pairs>", eng.last_kernel
            st = eng.read_state()
            for c, ws in enumerate(sets):
                y = orc.forward(x, ws, "tanh", None, "softmax")
                assert rel_close(st.logLik[c], orc.loglik_categorical(y, labels)), c
                nc, ck, _, hist = orc.class_counters(y, labels)
                assert st.n_correct[c] == nc and np.array_equal(st.class_correct[c], ck) and np.array_equal(st.pred_hist[c], hist)
        else:
            assert not eng.last_kernel.startswith("k_fwd_sparse"), eng.last_kernel
        eng.mh_steps(12)
        states.append(eng.read_state())
        eng.close()
    a, b = states
    assert np.array_equal(a.n_accepted, b.n_accepted) and 0 < a.n_accepted.sum() < 12 * C
    assert np.array_equal(a.w, b.w)
    assert rel_close(a.logLik, b.logLik)
    assert np.array_equal(a.n_correct, b.n_correct) and np.array_equal(a.pred_hist, b.pred_hist)
    for c in range(C):
        for wl_, m in zip(a.weights(c), mask):
            assert np.all(wl_[m == 0] == 0)


def test_chain_loop_is_taken_where_it_pays():
    """Automatic mode (option chain_loop = 1, the default): the persistent loop is chosen for the reference's example sizes
    (a few thousand rows, a few chains whose clusters are resident together) and NOT for mid-size data, where the
    grid-wide launch sequence is faster (profiles/r02_chain_loop_threshold.json)."""
    from npbnn_b200.engine import Engine, NetShape
    rng = np.random.default_rng(3)
    shapes = [(5, 129), (5, 6), (5, 5)]
    net = NetShape(128, shapes, act="tanh", lik=0)
    for n, chains, want in ((2500, 1, "k_chain_loop"), (2500, 2, "k_chain_loop"), (20000, 1, "k_fwd_generic"),
                            (20000, 8, "k_fwd_generic"), (400, 32, "k_chain_loop")):
        x = rng.standard_normal((n, 128))
        y = rng.integers(0, 5, n)
        eng = Engine(net)
        eng.set_data(x, y)
        eng.chains_init([[rng.normal(0, 0.1, s) for s in shapes] for _ in range(chains)], seed=5)
        eng.mh_steps(3)
        assert eng.last_kernel == want, (n, chains, eng.last_kernel)
        eng.close()


@pytest.mark.parametrize("n", [1, 2, 15, 17, 33])
def test_tiny_and_ragged_row_counts(n):
    """Edge sizes: fewer rows than one 16-row tile, one row more / less than a tile boundary.  The reference has no
    size restriction (np.dot on [N, F], BNN_lib.py:154-162); the padded rows of the device layout must not reach the
    likelihood, the counters or the predictions -- on the specialised kernel, the generic kernel and inside the
    persistent chain loop."""
    from npbnn_b200.engine import Engine, NetShape
    # (a) the c4 network: k_fwd3 and the generic kernel against the oracle
    x, labels, sets = _c4_like(n, 3, seed=n)
    m = orc.Model(x=x, labels=labels, weights=sets[0], act="swish", mode="classification")
    eng = Engine(NetShape.from_weights(sets[0], 64, act="swish", lik=0))
    eng.set_data(x, labels)
    res = eng.forward_lik(sets)
    assert eng.last_kernel.startswith("k_fwd3"), eng.last_kernel
    eng.set_option("force_generic", 1)
    gen = eng.forward_lik(sets)
    assert eng.last_kernel == "k_fwd_generic"
    eng.set_option("force_generic", 0)
    for i, w in enumerate(sets):
        ref = oracle_score(m, w)
        for r in (res, gen):
            assert rel_close(r["loglik"][i], ref["loglik"]), (n, i, r["loglik"][i], ref["loglik"])
            assert r["counts"][i][0] == ref["n_correct"]
            assert np.array_equal(r["counts"][i][12:22], ref["pred_hist"]) and ref["pred_hist"].sum() == n
    out = eng.predict(x, sets, mean=True, votes=True, dense=True)
    dense_ref, mean_ref = orc.posterior_predict(x, sets, "swish", None, "softmax", 1)
    assert out["dense"].shape == dense_ref.shape and np.allclose(out["dense"], dense_ref, rtol=1e-10, atol=1e-300)
    assert np.allclose(out["mean"], mean_ref, rtol=1e-10, atol=1e-300)
    eng.close()
    # (b) a small tanh classifier: the persistent chain loop against the per-step launch sequence, bit for bit
    rng = np.random.default_rng(100 + n)
    xs = rng.standard_normal((n, 7))
    ys = rng.integers(0, 3, n).astype(np.int64)
    ws = [[rng.normal(0, 0.4, s) for s in ((5, 8), (4, 6), (3, 4))] for _ in range(2)]
    ms = orc.Model(x=xs, labels=ys, weights=ws[0], act="tanh", mode="classification")
    states = []
    for mode in (2, 0):
        eng = Engine(NetShape.from_weights(ws[0], 7, act="tanh", lik=0))
        eng.set_data(xs, ys)
        if mode == 2:
            sc = eng.forward_lik(ws)
            for i, w in enumerate(ws):
                ref = oracle_score(ms, w)
                assert rel_close(sc["loglik"][i], ref["loglik"]) and sc["counts"][i][0] == ref["n_correct"]
        eng.chains_init(ws, seed=5)
        eng.set_option("chain_loop", mode)
        eng.mh_steps(12)
        assert eng.last_kernel == ("k_chain_loop" if mode == 2 else "k_fwd_generic"), eng.last_kernel
        st = eng.read_state()
        states.append((st.f64.copy(), st.i32.copy(), st.w.copy()))
        eng.close()
    for a, b in zip(*states):
        assert np.array_equal(a, b, equal_nan=True)


def test_empty_training_set_is_refused():
    """Zero rows: the reference fails inside numpy (np.argmax of an empty axis, BNN_lib.py:203-209); the library
    refuses the data set up front instead of launching over nothing."""
    from npbnn_b200.engine import Engine, NetShape
    ws = [np.zeros(s) for s in ((5, 8), (3, 6))]
    eng = Engine(NetShape.from_weights(ws, 7, act="tanh", lik=0))
    with pytest.raises(Exception):
        eng.set_data(np.zeros((0, 7)), np.zeros(0, dtype=np.int64))
    eng.close()
