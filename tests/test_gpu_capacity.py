"""GPU: the size limits of the dense path against the oracle, on both sides of every threshold where the code changes
path or sizes a launch -- hidden layers wider than four (and two) warps of k_fwd_generic staging fit, the widest hidden
layer a network may have, 65,537 weight sets in one call, proposals of more than UPD_DRAW_CAP (1,024) draws, the
256 / 1,024-thread update kernels and the persistent chain loop at 2,048 / 2,049 weights, 1 and 8 layers, and 32 output
columns (class counters full, scoring split into passes, partials folded by k_reduce_part)."""
import copy
import dataclasses

import numpy as np
import pytest

from oracle import npbnn_oracle as orc
from tests.test_gpu_parity import make_engine, oracle_score, rel_close

pytestmark = pytest.mark.gpu

MAX_DYN_SMEM = 232448       # BNN_MAX_DYN_SMEM (csrc/bnn_kernels.h)


def _shapes(f, hidden, out, last_bias=True):
    """Weight shapes of a dense network, bias column on every layer (on the last one if last_bias)."""
    widths = [f] + list(hidden)
    sh = [(widths[i + 1], widths[i] + 1) for i in range(len(hidden))]
    return sh + [(out, widths[-1] + int(last_bias))]


def _problem(f, hidden, k, n, act="tanh", seed=0, n_sets=1, mode="classification", last_bias=True, alphas=None,
             n_test=0, w_sd=0.3):
    rng = np.random.default_rng(seed)
    out = 2 * k if mode == "regression-error" else k
    shapes = _shapes(f, hidden, out, last_bias)
    x = rng.standard_normal((n + n_test, f))
    teacher = [rng.normal(0, 0.5, s) for s in shapes]
    okind = {"classification": "softmax", "regression": "identity", "regression-error": "regress-error"}[mode]
    yt = orc.forward(x, teacher, act, alphas, okind)
    if mode == "classification":
        lab = np.argmax(yt, axis=1)
        lab[:k] = np.arange(k)               # every class present, in the training rows
    else:
        lab = yt[:, :k] + 0.2 * rng.standard_normal((n + n_test, k))
    sets = [[rng.normal(0, w_sd, s) for s in shapes] for _ in range(n_sets)]
    m = orc.Model(x=x[:n], labels=lab[:n], weights=sets[0], act=act, alphas=alphas, mode=mode,
                  x_test=x[n:] if n_test else None, labels_test=lab[n:] if n_test else None,
                  error_prm=np.ones(k) if mode == "regression" else 1.0)
    return m, sets


def _check_scores(eng, m, sets, alphas=None):
    al = None if alphas is None else np.tile(alphas, (len(sets), 1))
    res = eng.forward_lik(sets, alphas=al)
    assert eng.last_kernel == "k_fwd_generic", eng.last_kernel
    for i, w in enumerate(sets):
        ref = oracle_score(m, w)
        assert rel_close(res["loglik"][i], ref["loglik"]), (i, res["loglik"][i], ref["loglik"])
        if m.mode == "classification":
            K = eng.K
            c = res["counts"][i]
            assert c[0] == ref["n_correct"], i
            assert np.array_equal(c[2:2 + K], ref["class_correct"]) and np.array_equal(c[2 + K:2 + 2 * K], ref["pred_hist"]), i
            if m.x_test is not None:
                assert c[1] == ref["n_correct_test"], i
        else:
            assert np.allclose(res["sums"][i][0], ref["sum_r"], rtol=1e-9, atol=1e-9), i
            assert rel_close(res["sums"][i][1], ref["sum_r2"]), i
    return res


def _check_predict(eng, m, sets, alphas=None):
    al = None if alphas is None else np.tile(alphas, (len(sets), 1))
    cat = m.mode == "classification"
    out = eng.predict(m.x, sets, alphas=al, mean=True, votes=cat, dense=True)
    assert eng.last_kernel == "k_fwd_generic", eng.last_kernel
    pa = None if alphas is None else [alphas] * len(sets)
    dense_ref, mean_ref = orc.posterior_predict(m.x, sets, m.act, pa, m.out_kind, 1)
    atol = 1e-300 if cat else 1e-11
    assert np.allclose(out["dense"], dense_ref, rtol=1e-10, atol=atol)
    assert np.allclose(out["mean"], mean_ref, rtol=1e-10, atol=atol)
    if cat:
        _, votes_ref = orc.posterior_predict(m.x, sets, m.act, pa, "softmax", 0)
        assert np.array_equal(out["votes"], votes_ref)


def _step_arrays(injs, nl):
    """Injection arrays of ONE MH iteration for len(injs) chains (one orc.StepInjection per chain)."""
    C = len(injs)
    cap = max(1, max(sum(len(l[0]) for l in inj.layers if l is not None) for inj in injs))
    arr = {"proposed": np.zeros((1, C, nl), np.int32), "count": np.zeros((1, C, nl), np.int32),
           "ix": np.zeros((1, C, cap), np.int32), "iy": np.zeros((1, C, cap), np.int32),
           "dz": np.zeros((1, C, cap)), "log_u": np.array([[inj.log_u for inj in injs]])}
    for c, inj in enumerate(injs):
        o = 0
        for l, lay in enumerate(inj.layers):
            if lay is None:
                continue
            cnt = len(lay[0])
            arr["proposed"][0, c, l], arr["count"][0, c, l] = 1, cnt
            arr["ix"][0, c, o:o + cnt], arr["iy"][0, c, o:o + cnt], arr["dz"][0, c, o:o + cnt] = lay
            o += cnt
    if injs[0].alpha_ix is not None:
        arr["alpha_ix"] = np.array([[inj.alpha_ix for inj in injs]], np.int32)
        arr["alpha_dz"] = np.array([[inj.alpha_dz for inj in injs]])
    return arr


def _stack(steps):
    """Injection arrays of consecutive iterations (each from _step_arrays) as one multi-step injection."""
    cap = max(a["ix"].shape[2] for a in steps)
    out = {}
    for key in steps[0]:
        parts = []
        for a in steps:
            v = a[key]
            if key in ("ix", "iy", "dz") and v.shape[2] < cap:
                v = np.concatenate([v, np.zeros(v.shape[:2] + (cap - v.shape[2],), v.dtype)], axis=2)
            parts.append(v)
        out[key] = np.concatenate(parts, axis=0)
    return out


def _draw(m, s, rs):
    """The draws of the next iteration: mh_step adapts before it proposes, so they follow the adapted update_n / ws."""
    s_next = copy.deepcopy(s)
    orc.adapt(m, s_next)
    return orc.draw_injection(m, s_next, rs)


def _chain(m, update_f=None, update_ws=None, prior_scale=None, n_act_prm=0, adapt=(0.0, 1.0, 1000, 0)):
    """Keyword arguments of Engine.chains_init and the oracle sampler for one chain started at m.weights."""
    nl = len(m.weights)
    uf = [0.05] * nl if update_f is None else list(update_f)
    uws = [0.075] * nl if update_ws is None else list(update_ws)
    af, afm, afreq, astop = adapt
    kw = dict(update_f=uf, update_ws=uws, prior_scale=np.ones(nl) if prior_scale is None else prior_scale,
              adapt_f=af, adapt_fM=afm, adapt_freq=afreq, adapt_stop=astop, n_act_prm=n_act_prm,
              alphas=None if m.alphas is None else np.asarray(m.alphas, dtype=np.float64))
    s = orc.make_sampler(m, update_f=uf, update_ws=uws, adapt_f=af, adapt_fM=afm, adapt_freq=afreq, adapt_stop=astop)
    return kw, s


def _replay(eng, m, s, n_steps, kernel, seed=2, on_step=None):
    """n_steps injected MH iterations of chain 0, one call each, against the oracle: proposal scores, accept decisions,
    the accepted state, and at the end bit-identical weights."""
    rs = np.random.default_rng(seed)
    nl = len(m.weights)
    st = eng.read_state()
    assert rel_close(st.logLik[0], s.logLik) and rel_close(st.logPrior[0], s.logPrior)
    for it in range(n_steps):
        inj = _draw(m, s, rs)
        d = orc.mh_step(m, s, inj)
        eng.mh_steps(1, _step_arrays([inj], nl))
        assert eng.last_kernel == kernel, (it, eng.last_kernel)
        st = eng.read_state()
        assert st.last_accepted[0] == d["accepted"], it
        assert rel_close(st.logLik_prop[0], d["logLik_prime"]), (it, st.logLik_prop[0], d["logLik_prime"])
        assert rel_close(st.logPrior_prop[0], d["logPrior_prime"]), (it, st.logPrior_prop[0], d["logPrior_prime"])
        assert rel_close(st.logLik[0], s.logLik) and rel_close(st.logPrior[0], s.logPrior), it
        assert np.array_equal(st.update_n[0], s.update_n), (it, st.update_n[0], s.update_n)
        if on_step:
            on_step(it, st)
    for a, b in zip(st.weights(0), m.weights):
        assert np.array_equal(a, b)
    if m.act_trainable:
        assert np.allclose(st.alpha[0][:len(m.alphas)], m.alphas, rtol=1e-14, atol=0)
    return st


def _same_state(a, b):
    assert np.array_equal(a.f64, b.f64, equal_nan=True)
    assert np.array_equal(a.i32, b.i32)
    assert np.array_equal(a.w, b.w)


def _widest_hidden(k, out, categorical):
    """Widest hidden layer (a multiple of 8) whose k_fwd_generic staging fits one warp per CTA in both modes:
    a full pass of likelihood counters (sets_per_pass) and the prediction accumulators."""
    zs = (out + 7) // 8 * 8 + 1
    pw = k if categorical else out
    per_pass = max(1, min(64, 16384 // ((2 + 2 * k) * 4)))
    best = 0
    for w in range(8, 4096, 8):
        lik = 8 * (256 + 32 * w + 16 * zs) + 4 * (per_pass * (2 + 2 * k) if categorical else 0)
        pred = 8 * (256 + 32 * w + 16 * zs + 16 * pw) + 4 * 16 * pw
        if max(lik, pred) > MAX_DYN_SMEM:
            break
        best = w
    return best


# ----------------------------------------------------------------------------------------------------------------------
# wide hidden layers: k_fwd_generic with 4, 2 and 1 warps per CTA
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 32])
@pytest.mark.parametrize("hidden", [200, 216, 224, 256, 512])
def test_wide_hidden_layer(hidden, k):
    """One hidden layer of 200 - 512 units (the staging of four warps fits up to 216 units at K = 2; wider layers run two
    or one warps per CTA): scoring of 1 and 40 sets with every counter, prediction summaries and 4 injected MH steps against the oracle."""
    m, sets = _problem(16, [hidden], k, 2000, act="tanh", seed=hidden + k, n_sets=40, n_test=97)
    eng = make_engine(m)
    _check_scores(eng, m, sets[:1])
    _check_scores(eng, m, sets)
    _check_predict(eng, dataclasses.replace(m, x=m.x[:300], labels=m.labels[:300]), sets[:8])
    kw, s = _chain(m, update_f=[0.02, 0.05])
    eng.chains_init([m.weights], **kw)
    _replay(eng, m, s, 4, "k_fwd_generic")
    eng.close()


@pytest.mark.parametrize("k,out,mode,expected", [(2, 2, "classification", 888), (32, 32, "classification", 816),
                                                 (32, 32, "regression", 856), (16, 32, "regression-error", 856)])
def test_widest_hidden_layer_runs_and_one_more_unit_is_refused(k, out, mode, expected):
    """The widest hidden layer the forward kernel supports for the output layer (816 units at 32 classes, 888 at 2)
    scores a full pass of sets and predicts; 8 more units, or a hidden layer of 2,048 anywhere in the network, are
    refused when the network is set, with a message that names the limit."""
    from npbnn_b200._lib import NpbnnError
    from npbnn_b200.engine import Engine, NetShape
    from tests.test_gpu_parity import LIK
    cat = mode == "classification"
    widest = _widest_hidden(k, out, cat)
    assert widest == expected                # the limits DESIGN.md states
    m, sets = _problem(12, [widest], k, 150, act="swish", seed=widest, n_sets=62, mode=mode, w_sd=0.1)
    eng = make_engine(m)
    _check_scores(eng, m, sets)
    _check_predict(eng, m, sets[:4])
    eng.close()
    for hidden in ([widest + 1], [widest + 8], [16, 2048, 16]):
        net = NetShape(12, _shapes(12, hidden, out), act="swish", lik=LIK[mode])
        with pytest.raises(NpbnnError, match=r"at most %d units per hidden layer" % widest):
            Engine(net)


# ----------------------------------------------------------------------------------------------------------------------
# more weight sets in one call than a grid dimension holds
# ----------------------------------------------------------------------------------------------------------------------
def _tiny_forward(x, W1, W2):
    """[S, N, K] softmax outputs of S sets of the network F -> 4 (tanh) -> K, vectorised over the sets."""
    z = np.einsum("nf,shf->snh", x, W1[:, :, 1:]) + W1[:, None, :, 0]
    h = orc.activation(z, "tanh")
    o = np.einsum("snh,skh->snk", h, W2[:, :, 1:]) + W2[:, None, :, 0]
    return orc.softmax_rows(o.reshape(-1, o.shape[2])).reshape(o.shape)


def test_65537_weight_sets_in_one_call():
    """S = 65,537 sets of a tiny network (3 -> 4 -> 3) over 33 rows: posterior mean and vote shares, and scoring of every
    set (1,025 passes) -- every set's counters, the log-likelihood of a sample of sets -- against the oracle."""
    S, n = 65537, 33
    rng = np.random.default_rng(17)
    x = rng.standard_normal((n, 3))
    W1, W2 = rng.normal(0, 0.8, (S, 4, 4)), rng.normal(0, 0.8, (S, 3, 5))
    lab = rng.integers(0, 3, n)
    lab[:3] = np.arange(3)
    m = orc.Model(x=x, labels=lab, weights=[W1[0], W2[0]], act="tanh")
    y = _tiny_forward(x, W1, W2)
    pref = [[W1[i], W2[i]] for i in range(40)]
    dense_ref, _ = orc.posterior_predict(x, pref, "tanh", None, "softmax", 1)
    assert np.allclose(y[:40], dense_ref, rtol=1e-13, atol=1e-300)      # the vectorised restatement is the oracle's
    flat = np.concatenate([W1.reshape(S, -1), W2.reshape(S, -1)], axis=1)
    eng = make_engine(m)
    out = eng.predict(x, flat, mean=True, votes=True)
    assert eng.last_kernel == "k_fwd_generic"
    assert np.allclose(out["mean"], y.mean(axis=0), rtol=1e-10, atol=1e-300)
    am = np.argmax(y, axis=2)
    votes = np.stack([np.sum(am == c, axis=0) for c in range(3)], axis=1) / S
    assert np.array_equal(out["votes"], votes)
    res = eng.forward_lik(flat)
    assert eng.last_kernel == "k_fwd_generic"
    ok = am == lab[None, :]
    assert np.array_equal(res["counts"][:, 0], ok.sum(axis=1))
    for c in range(3):
        assert np.array_equal(res["counts"][:, 2 + c], (ok & (lab[None, :] == c)).sum(axis=1)), c
        assert np.array_equal(res["counts"][:, 5 + c], (am == c).sum(axis=1)), c
    ll = np.log(y[:, np.arange(n), lab]).sum(axis=1)
    assert rel_close(res["loglik"], ll)
    for i in list(range(0, S, 4099)) + [65535, 65536]:
        assert rel_close(res["loglik"][i], oracle_score(m, [W1[i], W2[i]])["loglik"]), i
    eng.close()


# ----------------------------------------------------------------------------------------------------------------------
# proposals past the shared-memory draw cache (UPD_DRAW_CAP = 1,024)
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("f,hidden,draws", [(255, 128, 1651), (164, 120, 1002)])
def test_large_proposals_on_the_launch_sequence(f, hidden, draws):
    """A first layer of 32,768 entries at the default update_f proposes 1,651 entries per iteration (drawn three times,
    uncached); one of 19,800 proposes 1,002 (cached).  5 injected iterations against the oracle, and free-running chains
    (device draws) that are bit-identical when run twice and whose state the oracle scores alike."""
    m, _ = _problem(f, [hidden], 2, 600, act="ReLU", seed=f, w_sd=0.05)
    kw, s = _chain(m)
    assert int(np.sum(s.update_n)) == draws
    eng = make_engine(m)
    eng.chains_init([m.weights], **kw)
    _replay(eng, m, s, 5, "k_fwd_generic")
    m0, _ = _problem(f, [hidden], 2, 600, act="ReLU", seed=f, w_sd=0.05)
    states = []
    for _ in range(2):
        eng.chains_init([m0.weights] * 2, seed=99, **kw)
        eng.mh_steps(5)
        assert eng.last_kernel == "k_fwd_generic"
        states.append(eng.read_state())
    _same_state(*states)
    st = states[0]
    assert np.all(np.sum(st.update_n, axis=1) == draws)
    for c in range(2):
        w = st.weights(c)
        assert rel_close(st.logLik[c], oracle_score(m0, w)["loglik"]), c
        assert rel_close(st.logPrior[c], orc.log_prior(w, 1, np.ones(2))), c
    eng.close()


def test_draw_cap_crossed_by_adaptation():
    """1,682 weights, update_f 0.6 / 0.05: 955 draws per iteration until the adaptation at iteration 2 raises update_f,
    1,033 after it.  Injected iterations against the oracle with update_n read from the chain state on both sides; the
    persistent chain loop (whose pre-proposal of the next iteration gives up its draw cache there) and the launch
    sequence agree bit for bit, on injected and on device-drawn proposals."""
    m, _ = _problem(32, [48], 2, 500, act="swish", seed=4, w_sd=0.1)
    assert m.n_params == 1682
    kw, s = _chain(m, update_f=[0.6, 0.05], adapt=(0.0, 0.0, 2, 4))
    m_start = copy.deepcopy(m)
    s_start = copy.deepcopy(s)
    eng = make_engine(m)
    eng.set_option("chain_loop", 0)
    eng.chains_init([m.weights], **kw)
    seen = []
    _replay(eng, m, s, 5, "k_fwd_generic", on_step=lambda it, st: seen.append(int(np.sum(st.update_n[0]))))
    assert seen == [955, 955, 1033, 1033, 1033], seen
    # the same five iterations in one call: chain loop vs launch sequence
    rs = np.random.default_rng(2)
    mm, ss = copy.deepcopy(m_start), copy.deepcopy(s_start)
    steps = []
    for _ in range(5):
        inj = _draw(mm, ss, rs)
        orc.mh_step(mm, ss, inj)
        steps.append(_step_arrays([inj], 2))
    inj5 = _stack(steps)
    out = {}
    for mode, kernel in ((2, "k_chain_loop"), (0, "k_fwd_generic")):
        eng.set_option("chain_loop", mode)
        eng.chains_init([m_start.weights], **kw)
        eng.mh_steps(5, inj5)
        assert eng.last_kernel == kernel
        out[mode] = [eng.read_state()]
        eng.chains_init([m_start.weights] * 3, seed=7, **kw)
        eng.mh_steps(6)
        assert eng.last_kernel == kernel
        out[mode].append(eng.read_state())
    for a, b in zip(out[2], out[0]):
        _same_state(a, b)
    st = out[2][0]
    for a, b in zip(st.weights(0), m.weights):
        assert np.array_equal(a, b)
    assert np.all(np.sum(out[2][1].update_n, axis=1) == 1033)
    eng.close()


# ----------------------------------------------------------------------------------------------------------------------
# 2,048 / 2,049 weights: the update kernels' thread count and the chain loop's limit
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("f,hidden,k,last_bias,P", [(61, 32, 2, False, 2048), (62, 31, 3, True, 2049)])
def test_2048_and_2049_weights(f, hidden, k, last_bias, P):
    """Log-prior, scoring and 5 injected iterations against the oracle at 2,048 weights (256-thread update kernels,
    chain loop allowed) and 2,049 (1,024 threads, launch sequence only)."""
    m, sets = _problem(f, [hidden], k, 400, act="genReLU", seed=P, n_sets=6, last_bias=last_bias,
                       alphas=np.array([0.1, 0.0]))
    assert m.n_params == P
    m.prior_scale = [0.7, 1.3]
    eng = make_engine(m)
    for prior in (1, 2, 3):
        got = eng.log_prior(sets, prior, m.prior_scale)
        for i, w in enumerate(sets):
            assert rel_close(got[i], orc.log_prior(w, prior, m.prior_scale)), (prior, i)
    _check_scores(eng, m, sets, m.alphas)
    eng.set_option("chain_loop", 2)
    kw, s = _chain(m, update_f=[0.1, 0.3], prior_scale=m.prior_scale)
    eng.chains_init([m.weights], **kw)
    _replay(eng, m, s, 5, "k_chain_loop" if P <= 2048 else "k_fwd_generic")
    eng.close()


# ----------------------------------------------------------------------------------------------------------------------
# depth: 1 layer and BNN_MAX_LAYERS = 8
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hidden", [[], [24, 7, 40, 17, 9, 33, 5]])
def test_one_and_eight_layers(hidden):
    """A network without hidden layers and one of 8 layers of ragged widths: genReLU with trainable slopes on every
    layer (n_act_prm = number of layers) and a prior scale per layer.  Scoring, prediction, and 5 injected iterations
    with slope proposals against the oracle."""
    nl = len(hidden) + 1
    alphas = np.linspace(0.05, 0.4, nl)
    m, sets = _problem(13, hidden, 4, 700, act="genReLU", seed=nl, n_sets=5, alphas=alphas, n_test=50)
    m.prior_scale = list(np.linspace(0.5, 1.5, nl))
    m.act_trainable = True
    eng = make_engine(m)
    _check_scores(eng, m, sets, alphas)
    _check_predict(eng, m, sets, alphas)
    kw, s = _chain(m, update_f=[0.1] * nl, prior_scale=m.prior_scale, n_act_prm=nl)
    eng.set_option("chain_loop", 0)
    eng.chains_init([m.weights], **kw)
    _replay(eng, m, s, 5, "k_fwd_generic")
    eng.close()


def test_nine_layers_are_refused():
    from npbnn_b200._lib import NpbnnError
    from npbnn_b200.engine import Engine, NetShape
    with pytest.raises(NpbnnError, match=r"n_layers must be in \[1, 8\]"):
        Engine(NetShape(5, _shapes(5, [6] * 8, 3)))


# ----------------------------------------------------------------------------------------------------------------------
# 32 output columns (BNN_MAX_OUT)
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,mode", [(32, "classification"), (32, "regression"), (16, "regression-error")])
def test_32_outputs_score_in_passes(k, mode):
    """32 output columns: 130 sets are scored in three passes (62 sets per pass); every set against the oracle."""
    m, sets = _problem(9, [20], k, 1500, act="tanh", seed=k, n_sets=130, mode=mode, n_test=0)
    eng = make_engine(m)
    _check_scores(eng, m, sets)
    _check_predict(eng, dataclasses.replace(m, x=m.x[:200], labels=m.labels[:200]), sets[:3])
    eng.close()


def test_33_outputs_are_refused():
    from npbnn_b200._lib import NpbnnError
    from npbnn_b200.engine import Engine, NetShape
    with pytest.raises(NpbnnError, match="wider than BNN_MAX_OUT"):
        Engine(NetShape(5, _shapes(5, [6], 33)))


def test_32_classes_70_chains_on_70000_rows():
    """70 chains at 32 classes on 70,000 rows: the chains' forward pass runs in two passes (62 + 8) and k_reduce_part
    folds the partials of 4,375 row tiles.  Initial log-likelihood and counters of every chain, then 2 injected
    iterations of every chain, against the oracle."""
    C, n, k = 70, 70000, 32
    m, sets = _problem(8, [16], k, n, act="ReLU", seed=70, n_sets=C, w_sd=0.4)
    eng = make_engine(m)
    models, samplers = [], []
    for c in range(C):
        mc = copy.copy(m)
        mc.weights = sets[c]
        kw, s = _chain(mc, update_f=[0.05, 0.02])
        models.append(mc)
        samplers.append(s)
    eng.chains_init(sets, **kw)
    st = eng.read_state()
    for c in range(C):
        s = samplers[c]
        assert rel_close(st.logLik[c], s.logLik) and rel_close(st.logPrior[c], s.logPrior), c
        ref = oracle_score(models[c], sets[c])
        assert st.n_correct[c] == ref["n_correct"], c
        assert np.array_equal(st.pred_hist[c], ref["pred_hist"]), c
        assert np.array_equal(st.class_correct[c], ref["class_correct"]), c
    rs = np.random.default_rng(5)
    for it in range(2):
        injs = [_draw(models[c], samplers[c], rs) for c in range(C)]
        ds = [orc.mh_step(models[c], samplers[c], injs[c]) for c in range(C)]
        eng.mh_steps(1, _step_arrays(injs, 2))
        assert eng.last_kernel == "k_fwd_generic"
        st = eng.read_state()
        for c in range(C):
            assert st.last_accepted[c] == ds[c]["accepted"], (it, c)
            assert rel_close(st.logLik_prop[c], ds[c]["logLik_prime"]), (it, c)
            assert rel_close(st.logLik[c], samplers[c].logLik), (it, c)
            ref = oracle_score(models[c], models[c].weights)
            assert st.n_correct[c] == ref["n_correct"] and np.array_equal(st.pred_hist[c], ref["pred_hist"]), (it, c)
    for c in range(C):
        for a, b in zip(st.weights(c), models[c].weights):
            assert np.array_equal(a, b), c
    eng.close()
