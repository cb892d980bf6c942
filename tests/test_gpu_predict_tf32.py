"""GPU: opt-in reduced-precision posterior prediction (option predict_tf32) on every dense network.

Every case is compared with the FP64 kernels on the same engine and inputs.  Stated tolerances (include/npbnn_b200.h):
3xTF32 (option 1) class probabilities within 5e-6 absolute, regression / sigma-head / count means within
1e-5 * max(1, |y_fp64|), vote flips at most 1e-4 * n * S; plain TF32 (option 2) 5e-3 in the same forms.  A resampled
class may differ from the FP64 draw only where the FP64 running sum lies within 1e-5 of u at a class boundary (5e-3 for
plain TF32)."""
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

from tests.test_gpu_parity import _random_block_net

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {1: 5e-6, 2: 5e-3}
REG_TOL = {1: 1e-5, 2: 5e-3}
DRAW_TOL = {1: 1e-5, 2: 5e-3}
KNAME = {"ReLU": "relu", "genReLU": "leaky", "swish": "swish", "tanh": "tanh"}

# name: (features, hidden widths, output width, activation, likelihood)
NETS = {
    "config1": (128, [5, 5], 5, "tanh", 0),
    "n50_5_k10": (20, [50, 5], 10, "tanh", 0),
    "config2_regression": (3, [10, 5], 2, "ReLU", 1),
    "block_dense_40_120_80_5": (40, [120, 80], 5, "tanh", 0),
    "wide_swish": (64, [256, 128], 10, "swish", 0),
    "sigma_head": (10, [32, 16], 4, "swish", 2),
    "no_hidden": (12, [], 3, "ReLU", 0),
    "deep_genrelu": (9, [13, 7, 21, 5, 16, 9, 11], 4, "genReLU", 0),
    "widest_816_k32": (16, [816], 32, "tanh", 0),
    "k32": (20, [40], 32, "swish", 0),
    "poisson": (6, [12, 8], 1, "tanh", 3),
    "negbin": (6, [12, 8], 4, "ReLU", 4),
}


def make(name, S, rng, bias=True):
    from npbnn_b200.engine import NetShape, flatten_weights
    f, hidden, out, act, lik = NETS[name] if isinstance(name, str) else name
    shapes, width = [], f
    for o in hidden + [out]:
        shapes.append((o, width + int(bias)))
        width = o
    net = NetShape(f, shapes, act=act, lik=lik)
    sets = np.stack([flatten_weights([rng.normal(0, 1.0 / np.sqrt(c), s) for s, c in zip(shapes, [c for _, c in shapes])])
                     for _ in range(S)])
    alphas = rng.uniform(0.0, 0.3, (S, len(shapes))) if act == "genReLU" else None
    return net, sets, alphas


def check_summaries(ref, lp, lik, n, S, mode):
    if lik == 0:
        err = np.abs(lp["mean"] - ref["mean"]).max()
        assert err < TOL[mode], err
        flips = np.abs(np.rint(lp["votes"] * S) - np.rint(ref["votes"] * S)).sum() / 2
        assert flips <= (1e-4 if mode == 1 else 5e-3) * n * S, flips
    else:
        err = (np.abs(lp["mean"] - ref["mean"]) / np.maximum(1.0, np.abs(ref["mean"]))).max()
        assert err < REG_TOL[mode], err


CASES = [(name, 2003, 7) for name in NETS] + [("config1", 5, 1), ("n50_5_k10", 37, 300), ("deep_genrelu", 13, 300),
                                              ("sigma_head", 37, 1), ("widest_816_k32", 21, 7)]


@pytest.mark.parametrize("name,n,S", CASES)
def test_shape_matrix(name, n, S):
    """Every dense network kind on the generic reduced-precision kernel, options 1 and 2, against the FP64 kernel."""
    from npbnn_b200.engine import Engine
    rng = np.random.default_rng(zlib.crc32(name.encode()) + n + S)
    net, sets, alphas = make(name, S, rng)
    x = rng.standard_normal((n, net.n_features))
    eng = Engine(net)
    cat = net.lik == 0
    ref = eng.predict(x, sets, alphas=alphas, mean=True, votes=cat)
    fp64 = eng.last_kernel
    assert fp64 == "k_fwd_generic" or fp64.startswith("k_fwd3<"), fp64
    for mode in (1, 2):
        eng.set_option("predict_tf32", mode)
        lp = eng.predict(x, sets, alphas=alphas, mean=True, votes=cat)
        want = "k_pred_tf32x%d_generic<%s>" % (3 if mode == 1 else 1, KNAME[net.act])
        assert eng.last_kernel == want, (eng.last_kernel, want)
        check_summaries(ref, lp, net.lik, n, S, mode)
    eng.set_option("predict_tf32", 0)
    again = eng.predict(x, sets, alphas=alphas, mean=True, votes=cat)
    assert eng.last_kernel == fp64
    for k in ref:
        assert np.array_equal(ref[k], again[k])
    eng.close()


def test_no_bias_network():
    """Layers without a bias column (a weight matrix as wide as its input)."""
    from npbnn_b200.engine import Engine
    rng = np.random.default_rng(3)
    net, sets, _ = make((11, [17, 9], 6, "swish", 0), 9, rng, bias=False)
    x = rng.standard_normal((300, 11))
    eng = Engine(net)
    ref = eng.predict(x, sets, mean=True, votes=True)
    eng.set_option("predict_tf32", 1)
    lp = eng.predict(x, sets, mean=True, votes=True)
    assert eng.last_kernel == "k_pred_tf32x3_generic<swish>"
    check_summaries(ref, lp, 0, 300, 9, 1)
    eng.close()


def _c4_sets(rng, S):
    from npbnn_b200.engine import flatten_weights
    from npbnn_b200 import workloads as wl
    base = flatten_weights(wl.c4_init_weights(1)[0])
    return base[None, :] + rng.normal(0, 0.15, (S, base.size))


def _resampling_nets():
    """(label, net, sets, alphas, x, reduced-precision kernel prefix): a generic network and the 64-64-32-16 family."""
    from npbnn_b200.engine import NetShape
    from npbnn_b200 import workloads as wl
    rng = np.random.default_rng(21)
    net, sets, alphas = make("n50_5_k10", 23, rng)
    yield "generic", net, sets, alphas, rng.standard_normal((1501, net.n_features)), "k_pred_tf32x%d_generic<tanh>"
    x, _ = wl.c4_data(1501, seed=6)
    yield "family_a", NetShape(64, list(wl.C4_SHAPES), act="swish", lik=0), _c4_sets(rng, 23), None, x, "k_pred_tf32x%d<swish>"


def _draws_are_near_ties(dense, u, pp_ref, pp_lp, tol):
    """Every (row, set) whose drawn class differs: the FP64 running sum is within tol of u at some class boundary."""
    rows, sets = np.nonzero(pp_ref != pp_lp)
    for r, s in zip(rows, sets):
        cum = np.cumsum(dense[s, r])
        assert np.min(np.abs(cum - u[r, s])) < tol, (r, s, pp_ref[r, s], pp_lp[r, s])
    return len(rows)


def philox_uniforms(seed, n, S, row0=0, set0=0):
    """The in-kernel uniforms of bnn_predict_sample_philox_at (bnn_samp_uniform: Philox4x32-10, counter
    (row, row >> 32, set, 9), key = seed, 53 bits of the first two words), [n, S]."""
    M0, M1, W0, W1, MASK = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF
    row = np.arange(row0, row0 + n, dtype=np.uint64)[:, None] + np.zeros((1, S), dtype=np.uint64)
    st = np.arange(set0, set0 + S, dtype=np.uint64)[None, :] + np.zeros((n, 1), dtype=np.uint64)
    c = [row & MASK, row >> np.uint64(32), st, np.full((n, S), 9, dtype=np.uint64)]
    k0, k1 = seed & MASK, (seed >> 32) & MASK
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c[0], np.uint64(M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & MASK]
        k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
    return ((c[0] >> np.uint64(5)).astype(np.float64) * 67108864.0 + (c[1] >> np.uint64(6)).astype(np.float64)) / 2.0 ** 53


def test_resampling_injected_and_philox():
    """Mode-2 resampling (injected and Philox uniforms) in reduced precision: kernel names, differing draws only at
    near-ties of the FP64 probabilities, est and class_counts consistent with post_predictions."""
    from npbnn_b200.engine import Engine
    for label, net, sets, alphas, x, kname in _resampling_nets():
        n, S = x.shape[0], sets.shape[0]
        eng = Engine(net)
        dense = eng.predict(x, sets, alphas=alphas, mean=False, dense=True)["dense"]
        u = np.random.default_rng(4).random((n, S))
        ref_u = eng.predict_sample(x, sets, u=u, alphas=alphas)
        ref_p = eng.predict_sample(x, sets, alphas=alphas, seed=77)
        for mode in (1, 2):
            eng.set_option("predict_tf32", mode)
            lp_u = eng.predict_sample(x, sets, u=u, alphas=alphas)
            assert eng.last_kernel == kname % (3 if mode == 1 else 1), (label, eng.last_kernel)
            _draws_are_near_ties(dense, u, ref_u["post_predictions"], lp_u["post_predictions"], DRAW_TOL[mode])
            lp_p = eng.predict_sample(x, sets, alphas=alphas, seed=77)
            assert eng.last_kernel == kname % (3 if mode == 1 else 1), (label, eng.last_kernel)
            up = philox_uniforms(77, n, S)
            assert np.array_equal(np.argmax(np.cumsum(dense, 2) - up.T[:, :, None] >= 0, 2).T, ref_p["post_predictions"])
            m = _draws_are_near_ties(dense, up, ref_p["post_predictions"], lp_p["post_predictions"], DRAW_TOL[mode])
            assert m <= max(2, 1e-3 * n * S), (label, m)
            for res in (lp_u, lp_p):
                pp = res["post_predictions"].astype(int)
                K = res["predictions"].shape[1]
                share = np.stack([(pp == k).sum(1) for k in range(K)], 1) / S
                assert np.allclose(res["predictions"], share, rtol=0, atol=1e-12), label
                counts = np.stack([(pp == k).sum(0) for k in range(K)], 1)
                assert np.array_equal(res["class_counts"], counts), label
        eng.close()


def test_resampling_row_and_sample_split_matches_one_call():
    """predict_sample(row0=, set0=) over a 2 x 2 row x sample split reproduces the one-call post_predictions bit for bit
    on both reduced-precision kernels (the Philox uniforms are keyed on the global row and set)."""
    from npbnn_b200.engine import Engine
    for label, net, sets, alphas, x, kname in _resampling_nets():
        n, S = x.shape[0], sets.shape[0]
        eng = Engine(net)
        eng.set_option("predict_tf32", 1)
        one = eng.predict_sample(x, sets, alphas=alphas, seed=1234)["post_predictions"]
        r2, s2 = 700, 10
        got = np.empty_like(one)
        for r0, r1 in ((0, r2), (r2, n)):
            for s0, s1 in ((0, s2), (s2, S)):
                a = None if alphas is None else alphas[s0:s1]
                part = eng.predict_sample(x[r0:r1], sets[s0:s1], alphas=a, seed=1234, row0=r0, set0=s0)
                assert eng.last_kernel == kname % 3, (label, eng.last_kernel)
                got[r0:r1, s0:s1] = part["post_predictions"]
        assert np.array_equal(got, one), label
        eng.close()


def test_identical_calls_give_identical_bytes():
    """Two identical calls return identical bytes: summaries of a generic network (every likelihood kind here is summed
    the same way) and of the family-A kernel, and resampled classes."""
    from npbnn_b200.engine import Engine
    for label, net, sets, alphas, x, kname in _resampling_nets():
        eng = Engine(net)
        for mode in (1, 2):
            eng.set_option("predict_tf32", mode)
            a = eng.predict(x, sets, alphas=alphas, mean=True, votes=True)
            b = eng.predict(x, sets, alphas=alphas, mean=True, votes=True)
            assert a["mean"].tobytes() == b["mean"].tobytes() and a["votes"].tobytes() == b["votes"].tobytes(), label
            c = eng.predict_sample(x, sets, alphas=alphas, seed=5)
            d = eng.predict_sample(x, sets, alphas=alphas, seed=5)
            for k in c:
                assert c[k].tobytes() == d[k].tobytes(), (label, k)
        eng.close()
    rng = np.random.default_rng(9)
    net, sets, _ = make("sigma_head", 31, rng)
    x = rng.standard_normal((999, net.n_features))
    eng = Engine(net)
    eng.set_option("predict_tf32", 1)
    a, b = eng.predict(x, sets)["mean"], eng.predict(x, sets)["mean"]
    assert a.tobytes() == b.tobytes()
    eng.close()


def test_dense_output_stays_fp64():
    """With option 1 a call that asks for the dense [S, N, K] tensor runs the FP64 kernel and returns the bytes of
    option 0, summaries included."""
    from npbnn_b200.engine import Engine
    rng = np.random.default_rng(17)
    for name in ("config1", "sigma_head"):
        net, sets, alphas = make(name, 6, rng)
        x = rng.standard_normal((500, net.n_features))
        eng = Engine(net)
        ref = eng.predict(x, sets, alphas=alphas, mean=True, dense=True)
        k0 = eng.last_kernel
        eng.set_option("predict_tf32", 1)
        lp = eng.predict(x, sets, alphas=alphas, mean=True, dense=True)
        assert eng.last_kernel == k0 == "k_fwd_generic", (eng.last_kernel, k0)
        for k in ref:
            assert ref[k].tobytes() == lp[k].tobytes(), (name, k)
        eng.close()
    from npbnn_b200.engine import NetShape
    from npbnn_b200 import workloads as wl
    x, _ = wl.c4_data(400, seed=3)
    eng = Engine(NetShape(64, list(wl.C4_SHAPES), act="swish", lik=0))
    sets = _c4_sets(rng, 4)
    ref = eng.predict(x, sets, mean=True, votes=True, dense=True)
    eng.set_option("predict_tf32", 1)
    lp = eng.predict(x, sets, mean=True, votes=True, dense=True)
    assert eng.last_kernel.startswith("k_fwd3<"), eng.last_kernel
    for k in ref:
        assert ref[k].tobytes() == lp[k].tobytes(), k
    eng.close()


def test_block_masked_network_stays_on_the_sparse_kernels():
    """A block-masked network with its pattern set keeps the block-sparse prediction kernels (FP64) under option 1,
    with the bytes of option 0."""
    from npbnn_b200 import predshard
    from npbnn_b200.engine import Engine, NetShape, flatten_weights
    rng = np.random.default_rng(43)
    shapes, mask, w = _random_block_net(rng, 12, 3, 2, 4)
    net = NetShape(12, shapes, act="tanh", lik=0)
    sets = np.stack([flatten_weights([a + rng.normal(0, 0.3, a.shape) * m for a, m in zip(w, mask)]) for _ in range(5)])
    pattern = predshard.zero_pattern(sets, net)
    x = rng.standard_normal((300, 12))
    eng = Engine(net)
    ref = eng.predict(x, sets, mean=True, votes=True, pattern=pattern)
    k0 = eng.last_kernel
    ref_s = eng.predict_sample(x, sets, seed=3, pattern=pattern)
    eng.set_option("predict_tf32", 1)
    lp = eng.predict(x, sets, mean=True, votes=True, pattern=pattern)
    assert eng.last_kernel == k0 and k0 in ("k_fwd_sparse<pairs,predict>", "k_fwd_sparse<predict>"), (eng.last_kernel, k0)
    lp_s = eng.predict_sample(x, sets, seed=3, pattern=pattern)
    assert eng.last_kernel.startswith("k_fwd_sparse<"), eng.last_kernel
    for k in ref:
        assert ref[k].tobytes() == lp[k].tobytes(), k
    for k in ref_s:
        assert ref_s[k].tobytes() == lp_s[k].tobytes(), k
    eng.close()


SURFACE = r'''
import os, sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import npbnn_b200 as bn
import npbnn_b200.api as api
rng = np.random.default_rng(51)
n, f = 600, 7
x = rng.standard_normal((n, f))
labels = np.argmax(x[:, :3] + 0.3 * rng.standard_normal((n, 3)), 1)
res, kern = {}, {}
fun = api.ActFun(fun="tanh")
shapes = [(20, f + 1), (6, 21), (3, 7)]
ps = [{"weights": [rng.normal(0, 0.6, s) for s in shapes], "alphas": [0.0]} for _ in range(25)]
for mode in (0, 1, 2):
    for kind in (("host", "philox") if mode == 2 else (None,)):
        np.random.seed(8)
        _, s = api.get_posterior_cat_prob(x, ps, post_summary_mode=mode, actFun=fun, output_act_fun=api.SoftMax,
                                          return_dense=False, rng=kind)
        res["cat%d_%s" % (mode, kind)] = s
        kern["cat%d_%s" % (mode, kind)] = api._predict_engine(ps[0]["weights"], f, fun, api.SoftMax).last_kernel
w = [p["weights"] for p in ps]
res["pdp_cls"] = api.get_pdp(x, [2], "classification", 3, fun, api.SoftMax, w, [p["alphas"] for p in ps], None)["pdp"]
kern["pdp_cls"] = api._predict_engine(w[0], f, fun, api.SoftMax).last_kernel
rshapes = [(12, f + 1), (2, 13)]
wr = [[rng.normal(0, 0.5, s) for s in rshapes] for _ in range(19)]
res["pdp_reg"] = api.get_pdp(x, [1], "regression", 2, fun, api.RegressTransform, wr, [[0.0]] * 19, None)["pdp"]
kern["pdp_reg"] = api._predict_engine(wr[0], f, fun, api.RegressTransform).last_kernel
dat = {"data": x[:500], "labels": labels[:500], "test_data": x[500:], "test_labels": labels[500:]}
np.random.seed(3)
bnn = bn.npBNN(dat, n_nodes=[8, 4], actFun=bn.ActFun(fun="tanh"), use_bias_node=1, seed=3)
mcmc = bn.MCMC(bnn, n_iteration=10, sampling_f=5, print_f=1000, n_post_samples=2)
res["mcmc_y"] = np.asarray(mcmc._y)
np.savez(sys.argv[2], kernels=np.array([k + "=" + v for k, v in sorted(kern.items())]), **res)
'''


def test_python_surface_with_environment_option(tmp_path):
    """NPBNN_PREDICT_TF32=1 in a fresh process: get_posterior_cat_prob(return_dense=False) in modes 0/1/2 and get_pdp
    (classification and regression) run the reduced-precision kernel and agree with the FP64 process within the stated
    tolerances; mcmc._y (the dense prediction table) has the FP64 bytes."""
    script = tmp_path / "surface.py"
    script.write_text(SURFACE)
    out = {}
    for opt in ("0", "1"):
        env = dict(os.environ, NPBNN_PREDICT_TF32=opt)
        path = tmp_path / ("res%s.npz" % opt)
        subprocess.run([sys.executable, str(script), ROOT, str(path)], cwd=ROOT, env=env, check=True, timeout=600)
        out[opt] = dict(np.load(path))
    a, b = out["0"], out["1"]
    kb = dict(s.split("=") for s in b["kernels"])
    ka = dict(s.split("=") for s in a["kernels"])
    assert all(v == "k_pred_tf32x3_generic<tanh>" for v in kb.values()), kb
    assert not any(v.startswith("k_pred") for v in ka.values()), ka
    n, S = 600, 25
    assert np.abs(a["cat1_None"] - b["cat1_None"]).max() < 5e-6
    assert np.abs(np.rint(a["cat0_None"] * S) - np.rint(b["cat0_None"] * S)).sum() / 2 <= max(1, 1e-4 * n * S)
    for kind in ("host", "philox"):
        moved = np.abs(np.rint(a["cat2_%s" % kind] * S) - np.rint(b["cat2_%s" % kind] * S)).sum() / 2
        assert moved <= max(2, 1e-3 * n * S), (kind, moved)
    # the PDP curves are row means / quantiles of the mean probabilities (cumulated over classes) and regression means
    assert np.abs(a["pdp_cls"] - b["pdp_cls"]).max() < 3 * 5e-6
    assert (np.abs(a["pdp_reg"] - b["pdp_reg"]) / np.maximum(1, np.abs(a["pdp_reg"]))).max() < 1e-5
    assert a["mcmc_y"].tobytes() == b["mcmc_y"].tobytes()


def test_measured_exclusion_keeps_fp64_where_3xtf32_is_slower():
    """Config 2 (3 -> 10 -> 5 -> 2 ReLU regression) on enough rows to be padded to the 32-32-16 width family: option 1
    keeps the FP64 k_fwd3 kernel (the bytes of option 0; 3xTF32 measured slower there), option 2 runs the generic
    reduced-precision kernel within its tolerance."""
    from npbnn_b200.engine import Engine
    rng = np.random.default_rng(61)
    net, sets, _ = make("config2_regression", 3, rng)
    x = rng.standard_normal((16 * 148 * 12 + 5, 3))
    eng = Engine(net)
    ref = eng.predict(x, sets)
    k0 = eng.last_kernel
    assert k0.startswith("k_fwd3<relu,32,32,16"), k0
    eng.set_option("predict_tf32", 1)
    lp = eng.predict(x, sets)
    assert eng.last_kernel == k0 and ref["mean"].tobytes() == lp["mean"].tobytes(), eng.last_kernel
    eng.set_option("predict_tf32", 2)
    lp = eng.predict(x, sets)
    assert eng.last_kernel == "k_pred_tf32x1_generic<relu>", eng.last_kernel
    check_summaries(ref, lp, net.lik, x.shape[0], 3, 2)
    eng.close()
