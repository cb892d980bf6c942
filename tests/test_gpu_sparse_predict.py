"""GPU: posterior prediction of block-masked networks on the block-sparse kernels (bnn_set_predict_mask).

Every case is compared with the same engine under option sparse=0 (the dense kernels): means and dense outputs to 1e-12
relative (1e-300 floor; regression outputs: 1e-14 absolute below 1e-2, where a sum of O(1) terms cancels; only the
order of the sums differs), vote shares, resampled classes and class counts exactly."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import npbnn_oracle as orc
from tests.test_gpu_parity import _random_block_net

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAIRS, PROGRAM = "k_fwd_sparse<pairs,predict>", "k_fwd_sparse<predict>"


def close(a, b, rtol=1e-12, floor=1e-300):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(b), floor)))


def uneven_block_net(rng, f=10, k=3):
    """Feature g -> n1[g] nodes -> n2[g] nodes: blocks of different heights (the general program, not uniform pairs)."""
    n1 = [1 + g % 4 for g in range(f)]
    n2 = [1 + (g * 3) % 5 for g in range(f)]
    h1, h2 = sum(n1), sum(n2)
    shapes = [(h1, f), (h2, h1), (k, h2 + 1)]
    mask = [np.zeros(s) for s in shapes]
    r1 = r2 = 0
    for g in range(f):
        mask[0][r1:r1 + n1[g], g] = 1
        mask[1][r2:r2 + n2[g], r1:r1 + n1[g]] = 1
        r1, r2 = r1 + n1[g], r2 + n2[g]
    mask[2][:] = 1
    return shapes, mask, [rng.normal(0, 0.4, s) * m for s, m in zip(shapes, mask)]


def c3_net():
    import npbnn_b200.api as api
    shapes = [(120, 40), (80, 120), (5, 81)]
    idx = [list(range(40)), sum(([g] * 3 for g in range(40)), []), []]
    return shapes, api.create_mask([np.zeros(s) for s in shapes], idx, [[3] * 40, [2] * 40, []])


def posterior(rng, w, mask, S):
    """S samples inside the mask, as [S, n_params]."""
    from npbnn_b200.engine import flatten_weights
    return np.stack([flatten_weights([a + rng.normal(0, 0.3, a.shape) * m for a, m in zip(w, mask)]) for _ in range(S)])


def engines(f, shapes, act, lik):
    from npbnn_b200.engine import Engine, NetShape
    out = []
    for sparse in (1, 0):
        e = Engine(NetShape(f, shapes, act=act, lik=lik))
        e.set_option("sparse", sparse)
        out.append(e)
    return out


def both(f, shapes, act, lik, x, sets, alphas=None, pattern="auto", **kw):
    """(sparse engine's outputs, its kernel, dense engine's outputs) of Engine.predict."""
    from npbnn_b200 import predshard
    from npbnn_b200.engine import NetShape
    if isinstance(pattern, str):
        pattern = predshard.zero_pattern(sets, NetShape(f, shapes, act=act, lik=lik))
    sp, de = engines(f, shapes, act, lik)
    a = sp.predict(x, sets, alphas=alphas, pattern=pattern, **kw)
    kern = sp.last_kernel
    b = de.predict(x, sets, alphas=alphas, pattern=pattern, **kw)
    assert not de.last_kernel.startswith("k_fwd_sparse")
    sp.close(), de.close()
    return a, kern, b


NETS = {"pairs": (lambda rng: (12,) + _random_block_net(rng, 12, 3, 2, 4), PAIRS),
        "program": (lambda rng: (10,) + uneven_block_net(rng), PROGRAM)}


@pytest.mark.parametrize("act", ["tanh", "ReLU", "swish", "genReLU"])
@pytest.mark.parametrize("net", ["pairs", "program"])
def test_categorical_matches_dense_kernels(net, act):
    rng = np.random.default_rng(3)
    make, kernel = NETS[net]
    f, shapes, mask, w = make(rng)
    x = rng.standard_normal((300, f))
    sets = posterior(rng, w, mask, 23)
    al = rng.uniform(0.01, 0.3, (23, 3)) if act == "genReLU" else None
    a, kern, b = both(f, shapes, act, 0, x, sets, alphas=al, mean=True, votes=True, dense=True)
    assert kern == kernel
    assert close(a["mean"], b["mean"]) and close(a["dense"], b["dense"])
    assert np.array_equal(a["votes"], b["votes"])


@pytest.mark.parametrize("lik", [1, 2, 3])                  # Gaussian, sigma head, Poisson
@pytest.mark.parametrize("net", ["pairs", "program"])
def test_regression_outputs_match_dense_kernels(net, lik):
    from npbnn_b200 import _lib as L
    rng = np.random.default_rng(5)
    make, kernel = NETS[net]
    f, shapes, mask, w = make(rng)
    out = 4 if lik in (L.LIK_GAUSSIAN_HEAD, L.LIK_POISSON) else 2
    shapes = shapes[:2] + [(out, shapes[2][1])]
    mask = mask[:2] + [np.ones(shapes[2])]
    w = w[:2] + [rng.normal(0, 0.4, shapes[2])]
    x = rng.standard_normal((200, f))
    sets = posterior(rng, w, mask, 9)
    a, kern, b = both(f, shapes, "swish", lik, x, sets, mean=True, dense=True)
    assert kern == kernel
    # an output is a sum of O(1) terms: where it cancels to near zero, the two summation orders differ by its rounding,
    # ~1e-16 absolute, so relative agreement is asked above 1e-2 and 1e-14 absolute below
    assert close(a["mean"], b["mean"], floor=1e-2) and close(a["dense"], b["dense"], floor=1e-2)


def test_c3_mask_matches_dense_kernels_and_repeats_bit_for_bit():
    from npbnn_b200 import predshard
    from npbnn_b200.engine import NetShape
    rng = np.random.default_rng(7)
    shapes, mask = c3_net()
    w = [rng.normal(0, 0.5, s) * m for s, m in zip(shapes, mask)]
    x = rng.standard_normal((3000, 40))
    sets = posterior(rng, w, mask, 37)
    pat = predshard.zero_pattern(sets, NetShape(40, shapes, act="tanh", lik=0))
    assert np.array_equal(pat, np.concatenate([m.ravel() for m in mask]))
    sp, de = engines(40, shapes, "tanh", 0)
    a = sp.predict(x, sets, pattern=pat, mean=True, votes=True)
    assert sp.last_kernel == PAIRS
    a2 = sp.predict(x, sets, pattern=pat, mean=True, votes=True)
    b = de.predict(x, sets, pattern=pat, mean=True, votes=True)
    assert close(a["mean"], b["mean"]) and np.array_equal(a["votes"], b["votes"])
    assert np.array_equal(a["mean"], a2["mean"]) and np.array_equal(a["votes"], a2["votes"])
    sp.close(), de.close()


def test_small_case_matches_the_oracle():
    rng = np.random.default_rng(9)
    f, shapes, mask, w = NETS["pairs"][0](rng)
    x = rng.standard_normal((50, f))
    sets = posterior(rng, w, mask, 5)
    al = rng.uniform(0.01, 0.3, (5, 3))
    a, kern, _ = both(f, shapes, "genReLU", 0, x, sets, alphas=al, mean=True)
    from npbnn_b200.engine import unflatten_weights
    ref = np.mean([orc.forward(x, unflatten_weights(s, shapes), "genReLU", al[i], "softmax") for i, s in enumerate(sets)], 0)
    assert kern == PAIRS and close(a["mean"], ref, 1e-9)


def _no_ties(u, dense):
    """u with every draw that falls within 1e-9 of a cumulative probability moved to 0 (class 0, no tie)."""
    cum = np.cumsum(dense, 2).transpose(1, 0, 2)               # [n, S, K]
    u = u.copy()
    u[np.any(np.abs(cum - u[:, :, None]) < 1e-9, axis=2)] = 0.0
    return u


@pytest.mark.parametrize("net", ["pairs", "program"])
def test_resampling_matches_dense_kernels(net):
    from npbnn_b200 import predshard
    from npbnn_b200.engine import NetShape
    rng = np.random.default_rng(13)
    make, kernel = NETS[net]
    f, shapes, mask, w = make(rng)
    n, S = 500, 31
    x = rng.standard_normal((n, f))
    sets = posterior(rng, w, mask, S)
    pat = predshard.zero_pattern(sets, NetShape(f, shapes, act="tanh", lik=0))
    sp, de = engines(f, shapes, "tanh", 0)
    u = _no_ties(rng.random((n, S)), de.predict(x, sets, mean=False, dense=True)["dense"])
    a = sp.predict_sample(x, sets, u=u, pattern=pat)
    assert sp.last_kernel == kernel
    b = de.predict_sample(x, sets, u=u, pattern=pat)
    for k in ("post_predictions", "class_counts", "predictions"):
        assert np.array_equal(a[k], b[k]), k
    a = sp.predict_sample(x, sets, seed=1234567, pattern=pat)
    assert sp.last_kernel == kernel
    b = de.predict_sample(x, sets, seed=1234567, pattern=pat)
    for k in ("post_predictions", "class_counts", "predictions"):
        assert np.array_equal(a[k], b[k]), k
    # a rows x samples block is that block of the full call, bit for bit
    blk = sp.predict_sample(x[100:333], sets[4:19], seed=1234567, row0=100, set0=4, pattern=pat)
    assert sp.last_kernel == kernel
    assert np.array_equal(blk["post_predictions"], a["post_predictions"][100:333, 4:19])
    sp.close(), de.close()


@pytest.mark.parametrize("n,S", [(1, 1), (17, 7), (33, 2), (33, 700), (1000, 701)])
def test_edge_sizes(n, S):
    rng = np.random.default_rng(n * 1000 + S)
    f, shapes, mask, w = NETS["pairs"][0](rng)
    x = rng.standard_normal((n, f))
    sets = posterior(rng, w, mask, S)
    a, kern, b = both(f, shapes, "tanh", 0, x, sets, mean=True, votes=True, dense=S <= 7)
    assert kern == PAIRS
    assert close(a["mean"], b["mean"]) and np.array_equal(a["votes"], b["votes"])
    if S <= 7:
        assert close(a["dense"], b["dense"])


def test_wide_output_and_dense_network_stay_on_dense_kernels_bit_for_bit():
    from npbnn_b200 import predshard
    from npbnn_b200.engine import NetShape
    rng = np.random.default_rng(21)
    f = 12
    shapes, mask, w = _random_block_net(rng, f, 3, 2, 10)          # 10 classes: wider than 8
    x = rng.standard_normal((100, f))
    sets = posterior(rng, w, mask, 4)
    a, kern, b = both(f, shapes, "tanh", 0, x, sets, mean=True, votes=True)
    assert kern == "k_fwd_generic"
    assert np.array_equal(a["mean"], b["mean"]) and np.array_equal(a["votes"], b["votes"])
    shapes = [(16, f), (8, 16), (3, 9)]                             # dense network: the pattern shortcut says dense
    sets = np.stack([np.concatenate([rng.normal(0, 0.4, s).ravel() for s in shapes]) for _ in range(4)])
    assert predshard.zero_pattern(sets, NetShape(f, shapes, act="tanh", lik=0)) is None
    a, kern, b = both(f, shapes, "tanh", 0, x, sets, pattern=np.ones(sets.shape[1]), mean=True, votes=True)
    assert kern == "k_fwd_generic"
    assert np.array_equal(a["mean"], b["mean"]) and np.array_equal(a["votes"], b["votes"])


def test_weights_outside_the_pattern_fall_back_to_dense_kernels():
    from npbnn_b200 import predshard
    from npbnn_b200.engine import NetShape
    rng = np.random.default_rng(23)
    f, shapes, mask, w = NETS["pairs"][0](rng)
    x = rng.standard_normal((64, f))
    sets = posterior(rng, w, mask, 6)
    pat = predshard.zero_pattern(sets, NetShape(f, shapes, act="tanh", lik=0))
    bad = sets.copy()
    bad[3, 5] = 0.25                                               # layer 0, row 0, feature 5: outside the mask
    assert pat[5] == 0
    a, kern, b = both(f, shapes, "tanh", 0, x, bad, pattern=pat, mean=True, votes=True)
    assert kern == "k_fwd_generic"
    assert np.array_equal(a["mean"], b["mean"]) and np.array_equal(a["votes"], b["votes"])
    from npbnn_b200.engine import unflatten_weights
    ref = np.mean([orc.forward(x, unflatten_weights(s, shapes), "tanh", None, "softmax") for s in bad], 0)
    assert close(a["mean"], ref, 1e-9)


def test_cached_engine_takes_each_calls_pattern():
    """Two networks of the same shape and different masks through the cached prediction engine of the API."""
    import npbnn_b200.api as api
    rng = np.random.default_rng(29)
    f, shapes, mask, w = NETS["pairs"][0](rng)
    x = rng.standard_normal((200, f))
    mask2 = [np.roll(m, 1, axis=1) if i == 0 else m for i, m in enumerate(mask)]
    results = []
    for m in (mask, mask2, mask):
        ws = [[rng.normal(0, 0.5, s) * mm for s, mm in zip(shapes, m)] for _ in range(5)]
        ps = [{"weights": v, "alphas": [0.0]} for v in ws]
        fun = api.ActFun(fun="tanh")
        _, mean = api.get_posterior_cat_prob(x, ps, post_summary_mode=1, actFun=fun, output_act_fun=api.SoftMax)
        eng = api._predict_engine(ws[0], f, fun, api.SoftMax)
        assert eng.last_kernel == PAIRS
        ref = np.mean([orc.forward(x, v, "tanh", None, "softmax") for v in ws], 0)
        assert close(mean, ref, 1e-9)
        results.append(mean)


def _callers(x, ps, fun, labels, pkl, tmp):
    import npbnn_b200 as bn
    import npbnn_b200.api as api
    eng = api._predict_engine(ps[0]["weights"], x.shape[1], fun, api.SoftMax)
    out, kernels = {}, []
    for mode in (0, 1, 2):
        np.random.seed(4)
        d, s = api.get_posterior_cat_prob(x, ps, post_summary_mode=mode, actFun=fun, output_act_fun=api.SoftMax)
        out["cat%d" % mode], out["dense%d" % mode] = s, d
        kernels.append(eng.last_kernel)
    np.random.seed(5)
    out["fi"] = api.feature_importance(x, weights_posterior=ps, true_labels=labels, n_permutations=2, actFun=fun,
                                       output_act_fun=api.SoftMax, write_to_file=False,
                                       feature_blocks={"a": [0, 1], "b": [2]})
    kernels.append(eng.last_kernel)
    out["pdp"] = bn.pdp(pkl, [[3]])[0]["pdp"]
    kernels.append(eng.last_kernel)
    est = bn.get_posterior_est(pkl)
    out["est"], out["est_mean"] = est["post_est"], est["prm_mean"]
    kernels.append(eng.last_kernel)
    res = bn.predictBNN(x, pkl, test_labels=labels, post_summary_mode=1, wd=str(tmp), verbose=0)
    out["pbnn"] = res["post_prob_predictions"]
    kernels.append(eng.last_kernel)
    return out, kernels


def test_prediction_callers_on_a_pickled_block_net_run_match_sparse_off(tmp_path):
    """A block-masked run pickled by run_mcmc: get_posterior_cat_prob modes 0/1/2, feature_importance, pdp,
    get_posterior_est and predictBNN run the block-sparse kernel and agree with option sparse=0."""
    import npbnn_b200 as bn
    import npbnn_b200.api as api
    rng = np.random.default_rng(31)
    x = rng.standard_normal((600, 8))
    labels = np.argmax(x[:, :3] + 0.3 * rng.standard_normal((600, 3)), 1)
    dat = {"data": x[:500], "labels": labels[:500], "test_data": x[500:], "test_labels": labels[500:]}
    np.random.seed(7)
    bnn = bn.npBNN(dat, n_nodes=[24, 16], actFun=bn.ActFun(fun="tanh"), use_bias_node=-1, seed=7)
    m = bn.create_mask(bnn._w_layers, indx_input_list=[list(range(8)), sum(([g] * 3 for g in range(8)), []), []],
                       nodes_per_feature_list=[[3] * 8, [2] * 8, []])
    bnn.apply_mask(m)
    mcmc = bn.MCMC(bnn, n_iteration=200, sampling_f=20, print_f=1000, n_post_samples=8, rng="philox")
    logger = bn.postLogger(bnn, filename="blk", wdir=str(tmp_path))
    bn.run_mcmc(bnn, mcmc, logger)
    _, _, lg = bn.load_obj(logger._pklfile)
    ps = lg._post_weight_samples
    fun = bnn._act_fun
    eng = api._predict_engine(ps[0]["weights"], 8, fun, api.SoftMax)
    a, ka = _callers(x, ps, fun, labels, logger._pklfile, tmp_path)
    assert all(k == PAIRS for k in ka), ka
    eng.set_option("sparse", 0)
    try:
        b, kb = _callers(x, ps, fun, labels, logger._pklfile, tmp_path)
    finally:
        eng.set_option("sparse", 1)
    assert not any(k.startswith("k_fwd_sparse") for k in kb), kb
    for k in ("cat1", "dense0", "dense1", "dense2", "pdp", "est", "est_mean", "pbnn"):
        assert close(a[k], b[k]), k
    for k in ("cat0", "cat2"):
        assert np.array_equal(a[k], b[k]), k
    assert a["fi"].equals(b["fi"])


def test_set_net_drops_the_previous_networks_pattern():
    """bnn_set_net on a context that holds a prediction pattern: the next network (more parameters) predicts on the
    dense kernels with the values of a fresh context."""
    from npbnn_b200 import _lib as L
    from npbnn_b200 import predshard
    from npbnn_b200.engine import Engine, NetShape
    import ctypes as C
    import torch
    rng = np.random.default_rng(41)
    f, shapes_a, mask_a, w_a = NETS["pairs"][0](rng)
    net_a = NetShape(f, shapes_a, act="tanh", lik=0)
    eng = Engine(net_a)
    eng._set_pattern(predshard.zero_pattern(posterior(rng, w_a, mask_a, 3), net_a))
    shapes_b, mask_b, w_b = _random_block_net(rng, 16, 4, 2, 4)          # more parameters than network A
    net_b = NetShape(16, shapes_b, act="tanh", lik=0)
    spec = L.NetSpec()
    spec.n_layers, spec.n_features = net_b.n_layers, net_b.n_features
    for i, ((r, c), hb) in enumerate(zip(net_b.shapes, net_b.has_bias())):
        spec.out_dim[i], spec.has_bias[i] = int(r), int(hb)
    spec.act, spec.lik = L.ACT["tanh"], 0
    L.check(eng.lib.bnn_set_net(eng._h, C.byref(spec)))
    x = rng.standard_normal((200, 16))
    sets = posterior(rng, w_b, mask_b, 5)
    xd = torch.as_tensor(x, device="cuda")
    wd = torch.as_tensor(sets, device="cuda")
    md = torch.empty((200, 4), dtype=torch.float64, device="cuda")
    L.check(eng.lib.bnn_predict(eng._h, C.c_void_p(xd.data_ptr()), 200, C.c_void_p(wd.data_ptr()), 5, None, None, None,
                                0, C.c_void_p(md.data_ptr()), None, None, eng._stream()))
    torch.cuda.synchronize()
    assert eng.last_kernel == "k_fwd_generic", eng.last_kernel
    fresh = Engine(net_b)
    ref = fresh.predict(x, sets, mean=True)["mean"]
    assert np.array_equal(md.cpu().numpy(), ref)
    fresh.close(), eng.close()


WORKER = r'''
import os, sys
sys.path.insert(0, sys.argv[3])
import numpy as np, torch.distributed as dist
rank, world = int(sys.argv[1]), int(sys.argv[2])
if world > 1:
    dist.init_process_group("gloo", store=dist.FileStore(sys.argv[4], world), rank=rank, world_size=world)
import npbnn_b200.api as api
from tests.test_gpu_parity import _random_block_net
rng = np.random.default_rng(37)
shapes, mask, w = _random_block_net(rng, 12, 3, 2, 4)
x = rng.standard_normal((700, 12))
ps = [{"weights": [a + rng.normal(0, 0.3, a.shape) * m for a, m in zip(w, mask)], "alphas": [0.0]} for _ in range(21)]
fun = api.ActFun(fun="tanh")
res = {}
for mode in (0, 1, 2):
    for rng_kind in (("host", "philox") if mode == 2 else (None,)):
        np.random.seed(8)
        d, s = api.get_posterior_cat_prob(x, ps, post_summary_mode=mode, actFun=fun, output_act_fun=api.SoftMax,
                                          return_dense=False, rng=rng_kind)
        res["m%d_%s" % (mode, rng_kind)] = s
res["kernel"] = np.array(api._predict_engine(ps[0]["weights"], 12, fun, api.SoftMax).last_kernel)
if rank == 0:
    np.savez(os.path.join(sys.argv[5], "res%d.npz" % world), **res)
if world > 1:
    dist.destroy_process_group()
'''


def test_two_gloo_ranks_return_the_single_process_results(tmp_path):
    """get_posterior_cat_prob modes 0/1/2 of a block network on two gloo ranks sharing the GPU against one process:
    votes and draws bit for bit, means to 1e-13; both run the block-sparse kernel."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out = {}
    for world in (1, 2):
        store = tmp_path / ("store%d" % world)
        procs = [subprocess.Popen([sys.executable, str(script), str(r), str(world), ROOT, str(store), str(tmp_path)],
                                  cwd=ROOT) for r in range(world)]
        try:
            for p in procs:
                p.wait(timeout=600)
        finally:
            for p in procs:          # a rank left waiting for its peer does not outlive the test
                if p.poll() is None:
                    p.kill()
                    p.wait()
        assert all(p.returncode == 0 for p in procs)
        out[world] = dict(np.load(tmp_path / ("res%d.npz" % world)))
    one, two = out[1], out[2]
    assert str(one["kernel"]) == PAIRS and str(two["kernel"]) == PAIRS
    assert np.array_equal(one["m0_None"], two["m0_None"])
    assert close(two["m1_None"], one["m1_None"], 1e-13)
    assert np.array_equal(one["m2_host"], two["m2_host"]) and np.array_equal(one["m2_philox"], two["m2_philox"])
