"""CPU (gloo, no GPU): the host logic of the collective posterior prediction (predshard.predict_ranks and the
api callers on top of it).  A numpy stand-in for the engine computes softmax(x @ W_s) per sample with the engine's
output conventions, so that every rank layout can be compared with the single-process call:
  * the combine and gather of row x sample blocks, empty row blocks (N < world) and empty sample blocks (S < Q) included;
  * the draws of rank 0 (permutations of shuffled feature blocks, host uniforms, Philox seeds) reach every rank, are the
    draws the single-process call makes, and leave the other ranks' np.random state as it was;
  * ranks called with different arguments all raise ValueError;
  * one rank, with no process group or in a group of one, returns the engine's own results for the whole problem, makes
    the reference's draws and no collective call."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FAKE_ENGINE = r'''
import numpy as np, torch
from types import SimpleNamespace


class FakeEngine:
    """Engine.predict / predict_sample with numpy arithmetic: weight set s is a flat [F * K] matrix, class probabilities
    softmax(x @ W_s); means add the samples in order and divide by their count, as the kernels do; the in-kernel
    uniform of (row, set) is a fixed function of the GLOBAL (row0 + row, set0 + set) and the seed."""

    def __init__(self, F, K):
        self.K, self.O = K, K
        self.net = SimpleNamespace(n_params=F * K, act="swish", lik=0)

    def _probs(self, x, w):
        x = np.asarray(x.cpu() if isinstance(x, torch.Tensor) else x, dtype=np.float64)
        ws = np.stack([np.concatenate([np.ravel(a) for a in s]) if isinstance(s, list) else np.ravel(s) for s in w])
        z = np.einsum("nf,sfk->snk", x, ws.reshape(len(ws), x.shape[1], self.K))
        e = np.exp(z - z.max(2, keepdims=True))
        return e / e.sum(2, keepdims=True)

    @staticmethod
    def _out(d, device_out):
        return {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)) if device_out else v) for k, v in d.items()}

    def predict(self, x, w, alphas=None, override=None, mean=True, votes=False, dense=False, device_out=False):
        x = np.array(x, dtype=np.float64)
        if override is not None:
            x[:, list(override[0])] = list(override[1])
        p = self._probs(x, w)
        out = {}
        if mean:
            acc = np.zeros(p.shape[1:])
            for s in range(len(p)):
                acc += p[s]
            out["mean"] = acc / len(p)
        if votes:
            cnt = np.zeros(p.shape[1:])
            for s in range(len(p)):
                cnt[np.arange(p.shape[1]), p[s].argmax(1)] += 1
            out["votes"] = cnt / len(p)
        if dense:
            out["dense"] = p
        return self._out(out, device_out)

    def predict_sample(self, x, w, u=None, alphas=None, post_predictions=True, seed=None, row0=0, set0=0,
                       device_out=False):
        p = self._probs(x, w)
        S, n, K = p.shape
        if u is None:
            r = (row0 + np.arange(n))[:, None] * 7919 + (set0 + np.arange(S))[None, :] * 104729 + seed % 1000003
            u = np.modf(np.sin(r.astype(np.float64)) * 43758.5453)[0] % 1.0
        u = np.asarray(u.cpu() if isinstance(u, torch.Tensor) else u)
        cum = np.cumsum(p, 2).transpose(1, 0, 2)                       # [n, S, K]
        drawn = np.argmax(cum - u[:, :, None] >= 0.0, axis=2)
        drawn[~np.any(cum - u[:, :, None] >= 0.0, axis=2)] = 0
        est = np.stack([(drawn == k).sum(1) for k in range(K)], axis=1) / S
        cc = np.stack([(drawn == k).sum(0) for k in range(K)], axis=1).astype(np.float64)
        return self._out({"predictions": est, "class_counts": cc,
                          "post_predictions": drawn.astype(np.float64) if post_predictions else None}, device_out)
'''

WORKER = r'''
import os, sys, json
sys.path.insert(0, %(root)r)
exec(open(%(fake)r).read())
import numpy as np, torch
import torch.distributed as dist
rank, world, port, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4]
if world > 1:
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
import npbnn_b200 as bn
from npbnn_b200 import api, predshard

F, K = 6, 4
eng = FakeEngine(F, K)
api._predict_engine = lambda *a, **k: eng
af = bn.ActFun(fun="swish")


def post(S, seed):
    rs = np.random.default_rng(seed)
    return [{"weights": [rs.normal(0, 1.0, (F, K))], "alphas": [0.0]} for _ in range(S)]


res, info = {}, {}
for n, S in ((1, 1), (3, 2), (37, 5), (200, 12), (203, 1)):        # N < world and S < world included
    x = np.random.default_rng(n).standard_normal((n, F))
    ps = post(S, S)
    tag = "n%%d_s%%d" %% (n, S)
    for mode in (0, 1):
        d, s = bn.get_posterior_cat_prob(x, ps, post_summary_mode=mode, actFun=af, output_act_fun=bn.SoftMax)
        res[tag + "_mode%%d" %% mode], res[tag + "_dense%%d" %% mode] = s, d
    # the callers that draw nothing: partial dependence (a column override per grid step)
    res[tag + "_pdp_mean"] = bn.get_pdp(x, [1], "classification", K, af, bn.SoftMax, [p["weights"] for p in ps],
                                        [p["alphas"] for p in ps], None)["pdp"]
    for rng in ("host", "philox"):
        np.random.seed(11 + rank * (world > 1))      # ranks other than 0 hold other global states
        before = np.random.get_state()[1].copy()
        r = bn.sample_from_categorical(x, ps, actFun=af, output_act_fun=bn.SoftMax, rng=rng)
        after = np.random.get_state()[1]
        for k in ("predictions", "class_counts", "post_predictions"):
            res["%%s_%%s_%%s" %% (tag, rng, k)] = r[k]
        if rank == 0:
            res["%%s_%%s_state" %% (tag, rng)] = after.copy()
        else:
            info["%%s_%%s_state_kept" %% (tag, rng)] = bool(np.array_equal(before, after))
    # shuffled feature blocks: a list of single features (unlinked), a 2-D block and a repeated column, then mode-2
    # uniforms from the same stream
    for i, (fis, unlink) in enumerate((([0, 3], True), ([1, 2, 4], False), ([5, 5], True), (2, False))):
        np.random.seed(5 + rank * (world > 1))
        before = np.random.get_state()[1].copy()
        _, s = bn.get_posterior_cat_prob(x, ps, feature_index_to_shuffle=fis, unlink_features_within_block=unlink,
                                         post_summary_mode=2, actFun=af, output_act_fun=bn.SoftMax, return_dense=False,
                                         rng="host")
        res["%%s_shuffle%%d" %% (tag, i)] = s
        if rank:
            info["%%s_shuffle%%d_state_kept" %% (tag, i)] = bool(np.array_equal(before, np.random.get_state()[1]))
    # sample groups with no sample (S < Q) and row groups with no row on an explicit grid
    if world > 1:
        for i, grid in enumerate(((1, world), (world, 1))):
            o = predshard.predict_ranks(eng, x, [p["weights"] for p in ps], mean=True, votes=True, dense=True,
                                        sample="philox", post_predictions=True, draw=lambda: ([], None, 4242), grid=grid)
            for k, v in o.items():
                res["%%s_grid%%d_%%s" %% (tag, i, k)] = v
    else:
        full = eng.predict(x, [p["weights"] for p in ps], mean=True, votes=True, dense=True)
        smp = eng.predict_sample(x, [p["weights"] for p in ps], seed=4242)
        for i in range(2):
            for k, v in list(full.items()) + list(smp.items()):
                res["%%s_grid%%d_%%s" %% (tag, i, k)] = v
# different arguments on different ranks
if world > 1:
    try:
        bn.get_posterior_cat_prob(np.zeros((10 + rank, F)), post(3, 0), post_summary_mode=1, actFun=af,
                                  output_act_fun=bn.SoftMax)
        info["mismatch_raised"] = False
    except ValueError:
        info["mismatch_raised"] = True
    dist.barrier()
if rank == 0:
    np.savez(out + "/res.npz", **{k: (np.array(np.nan) if v is None else v) for k, v in res.items()})
json.dump(info, open(out + "/info%%d.json" %% rank, "w"))
if world > 1:
    dist.destroy_process_group()
'''


def _run(tmp_path, world):
    out = tmp_path / ("w%d" % world)
    out.mkdir()
    fake = tmp_path / "fake_engine.py"
    fake.write_text(FAKE_ENGINE)
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT, "fake": str(fake)})
    port = str(35500 + (os.getpid() + 13 * world) % 2000)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    procs = [subprocess.Popen([sys.executable, str(script), str(r), str(world), port, str(out)], env=env)
             for r in range(world)]
    for p in procs:
        assert p.wait(timeout=300) == 0
    res = dict(np.load(out / "res.npz"))
    infos = [json.load(open(out / ("info%d.json" % r))) for r in range(world)]
    return res, infos


def test_permuted_rows_are_the_reference_permutation():
    """x[:, fi] = np.random.permutation(x[:, fi]) for an index, a 2-D block and a repeated column, in sequence: the
    rows a rank builds from np.random.permutation(N) and the full host copy are those rows of the permuted array."""
    from npbnn_b200 import predshard
    x = np.random.default_rng(0).standard_normal((57, 6))
    for shuffle in ([0, 3], [[1, 2, 4]], [5, 5], [2, [2, 3], -1]):
        np.random.seed(9)
        ref = x.copy()
        for fi in shuffle:
            ref[:, fi] = np.random.permutation(ref[:, fi])
        np.random.seed(9)
        perms = [np.random.permutation(len(x)) for _ in shuffle]
        for lo, hi in ((0, 57), (0, 0), (10, 31), (56, 57)):
            assert np.array_equal(predshard.permuted_rows(x, lo, hi, shuffle, perms), ref[lo:hi]), (shuffle, lo, hi)


@pytest.mark.parametrize("world", [2, 3, 4])
def test_rank_layouts_return_the_single_process_results(world, tmp_path):
    one, _ = _run(tmp_path, 1)
    many, infos = _run(tmp_path, world)
    assert set(one) == set(many)
    for k in one:
        a, b = one[k], many[k]
        assert a.shape == b.shape, k
        if k.endswith("mode1") or k.endswith("_mean"):
            # sample groups add in another order than one pass over the samples
            assert np.allclose(a, b, rtol=1e-13, atol=0), k
        else:
            assert np.array_equal(a, b, equal_nan=True), k
    for r, info in enumerate(infos):
        if r:
            kept = [k for k in info if k.endswith("_kept")]
            assert len(kept) == 5 * 6 and all(info[k] for k in kept), (r, info)
        assert info["mismatch_raised"], (r, info)


def _forbidden(name):
    def call(*a, **k):
        raise AssertionError("one rank made a collective call: torch.distributed.%s" % name)
    return call


def _one_rank_is_the_engine(eng):
    """The callers on one rank against the engine calls on a copy of x permuted in place by
    x[:, fi] = np.random.permutation(x[:, fi]): the same bits, and the same np.random state afterwards."""
    import npbnn_b200 as bn
    n, S = 37, 5
    x = np.random.default_rng(2).standard_normal((n, 6))
    rs = np.random.default_rng(3)
    ps = [{"weights": [rs.normal(0, 1.0, (6, 4))], "alphas": [0.0]} for _ in range(S)]
    w = [p["weights"] for p in ps]
    af = bn.ActFun(fun="swish")
    kw = dict(actFun=af, output_act_fun=bn.SoftMax)

    def same(call, ref, seed):
        np.random.seed(seed)
        want = ref()
        state = np.random.get_state()
        np.random.seed(seed)
        got = call()
        assert np.array_equal(np.random.get_state()[1], state[1]) and np.random.get_state()[2] == state[2]
        return got, want

    for fis, unlink in ((None, False), ([0, 3], True), ([1, 2, 4], False), ([5, 5], True), (2, False)):
        def ref_cat_prob(mode):
            xr = x.copy()
            if fis:
                for fi in (fis if unlink and type(fis) == list else [fis]):
                    xr[:, fi] = np.random.permutation(xr[:, fi])
            if mode == 2:
                dense = eng.predict(xr, w, mean=False, dense=True)["dense"]
                return dense, eng.predict_sample(xr, w, np.random.random((n, S)), post_predictions=False)["predictions"]
            o = eng.predict(xr, w, mean=mode == 1, votes=mode == 0, dense=True)
            return o["dense"], o["votes" if mode == 0 else "mean"]

        for mode in (0, 1, 2):
            got, want = same(lambda: bn.get_posterior_cat_prob(x, ps, feature_index_to_shuffle=fis,
                                                                unlink_features_within_block=unlink,
                                                                post_summary_mode=mode, rng="host", **kw),
                             lambda: ref_cat_prob(mode), 5)
            assert all(np.array_equal(g, r) for g, r in zip(got, want)), (fis, mode)
    # an invalid mode raises before any draw
    np.random.seed(5)
    state = np.random.get_state()[1].copy()
    with pytest.raises(ValueError):
        bn.get_posterior_cat_prob(x, ps, feature_index_to_shuffle=[0, 3], post_summary_mode=3, **kw)
    assert np.array_equal(np.random.get_state()[1], state)

    def ref_sample(rng):
        if rng == "host":
            return eng.predict_sample(x, w, np.random.random((n, S)))
        return eng.predict_sample(x, w, seed=int(np.random.randint(0, 2 ** 31 - 1)) * 2654435761 + 1)

    for rng in ("host", "philox"):
        got, want = same(lambda: bn.sample_from_categorical(x, ps, rng=rng, **kw), lambda: ref_sample(rng), 11)
        assert set(got) == set(want) and all(np.array_equal(got[k], want[k]) for k in want), rng

    def ref_pdp():
        grid = bn.make_pdp_features(x, [1])
        out = np.zeros((len(grid), 4, 3))
        for i, v in enumerate(grid[:, 0]):
            m = np.cumsum(eng.predict(x, w, override=([1], [float(v)]), mean=True)["mean"], axis=1)
            out[i, :, 0] = np.mean(m, axis=0)
            out[i, :, 1], out[i, :, 2] = np.quantile(m, q=(0.025, 0.975), axis=0)
        return out

    got, want = same(lambda: bn.get_pdp(x, [1], "classification", 4, af, bn.SoftMax, w, [p["alphas"] for p in ps],
                                        None)["pdp"], ref_pdp, 13)
    assert np.array_equal(got, want)


@pytest.fixture
def fake_engine(monkeypatch):
    from npbnn_b200 import api
    ns = {}
    exec(FAKE_ENGINE, ns)
    eng = ns["FakeEngine"](6, 4)
    monkeypatch.setattr(api, "_predict_engine", lambda *a, **k: eng)
    return eng


def test_one_process_returns_the_engine_results(fake_engine):
    import torch.distributed as dist
    assert not dist.is_initialized()
    _one_rank_is_the_engine(fake_engine)


def test_group_of_one_rank_makes_no_collective_call(fake_engine, monkeypatch, tmp_path):
    import torch.distributed as dist
    from npbnn_b200 import predshard
    dist.init_process_group("gloo", init_method="file://%s" % (tmp_path / "store"), rank=0, world_size=1)
    try:
        assert predshard.ranks() == (1, 0)
        for name in ("all_gather", "all_gather_object", "broadcast", "broadcast_object_list", "all_reduce"):
            monkeypatch.setattr(dist, name, _forbidden(name))
        _one_rank_is_the_engine(fake_engine)
    finally:
        dist.destroy_process_group()
