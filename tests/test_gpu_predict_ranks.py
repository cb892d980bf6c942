"""GPU: posterior prediction on every rank of a torch.distributed group.  The prediction callers (get_posterior_cat_prob,
sample_from_categorical, get_posterior_est, pdp, predictBNN, get_posterior_threshold, feature_importance) split rows and
samples over the ranks (predshard.predict_ranks) and must return the single-process results; the in-kernel uniforms of
the resampling are keyed on the global (row, sample), so a block of the prediction draws the whole call's uniforms
(bnn_predict_sample_philox_at)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("force_generic", [0, 1])
def test_philox_block_draws_the_full_calls_uniforms(force_generic):
    """bnn_predict_sample_philox_at over rows [a, b) x sets [c, d) with offsets (a, c) reproduces that block of the full
    call's post_predictions bit for bit, on k_fwd3 and on the generic kernel; shares and class counts are the block's."""
    from npbnn_b200 import _lib as L
    from npbnn_b200 import workloads as wl
    from npbnn_b200.engine import Engine, NetShape, flatten_weights
    rng = np.random.default_rng(21)
    n, S, K = 5000, 40, 10
    x, _ = wl.c4_data(n, seed=5)
    base = flatten_weights(wl.c4_init_weights(1)[0])
    w = base[None, :] + rng.normal(0, 0.1, (S, base.size))
    eng = Engine(NetShape(64, list(wl.C4_SHAPES), act="swish", lik=L.LIK_CATEGORICAL))
    eng.set_option("force_generic", force_generic)
    full = eng.predict_sample(x, w, seed=99)
    kernel = eng.last_kernel
    assert kernel == "k_fwd_generic" if force_generic else kernel.startswith("k_fwd3<"), kernel
    assert np.array_equal(full["post_predictions"], eng.predict_sample(x, w, seed=99, row0=0, set0=0)["post_predictions"])
    for (a, b), (c, d) in (((0, 5000), (7, 40)), ((1234, 4321), (0, 40)), ((17, 2049), (3, 29)), ((4999, 5000), (39, 40))):
        blk = eng.predict_sample(x[a:b], w[c:d], seed=99, row0=a, set0=c)
        assert eng.last_kernel == kernel
        pp = blk["post_predictions"]
        assert np.array_equal(pp, full["post_predictions"][a:b, c:d]), (a, b, c, d)
        assert np.array_equal(blk["predictions"], np.stack([(pp == k).sum(1) for k in range(K)], 1) / (d - c))
        assert np.array_equal(blk["class_counts"], np.stack([(pp == k).sum(0) for k in range(K)], 1))
    # without the offsets the block draws other uniforms
    blk = eng.predict_sample(x[100:600], w[5:20], seed=99)
    assert np.mean(blk["post_predictions"] == full["post_predictions"][100:600, 5:20]) < 0.9
    eng.close()


def _run(outdir, world):
    tool = os.path.join(ROOT, "tools", "predict_ranks_multi.py")
    if world == 1:
        cmd = [sys.executable, tool, outdir]
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
               "--master-port", str(37500 + (os.getpid() + 11 * world) % 2000), tool, outdir]
    subprocess.run(cmd, check=True, timeout=900)
    res = dict(np.load(os.path.join(outdir, "results.npz")))
    infos = [json.load(open(os.path.join(outdir, "rank%d.json" % r))) for r in range(world)]
    return res, infos


_ONE = {}


def _single(tmp_path_factory):
    if "res" not in _ONE:
        _ONE["dir"] = str(tmp_path_factory.mktemp("predict_one"))
        _ONE["res"] = _run(_ONE["dir"], 1)
    return _ONE["dir"], _ONE["res"]


def _worlds():
    import torch
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    return [2, 4] + ([8] if n >= 8 else [])


@pytest.mark.parametrize("world", [2, 4, 8])
def test_callers_on_ranks_return_the_single_process_results(world, tmp_path, tmp_path_factory):
    """The worker (tools/predict_ranks_multi.py) once as one process and once on `world` ranks (NCCL with a GPU per
    rank, gloo where ranks share GPUs):
      * the 64 -> 64 -> 32 -> 10 swish network (a k_fwd3 family at every row count): votes, mode-2 predictions /
        class_counts / post_predictions (Philox and host uniforms), dense, get_posterior_est's dense and the
        feature_importance table are bit-identical; means and pdp curves agree to 1e-13 relative (the sample groups add
        in another order); predictBNN's and feature_importance's files are byte-identical and written by rank 0 alone;
      * a [8, 5] tanh network on 40,000 rows, above kFwd3PromoteRows: the single process runs it as a k_fwd3 family,
        a rank's block of 20,000 rows or fewer on the generic kernel, so it is compared to a tolerance: means to 1e-11
        relative, votes and Philox draws in all but a 1e-4 share of cells (rounding ties of the two kernels);
      * edge cases: fewer rows than ranks (empty row blocks) and, on an explicit grid, fewer samples than sample groups;
      * numpy's global stream: rank 0 ends in the single-process state, every other rank's state is untouched;
      * a call whose arguments differ between the ranks raises ValueError on every rank, and every rank exits."""
    import torch
    if world not in _worlds():
        pytest.skip("%d ranks need %d GPUs (this machine has %d)" % (world, world, torch.cuda.device_count()))
    one_dir, (one, _) = _single(tmp_path_factory)
    many_dir = str(tmp_path / ("w%d" % world))
    many, infos = _run(many_dir, world)
    assert set(one) == set(many)
    close13 = {"c4_mode1", "c4_est_prm_mean", "c4_est_prm_mean_test", "c4_pdp0", "c4_pdp1", "c4_predictBNN",
               "edge_n1_s1_mode1", "edge_n3_s2_mode1", "edge_q_mean"}
    for k in sorted(one):
        a, b = one[k], many[k]
        assert a.shape == b.shape, k
        if k.startswith("tanh_"):
            if k == "tanh_mode1":
                assert np.allclose(a, b, rtol=1e-11, atol=1e-15), k
            else:
                assert np.mean(a != b) <= 1e-4, (k, np.mean(a != b))
        elif k in close13:
            assert np.allclose(a, b, rtol=1e-13, atol=1e-300, equal_nan=True), (k, np.nanmax(np.abs(a - b)))
        else:
            assert np.array_equal(a, b, equal_nan=True), k
    assert one["c4_sfc_philox_post_predictions"].shape == (3000, 24)
    # only rank 0 writes, the same files as the single process, with the same bytes
    single_written = json.load(open(os.path.join(one_dir, "rank0.json")))["written"]
    assert infos[0]["written"] == single_written and len(single_written) >= 4
    for r, info in enumerate(infos):
        assert info["mismatch_raised"], r
        if r:
            assert info["written"] == [], (r, info["written"])
            assert len(info["state_kept"]) == 6 and all(info["state_kept"].values()), (r, info["state_kept"])
    for f in sorted(set(single_written)):
        a = open(os.path.join(one_dir, "files", f), "rb").read()
        b = open(os.path.join(many_dir, "files", f), "rb").read()
        assert a == b, f
