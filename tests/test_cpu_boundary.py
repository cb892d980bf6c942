"""CPU: the C-ABI library loads and exports every symbol include/npbnn_b200.h declares; host-side
logic (MC3 partition / swap, net-shape inference, weight (un)flattening); product path has no CPU fallback."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "npbnn_b200.h")).read()
    return sorted(set(re.findall(r"\b(bnn_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_header_symbols_of_abi_2():
    """ABI version 2: the header's entry points, and not the two debugging entry points of the removed tensor-core
    first layer that version 1 exported."""
    import __graft_entry__ as ge
    ge.build()
    from npbnn_b200 import _lib
    import ctypes
    h = ctypes.CDLL(_lib.LIB_PATH)
    names = header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(h, n), "library does not export %s" % n
    # the ctypes binding covers exactly the header
    assert set(_lib.EXPORTED_SYMBOLS) == set(names)
    assert h.bnn_abi_version() == 2
    for n in ("bnn_debug_counters", "bnn_debug_set_trace"):
        assert not hasattr(h, n), n


def test_state_slot_constants_match_header():
    from npbnn_b200 import _lib
    src = open(os.path.join(ROOT, "include", "npbnn_b200.h")).read()
    consts = dict((k, int(v)) for k, v in re.findall(r"\b(BNN_[FI]_[A-Z0-9_]+)\s*=\s*(\d+)", src))
    for k, v in consts.items():
        py = k.replace("BNN_", "")
        assert getattr(_lib, py) == v, k
    assert _lib.MAX_LAYERS == 8 and _lib.MAX_OUT == 32


def test_no_cpu_fallback_engine_raises_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from npbnn_b200.engine import Engine, NetShape
    from npbnn_b200 import _lib
    with pytest.raises(_lib.NpbnnError):
        Engine(NetShape(4, [(3, 4), (2, 3)]))


def test_product_code_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "npbnn_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("no oracle", ""), os.path.join(dirpath, f)


def test_net_shape_bias_inference_and_flatten_roundtrip():
    from npbnn_b200.engine import NetShape, flatten_weights, unflatten_weights
    rng = np.random.default_rng(0)
    w = [rng.normal(size=(5, 129)), rng.normal(size=(5, 6)), rng.normal(size=(5, 5))]
    net = NetShape.from_weights(w, 128)
    assert net.has_bias() == [1, 1, 0] and net.n_params == 700
    back = unflatten_weights(flatten_weights(w), net.shapes)
    assert all(np.array_equal(a, b) for a, b in zip(w, back))
    with pytest.raises(ValueError):
        NetShape(10, [(4, 13)]).has_bias()


def test_mc3_partition_and_swap_rule():
    from npbnn_b200 import mc3
    from oracle import npbnn_oracle as orc
    for n, world in [(32, 1), (32, 8), (5, 2), (3, 4)]:
        parts = [mc3.chain_partition(n, world, r) for r in range(world)]
        assert parts[0][0] == 0 and sum(p[1] for p in parts) == n
        for a, b in zip(parts, parts[1:]):
            assert a[0] + a[1] == b[0]
    assert np.array_equal(mc3.default_temperatures(4, 0.8), np.linspace(0.8, 1, 4))
    assert mc3.default_temperatures(1)[0] == 1.0
    rng = np.random.default_rng(0)
    for _ in range(50):
        lp = rng.normal(-100, 5, 6)
        t = np.linspace(0.8, 1, 6)
        j, k = rng.choice(6, 2, replace=False)
        lu = float(np.log(rng.random()))
        got, sw = mc3.swap_temperatures(lp, t, int(j), int(k), lu)
        exp, sw2, _ = orc.mc3_swap(lp, t, int(j), int(k), lu)
        assert sw == sw2 and np.array_equal(got, exp)


def test_mc3_swaps_match_reference_golden():
    from npbnn_b200 import mc3
    from tests import _golden as G
    z, meta = G.load("mc3")
    for it in range(meta["n_mc3_iterations"]):
        j, k = [int(v) for v in z["it%d_pair" % it]]
        t, _ = mc3.swap_temperatures(z["it%d_logPost" % it], z["it%d_temps_before" % it], j, k, float(z["it%d_log_u" % it]))
        assert np.array_equal(t, z["it%d_temps_after" % it])


WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
from npbnn_b200 import mc3
rank, world = int(sys.argv[1]), 2
os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = sys.argv[2]
dist.init_process_group("gloo", rank=rank, world_size=world)
n = 5
lp_all = np.array([-10.0, -12.5, -9.25, -11.0, -8.75])
temps = mc3.default_temperatures(n, 0.8)
rng = mc3.SwapRNG(7)
start, cnt = mc3.chain_partition(n, world, rank)
log = []
for it in range(20):
    local = torch.tensor(lp_all[start:start + cnt] + 0.1 * it * (np.arange(cnt) + start))
    temps, swapped, pair, lp = mc3.exchange(local, temps, rng, None, world)
    log.append((pair, swapped, temps.copy(), lp.copy()))
np.save(sys.argv[3] + "/temps_%%d.npy" %% rank, np.array([l[2] for l in log]))
np.save(sys.argv[3] + "/lp_%%d.npy" %% rank, np.array([l[3] for l in log]))
dist.destroy_process_group()
'''


def test_mc3_exchange_two_ranks_gloo(tmp_path):
    """world_size-2 run of the swap step on CPU (gloo): both ranks gather the same log-posteriors and
    reach identical temperature vectors, equal to a single-process replay."""
    from npbnn_b200 import mc3
    script = tmp_path / "w.py"
    script.write_text(WORKER % {"root": ROOT})
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), port, str(tmp_path)]) for r in range(2)]
    for p in procs:
        assert p.wait(timeout=240) == 0
    t0, t1 = np.load(tmp_path / "temps_0.npy"), np.load(tmp_path / "temps_1.npy")
    l0, l1 = np.load(tmp_path / "lp_0.npy"), np.load(tmp_path / "lp_1.npy")
    assert np.array_equal(t0, t1) and np.array_equal(l0, l1)
    # single-process replay
    n = 5
    lp_all = np.array([-10.0, -12.5, -9.25, -11.0, -8.75])
    temps = mc3.default_temperatures(n, 0.8)
    rng = mc3.SwapRNG(7)
    for it in range(20):
        lp = lp_all + 0.1 * it * np.arange(n)
        assert np.allclose(l0[it], lp)
        j, k = rng.pair(n)
        temps, _ = mc3.swap_temperatures(lp, temps, j, k, rng.log_uniform())
        assert np.array_equal(temps, t0[it])
    assert sorted(t0[-1]) == sorted(mc3.default_temperatures(n, 0.8))


def test_row_partition_covers_all_rows_once():
    from npbnn_b200 import rowshard
    for n, w in ((10, 3), (1_000_003, 8), (5, 8), (64, 1)):
        spans = [rowshard.row_partition(n, w, r) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
        assert max(b - a for a, b in spans) - min(b - a for a, b in spans) <= 1


RS_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
from npbnn_b200 import rowshard
rank, world = int(sys.argv[1]), 2
os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = sys.argv[2]
dist.init_process_group("gloo", rank=rank, world_size=world)
per_row = np.load(sys.argv[3] + "/per_row.npy")            # [C, n_rows, n_values]
a, b = rowshard.row_partition(per_row.shape[1], world, rank)
out = []
for it in range(3):
    red = torch.from_numpy(per_row[:, a:b].sum(axis=1) * (it + 1))
    rowshard.dist_all_reduce_sum(red)
    out.append(red.numpy().copy())
np.save(sys.argv[3] + "/red_%%d.npy" %% rank, np.array(out))
dist.destroy_process_group()
'''


def test_rowshard_exchange_two_ranks_gloo(tmp_path):
    """world_size-2 run of the row-sharding exchange on CPU (gloo): each rank sums its own rows' contributions, the
    all-reduce leaves the same bits on both ranks (so both take the same accept decision) and they equal the
    unsharded sums."""
    rs = np.random.default_rng(5)
    per_row = rs.normal(size=(3, 1001, 23))
    np.save(tmp_path / "per_row.npy", per_row)
    script = tmp_path / "w.py"
    script.write_text(RS_WORKER % {"root": ROOT})
    port = str(31500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), port, str(tmp_path)]) for r in range(2)]
    for p in procs:
        assert p.wait(timeout=240) == 0
    r0, r1 = np.load(tmp_path / "red_0.npy"), np.load(tmp_path / "red_1.npy")
    assert np.array_equal(r0, r1)
    for it in range(3):
        np.testing.assert_allclose(r0[it], per_row.sum(axis=1) * (it + 1), rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------------------
# host-side logic of the Python surface that needs no device
# ------------------------------------------------------------------------------------------------------
def _toy_model(hyper_p=0, feature_indicators=None):
    import npbnn_b200 as bn
    rng = np.random.default_rng(0)
    x = rng.standard_normal((60, 5))
    y = rng.integers(0, 3, 60)
    y[:3] = [0, 1, 2]
    dat = {"data": x, "labels": y, "test_data": [], "test_labels": []}
    np.random.seed(3)
    return bn, bn.npBNN(dat, n_nodes=[4, 3], actFun=bn.ActFun(fun="tanh"), use_bias_node=2, hyper_p=hyper_p,
                        feature_indicators=feature_indicators)


@pytest.mark.parametrize("hp", [1, 2, 3])
def test_sample_prior_scale_is_the_oracle_draw(hp):
    """npBNN.sample_prior_scale (host arithmetic, numpy's global generator) against the oracle's restatement of
    BNN_mcmc.py:124-141 from the same generator state; the broadcast to one scale per entry follows calc_prior."""
    from oracle import npbnn_oracle as orc
    bn, bnn = _toy_model(hyper_p=hp)
    assert bnn._scales_per_layer()
    np.random.seed(11)
    bnn.sample_prior_scale()
    np.random.seed(11)
    ref = orc.gibbs_prior_scales(bnn._w_layers, hp)
    for a, b in zip(bnn._prior_scale, ref):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    e = bnn._entry_scales()
    assert e.shape == (sum(w.size for w in bnn._w_layers),)
    off = 0
    for w, sc in zip(bnn._w_layers, ref):
        assert np.array_equal(e[off:off + w.size].reshape(w.shape), np.broadcast_to(sc, w.shape))
        off += w.size


def test_data_transform_override_and_feature_means():
    bn, bnn = _toy_model(feature_indicators=True)
    assert np.array_equal(bnn._feature_indicators, np.ones(5, dtype=int))
    assert np.allclose(bnn._feature_means, bnn._data.mean(axis=0))
    dt = bn.data_transform_obj(np.array([1, 0, 1, 0, 1]), bnn._feature_means)
    cols, vals = dt.override()
    assert list(cols) == [1, 3] and np.array_equal(vals, bnn._feature_means[[1, 3]])


def test_run_mcmc_stop_points_follow_the_reference_loop():
    """run_mcmc batches iterations up to the next point at which the reference's loop does something: iteration 1
    (first print), multiples of print_f and sampling_f, and the last iteration (BNN_mcmc.py:153-170)."""
    from npbnn_b200 import api

    class M:
        _n_iterations, _print_f, _sampling_f = 95, 40, 25

    it, stops = 0, []
    while it < M._n_iterations:
        it += api._next_stop(M, it)
        stops.append(it)
    assert stops == [1, 25, 40, 50, 75, 80, 95]


class _FakeMCMC:                          # the attributes log_sample / log_weights read (module level: it is pickled)
    def __init__(self):
        self._logPost = self._logLik = self._logPrior = -1.0
        self._accuracy = self._test_accuracy = 0.5
        self._label_acc = np.array([0.5, 0.5, 0.5])
        self._acceptance_rate, self._mcmc_id, self._n_post_samples = 0.3, 0, 5
        self._current_iteration = 0


def test_background_pickle_writer_keeps_the_newest_state(tmp_path):
    """postLogger.begin_async / end_async: log_weights hands shallow snapshots to a writer thread that always writes the
    newest one; after end_async the pickle on disk is the last logged state, and the logger pickles without its
    thread state."""
    import pickle
    bn, bnn = _toy_model()

    mc = _FakeMCMC()
    logger = bn.postLogger(bnn, filename="bg", wdir=str(tmp_path))
    logger.begin_async()
    for it in range(1, 41):
        mc._current_iteration = it
        bnn._w_layers = [w + 1.0 for w in bnn._w_layers]          # rebinding, as _sync does
        logger.log_sample(bnn, mc)
        logger.log_weights(bnn, mc)
    written = logger.end_async()
    assert 1 <= written <= 40
    with open(logger._pklfile, "rb") as f:
        b2, m2, l2 = pickle.load(f)
    assert m2._current_iteration == 40 and len(l2._post_weight_samples) == 5
    assert [s["mcmc_it"] for s in l2._post_weight_samples] == [36, 37, 38, 39, 40]
    for a, b in zip(b2._w_layers, bnn._w_layers):
        assert np.array_equal(a, b)
    assert "_async" not in l2.__dict__ or l2.__dict__["_async"] is None
    assert len(open(logger._logfile).read().splitlines()) == 41
    # synchronous mode again after end_async
    mc._current_iteration = 41
    logger.log_weights(bnn, mc)
    with open(logger._pklfile, "rb") as f:
        assert pickle.load(f)[1]._current_iteration == 41


PRED_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch
import torch.distributed as dist
rank, port, out = int(sys.argv[1]), sys.argv[2], sys.argv[3]
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
dist.init_process_group("gloo", rank=rank, world_size=2)
from npbnn_b200 import predshard
n, S, K = 1000, 7, 3
rng = np.random.default_rng(0)
probs = rng.random((S, n, K))                            # stands for the per-sample predictions of the kernel
rows, sets, grid, rg, sg = predshard.partition(n, S, 2, rank, grid=(1, 2))
local = torch.from_numpy(probs[sets[0]:sets[1], rows[0]:rows[1]].sum(0))
mean = predshard.combine(local, S, 2, rank, grid)
np.save(out + "/pred_%%d.npy" %% rank, mean.numpy())
dist.destroy_process_group()
'''


def test_prediction_grid_and_combine_two_ranks_gloo(tmp_path):
    """2-D sharding of the posterior prediction (npbnn_b200/predshard.py): grid choice by rounds of warp tiles, exact
    cover of rows x samples, and the all-reduce of the partial sums over a sample group on two gloo ranks."""
    from npbnn_b200 import predshard as ps
    assert ps.grid_for(1_000_000, 10_000, 8) == (4, 2)       # 125k rows: 4.4 rounds executed as 5 -> 250k rows x half the samples
    assert ps.grid_for(1_000_000, 10_000, 4) == (4, 1) and ps.grid_for(1_000_000, 10_000, 1) == (1, 1)
    assert ps.grid_for(1_000_000, 1, 8) == (8, 1)            # a single sample cannot be split
    for n, S, world in ((1_000_003, 77, 8), (999, 5, 4), (50_000, 64, 2)):
        grid = ps.grid_for(n, S, world)
        cover = np.zeros((n, S), dtype=np.int8) if n * S < 10 ** 7 else None
        cells = 0
        for r in range(world):
            rows, sets, g, rg, sg = ps.partition(n, S, world, r, grid)
            assert g == grid and r == rg * grid[1] + sg
            cells += (rows[1] - rows[0]) * (sets[1] - sets[0])
            if cover is not None:
                cover[rows[0]:rows[1], sets[0]:sets[1]] += 1
        assert cells == n * S and (cover is None or np.all(cover == 1))
    script = tmp_path / "p.py"
    script.write_text(PRED_WORKER % {"root": ROOT})
    port = str(33500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), port, str(tmp_path)]) for r in range(2)]
    for p in procs:
        assert p.wait(timeout=240) == 0
    a, b = np.load(tmp_path / "pred_0.npy"), np.load(tmp_path / "pred_1.npy")
    probs = np.random.default_rng(0).random((7, 1000, 3))
    assert np.array_equal(a, b) and np.allclose(a, probs.mean(0), rtol=1e-14)


def test_host_draws_do_not_depend_on_how_a_stretch_is_sliced():
    """MC3 with the reference's generator (randomize_seed: default_rng(iteration + chain id) per step, BNN_env.py:383-384)
    draws slice j + 1 on a worker thread while the device runs slice j: the draws of an adaptation-free stretch must be
    the same whether they are made in one call or in slices (draw_steps(..., step0=...))."""
    from types import SimpleNamespace
    from npbnn_b200 import api
    shapes = [(6, 9), (4, 7), (3, 5)]
    g = object.__new__(api._ChainGroup)
    g.net = SimpleNamespace(n_layers=3, shapes=shapes, n_features=8)
    g.n, g.n_act_prm, g.freq_indicator, g.use_fi = 3, 0, 0.0, False
    st = SimpleNamespace(update_n=np.array([[5, 3, 2]] * 3), freq_layer_update=np.array([[0.6, 0.5, 0.4]] * 3),
                         update_ws=np.array([[0.07, 0.08, 0.09]] * 3), update_f=np.array([[0.05] * 3] * 3),
                         iteration=np.array([40, 40, 40]))
    reseed = lambda cid, i: np.random.default_rng(i + cid)
    ids = [4, 5, 6]
    whole = g.draw_steps([None] * 3, st, ids, 10, reseed=reseed)
    parts = [g.draw_steps([None] * 3, st, ids, m, reseed=reseed, step0=s0) for s0, m in ((0, 4), (4, 4), (8, 2))]
    assert whole["proposed"].sum() > 0
    for k in whole:
        assert np.array_equal(whole[k], np.concatenate([p[k] for p in parts], axis=0)), k
    with pytest.raises(AssertionError):                        # a stateful generator cannot be sliced out of order
        g.draw_steps([np.random.default_rng(0)] * 3, st, ids, 2, step0=3)
