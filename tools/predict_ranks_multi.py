#!/usr/bin/env python
"""The posterior-prediction callers through the reference-facing surface (`import np_bnn as bn`) on 1 or N ranks.  Run
once as a plain process and once under torchrun: every rank must return the single-process results, and only rank 0
may write files.

    python tools/predict_ranks_multi.py OUTDIR
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/predict_ranks_multi.py OUTDIR

Writes OUTDIR/results.npz (rank 0: every caller's outputs), OUTDIR/files/ (predictBNN and feature_importance output)
and OUTDIR/rank<r>.json (per rank: the files it wrote, whether its np.random state was left alone, whether a call with
arguments that differ between the ranks raised ValueError).  Ranks use NCCL when each has a GPU of its own and gloo when
ranks share GPUs (rank r runs on GPU r mod the GPU count)."""
import builtins
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import np_bnn as bn
from npbnn_b200 import api, predshard
from npbnn_b200 import workloads as wl

outdir = sys.argv[1]
world = int(os.environ.get("WORLD_SIZE", "1"))
device = int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count()
if world > 1:
    torch.cuda.set_device(device)
    dist.init_process_group("nccl" if world <= torch.cuda.device_count() else "gloo")
rank = dist.get_rank() if world > 1 else 0
files = os.path.join(outdir, "files")
os.makedirs(files, exist_ok=True)

# every write of this process under OUTDIR/files: np.save / np.savetxt / DataFrame.to_csv / open(..., "w")
written = []
_open, _save, _savetxt = builtins.open, np.save, np.savetxt


def _note(path):
    if isinstance(path, str) and os.path.abspath(path).startswith(os.path.abspath(files)):
        written.append(os.path.basename(path))


def _open_w(path, mode="r", *a, **k):
    if "w" in mode or "a" in mode:
        _note(path)
    return _open(path, mode, *a, **k)


builtins.open = _open_w
np.save = lambda path, *a, **k: (_note(path), _save(path, *a, **k))[1]
np.savetxt = lambda path, *a, **k: (_note(path), _savetxt(path, *a, **k))[1]
import pandas as pd  # noqa: E402
_to_csv = pd.DataFrame.to_csv
pd.DataFrame.to_csv = lambda self, *a, **k: (_note(a[0] if a else k.get("path_or_buf")), _to_csv(self, *a, **k))[1]

res, info = {}, {"rank": rank, "world": world}


def keep_state(tag, fn):
    """Run fn after seeding numpy's global stream with 100 on rank 0 (and in the single process) and with another seed on
    every other rank; those ranks must find their state unchanged afterwards."""
    np.random.seed(100 + rank)
    before = np.random.get_state()[1].copy()
    out = fn()
    if rank:
        info.setdefault("state_kept", {})[tag] = bool(np.array_equal(before, np.random.get_state()[1]))
    return out


# ---- a 64 -> 64 -> 32 -> 10 swish classifier (a k_fwd3 family: every block runs the whole data set's kernel)
n, S = 3000, 24
x, y = wl.c4_data(n, seed=4)
y[:10] = np.arange(10)
rs = np.random.default_rng(6)
base = wl.c4_init_weights(1)[0]
post = [{"weights": [w + rs.normal(0, 0.1, w.shape) for w in base], "alphas": [0.0]} for _ in range(S)]
af = bn.ActFun(fun="swish")
kw = dict(actFun=af, output_act_fun=bn.SoftMax)
for mode in (0, 1):
    d, s = bn.get_posterior_cat_prob(x, post, post_summary_mode=mode, **kw)
    res["c4_mode%d" % mode], res["c4_dense%d" % mode] = s, d
for rng in ("philox", "host"):
    d, s = keep_state("cat2_" + rng, lambda: bn.get_posterior_cat_prob(x, post, post_summary_mode=2, rng=rng, **kw))
    res["c4_mode2_%s" % rng], res["c4_mode2_dense_%s" % rng] = s, d
    r = keep_state("sfc_" + rng, lambda: bn.sample_from_categorical(x, post, rng=rng, **kw))
    for k in ("predictions", "class_counts", "post_predictions"):
        res["c4_sfc_%s_%s" % (rng, k)] = r[k]
    res["c4_state_%s" % rng] = np.random.get_state()[1].copy()
_, s = keep_state("shuffle", lambda: bn.get_posterior_cat_prob(x, post, feature_index_to_shuffle=[3, 7, 11],
                                                               unlink_features_within_block=True, post_summary_mode=0, **kw))
res["c4_shuffle"] = s

# the pickle the file-based callers read: [bnn, mcmc, logger] as postLogger writes it
dat = {"data": x[:2000], "labels": y[:2000], "test_data": x[2000:], "test_labels": y[2000:]}
np.random.seed(1)
bnn = bn.npBNN(dat, n_nodes=[64, 32], use_bias_node=-1, actFun=af, seed=1)
pkl = os.path.join(outdir, "c4.pkl")
if rank == 0:
    logger = bn.postLogger(bnn, filename="c4", wdir=outdir)
    logger.replace_post_weight_samples(post)
    bn.SaveObject([bnn, None, logger], pkl)
if world > 1:
    dist.barrier()
est = bn.get_posterior_est(pkl)
for k in ("post_est", "prm_mean", "post_est_test", "prm_mean_test"):
    res["c4_est_" + k] = est[k]
for i, pd_ in enumerate(bn.pdp(pkl, [[0], [3, 5]])):
    res["c4_pdp%d" % i] = pd_["pdp"]
pr = bn.predictBNN(x[2000:], pkl, test_labels=y[2000:], post_summary_mode=1, wd=files, verbose=0)
res["c4_predictBNN"] = pr["post_prob_predictions"]
res["c4_threshold"] = bn.get_posterior_threshold(pkl, target_acc=0.05, post_summary_mode=0,
                                                 output_file=os.path.join(files, "c4_threshold.txt"))
df = keep_state("fi", lambda: bn.feature_importance(x[:2000], weights_pkl=pkl, true_labels=y[:2000], fname_stem="fi",
                                                    n_permutations=3, feature_blocks={"a": [0, 1], "b": [2], "c": [5, 9]},
                                                    predictions_outdir=files))
res["c4_fi"] = df[["delta_acc_mean", "delta_acc_std", "acc_with_feature_randomized_mean"]].to_numpy()

# ---- a [8, 5] tanh network above kFwd3PromoteRows: one process promotes it to k_fwd3, a rank's block may not be
n2, S2 = 40_000, 16
rs = np.random.default_rng(8)
x2 = rs.standard_normal((n2, 12))
w2 = [rs.normal(0, 0.4, s) for s in ((8, 13), (5, 9), (3, 6))]
post2 = [{"weights": [w + rs.normal(0, 0.05, w.shape) for w in w2], "alphas": [0.0]} for _ in range(S2)]
kw2 = dict(actFun=bn.ActFun(fun="tanh"), output_act_fun=bn.SoftMax, return_dense=False)
for mode in (0, 1):
    res["tanh_mode%d" % mode] = bn.get_posterior_cat_prob(x2, post2, post_summary_mode=mode, **kw2)[1]
np.random.seed(3)
r = bn.sample_from_categorical(x2, post2, actFun=kw2["actFun"], output_act_fun=bn.SoftMax, rng="philox")
res["tanh_sfc_predictions"], res["tanh_sfc_post_predictions"] = r["predictions"], r["post_predictions"]

# ---- edge cases: fewer rows than ranks, fewer samples than ranks
for nn, ss in ((1, 1), (3, 2)):
    for mode in (0, 1):
        res["edge_n%d_s%d_mode%d" % (nn, ss, mode)] = bn.get_posterior_cat_prob(x[:nn], post[:ss], post_summary_mode=mode,
                                                                               **kw)[1]
    np.random.seed(9)
    r = bn.sample_from_categorical(x[:nn], post[:ss], rng="philox", **kw)
    for k in ("predictions", "class_counts", "post_predictions"):
        res["edge_n%d_s%d_%s" % (nn, ss, k)] = r[k]
# sample groups without a sample (S < Q): an explicit grid of world sample groups over S = 1
eng = api._predict_engine(post[0]["weights"], 64, af, bn.SoftMax)
ws = [p["weights"] for p in post[:1]]
if world > 1:
    o = predshard.predict_ranks(eng, x[:500], ws, mean=True, votes=True, sample="philox", post_predictions=True,
                                draw=lambda: ([], None, 777), grid=(1, world))
else:
    o = dict(eng.predict(x[:500], ws, mean=True, votes=True))
    o.update(eng.predict_sample(x[:500], ws, seed=777))
for k in ("mean", "votes", "predictions", "class_counts", "post_predictions"):
    res["edge_q_" + k] = o[k]

# ---- arguments that differ between the ranks
if world > 1:
    try:
        bn.get_posterior_cat_prob(x[:100 + rank], post, post_summary_mode=1, **kw)
        info["mismatch_raised"] = False
    except ValueError:
        info["mismatch_raised"] = True
    dist.barrier()

torch.cuda.synchronize()
info["written"] = written
if rank == 0:
    np.savez(os.path.join(outdir, "results.npz"), **{k: np.asarray(v, dtype=np.float64) for k, v in res.items()})
json.dump(info, _open(os.path.join(outdir, "rank%d.json" % rank), "w"))
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
