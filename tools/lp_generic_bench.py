#!/usr/bin/env python
"""Opt-in reduced-precision prediction (option predict_tf32) against the FP64 kernels on every kind of dense network:
1,000,000 rows x 1,024 posterior samples per call, FP64 / 3xTF32 / plain TF32 through the same Engine.predict or
Engine.predict_sample call, after a warm-up of every mode.  A call is timed with a host clock around the call, which
ends in a device synchronise; each mode runs twice, alternating with the others, and both times are kept.  Agreement
with the FP64 call: largest difference of the means (absolute for class probabilities, relative to max(1, |y|) for
regression outputs), vote flips, and for resampling the number of differing draws.  The card's name and power limit
are read in the same run.  Output: r03_predict_tf32_generic.json in --out (default profiles/).

    python tools/lp_generic_bench.py [--rows N] [--samples S] [--out DIR]
"""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from npbnn_b200 import _lib as L, workloads as wl
from npbnn_b200.engine import Engine, NetShape, flatten_weights

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=1_000_000)
ap.add_argument("--samples", type=int, default=1024)
ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles"))
ARGS = ap.parse_args()
N, S = ARGS.rows, ARGS.samples
MODES = ("fp64", "tf32x3", "tf32x1")

# label: (features, hidden widths, outputs, activation, likelihood, call); the reference's example networks (config 1:
# bnn_classify.py, config 2: bnn_regress.py), npBNN's default n_nodes=[50, 5], a block-masked shape evaluated densely,
# a wide network, a sigma-head regression and the config-5 shape's categorical resampling (post_summary_mode=2)
SHAPES = {
    "config1_128_5_5_5_tanh": (128, [5, 5], 5, "tanh", L.LIK_CATEGORICAL, "summary"),
    "npbnn_default_50_5_tanh_k10": (20, [50, 5], 10, "tanh", L.LIK_CATEGORICAL, "summary"),
    "config2_regression_3_10_5_2_relu": (3, [10, 5], 2, "ReLU", L.LIK_GAUSSIAN, "summary"),
    "dense_40_120_80_5_tanh": (40, [120, 80], 5, "tanh", L.LIK_CATEGORICAL, "summary"),
    "wide_64_256_128_10_swish": (64, [256, 128], 10, "swish", L.LIK_CATEGORICAL, "summary"),
    "sigma_head_10_32_16_2_swish": (10, [32, 16], 2, "swish", L.LIK_GAUSSIAN_HEAD, "summary"),
    "family_a_mode2_philox": (64, [64, 32], 16, "swish", L.LIK_CATEGORICAL, "sample"),
}


def problem(label, rng):
    f, hidden, out, act, lik, call = SHAPES[label]
    if label.startswith("family_a"):
        x, _ = wl.c4_data(N, seed=0)
        base = flatten_weights(wl.c4_init_weights(1)[0])
        return NetShape(64, list(wl.C4_SHAPES), act=act, lik=lik), x, base[None, :] + rng.normal(0, 0.05, (S, base.size))
    shapes, width = [], f
    for o in hidden + [out]:
        shapes.append((o, width + 1))
        width = o
    sets = np.stack([flatten_weights([rng.normal(0, 1.0 / np.sqrt(c), (r, c)) for r, c in shapes]) for _ in range(S)])
    return NetShape(f, shapes, act=act, lik=lik), rng.standard_normal((N, f)), sets


def run(eng, call, cat, xd, wd):
    if call == "sample":
        return eng.predict_sample(xd, wd, seed=2024, device_out=True)
    return eng.predict(xd, wd, mean=True, votes=cat, device_out=True)


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = {"rows": N, "samples": S, "device": torch.cuda.get_device_name(0), "nvidia_smi": smi[:1], "shapes": {}}
    rng = np.random.default_rng(5)
    for label in SHAPES:
        net, x, w = problem(label, rng)
        call, cat = SHAPES[label][5], net.lik == L.LIK_CATEGORICAL
        eng = Engine(net)
        xd, wd = torch.from_numpy(x).cuda(), torch.from_numpy(w).cuda()
        rec, res = {m: {"seconds": []} for m in MODES}, {}
        for m in range(3):                                      # warm-up of every mode (modules, kernel attributes)
            eng.set_option("predict_tf32", m)
            run(eng, call, cat, xd, wd[:32])
        for rep in range(2):
            for m in range(3):
                eng.set_option("predict_tf32", m)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = run(eng, call, cat, xd, wd)
                torch.cuda.synchronize()
                rec[MODES[m]]["seconds"].append(time.perf_counter() - t0)
                rec[MODES[m]]["kernel"] = eng.last_kernel
                res[m] = r
        for m in (1, 2):
            a, b = res[0], res[m]
            d = rec[MODES[m]]
            d["speedup"] = min(rec["fp64"]["seconds"]) / min(d["seconds"])
            if call == "sample":
                d["differing_draws"] = int((a["post_predictions"] != b["post_predictions"]).sum().item())
                d["draws"] = N * S
            elif cat:
                d["max_abs_diff_mean_prob"] = (a["mean"] - b["mean"]).abs().max().item()
                d["vote_flips"] = ((a["votes"] * S).round() - (b["votes"] * S).round()).abs().sum().item() / 2
            else:
                d["max_rel_diff_mean"] = ((a["mean"] - b["mean"]).abs() / a["mean"].abs().clamp(min=1.0)).max().item()
        out["shapes"][label] = rec
        print(label, json.dumps(rec), flush=True)
        eng.close()
        del xd, wd, res
        torch.cuda.empty_cache()
    os.makedirs(ARGS.out, exist_ok=True)
    json.dump(out, open(os.path.join(ARGS.out, "r03_predict_tf32_generic.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
