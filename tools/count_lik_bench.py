#!/usr/bin/env python
"""Cost of the count-likelihood epilogue (estimation_mode="custom"): free-running MH chain-steps/s of the Poisson and
negative-binomial likelihoods against Gaussian regression on the same network and data size, on the two paths the
dispatcher takes for them:
  - family A (64 -> 64 -> 32 -> 2, swish, bias on the last layer), 32 chains x 1,000,000 rows: k_fwd3 + k_mh_update;
  - the small-data case (config-1 sized: 24 features, [5, 5] tanh, 2 outputs, 400 rows), 4 chains: k_chain_loop.
Kinds are timed in alternation (three rounds, median reported) so that drift of the shared machine hits all alike.
Also the forward-kernel time per launch of forward_lik on the family-A data (option time_forward, 32 weight sets).
    python tools/count_lik_bench.py [out.json]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch  # noqa: E401,E402
from npbnn_b200 import _lib as L  # noqa: E402
from npbnn_b200.engine import Engine, NetShape  # noqa: E402

KINDS = [("gaussian", L.LIK_GAUSSIAN), ("poisson", L.LIK_POISSON), ("negbin", L.LIK_NEGBIN)]


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")]
    except Exception as e:          # the numbers still stand; the reader sees that the card settings are unknown
        info["power_limit"] = "unknown (%s)" % type(e).__name__
    return info


def make_case(kind, f, shapes, rows, act, n_chains, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(rows, f, dtype=torch.float64, device="cuda", generator=g)
    if kind == L.LIK_GAUSSIAN:
        y = torch.randn(rows, shapes[-1][0], dtype=torch.float64, device="cuda", generator=g)
    else:
        y = torch.poisson(torch.full((rows, 1), 3.0, dtype=torch.float64, device="cuda"), generator=g)
    eng = Engine(NetShape(f, shapes, act=act, lik=kind))
    eng.set_data(x, y)
    rs = np.random.RandomState(seed)
    w0 = np.stack([np.concatenate([rs.normal(0, 0.1, s).ravel() for s in shapes]) for _ in range(n_chains)])
    eng.chains_init(w0, seed=seed)
    return eng, w0


def chain_rate(eng, n_chains, steps):
    eng.mh_steps(steps)                       # warm-up: graph capture / module load
    eng.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.mh_steps(steps)
    e1.record()
    e1.synchronize()
    return n_chains * steps / (e0.elapsed_time(e1) * 1e-3)


def forward_ms(eng, w, reps=6):
    eng.forward_lik(w)
    eng.set_option("time_forward", 1)
    eng.forward_time(True)
    for _ in range(reps):
        eng.forward_lik(w)
    ms, n = eng.forward_time(True)
    eng.set_option("time_forward", 0)
    return ms / n, eng.last_kernel


def run_case(name, f, shapes, rows, act, n_chains, steps, timed_forward):
    engines = {k: make_case(kind, f, shapes, rows, act, n_chains, 7) for k, kind in KINDS}
    rates = {k: [] for k, _ in KINDS}
    kernels = {}
    for _ in range(3):
        for k, _ in KINDS:
            eng = engines[k][0]
            rates[k].append(chain_rate(eng, n_chains, steps))
            kernels[k] = eng.last_kernel
    res = {"case": name, "rows": rows, "chains": n_chains, "steps_per_window": steps, "kinds": {}}
    for k, _ in KINDS:
        r = {"chain_steps_per_s": float(np.median(rates[k])), "rounds": [float(v) for v in rates[k]],
             "mh_kernel": kernels[k]}
        if timed_forward:
            ms, kern = forward_ms(engines[k][0], engines[k][1])
            r["forward_ms_per_launch_32_sets"], r["forward_kernel"] = ms, kern
        res["kinds"][k] = r
    g = res["kinds"]["gaussian"]["chain_steps_per_s"]
    for k in ("poisson", "negbin"):
        res["kinds"][k]["slowdown_vs_gaussian"] = g / res["kinds"][k]["chain_steps_per_s"] - 1.0
    for eng, _ in engines.values():
        eng.close()
    return res


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r03_count_lik.json")
    assert torch.cuda.is_available(), "count_lik_bench needs the GPU"
    results = {"gpu": gpu_info(), "cases": []}
    a_shapes = [(64, 64), (32, 64), (2, 33)]
    results["cases"].append(run_case("family A 64-64-32-2 swish, 1M rows", 64, a_shapes, 1_000_000, "swish", 32, 200, True))
    c1_shapes = [(5, 25), (5, 6), (2, 5)]
    results["cases"].append(run_case("config-1 sized 24-5-5-2 tanh, 400 rows (k_chain_loop)", 24, c1_shapes, 400, "tanh",
                                     4, 4000, False))
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as fh:
        json.dump(results, fh, indent=1)
    print(json.dumps(results, indent=1))


if __name__ == "__main__":
    main()
