#!/usr/bin/env python
"""Benchmark of the npBNN Metropolis-Hastings hot path on B200 (contract: task brief, section 4).

Workload (BASELINE.json configs[3], SURVEY.md 8d "c4"): MC3 with 32 tempered chains on a synthetic
1,000,000 x 64 float64 feature matrix, [64,32] swish hidden layers, 10 classes, bias on the last layer,
Normal(0,1) prior, update_f 0.05, update_ws 0.075.  A "step" is one MH iteration of every chain.
  value  = chains x steps / s with X resident in HBM, proposals generated on the device (Philox)
  e2e    = the same metric through the C ABI with HOST buffers: every step the host draws the proposals of all
           chains (numpy), bnn_mh_steps copies them in from pinned host memory and runs one MH iteration, and the
           chain state is copied back; X is staged once from pinned host memory before the timed region
           (setup_seconds in the e2e object), like the reference's data loading and MCMC.__init__
Chains are sharded over ranks (32 / N per GPU, strong scaling); the only exchange is the MC3 swap
(all-gather of 32 log-posteriors every swap_frequency steps).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the UNMODIFIED reference (oracle/_ref, oracle/make_ref.py) on the host cores
    python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs DIR

--dump-outputs DIR writes, after the run, what each timed leg computed in its last step as DIR/<name>.npy (float64):
mh_* and e2e_* are the chain state a caller reads back after the last of the K steps (every chain's logLik, logPrior,
logPost, temperature, acceptance_rate, n_accepted; the weights of the first DUMP_CHAINS chains), predict_mean /
predict_votes the posterior summaries of DUMP_ROWS rows drawn once with default_rng(0).  Inputs, seeds and the step
count depend only on the arguments, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ROWS = 1_000_000
N_CHAINS = 32
SWAP_FREQUENCY = 100
CPU_SAMPLE_ROWS = 100_000
DUMP_CHAINS = 256            # --dump-outputs keeps the weights of at most this many chains (13 MB per leg) and the
DUMP_ROWS = 65_536           # summaries of at most this many rows (10 MB), so that the dump stays under 64 MB
PRED_SAMPLES = 1024          # posterior samples of the forward rows/s leg (c5 shape; S >= 1,000 so that the sample upload and the
                              # one all-reduce of the rows x samples grid are amortised as they are at the full 10k)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=N_ROWS)
    ap.add_argument("--chains", type=int, default=N_CHAINS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-mc3-leg", action="store_true", help="reference arm: skip the np_bnn.MC3.run_mcmc() swap period")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed legs computed in their last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm runs in a subprocess and returns only its rate)")
    return args


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, line in self.rows:
            f = [v.strip() for v in line.split(",")]
            if len(f) < 8:
                continue
            try:
                clk, mxv = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = mxv
            if t0 <= t <= t1:
                sm.append(clk)
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def run_reference(rows, steps, warmup, chains=N_CHAINS, mc3_period=0, timeout=3000):
    """The UNMODIFIED reference (oracle/_ref/np_bnn, installed by oracle/make_ref.py) on the host cores, in a
    subprocess so that `import np_bnn` is the reference and not this repository's drop-in.  Returns the JSON object
    of oracle/ref_baseline.py, or None when oracle/_ref is absent."""
    if not os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "np_bnn", "__init__.py")):
        return None
    env = dict(os.environ)
    for k in ("PYTHONPATH", "RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_baseline.py"), "--rows", str(rows), "--steps", str(steps),
           "--warmup", str(warmup), "--chains", str(chains), "--mc3-period", str(mc3_period)]
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        r = subprocess.run(cmd, cwd=tmp, env=env, capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        sys.stderr.write(r.stderr[-2000:])
        raise RuntimeError("oracle/ref_baseline.py failed (rc %d)" % r.returncode)
    return json.loads(r.stdout.strip().splitlines()[-1])


def port_baseline(rows, steps, seconds):
    """Fallback when oracle/_ref is absent: the numpy oracle port on a row sample (kind "port")."""
    from npbnn_b200 import workloads as wl
    from oracle import cpu_baseline
    x, labels = wl.c4_data(min(rows, CPU_SAMPLE_ROWS), seed=0)
    res = cpu_baseline.mh_rate(x, labels.astype(np.int64), wl.C4_SHAPES, "swish", rows, steps_per_proc=steps, seconds=seconds)
    return {"value": res["value"], "unit": "chain-steps/s", "cores": res["cores"], "kind": "port", "sample": res["sample"]}


def reference_arm(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores.
    A "step" is one np_bnn.MCMC.mh_step of every chain (min(32, cores) forked chains, all 1,000,000 rows)."""
    if rank != 0:
        return
    K, W = max(1, args.steps), max(0, args.warmup)
    t0 = time.perf_counter()
    ref = run_reference(args.rows, K, W, chains=args.chains, mc3_period=min(K, 5) if not args.no_mc3_leg else 0)
    wall = time.perf_counter() - t0
    if ref is None:
        cpu = port_baseline(args.rows, K, 30.0 + 5.0 * K)
        value, ms_per_step, extra = cpu["value"], 1e3 * cpu["cores"] / cpu["value"], {}
    else:
        value = ref["value"]
        ms_per_step = 1e3 * ref["chains_leg"]["wall_s"] / K
        cpu = {"value": value, "unit": "chain-steps/s", "cores": ref["chains"], "kind": "reference", "sample": ref["sample"]}
        extra = {"reference": {k: ref.get(k) for k in ("reference_version", "cores", "chains", "numpy",
                                                       "blas_threads_per_process", "chains_leg", "mc3_leg")}}
    cfg = workload_config(args)
    line = {"impl": "reference", "metric": "MH iterations/sec (chains x steps / s)", "value": value,
            "unit": "chain-steps/s", "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg, "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": "chain-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": wall}
    line.update(extra)
    _emit(line)


def workload_config(args):
    return {"workload": "c4: MC3 %d tempered chains, synthetic %dx64 f64, [64,32] swish, 10 classes, bias on last layer"
                        % (args.chains, args.rows),
            "rows": args.rows, "features": 64, "chains": args.chains, "swap_frequency": SWAP_FREQUENCY,
            "update_f": 0.05, "update_ws": 0.075, "prior": "Normal(0,1)", "parallelism": "chains sharded over GPUs",
            "l2": "inputs larger than L2 (X = %.0f MB streamed once per step)" % (args.rows * 64 * 8 / 1e6)}


def chain_outputs(prefix, st, first_chain):
    """What bnn_chains_read hands back for the local chains first_chain, ... as float64 arrays '<prefix>_<field>';
    weights only of the chains below DUMP_CHAINS."""
    out = {k: getattr(st, k) for k in ("logLik", "logPrior", "logPost", "temperature", "acceptance_rate", "n_accepted")}
    out["weights"] = st.w[:max(0, DUMP_CHAINS - first_chain)]
    return {"%s_%s" % (prefix, k): np.asarray(v, dtype=np.float64) for k, v in out.items()}


def write_outputs(path, parts):
    """parts: every rank's dict of arrays, in rank order (chains and row blocks are contiguous in rank order)."""
    arrays = {name: np.concatenate([p[name] for p in parts if name in p]) for name in parts[0]}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "--dump-outputs would exceed 64 MB"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout: libraries (NCCL prints its version banner there) get stderr for the
    whole run, the JSON line is written to the saved descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    args = parse()
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from npbnn_b200 import _lib as L
    from npbnn_b200 import mc3, workloads as wl
    from npbnn_b200.engine import Engine, NetShape, flatten_weights

    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"       # keep NCCL's version banner off stdout: one JSON line only
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ------------------------------------------------------------------ workload (host, pinned)
    x_np, y_np = wl.c4_data(args.rows, seed=0)
    x_pin = torch.from_numpy(x_np).pin_memory()
    y_pin = torch.from_numpy(y_np).pin_memory()
    start, n_local = mc3.chain_partition(args.chains, world, rank)
    temps_all = mc3.default_temperatures(args.chains, 0.8)
    w0 = np.stack([flatten_weights(w) for w in wl.c4_init_weights(n_local, start)])
    net = NetShape(64, list(wl.C4_SHAPES), act="swish", lik=L.LIK_CATEGORICAL)
    K, W = args.steps, max(args.warmup, 3)
    dump = {} if args.dump_outputs else None          # name -> this rank's share of the array (--dump-outputs)

    # ------------------------------------------------------------------ device-resident leg (value)
    eng = Engine(net, device=local_rank)
    eng.set_data(x_pin.to(dev), y_pin.to(dev))
    eng.chains_init(w0, temperature=temps_all[start:start + n_local], seed=1234 + rank)
    rng = mc3.SwapRNG(4321)
    step_ctr = [0]

    n_swaps = [0]

    def swap(temps):
        temps, _, _, _ = mc3.exchange(eng.gather(L.F_LOGPOST), temps, rng, None, world)
        eng.set_temperature(temps[start:start + n_local])
        n_swaps[0] += 1
        return temps

    def run_steps(n, temps, force_swap=False):
        """n MH iterations of every chain with the MC3 swap (all-gather of the log-posteriors + temperature
        update) every SWAP_FREQUENCY steps; force_swap adds one at the end if none fell inside the n steps."""
        done, swaps0 = 0, n_swaps[0]
        while done < n:
            chunk = min(n - done, SWAP_FREQUENCY - step_ctr[0] % SWAP_FREQUENCY)
            eng.mh_steps(chunk)
            done += chunk
            step_ctr[0] += chunk
            if step_ctr[0] % SWAP_FREQUENCY == 0 and args.chains > 1:
                temps = swap(temps)
        if force_swap and n_swaps[0] == swaps0 and args.chains > 1:
            temps = swap(temps)
        return temps

    peak_tf = eng.measure_fp64_peak()
    temps_all = run_steps(W, temps_all)
    barrier()
    eng.set_option("time_forward", 1)
    eng.forward_time(reset=True)
    clocks = ClockSampler(local_rank)
    clocks.start()
    time.sleep(0.25)
    # The timed region is EXACTLY K steps (barrier + synchronize on both sides, CUDA events, max over ranks), with at
    # least one MC3 swap in it even when K < SWAP_FREQUENCY.
    swaps_before = n_swaps[0]
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.perf_counter()
    ev0.record()
    temps_all = run_steps(K, temps_all, force_swap=True)
    ev1.record()
    barrier()
    t_wall1 = time.perf_counter()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = eng.launch_count - launches0
    clk = clocks.stop(t_wall0, t_wall1)
    fwd_ms, fwd_n = eng.forward_time(reset=True)
    eng.set_option("time_forward", 0)
    value = args.chains * K / (ms * 1e-3)
    st = eng.read_state(weights=dump is not None)
    if dump is not None:
        dump.update(chain_outputs("mh", st, start))
    kernel_name = eng.last_kernel

    # roofline of the dominant kernel (forward + likelihood): algorithmic FLOPs per launch / its mean duration
    flop_per_launch = float(n_local) * args.rows * wl.C4_FLOP_PER_ROW
    fwd_avg_ms = fwd_ms / max(fwd_n, 1)
    achieved_tf = flop_per_launch / (fwd_avg_ms * 1e-3) / 1e12 if fwd_n else None
    ncu = {}
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            ncu = json.load(f)
    except Exception:
        pass
    roofline = {"bound": "tensor", "pipe": "fp64 (DMMA and DFMA share one pipe on B200)", "kernel": kernel_name,
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": (achieved_tf / peak_tf) if achieved_tf else None,
                "peak_source": "measured live on this GPU: back-to-back FP64 DMMA (bnn_measure_fp64_peak); "
                               "MEASURED_PEAKS.json has no FP64 entry",
                "flop_per_launch": flop_per_launch, "launch_ms": fwd_avg_ms, "launches_timed": int(fwd_n),
                "kernel_share_of_step": fwd_ms / ms if fwd_n else None,
                "traffic": ncu.get("dram_bytes_per_launch"),
                "hbm": {"algorithmic_bytes_per_launch": args.rows * (64 * 8 + 4),
                        "achieved_gbs": args.rows * (64 * 8 + 4) / (fwd_avg_ms * 1e-3) / 1e9 if fwd_n else None}}

    # ------------------------------------------------------------------ forward rows/s (BASELINE metric, second half):
    # posterior prediction (c5 shape) for PRED_SAMPLES posterior samples, summaries mean + votes.  The ranks form a
    # (row groups x sample groups) grid chosen to minimise the rounds of warp tiles per GPU (npbnn_b200/predshard.py):
    # rows only (no collective) while that is balanced, otherwise the partial sums of a row block are added with one
    # all-reduce per summary inside the timed region.
    from npbnn_b200 import predshard
    predict = None
    try:
        rows_p, sets_p, grid_p, _, sg_p = predshard.partition(args.rows, PRED_SAMPLES, world, rank)
        xd = x_pin[rows_p[0]:rows_p[1]].to(dev)
        rs_p = np.random.default_rng(5)
        w_all = w0[:1].repeat(PRED_SAMPLES, 0) + rs_p.normal(0, 0.05, (PRED_SAMPLES, w0.shape[1])) if n_local else None
        if w_all is None:
            w_all = np.zeros((PRED_SAMPLES, net.n_params))
        if world > 1:       # every rank must hold the same posterior samples: rank 0's
            wt_ = torch.from_numpy(w_all).to(dev)
            dist.broadcast(wt_, 0)
            w_all = wt_.cpu().numpy()
        w_pin = torch.from_numpy(np.ascontiguousarray(w_all)).pin_memory()      # posterior samples in pinned host memory, like X

        def run_predict():
            return predshard.predict_sharded(eng, xd, w_pin, args.rows, rank, world, votes=True, grid=grid_p)
        out_p = run_predict()
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        out_p = run_predict()
        p1.record()
        barrier()
        pms = max_over_ranks(p0.elapsed_time(p1))
        tf = PRED_SAMPLES * args.rows * wl.C4_FLOP_PER_ROW / (pms * 1e-3) / 1e12
        predict = {"metric": "forward rows/s (posterior samples x rows / s)", "value": PRED_SAMPLES * args.rows / (pms * 1e-3),
                   "unit": "row-samples/s", "samples": PRED_SAMPLES, "rows": args.rows, "ms": pms, "tflops": tf,
                   "frac_of_fp64_peak_per_gpu": tf / world / peak_tf, "kernel": eng.last_kernel,
                   "grid": {"row_groups": grid_p[0], "sample_groups": grid_p[1],
                            "rounds_per_gpu": predshard.rounds(rows_p[1] - rows_p[0]),
                            "collective": "none" if grid_p[1] == 1 else "all-reduce of [rows, 10] partial sums within a row group"},
                   "includes": "upload (pinned host memory) + packing of the rank's posterior samples, the all-reduce of the grid, X row block resident",
                   "mean_prob_sum": float(out_p["mean"].sum().item()) / max(rows_p[1] - rows_p[0], 1)}
        if dump is not None:
            # the sampled rows of this rank's row block; the Q ranks of a row group hold the same summaries, the one of
            # sample group 0 contributes them
            idx = np.sort(np.random.default_rng(0).choice(args.rows, min(args.rows, DUMP_ROWS), replace=False))
            idx = idx[(idx >= rows_p[0]) & (idx < rows_p[1])] - rows_p[0] if sg_p == 0 else idx[:0]
            sel = torch.from_numpy(idx).to(dev)
            dump["predict_mean"] = out_p["mean"][sel].cpu().numpy()
            dump["predict_votes"] = out_p["votes"][sel].cpu().numpy()
        del xd, out_p
    except Exception as e:                                 # the headline must not depend on this leg
        predict = {"error": repr(e)}

    # ------------------------------------------------------------------ end-to-end leg (host buffers)
    e2e = None
    if not args.no_e2e:
        eng.close()
        del eng
        torch.cuda.empty_cache()
        host_rng = np.random.default_rng(99 + rank)
        sizes = [r * c for r, c in wl.C4_SHAPES]
        upd_n = [max(1, int(round(s * 0.05))) for s in sizes]
        cap = sum(upd_n)
        # set-up (not timed, reported as setup_seconds): context, X + labels staged from pinned host memory, chain
        # init.  The reference's counterpart is reading the data files and MCMC.__init__, which its own rate
        # (the reference arm / cpu_baseline) does not include either.
        barrier()
        ts = time.perf_counter()
        eng2 = Engine(net, device=local_rank)
        eng2.set_data(x_pin, y_pin)
        eng2.chains_init(w0, temperature=temps_all[start:start + n_local], seed=1)
        torch.cuda.synchronize(dev)
        t_setup = max_over_ranks(time.perf_counter() - ts)

        def pinned(shape, dtype):
            return torch.empty(shape, dtype=dtype, pin_memory=True).numpy()

        # this step's inputs live in pinned host memory (two buffers: while the device runs step s, a host thread draws
        # the proposals of step s+1 -- ctypes releases the GIL while bnn_mh_steps waits for the device); the library
        # copies them to the device inside bnn_mh_steps
        def make_inj():
            b = {"proposed": pinned((1, n_local, 3), torch.int32), "count": pinned((1, n_local, 3), torch.int32),
                 "ix": pinned((1, n_local, cap), torch.int32), "iy": pinned((1, n_local, cap), torch.int32),
                 "dz": pinned((1, n_local, cap), torch.float64), "log_u": pinned((1, n_local), torch.float64)}
            b["proposed"][:] = 1
            b["count"][:] = np.array(upd_n, np.int32)
            return b

        bufs = [make_inj(), make_inj()]

        def draw(b):
            # host side of one MH iteration: every chain's proposal (numpy, as the reference does)
            b["dz"][:] = host_rng.normal(0, 0.075, (1, n_local, cap))
            b["log_u"][:] = np.log(host_rng.random((1, n_local)))
            o = 0
            for l, (r, c) in enumerate(wl.C4_SHAPES):
                b["ix"][0, :, o:o + upd_n[l]] = host_rng.integers(0, r, (n_local, upd_n[l]))
                b["iy"][0, :, o:o + upd_n[l]] = host_rng.integers(0, c, (n_local, upd_n[l]))
                o += upd_n[l]
            return b

        from concurrent.futures import ThreadPoolExecutor
        pool = ThreadPoolExecutor(1)
        nxt = [pool.submit(draw, bufs[0]), 0]

        def e2e_step():
            # hand the drawn host buffers to the library (H2D inside), start drawing the next step's, read this
            # step's result back (D2H, synchronises)
            b = nxt[0].result()
            nxt[1] ^= 1
            nxt[0] = pool.submit(draw, bufs[nxt[1]])
            eng2.mh_steps(1, b)
            return eng2.read_state(weights=False)

        inj = bufs[0]
        for _ in range(max(3, W)):
            st2 = e2e_step()
        h2d = K * sum(a.nbytes for a in inj.values())
        d2h = K * (st2.f64.nbytes + st2.i32.nbytes)
        # as for `value`: the timed region is EXACTLY K steps (barrier + synchronize on both sides, max over ranks)
        torch.cuda.synchronize(dev)
        barrier()
        t0 = time.perf_counter()
        for s in range(K):
            st2 = e2e_step()
        torch.cuda.synchronize(dev)
        barrier()
        t_e2e = max_over_ranks(time.perf_counter() - t0)
        if dump is not None:
            dump.update(chain_outputs("e2e", eng2.read_state(), start))
        e2e = {"value": args.chains * K / t_e2e, "unit": "chain-steps/s", "h2d_bytes_per_step": h2d / K,
               "d2h_bytes_per_step": d2h / K,
               "includes": "every step, per rank: proposals of all local chains drawn on the host (numpy; a host thread "
                           "draws step s+1 while the device runs step s), copied from pinned host memory inside "
                           "bnn_mh_steps(1, inj), one MH iteration, chain state read back (bnn_chains_read, "
                           "synchronises); X is resident (staged once by bnn_set_data from pinned "
                           "host memory: setup_seconds, not timed)",
               "seconds": t_e2e, "setup_seconds": t_setup, "setup_h2d_bytes": x_pin.numel() * 8 + y_pin.numel() * 4 + w0.nbytes,
               "finite_logLik": bool(np.all(np.isfinite(st2.logLik)))}
        nxt[0].result()
        pool.shutdown()
        eng2.close()

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # bounded sample: 3 MH iterations per chain (after 1 warm-up) of the unmodified reference on all rows
        ref = run_reference(args.rows, 3, 1, chains=args.chains)
        if ref is None:
            cpu = port_baseline(args.rows, 3, 20.0)
        else:
            cpu = {"value": ref["value"], "unit": "chain-steps/s", "cores": ref["chains"], "kind": "reference",
                   "sample": ref["sample"], "wall_s": ref["chains_leg"]["wall_s"]}

    if dump is not None:
        parts = [dump]
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, dump)
        if rank == 0:
            write_outputs(args.dump_outputs, parts)

    if rank == 0:
        line = {"metric": "MH iterations/sec (chains x steps / s)", "value": value, "unit": "chain-steps/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(args), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": int(launches), "clocks": clk,
                "timing": {"timed_steps": K, "timed_seconds": ms * 1e-3}, "predict": predict,
                "swaps_in_timed_region": n_swaps[0] - swaps_before,
                "check": {"logLik_finite": bool(np.all(np.isfinite(st.logLik))),
                          "mean_acceptance": float(np.mean(st.n_accepted / np.maximum(st.iteration, 1)))}}
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
