"""Sharding of the posterior-prediction pass (BASELINE config 5: S posterior samples x N rows) over the ranks.

Prediction has no exchange on the data path when only ROWS are split (every rank owns the summaries of its rows,
SURVEY.md 8e).  But the kernel hands out whole 16-row warp tiles for all S samples: a GPU runs
ceil(tiles / (148 SMs x 12 warps)) rounds, and with 125,000 rows per GPU (8 GPUs at N = 1M) that is 4.4 rounds of work
executed as 5 -- 12 % idle (VERDICT r1).  A 2-D grid fixes the quantisation without touching the kernel: the ranks
form R row groups x Q sample groups (R Q = world); a rank predicts its row block for its share of the samples and
the Q partial sums of a row block ([rows, K] doubles, 20 MB at 250k rows) are added with ONE all-reduce over NCCL.
`grid_for` picks the (R, Q) with the fewest rounds per GPU; Q = 1 (rows only, no collective) wins whenever the row
split is already balanced.
"""
import math
from typing import Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

WARPS_PER_GPU = 148 * 12          # warp tiles a B200 works on at the same time (k_fwd3: one CTA per SM, 12 warps)


def rounds(n_rows: int) -> int:
    """Rounds of warp tiles the prediction kernel runs over n_rows rows."""
    return max(1, math.ceil(math.ceil(n_rows / 16) / WARPS_PER_GPU))


def grid_for(n_rows: int, n_sets: int, world: int) -> Tuple[int, int]:
    """(R, Q): row groups x sample groups with R * Q == world minimising the time of the slowest rank,
    rounds(rows per rank) * (samples per rank); ties go to the grid with fewer sample groups."""
    best = None
    for q in range(1, world + 1):
        if world % q or q > n_sets:
            continue
        r = world // q
        cost = rounds(math.ceil(n_rows / r)) * math.ceil(n_sets / q)
        if best is None or cost < best[0]:
            best = (cost, r, q)
    return best[1], best[2]


def partition(n_rows: int, n_sets: int, world: int, rank: int, grid: Optional[Tuple[int, int]] = None):
    """-> ((row_lo, row_hi), (set_lo, set_hi), (R, Q), row_group, sample_group).  Ranks of one row group are contiguous
    (rank = row_group * Q + sample_group), so a row group's all-reduce stays between neighbouring GPUs."""
    r, q = grid if grid is not None else grid_for(n_rows, n_sets, world)
    assert r * q == world
    rg, sg = rank // q, rank % q
    rows = (n_rows * rg // r, n_rows * (rg + 1) // r)
    sets = (n_sets * sg // q, n_sets * (sg + 1) // q)
    return rows, sets, (r, q), rg, sg


_GROUPS = {}


def block_group(world: int, size: int, index: int):
    """Process group of the `size` consecutive ranks of block `index` (ranks index * size ... + size - 1): the Q ranks
    that share a row group here, the R row shards of a chain block in MC3 (mc3.chain_grid).  Every rank creates all
    blocks' groups at its first call, in the same order, as torch.distributed requires."""
    key = (world, size)
    if key not in _GROUPS:
        _GROUPS[key] = [dist.new_group(list(range(g * size, (g + 1) * size))) for g in range(world // size)]
    return _GROUPS[key][index]


def combine(local_sum: torch.Tensor, n_sets_total: int, world: int, rank: int, grid: Tuple[int, int]) -> torch.Tensor:
    """local_sum [rows, K]: this rank's SUM over its samples (mean * its sample count, or vote counts).  Returns the
    mean over all n_sets_total samples of the row block, identical on the Q ranks of the row group."""
    r, q = grid
    if q > 1:
        dist.all_reduce(local_sum, op=dist.ReduceOp.SUM, group=block_group(world, q, rank // q))
    return local_sum / float(n_sets_total)


def predict_sharded(engine, x_rows, weight_sets, n_rows_total: int, rank: int, world: int, alphas=None, votes=False,
                    grid: Optional[Tuple[int, int]] = None):
    """Posterior mean (and vote shares) of this rank's row block from the posterior samples `weight_sets` (ALL S of
    them; the rank scores its sample share).  x_rows: the rank's rows (device tensor or array) as given by
    partition(...)[0].  Returns dict(mean [rows, K], votes?) as device tensors + the grid used."""
    import ctypes as C
    from . import _lib as L
    S = len(weight_sets)
    rows, sets, grid, rg, sg = partition(n_rows_total, S, world, rank, grid)
    w = engine._as_sets(weight_sets)[sets[0]:sets[1]]
    n_loc = sets[1] - sets[0]
    with torch.cuda.device(engine.device):
        xd = engine._dev(x_rows, torch.float64)
        n = xd.shape[0]
        assert n == rows[1] - rows[0]
        # Posterior samples in pinned host memory are uploaded in up to four chunks on a side stream, chunk i + 1 under
        # the kernel of chunk i (27 MB per rank at S = 1,024 on 8 GPUs would otherwise sit in front of a 68 ms kernel);
        # the chunk sums are exact multiples of the per-sample terms, so chunking only reorders the last additions.
        chunked = isinstance(w, torch.Tensor) and w.device.type == "cpu" and w.is_pinned() and n_loc >= 256
        n_chunks = min(4, n_loc // 128) if chunked else 1
        bounds = [n_loc * i // n_chunks for i in range(n_chunks + 1)]
        main = torch.cuda.current_stream(engine.device)
        side = torch.cuda.Stream(device=engine.device) if n_chunks > 1 else None
        al = None if alphas is None else np.asarray(alphas)[sets[0]:sets[1]]

        def upload(i):
            a, b = bounds[i], bounds[i + 1]
            if side is None:
                return engine._dev(w[a:b], torch.float64), None
            with torch.cuda.stream(side):
                t = w[a:b].to(device=engine.device, dtype=torch.float64, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(side)
            return t, ev

        msum = torch.zeros((n, engine.K), dtype=torch.float64, device=engine.device)
        vsum = torch.zeros((n, engine.K), dtype=torch.float64, device=engine.device) if votes else None
        md = torch.empty((n, engine.K), dtype=torch.float64, device=engine.device)
        vd = torch.empty((n, engine.K), dtype=torch.float64, device=engine.device) if votes else None
        nxt = upload(0)
        for i in range(n_chunks):
            wd, ev = nxt
            if i + 1 < n_chunks:
                nxt = upload(i + 1)
            if ev is not None:
                main.wait_event(ev)
                wd.record_stream(main)
            cnt = bounds[i + 1] - bounds[i]
            ad = engine._dev(None if al is None else al[bounds[i]:bounds[i + 1]], torch.float64)
            L.check(engine.lib.bnn_predict(engine._h, C.c_void_p(xd.data_ptr()), n, C.c_void_p(wd.data_ptr()), cnt,
                                           None if ad is None else C.c_void_p(ad.data_ptr()), None, None, 0,
                                           C.c_void_p(md.data_ptr()), None if vd is None else C.c_void_p(vd.data_ptr()), None,
                                           engine._stream()))
            msum.add_(md, alpha=float(cnt))
            if votes:
                vsum.add_(vd.mul_(float(cnt)).round_())
        out = {"mean": combine(msum, S, world, rank, grid), "grid": grid, "rows": rows, "sets": sets}
        if votes:
            out["votes"] = combine(vsum, S, world, rank, grid)
    return out
