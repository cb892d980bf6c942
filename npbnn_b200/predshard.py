"""Sharding of the posterior-prediction pass (BASELINE config 5: S posterior samples x N rows) over the ranks.

Prediction has no exchange on the data path when only ROWS are split (every rank owns the summaries of its rows,
SURVEY.md 8e).  But the kernel hands out whole 16-row warp tiles for all S samples: a GPU runs
ceil(tiles / (148 SMs x 12 warps)) rounds, and with 125,000 rows per GPU (8 GPUs at N = 1M) that is 4.4 rounds of work
executed as 5 -- 12 % idle (VERDICT r1).  A 2-D grid fixes the quantisation without touching the kernel: the ranks
form R row groups x Q sample groups (R Q = world); a rank predicts its row block for its share of the samples and
the Q partial sums of a row block ([rows, K] doubles, 20 MB at 250k rows) are added with ONE all-reduce over NCCL.
`grid_for` picks the (R, Q) with the fewest rounds per GPU; Q = 1 (rows only, no collective) wins whenever the row
split is already balanced.

`predict_ranks` is the same grid behind the reference's prediction callers (api.get_posterior_cat_prob and everything
built on it), in one process and on many ranks alike: every rank passes the caller's full arguments, scores its block
and gets back the full arrays one process computes.  It is collective: every rank of the process group calls it with
the same arguments.  One rank (no process group, or a group of one) scores the whole problem and makes no collective
call.
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
    engine._set_pattern(None)                 # the dense kernels, whatever pattern the engine's last call used
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


# ---------------------------------------------------------------------------------------------------------------------
# zero pattern of the posterior samples (block-masked networks run the block-sparse prediction kernels)
# ---------------------------------------------------------------------------------------------------------------------
def zero_pattern(weight_sets, net) -> Optional[np.ndarray]:
    """The union over the posterior samples of `w != 0`, as a canonical 0/1 vector [n_params] for
    Engine.predict(pattern=...), or None when the prediction should stay on the dense kernels.  Entries that are zero in
    every sample contribute nothing, so skipping them only changes the order of the sums.
    weight_sets: a list of per-layer weight lists, or an array / tensor [S, n_params].  The block cover of the pattern
    has at least as many multiply-adds as sample 0 has nonzero hidden-layer weights, and the program builder declines a
    cover above a quarter of the dense work: when sample 0 alone is past that, this returns None after looking at that
    one sample (dense networks pay O(n_params), not O(S n_params))."""
    shapes, hb = net.shapes, net.has_bias()
    if len(shapes) < 2 or len(weight_sets) == 0:
        return None
    dense = sum(r * (c - b) for (r, c), b in zip(shapes, hb))
    last = shapes[-1][0] * (shapes[-1][1] - hb[-1])
    flat = isinstance(weight_sets, (np.ndarray, torch.Tensor))
    host = (lambda t: t.detach().cpu().numpy()) if isinstance(weight_sets, torch.Tensor) else np.asarray
    if flat:
        w0 = host(weight_sets[0])                    # (a tensor is copied to the host only past the shortcut)
        offs = np.cumsum([0] + [r * c for r, c in shapes])
        layers0 = [w0[offs[l]:offs[l + 1]].reshape(shapes[l]) for l in range(len(shapes))]
    else:
        layers0 = [np.asarray(w) for w in weight_sets[0]]
    nnz = sum(int(np.count_nonzero(w[:, b:])) for w, b in zip(layers0[:-1], hb[:-1]))
    if 4 * (nnz + last) > dense:
        return None
    if flat:
        return np.any(host(weight_sets) != 0, axis=0).astype(np.float64)
    pat = [w != 0 for w in layers0]
    for s in weight_sets[1:]:
        for l, w in enumerate(s):
            pat[l] |= np.asarray(w) != 0
    return np.concatenate([p.ravel() for p in pat]).astype(np.float64)


def engine_pattern(engine, weight_sets) -> Optional[np.ndarray]:
    """zero_pattern for `engine`'s network; None for an engine whose network declares no layer shapes (it scores
    densely and is never handed a pattern)."""
    return zero_pattern(weight_sets, engine.net) if hasattr(engine.net, "shapes") else None


# ---------------------------------------------------------------------------------------------------------------------
# collective prediction behind the reference's prediction callers
# ---------------------------------------------------------------------------------------------------------------------
def ranks() -> Tuple[int, int]:
    """(world, rank) of the initialised default process group; (1, 0) without one."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def comm_device() -> torch.device:
    """Where the tensors of the collectives live: the current GPU under NCCL (one GPU per rank), host memory under
    gloo (ranks that share GPUs)."""
    if dist.get_backend() == "nccl":
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def agree(call) -> None:
    """Collective check that every rank passed the same arguments `call` (a small tuple of plain values).  Runs before
    any other collective of the call: ranks that disagree on a shape would otherwise hang in a later collective or
    exchange blocks of different problems.  A mismatch raises ValueError on every rank."""
    calls = [None] * dist.get_world_size()
    dist.all_gather_object(calls, call)
    bad = [r for r, c in enumerate(calls) if c != calls[0]]
    if bad:
        raise ValueError("collective prediction called with different arguments: rank 0 passed %r, rank %d passed %r"
                         % (calls[0], bad[0], calls[bad[0]]))


def from_rank0(value, shape, dtype: torch.dtype) -> torch.Tensor:
    """Rank 0's array `value` (ignored on the other ranks) on every rank, as a tensor of `shape` on comm_device()."""
    dev = comm_device()
    if dist.get_rank() == 0:
        t = torch.as_tensor(np.ascontiguousarray(value)).to(device=dev, dtype=dtype).reshape(shape).contiguous()
    else:
        t = torch.empty(shape, dtype=dtype, device=dev)
    dist.broadcast(t, src=0)
    return t


def _columns(selector, n_features: int):
    """Distinct column indices of a feature selector x[:, selector] (an index or a list of indices)."""
    return list(dict.fromkeys(int(c) % n_features for c in np.atleast_1d(np.asarray(selector)).ravel()))


def permuted_rows(x: np.ndarray, lo: int, hi: int, shuffle, perms) -> np.ndarray:
    """Rows lo..hi of x after `x[:, cols] = x[perm][:, cols]` for each (cols, perm) of zip(shuffle, perms), in order:
    the rows of the reference's `x[:, fi] = np.random.permutation(x[:, fi])` (np.random.permutation(N) draws the
    permutation np.random.permutation(x[:, fi]) applies), built from the full host copy without permuting it."""
    rows = np.array(x[lo:hi], copy=True)
    src = {}                      # column -> source row of each row after the permutations so far
    for cols, perm in zip(shuffle, perms):
        for col in _columns(cols, x.shape[1]):
            src[col] = perm if col not in src else src[col][perm]
    for col, s in src.items():
        rows[:, col] = x[s[lo:hi], col]
    return rows


# the outputs in the order a rank packs its blocks for the all-gather
_OUTPUTS = ("mean", "votes", "predictions", "class_counts", "post_predictions", "dense")


def predict_ranks(engine, x, weight_sets, alphas=None, override=None, mean=False, votes=False, dense=False,
                  sample=None, post_predictions=False, shuffle=(), draw=None, grid: Optional[Tuple[int, int]] = None,
                  pattern="auto"):
    """Posterior prediction of all N rows of x over all S posterior samples, split over the ranks of the default process
    group.  Collective: every rank passes the same arguments (checked first, ValueError on every rank otherwise) and
    returns the same dict of host arrays as the engine calls over the whole problem:
      mean [N, W], votes [N, W], dense [S, N, W]                     (Engine.predict; W = K, or the outputs)
      predictions [N, K], class_counts [S, K], post_predictions [N, S] (Engine.predict_sample, with sample set;
                                                                       post_predictions None unless asked for)
    x: the caller's full host features [N, F]; weight_sets: all S posterior samples; alphas: [S, L] or None; override:
    (cols, vals) column overwrite.  sample: None, "host" (reference uniforms) or "philox" (in-kernel uniforms, keyed on
    the global (row, sample) so the split does not change them).  shuffle: feature selectors whose rows are permuted.
    draw(): run on rank 0 only, returns (permutations of range(N), one per shuffle entry; uniforms [N, S] or None; seed
    or None) drawn from rank 0's numpy stream, which every rank then receives.  The engine scores with the zero pattern
    of all S samples: `pattern`, or zero_pattern(weight_sets) with pattern="auto" (callers that score the same samples
    many times compute it once and pass it).  Every rank computes the same pattern from the same full sample list, so a
    block-masked network runs the same block-sparse program on every rank.

    The rank scores rows x samples block `partition(N, S, world, rank, grid)`; a rank with an empty block makes no kernel
    call but joins every collective.  Combination (one all-gather of every rank's block): means are sums over each sample
    group, added in sample-group order and divided by S once (with one sample group: the block's own mean); votes and
    resampled shares are integer counts, added and divided by S once; class_counts are added over the row groups.
    With one rank the block is the whole problem and the engine's host outputs are returned as they are: no
    torch.distributed call, no rescaling."""
    from . import _lib as L
    world, rank = ranks()
    x = np.ascontiguousarray(x, dtype=np.float64)
    n, f = x.shape
    S = len(weight_sets)
    W = engine.K if engine.net.lik == L.LIK_CATEGORICAL else engine.O
    K = engine.K
    shuffle = list(shuffle)
    if world > 1:
        ov = None if override is None else (tuple(int(c) for c in override[0]), tuple(float(v) for v in override[1]))
        agree((n, f, S, W, engine.net.n_params, engine.net.act, engine.net.lik, bool(mean), bool(votes), bool(dense),
               sample, bool(post_predictions), [tuple(_columns(s, f)) for s in shuffle], ov, grid))
    if sample not in (None, "host", "philox"):
        raise ValueError("sample must be None, 'host' or 'philox'")
    rows, sets, grid, _, _ = partition(n, S, world, rank, grid)
    R, Q = grid
    (a, b), (c, d) = rows, sets
    n_loc, s_loc = b - a, d - c

    # draws from numpy's global stream: rank 0's, the ones one process makes
    perms, u, seed = draw() if rank == 0 and draw is not None else ([None] * len(shuffle), None, None)
    if world > 1:
        if shuffle:
            perms = list(from_rank0(np.stack(perms) if rank == 0 else None, (len(shuffle), n), torch.int64).cpu().numpy())
        if sample == "host":
            u = from_rank0(u, (n, S), torch.float64)
        elif sample == "philox":
            seed = int(from_rank0(np.array([seed if rank == 0 else 0], dtype=np.int64), (1,), torch.int64).item())

    out = {}
    if (n_loc and s_loc) or world == 1:       # one rank calls the engine even on an empty problem, which it refuses
        xb = permuted_rows(x, a, b, shuffle, perms) if shuffle else x[a:b]
        w = weight_sets[c:d]
        al = None if alphas is None else np.asarray(alphas)[c:d]
        # (passed only when there is one)
        pat = engine_pattern(engine, weight_sets) if isinstance(pattern, str) else pattern
        kw = {} if pat is None else {"pattern": pat}
        if mean or votes or dense:
            out.update(engine.predict(xb, w, alphas=al, override=override, mean=mean, votes=votes, dense=dense,
                                      device_out=world > 1, **kw))
        if sample:
            out.update(engine.predict_sample(xb, w, None if u is None else u[a:b, c:d], alphas=al,
                                             post_predictions=post_predictions, seed=seed, row0=a, set0=c,
                                             device_out=world > 1, **kw))
    if world == 1:
        return out

    # the block as the combination adds it: sums over the rank's samples, integer counts
    if out:
        if mean and Q > 1:
            out["mean"] = out["mean"] * float(s_loc)
        if votes:
            out["votes"] = torch.round(out["votes"] * float(s_loc))
        if sample:
            out["predictions"] = torch.round(out["predictions"] * float(s_loc))

    names = [k for k, on in zip(_OUTPUTS, (mean, votes, sample, sample, sample and post_predictions, dense)) if on]

    def sizes(nl, sl):
        return {"mean": (nl, W), "votes": (nl, W), "predictions": (nl, K), "class_counts": (sl, K),
                "post_predictions": (nl, sl), "dense": (sl, nl, W)}

    # one all-gather of every rank's blocks, packed into one vector padded to the longest
    dev = comm_device()
    blocks = [partition(n, S, world, q, grid)[:2] for q in range(world)]
    lens = [sum(int(np.prod(sizes(rb - ra, sb - sa)[k])) for k in names) for (ra, rb), (sa, sb) in blocks]
    send = torch.zeros(max(lens), dtype=torch.float64, device=dev)
    if out:
        send[:lens[rank]] = torch.cat([out[k].to(device=dev, dtype=torch.float64).reshape(-1) for k in names])
    recv = [torch.empty_like(send) for _ in range(world)]
    dist.all_gather(recv, send)

    def view(q):
        (ra, rb), (sa, sb) = blocks[q]
        out, o = {}, 0
        for k in names:
            shp = sizes(rb - ra, sb - sa)[k]
            m = int(np.prod(shp))
            out[k] = recv[q][o:o + m].reshape(shp)
            o += m
        return out

    views = [view(q) for q in range(world)]
    res = {}
    for k in names:
        if k in ("mean", "votes", "predictions"):
            full = torch.empty((n, W if k != "predictions" else K), dtype=torch.float64, device=dev)
            for g in range(R):
                (ra, rb), _ = blocks[g * Q]
                if rb == ra:
                    continue
                if k == "mean" and Q == 1:
                    full[ra:rb] = views[g][k]
                    continue
                acc = views[g * Q][k].clone()
                for q in range(1, Q):
                    acc += views[g * Q + q][k]
                full[ra:rb] = acc / float(S)
        elif k == "class_counts":
            full = torch.zeros((S, K), dtype=torch.float64, device=dev)
            for q in range(world):
                (ra, rb), (sa, sb) = blocks[q]
                if rb > ra:
                    full[sa:sb] += views[q][k]
        elif k == "post_predictions":
            full = torch.empty((n, S), dtype=torch.float64, device=dev)
            for q in range(world):
                (ra, rb), (sa, sb) = blocks[q]
                full[ra:rb, sa:sb] = views[q][k]
        else:
            full = torch.empty((S, n, W), dtype=torch.float64, device=dev)
            for q in range(world):
                (ra, rb), (sa, sb) = blocks[q]
                full[sa:sb, ra:rb] = views[q][k]
        res[k] = full.cpu().numpy()
    if sample and not post_predictions:
        res["post_predictions"] = None
    return res
