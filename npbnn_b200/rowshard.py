"""Row sharding of the MH step over ranks (SURVEY.md 8e-2): every rank holds a contiguous block of the training rows
and of the test rows and runs the SAME chains; per MH iteration one all-reduce of C * (slots + 2 + 2K) doubles (the
per-chain log-likelihood / residual sums and the accuracy counters) is the only exchange.  Chain sharding (mc3.py) is
the mode for many chains; this is the mode for one or a few chains on many rows (run_mcmc on several GPUs).  MC3 with
more ranks than chains combines both (mc3.chain_grid): the R ranks of a chain block row-shard it over their own
process group."""
import torch
import torch.distributed as dist


def row_partition(n_rows: int, world: int, rank: int):
    """Contiguous, balanced split: rank r owns rows [n r / world, n (r + 1) / world)."""
    return n_rows * rank // world, n_rows * (rank + 1) // world


def dist_all_reduce_sum(t: torch.Tensor, group=None) -> torch.Tensor:
    """In-place SUM over `group` (None: the default process group; NCCL over NVLink on a B200 box, gloo in the CPU
    tests).  The result is bit-identical on every rank, so the accept decisions are."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def exchange(shards, all_reduce_sum, accept_mode: int):
    """The exchange of one row-sharded iteration for `shards`, the engines of one chain block that this process drives
    (one in a run over ranks; all R of them when a test emulates the ranks in one process): local sums, all-reduce,
    commit, then the accept step (accept_mode 1) or the initial state (2).  all_reduce_sum(reds) sums the list of
    [C, n_values] device tensors, one per shard, in place over the block."""
    reds = [e.rowshard_local() for e in shards]
    all_reduce_sum(reds)
    for e, red in zip(shards, reds):
        e.rowshard_commit(red)
        e.rowshard_update(accept_mode, False)


def mh_steps(shards, n_steps: int, injection, all_reduce_sum):
    """n_steps row-sharded MH iterations of `shards` (see exchange), each from the same injected draws (or Philox)."""
    for s in range(n_steps):
        one = None if injection is None else {k: v[s:s + 1] for k, v in injection.items() if v is not None}
        for e in shards:
            e.rowshard_update(0, True, one)
        exchange(shards, all_reduce_sum, 1)


def shard_rows(x, y, world: int, rank: int):
    a, b = row_partition(len(x), world, rank)
    return x[a:b], y[a:b]
