"""MC3 (Metropolis-coupled MCMC) host logic: chain partitioning over ranks and the swap step.

Replaces the fork pool of the reference (BNN_mc3.py:87-126), which pickles every chain (with its copy
of the data) to a worker and back each swap period.  Here the chains never leave their GPU; the only
exchange is an all-gather of the per-chain log-posteriors (8 bytes per chain) over NCCL/NVLink, after
which every rank evaluates the same swap with the same seeded generator and updates the temperatures
of its own chains.  No tensor of the data path is communicated.  With more ranks than chains the ranks form a grid of
chain blocks x row shards (chain_grid): the ranks of a block run the same chains on their own rows (rowshard.py).
"""
from typing import Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist


def default_temperatures(n_chains: int, min_temperature: float = 0.8) -> np.ndarray:
    """np.linspace(min_temperature, 1, n_chains), [1] for a single chain (BNN_mc3.py:46-51)."""
    if n_chains == 1:
        return np.ones(1)
    return np.linspace(min_temperature, 1, n_chains)


def chain_partition(n_chains: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous block of chains owned by `rank` (sizes differ by at most one)."""
    base, rem = divmod(n_chains, world_size)
    start = rank * base + min(rank, rem)
    return start, base + (1 if rank < rem else 0)


def chain_grid(n_chains: int, world_size: int) -> Tuple[int, int]:
    """(Q, R): Q chain blocks x R row shards with Q * R == world_size.  Up to one rank per chain the ranks hold whole
    chains (R = 1, the partition of chain_partition over all ranks).  With more ranks than chains, Q is the largest
    divisor of world_size that does not exceed n_chains, and the R ranks of a block split its rows (rowshard.py), so
    every GPU has work: 4 chains on 8 GPUs run as 4 x 2, one chain on 8 GPUs as 1 x 8.  Rank = q * R + r: the R ranks
    of a block, which all-reduce every MH iteration, are neighbours."""
    if n_chains < 1 or world_size < 1:
        raise ValueError("chain_grid: %d chains on %d ranks" % (n_chains, world_size))
    if world_size <= n_chains:
        return world_size, 1
    q = max(d for d in range(1, n_chains + 1) if world_size % d == 0)
    return q, world_size // q


class SwapRNG:
    """The generator behind the swap step.  Every rank builds it from the same seed, so the pair and the
    uniform agree everywhere without communication (the reference uses the global np.random state,
    BNN_mc3.py:99,109)."""

    def __init__(self, seed: int = 4321):
        self._rs = np.random.RandomState(seed)

    def pair(self, n_chains: int):
        j, k = self._rs.choice(range(n_chains), 2, replace=False)
        return int(j), int(k)

    def log_uniform(self) -> float:
        return float(np.log(self._rs.random_sample()))


class GlobalSwapRNG:
    """Single-process default: the swap step consumes numpy's GLOBAL generator exactly as the reference does
    (np.random.choice(range(n), 2, replace=False) then np.log(np.random.random()), BNN_mc3.py:99,109), so a script that
    calls np.random.seed(...) first swaps the same pairs as the reference run."""

    def pair(self, n_chains: int):
        j, k = np.random.choice(range(n_chains), 2, replace=False)
        return int(j), int(k)

    def log_uniform(self) -> float:
        return float(np.log(np.random.random()))


def broadcast_from_rank0(obj, group: Optional[dist.ProcessGroup] = None):
    """Small host object of rank 0 on every rank (seeds); identity without a process group."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return obj
    box = [obj]
    dist.broadcast_object_list(box, src=0, group=group)
    return box[0]


def owner_of(chain: int, n_chains: int, world_size: int, R: int = 1) -> int:
    """Rank that holds global chain index `chain` under chain_partition over the world_size / R chain blocks: the r = 0
    rank of its block."""
    Q = world_size // R
    for q in range(Q):
        start, n = chain_partition(n_chains, Q, q)
        if start <= chain < start + n:
            return q * R
    raise ValueError("chain %d of %d" % (chain, n_chains))


def swap_temperatures(log_post: np.ndarray, temps: np.ndarray, j: int, k: int, log_u: float):
    """r = (lp_k - lp_j) T_j + (lp_j - lp_k) T_k; the two chains exchange temperatures (states stay put)
    iff r >= log u  (BNN_mc3.py:101-112)."""
    t = np.array(temps, dtype=np.float64, copy=True)
    r = (log_post[k] - log_post[j]) * t[j] + (log_post[j] - log_post[k]) * t[k]
    swapped = bool(r >= log_u)
    if swapped:
        t[j], t[k] = temps[k], temps[j]
    return t, swapped


def gather_log_post(local: torch.Tensor, counts, group: Optional[dist.ProcessGroup] = None) -> np.ndarray:
    """All-gather of the local chains' log-posteriors -> host vector over all chains (rank order).
    `counts[r]` = chains rank r contributes.  Uses the process group's backend (NCCL on GPUs, gloo in tests)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local.detach().cpu().numpy().astype(np.float64)
    world = dist.get_world_size(group)
    cmax = max(counts)
    send = torch.zeros(cmax, dtype=torch.float64, device=local.device)
    send[:local.numel()] = local
    recv = torch.empty(world * cmax, dtype=torch.float64, device=local.device)
    dist.all_gather_into_tensor(recv, send, group=group)
    recv = recv.cpu().numpy().reshape(world, cmax)
    return np.concatenate([recv[r, :counts[r]] for r in range(world)])


def exchange(local_log_post: torch.Tensor, temps_all: np.ndarray, rng: SwapRNG,
             group: Optional[dist.ProcessGroup] = None, world_size: int = 1, R: int = 1, gather=gather_log_post):
    """One swap step on a grid of world_size / R chain blocks x R row shards (chain_grid).  Returns (new temperatures of
    ALL chains, swapped?, (j, k), gathered log-posteriors).  The R ranks of a block hold bit-identical copies of its
    log-posteriors; only the r = 0 copy enters the swap (the others count zero chains in the gather).
    gather(local, counts, group): the all-gather (a test substitutes an in-process one)."""
    n = len(temps_all)
    Q = world_size // R
    counts = [chain_partition(n, Q, p // R)[1] if p % R == 0 else 0 for p in range(world_size)]
    lp = gather(local_log_post, counts, group)
    if n < 2:
        return np.array(temps_all, dtype=np.float64), False, (0, 0), lp
    j, k = rng.pair(n)
    t, swapped = swap_temperatures(lp, temps_all, j, k, rng.log_uniform())
    return t, swapped, (j, k), lp
