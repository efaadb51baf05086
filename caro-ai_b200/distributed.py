"""Multi-GPU plumbing (one process per GPU, ``torch.distributed``; NCCL over NVLink on the box, gloo in the CPU
tests).  Self-play needs no collective -- games shard by rank -- so the only exchanges are the ones SURVEY.md
section 8(e) lists: a flattened-gradient all-reduce per SGD step, the all-gather of the ranks' replay samples into the
step's batch, a weight broadcast before an evaluation / after a best-net promotion, the 3-integer W/L/D reduction of
the arena evaluation and the MIN-reduction behind every "do we train this step?" decision."""
from __future__ import annotations

from typing import Iterable, List, Tuple

import torch
import torch.distributed as dist


def world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_games(total_games: int, rank: int, world_size: int) -> Tuple[int, int]:
    """(first global game id, count) owned by ``rank``: contiguous, sizes differ by at most one."""
    base, extra = divmod(total_games, world_size)
    count = base + (1 if rank < extra else 0)
    first = rank * base + min(rank, extra)
    return first, count


def allreduce_gradients(params: Iterable[torch.nn.Parameter]) -> int:
    """Average the gradients over ranks with ONE all-reduce of a flattened fp32 bucket (188,301 elements for the
    Connect4 network = 753 KB: latency-bound, no bucketing needed).  Returns the bucket length."""
    plist: List[torch.nn.Parameter] = [p for p in params if p.grad is not None]
    if not plist:
        return 0
    flat = torch.cat([p.grad.reshape(-1).float() for p in plist])
    _, ws = world()
    if ws > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat /= ws
    off = 0
    for p in plist:
        n = p.grad.numel()
        p.grad.copy_(flat[off:off + n].view_as(p.grad))
        off += n
    return int(flat.numel())


class FlatGradients:
    """The same exchange without the per-step flatten / scatter: the parameters' ``.grad`` tensors are VIEWS into one
    persistent fp32 bucket, so a step's gradient averaging is exactly one NCCL all-reduce (+ one scale kernel) instead
    of ~75 small copy kernels around it (2 x B200: 459 us -> see tools/allreduce_bench.py).  Use ``zero()`` instead of
    ``optimizer.zero_grad()`` (which would drop the views)."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
        n = sum(p.numel() for p in self.params)
        dev = self.params[0].device if self.params else None
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        off = 0
        for p in self.params:
            assert p.dtype == torch.float32
            p.grad = self.flat[off:off + p.numel()].view_as(p)
            off += p.numel()

    def zero(self) -> None:
        self.flat.zero_()

    def allreduce(self) -> int:
        _, ws = world()
        if ws > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
            self.flat /= ws
        return int(self.flat.numel())


def broadcast_state_dict(module: torch.nn.Module, src: int = 0) -> None:
    """NetWrapper.sync() across ranks: every tensor of the state_dict (incl. BatchNorm running stats) from ``src``."""
    _, ws = world()
    if ws == 1:
        return
    for t in module.state_dict().values():
        dist.broadcast(t, src=src)


def all_min(value: int, device=None) -> int:
    """Smallest ``value`` over the ranks: collective decisions (train.py:199 "is the replay buffer large enough?") must be
    taken on a reduced quantity, or the ranks fall out of step with each other's collectives."""
    _, ws = world()
    if ws == 1:
        return int(value)
    t = torch.tensor([int(value)], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return int(t[0])


def all_gather_rows(tensors):
    """Concatenation over ranks (rank order) of every tensor's rows: the SGD batch assembled from the ranks' replay
    samples (BATCH_SIZE / world rows each).  One all-gather per tensor (planes, pi, z)."""
    _, ws = world()
    if ws == 1:
        return tuple(tensors)
    out = []
    for t in tensors:
        t = t.contiguous()
        full = torch.empty((ws * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(full, t)
        out.append(full)
    return tuple(out)


def reduce_tallies(wins: int, losses: int, draws: int, device=None) -> Tuple[int, int, int]:
    """Sum of the arena W/L/D counters over ranks (train.py:120-149 sharded over GPUs)."""
    _, ws = world()
    if ws == 1:
        return wins, losses, draws
    t = torch.tensor([wins, losses, draws], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return int(t[0]), int(t[1]), int(t[2])


def sum_counts(counts, device=None):
    """Element-wise sum over the ranks of an integer array (the resignation calibration's per-threshold tallies): one
    all-reduce, so every rank derives the same decision from the same numbers."""
    import numpy as np
    counts = np.asarray(counts, dtype=np.int64)
    _, ws = world()
    if ws == 1:
        return counts
    t = torch.from_numpy(counts.copy()).to(device if device is not None else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t.cpu().numpy()
