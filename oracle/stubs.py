"""Deterministic stand-ins for the policy/value network (TEST-ONLY, part of the oracle).

The reference's search accepts any callable ``net(planes) -> (logits, values)`` (lib/mcts.py:215);
``play_game`` additionally type-checks ``isinstance(net, model.Net)`` (lib/utils.py:52-53), which the
golden generator satisfies by subclassing the reference's Net and overriding ``forward`` with
``stub_forward`` below.

Two flavours, both pure functions of ONE board (no cross-row arithmetic), built from integer
hashes so that results are bit-identical on every machine:
  * ``stub_forward``  -- torch, returns (logits, values); the caller (reference / oracle) applies
                         its own softmax.  Used for the golden fixtures.
  * ``stub_priors``   -- numpy, returns (priors, values) directly with priors = w / sum(w) from
                         integer weights: one IEEE float32 division per entry, no exp().  Used
                         when the CUDA engine and the oracle must see *identical* network outputs.
"""
from __future__ import annotations

import numpy as np


def _weights(n_in: int, n_out: int, salt: int) -> np.ndarray:
    j = np.arange(n_in, dtype=np.uint64)[:, None]
    a = np.arange(n_out, dtype=np.uint64)[None, :]
    h = (j * np.uint64(2654435761) + a * np.uint64(40503) + np.uint64(salt)) & np.uint64(0xFFFFFFFF)
    h ^= h >> np.uint64(15)
    h = (h * np.uint64(2246822519)) & np.uint64(0xFFFFFFFF)
    h ^= h >> np.uint64(13)
    return (h >> np.uint64(20)).astype(np.int64)  # 0..4095


def _scores(planes: np.ndarray, actions_n: int):
    """Exact integer projections of the 0/1 planes: s[L,A] and t[L]."""
    x = np.asarray(planes).reshape(len(planes), -1).astype(np.int64)
    s = x @ _weights(x.shape[1], actions_n, 12345)
    t = (x @ _weights(x.shape[1], 1, 777))[:, 0]
    return s, t


def stub_forward(planes_tensor, actions_n: int):
    """(logits [L,A] in [-4,4), values [L,1] in [-1,1]) as float32 torch tensors."""
    import torch
    s, t = _scores(planes_tensor.detach().cpu().numpy(), actions_n)
    logits = torch.from_numpy(((s % 1024) - 512).astype(np.float32)) / 128.0
    values = torch.from_numpy(((t % 2001) - 1000).astype(np.float32)[:, None]) / 1000.0
    return logits, values


def stub_priors(planes: np.ndarray, actions_n: int):
    """(priors float32 [L,A] summing to ~1, values float32 [L])."""
    s, t = _scores(planes, actions_n)
    w = (1 + (s % 1024)).astype(np.int64)
    tot = w.sum(axis=1, keepdims=True)  # exact integer sum
    pri = w.astype(np.float32) / tot.astype(np.float32)
    val = ((t % 2001) - 1000).astype(np.float32) / np.float32(1000.0)
    return pri, val


CHAIN_PRIOR = 0.99


def chain_priors(planes: np.ndarray, actions_n: int):
    """(priors float32 [L,A], values float32 [L] = 0): CHAIN_PRIOR on ONE legal move picked by an integer hash of the
    planes, the rest spread evenly over the other actions.  A search driven by it keeps following that move, so its
    paths grow about one edge per visit of their end instead of staying a few plies deep.  Legal moves are read off the
    planes: an empty cell (m,n,k, one action per cell) or a column with an empty cell (Connect4, one action per column).
    On Connect4 the pick avoids a move that completes four for the side to move (plane 0) while another move is left,
    so that the chain can run to a nearly full board instead of ending in a win after a dozen plies."""
    x = np.asarray(planes).reshape(len(planes), 2, -1).astype(np.int64)
    occupied = x[:, 0] | x[:, 1]
    h = (x.reshape(len(planes), -1) @ _weights(x.shape[1] * x.shape[2], 1, 4242))[:, 0]
    pri = np.full((len(planes), actions_n), (1.0 - CHAIN_PRIOR) / (actions_n - 1), dtype=np.float32)
    for i in range(len(planes)):
        if occupied.shape[1] == actions_n:
            legal = np.flatnonzero(occupied[i] == 0)
        else:
            grid = occupied[i].reshape(-1, actions_n)  # row 0 = top
            legal = np.flatnonzero(grid[0] == 0)
            quiet = [c for c in legal if not _c4_completes_four(x[i, 0].reshape(grid.shape), grid, int(c))]
            legal = np.asarray(quiet) if quiet else legal
        if len(legal):
            pri[i, legal[h[i] % len(legal)]] = np.float32(CHAIN_PRIOR)
    return pri, np.zeros(len(planes), dtype=np.float32)


def _c4_completes_four(mine: np.ndarray, occupied: np.ndarray, col: int) -> bool:
    rows, cols = occupied.shape
    row = max(r for r in range(rows) if occupied[r, col] == 0)  # the token lands on the lowest empty cell
    for dr, dc in ((0, 1), (1, 0), (1, 1), (1, -1)):
        run = 1
        for sign in (1, -1):
            r, c = row + sign * dr, col + sign * dc
            while 0 <= r < rows and 0 <= c < cols and mine[r, c]:
                run += 1
                r, c = r + sign * dr, c + sign * dc
        if run >= 4:
            return True
    return False
