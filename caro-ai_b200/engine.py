"""Lock-step batched MCTS self-play engine (host wrapper over the ``caro_engine_*`` C ABI).

G independent games, each with its own tree arena(s), are advanced together: every
``search`` step is the reference's ``MCTS.search_minibatch`` (lib/mcts.py:248-287) for all games
at once, every ``advance`` one ply of ``play_game`` (lib/utils.py:76-99).  torch is used for device
memory and streams only.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _cabi
from .model import DeviceNet, IMPL_TCGEN05

_NP = {1: np.uint8, 4: np.int32, 8: np.int64}


class SelfPlayEngine:
    def __init__(self, game, games: int, trees_per_game: int = 1, max_batch: int = 8, node_capacity: int = 4096,
                 replay_capacity: int = 0, c_puct: float = 1.0, alpha: float = 0.30, explore: float = 0.25,
                 seed: int = 0, device: Optional[str] = None, virtual_loss: bool = False, mask_priors: bool = False,
                 fresh_tree: bool = False, recycle_tree: bool = False, compact_tree: bool = False):
        """``virtual_loss`` / ``mask_priors`` / ``fresh_tree`` / ``recycle_tree``: throughput-mode extensions that are NOT in the reference
        (include/caro_b200.h CARO_FLAG_*), all off by default; with any of them on the trees are no longer the
        reference's bit for bit.  ``compact_tree`` is different: after every move it drops the nodes that can no longer be
        reached and packs the arena -- every reachable statistic, policy and move stays bit-identical, only the arena demand
        changes (long games fit a small ``node_capacity``)."""
        _cabi.require_cuda()
        self.game = game
        self.G = int(games)
        self.A = game.action_space
        self.max_batch = int(max_batch)
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        flags = ((_cabi.FLAG_VIRTUAL_LOSS if virtual_loss else 0) | (_cabi.FLAG_MASK_PRIORS if mask_priors else 0) |
                 (_cabi.FLAG_FRESH_TREE if fresh_tree else 0) | (_cabi.FLAG_RECYCLE_TREE if recycle_tree else 0) |
                 (_cabi.FLAG_COMPACT_TREE if compact_tree else 0))
        self.cfg = _cabi.EngineConfig(game.game_kind, game.n, game.k, self.G, trees_per_game, max_batch, node_capacity,
                                      replay_capacity, c_puct, alpha, explore, seed, flags, 0)
        lib = _cabi.lib()
        nbytes = lib.caro_engine_workspace_bytes(C.byref(self.cfg))
        if nbytes == 0:
            raise _cabi.CaroError("bad engine config: " + lib.caro_last_error().decode())
        with torch.cuda.device(self.device):
            self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            handle = C.c_void_p()
            _cabi.check(lib.caro_engine_create(C.byref(self.cfg), self.workspace.data_ptr(), nbytes, C.byref(handle),
                                               self._stream()))
        self.handle = handle
        self.workspace_bytes = nbytes
        self._views: Dict[str, torch.Tensor] = {}

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    # fields of the per-descent record (csrc/engine.cuh DescRec): name -> (byte offset, bytes, dtype); the board follows at 32
    _DESC_FIELDS = {"desc_kind": (0, 1, torch.uint8), "desc_player": (1, 1, torch.uint8), "desc_path_len": (2, 2, torch.int16),
                    "desc_slot": (4, 4, torch.int32), "desc_value": (8, 4, torch.int32), "desc_key_lo": (16, 8, torch.int64),
                    "desc_key_hi": (24, 8, torch.int64)}

    def region(self, name: str) -> torch.Tensor:
        """Zero-copy torch view of a named workspace region (see include/caro_b200.h).  The per-descent fields
        ("desc_kind", "desc_slot", "desc_board", "desc_path_node", ...) are COPIES sliced out of the descent records
        ("desc": one 64 / 96-byte record per descent) and of the packed paths ("desc_path": node << 8 | action)."""
        if name in self._DESC_FIELDS or name == "desc_board":
            rec = self.region("desc")  # int64 [G, B, words]
            raw = rec.view(torch.uint8).view(rec.shape[0], rec.shape[1], rec.shape[2] * 8)
            if name == "desc_board":
                words = self.game.board_words
                return raw[:, :, 32:32 + 8 * words].contiguous().view(torch.int64).view(rec.shape[0], rec.shape[1], words)
            off, nbytes, dtype = self._DESC_FIELDS[name]
            out = raw[:, :, off:off + nbytes].contiguous().view(dtype).view(rec.shape[0], rec.shape[1])
            return out.to(torch.int32) if dtype == torch.int16 else out
        if name in ("desc_path_node", "desc_path_action"):
            path = self.region("desc_path")
            return ((path >> 8) & 0xFFFFFF) if name == "desc_path_node" else (path & 0xFF).to(torch.uint8)
        if name not in self._views:
            off, nbytes, elem = C.c_size_t(), C.c_size_t(), C.c_int32()
            dims = (C.c_int64 * 4)()
            _cabi.check(_cabi.lib().caro_engine_region(self.handle, name.encode(), C.byref(off), C.byref(nbytes),
                                                       C.byref(elem), C.byref(dims)))
            raw = self.workspace[off.value:off.value + nbytes.value]
            shape = [d for d in dims if d > 0]
            e = elem.value
            if e == 1:
                t = raw.view(shape)
            elif e == 2:
                t = raw.view(torch.int16).view(shape)
            elif e == 4:
                t = raw.view(torch.int32).view(shape)
            elif e == 8:
                t = raw.view(torch.int64).view(shape)
            else:  # boards / hash slots: expose as int64 words
                t = raw.view(torch.int64).view(shape + [e // 8])
            self._views[name] = t
        return self._views[name]

    def fregion(self, name: str) -> torch.Tensor:
        return self.region(name).view(torch.float32)

    def pool(self, name: str, lo: int = 0, hi: Optional[int] = None) -> torch.Tensor:
        """Rows [lo, hi) of one statistic of the node records (region "nodes": int32 [nodes, 4, Apad], rows N | W | P | C,
        csrc/engine.cuh): "N" visit counts, "W" total values, "P" priors, "C" cached child links, "f32" (bool: bit 31 of
        the N word, W has absorbed a float32 network value), "proof" (the solver's edge status, bits 29-30 of the N word:
        0 unknown, 1 win, 2 loss, 3 draw for the side to move at the node) and "Q" = f32(W / N) (0 where N == 0), which
        the engine does not store but recomputes with exactly this division wherever lib/mcts.py reads value_avg."""
        rec = self.region("nodes")
        rows = rec[lo:rec.shape[0] if hi is None else hi]
        raw = rows[:, 0, :]
        if name == "N":
            return raw & 0x1FFFFFFF
        if name == "f32":
            return raw < 0
        if name == "proof":
            return (raw >> 29) & 3
        if name == "W":
            return rows[:, 1, :].contiguous().view(torch.float32)
        if name == "P":
            return rows[:, 2, :].contiguous().view(torch.float32)
        if name == "C":
            return rows[:, 3, :]
        if name == "Q":  # IEEE float32 division on the host (numpy), the same rounding as __fdiv_rn
            n = (raw & 0x1FFFFFFF).cpu().numpy()
            w = rows[:, 1, :].contiguous().view(torch.float32).cpu().numpy()
            q = np.zeros_like(w)
            np.divide(w, n.astype(np.float32), out=q, where=n > 0)
            return torch.from_numpy(q)
        raise KeyError(name)

    def close(self):
        if getattr(self, "handle", None):
            _cabi.lib().caro_engine_destroy(self.handle)
            self.handle = None
            self._views = {}
            self.workspace = None  # the arenas go back to torch's allocator

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ game control
    def reset(self, mask: Optional[Sequence[int]] = None, first_player: int = -1):
        m = None
        if mask is not None:
            m = np.ascontiguousarray(np.asarray(mask, dtype=np.uint8))
            assert m.size == self.G
        _cabi.check(_cabi.lib().caro_engine_reset(self.handle, m.ctypes.data if m is not None else None, first_player,
                                                  self._stream()))
        if m is not None:
            torch.cuda.current_stream(self.device).synchronize()  # host mask buffer must outlive the copy

    def set_roots(self, states: Sequence[int], players: Sequence[int]):
        """search_batch's (state_int, player) arguments for every game (host ints -> one H2D copy)."""
        assert len(states) == self.G and len(players) == self.G
        boards = np.ascontiguousarray(self.game.boards_from_states(states))
        pl = np.ascontiguousarray(np.asarray(players, dtype=np.uint8))
        _cabi.check(_cabi.lib().caro_engine_set_roots(self.handle, boards.ctypes.data, pl.ctypes.data, self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def set_roots_pinned(self, boards_pinned: torch.Tensor, players_pinned: torch.Tensor):
        """Same, from caller-owned pinned host tensors (no sync; used by the end-to-end bench)."""
        _cabi.check(_cabi.lib().caro_engine_set_roots(self.handle, boards_pinned.data_ptr(), players_pinned.data_ptr(),
                                                      self._stream()))

    # ------------------------------------------------------------------ one minibatch, split
    def select(self, batch: int, minibatch_index: int = 0, noise: Optional[torch.Tensor] = None,
               noise_out: Optional[torch.Tensor] = None):
        _cabi.check(_cabi.lib().caro_engine_select(self.handle, batch, minibatch_index,
                                                   noise.data_ptr() if noise is not None else None,
                                                   noise_out.data_ptr() if noise_out is not None else None, self._stream()))

    def plan(self, batch: int):
        _cabi.check(_cabi.lib().caro_engine_plan(self.handle, batch, self._stream()))

    def leaf_count(self) -> int:
        return int(self.region("leaf_count").reshape(-1)[0].item())

    def leaf_planes(self, count: Optional[int] = None) -> torch.Tensor:
        """float32 [L,2,H,W] planes of the compact leaf batch (== states_to_training_batch)."""
        count = self.leaf_count() if count is None else count
        return self.game.planes_device(self.region("leaf_board"), self.region("leaf_player"), count)

    def expand_backup(self, batch: int, probs: torch.Tensor, values: torch.Tensor):
        assert probs.dtype == torch.float32 and values.dtype == torch.float32 and probs.is_contiguous()
        _cabi.check(_cabi.lib().caro_engine_expand_backup(self.handle, batch, probs.data_ptr(), values.data_ptr(),
                                                          self._stream()))

    # ------------------------------------------------------------------ fused paths
    def search(self, net: DeviceNet, count: int, batch: int, impl: int = None, first_minibatch: int = 0):
        """MCTS.search_batch(count, batch, ...) for all games with the built-in network.  ``first_minibatch`` numbers
        the minibatches for the Philox noise address (a running index when the same game / ply is searched again)."""
        impl = net.impl if impl is None else impl
        _cabi.check(_cabi.lib().caro_engine_search(self.handle, net.handle, count, batch, first_minibatch, impl, self._stream()))

    def search_with(self, evaluate, count: int, batch: int, noise_fn=None):
        """Same, with a caller-supplied evaluator ``evaluate(planes[L,2,H,W]) -> (priors[L,A], values[L])``
        (CUDA tensors).  One host sync per minibatch (the leaf count)."""
        for i in range(count):
            noise = noise_fn(i) if noise_fn is not None else None
            self.gumbel_plan(0, i, count, batch)
            self.select(batch, i, noise)
            self.plan(batch)
            n = self.leaf_count()
            if n:
                pri, val = evaluate(self.leaf_planes(n))
                self.expand_backup(batch, pri.contiguous().float(), val.contiguous().float())
            else:
                dummy = torch.zeros(1, dtype=torch.float32, device=self.device)
                self.expand_backup(batch, dummy, dummy)

    def root_policy(self, tau_mode: int = 1, tau_plies: int = 0) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        pi = torch.empty((self.G, self.A), dtype=torch.float64, device=self.device)
        q = torch.empty((self.G, self.A), dtype=torch.float32, device=self.device)
        n = torch.empty((self.G, self.A), dtype=torch.int32, device=self.device)
        _cabi.check(_cabi.lib().caro_engine_root_policy(self.handle, tau_mode, tau_plies, pi.data_ptr(), q.data_ptr(),
                                                        n.data_ptr(), self._stream()))
        return pi, q, n

    def advance(self, tau_plies: int, uniform: Optional[torch.Tensor] = None, auto_restart: bool = False,
                first_player: int = -1, want_actions: bool = True) -> Optional[torch.Tensor]:
        actions = torch.empty(self.G, dtype=torch.int32, device=self.device) if want_actions else None
        _cabi.check(_cabi.lib().caro_engine_advance(self.handle, tau_plies,
                                                    uniform.data_ptr() if uniform is not None else None,
                                                    1 if auto_restart else 0, first_player,
                                                    actions.data_ptr() if actions is not None else None, self._stream()))
        return actions

    def play(self, net_p0: DeviceNet, net_p1: DeviceNet, moves: int, count: int, batch: int, tau_plies: int,
             auto_restart: bool = True, first_player: int = -1, impl: int = None):
        impl = net_p0.impl if impl is None else impl
        _cabi.check(_cabi.lib().caro_engine_play(self.handle, net_p0.handle, net_p1.handle, moves, count, batch, tau_plies,
                                                 1 if auto_restart else 0, first_player, impl, self._stream()))

    def profile(self, level: int = 2):
        """0 = off, 1 = network kernel spans only (cheap), 2 = all four phases."""
        _cabi.check(_cabi.lib().caro_engine_profile(self.handle, int(level)))

    def profile_read(self) -> Dict[str, float]:
        """Summed CUDA-event milliseconds per search phase since the last read (+ kernel launches)."""
        ms = (C.c_double * 5)()
        launches = C.c_uint64()
        _cabi.check(_cabi.lib().caro_engine_profile_read(self.handle, C.byref(ms), C.byref(launches), self._stream()))
        return {"select_ms": ms[0], "plan_ms": ms[1], "net_ms": ms[2], "expand_backup_ms": ms[3], "noise_ms": ms[4],
                "launches": int(launches.value)}

    def step_host(self, boards_pinned: torch.Tensor, players_pinned: torch.Tensor, net: DeviceNet, count: int, batch: int,
                  tau_plies: int, out_pinned: Dict[str, torch.Tensor], impl: int = None):
        """One ply for all games through HOST buffers (the end-to-end path): roots H2D from pinned memory,
        search + advance on the device, then policy / actions / new roots D2H into pinned buffers."""
        self.set_roots_pinned(boards_pinned, players_pinned)
        self.search(net, count, batch, impl)
        pi, q, n = self.root_policy(2, tau_plies)
        actions = self.advance(tau_plies, None, auto_restart=True)
        out_pinned["pi"].copy_(pi, non_blocking=True)
        out_pinned["actions"].copy_(actions, non_blocking=True)
        out_pinned["boards"].copy_(self.region("root_board"), non_blocking=True)
        out_pinned["players"].copy_(self.region("root_player"), non_blocking=True)

    @staticmethod
    def play_multi(engines: Sequence["SelfPlayEngine"], net: DeviceNet, moves: int, count: int, batch: int, tau_plies: int,
                   auto_restart: bool = True, first_player: int = -1, impl: int = None):
        """Round-robin software pipeline over several engines (parts of the game batch): every part's tree kernels
        run on its own side stream underneath the other parts' network passes (caro_engine_play_multi)."""
        impl = net.impl if impl is None else impl
        arr = (C.c_void_p * len(engines))(*[e.handle for e in engines])
        _cabi.check(_cabi.lib().caro_engine_play_multi(arr, len(engines), net.handle, moves, count, batch, tau_plies,
                                                       1 if auto_restart else 0, first_player, impl, engines[0]._stream()))

    # ------------------------------------------------------------------ resignation (extension)
    def set_resign(self, threshold: Optional[float] = None, playthrough: float = 0.0):
        """Resignation (extension, off by default; include/caro_b200.h caro_engine_set_resign): from the next ply on, the
        side to move resigns when max(mean root value, Q of its most visited move) < ``threshold``.  ``threshold=None``
        switches it off; -1.0 never fires ("log only").  ``playthrough``: share of the games starting after this call that
        never resign and are logged instead (``resign_log``).  Enqueued on the current stream."""
        enable = threshold is not None
        _cabi.check(_cabi.lib().caro_engine_set_resign(self.handle, 1 if enable else 0, float(threshold) if enable else -1.0,
                                                       float(playthrough), self._stream()))

    # ------------------------------------------------------------------ MCTS solver (extension)
    def set_solver(self, players: int):
        """MCTS solver (extension, off by default; include/caro_b200.h caro_engine_set_solver): bit p of ``players`` makes
        the searches whose root player is p prove wins, losses and draws in the tree, stop descents at proven nodes and
        keep proven-losing moves out of pi and the move.  0 switches it off; 1 and 2 need two trees per game.  Enqueued on
        the current stream."""
        _cabi.check(_cabi.lib().caro_engine_set_solver(self.handle, int(players), self._stream()))

    def solver_counters(self) -> Dict[str, int]:
        """{"stopped": descents stopped at a proven node, "proven": edges proven}."""
        c = self.region("solver_counters").cpu().numpy()
        return {"stopped": int(c[0]), "proven": int(c[1])}

    # ------------------------------------------------------------------ Gumbel root search (extension)
    def set_gumbel(self, players: int, m: int = 16, c_visit: float = 50.0, c_scale: float = 0.1, scale: float = 1.0):
        """Gumbel root search (extension, off by default; include/caro_b200.h caro_engine_set_gumbel): bit p of ``players``
        makes the searches whose root player is p sample ``m`` root moves by Gumbel-top-k, split the descents over them
        by sequential halving, record softmax(log P + sigma(completed Q)) as pi and play the best survivor.  0 switches it
        off; 1 and 2 need two trees per game.  The defaults are the paper's and mctx's.  Enqueued on the current stream."""
        _cabi.check(_cabi.lib().caro_engine_set_gumbel(self.handle, int(players), int(m), float(c_visit), float(c_scale),
                                                       float(scale), self._stream()))

    def gumbel_plan(self, search_index: int, minibatch: int, count: int, batch: int):
        """The Gumbel step of the split API, before ``select`` of minibatch ``minibatch`` of a ``count``-minibatch search
        (no-op while Gumbel is off)."""
        _cabi.check(_cabi.lib().caro_engine_gumbel_plan(self.handle, int(search_index), int(minibatch), int(count), int(batch),
                                                        self._stream()))

    GUMBEL_STATE_DTYPE = np.dtype([("i0", np.int32), ("phase", np.int32), ("kstart", np.int32), ("m", np.int16),
                                   ("r", np.int16), ("surv", np.int16, (32,))])

    def gumbel_state(self) -> Dict[str, np.ndarray]:
        """Host copies of the Gumbel regions: "g" float64 [G, A] draws of the current search, "i0", "phase", "kstart", "m",
        "r" int [G] (i0 / phase -1: not yet), "survivors" (list per game, score order) and "forced" int [G, max_batch]
        (the coming minibatch's forced root actions, -1 = PUCT)."""
        st = self.region("gumbel_state").cpu().numpy().view(self.GUMBEL_STATE_DTYPE).reshape(-1)
        out = {k: st[k].astype(np.int64) for k in ("i0", "phase", "kstart", "m", "r")}
        out["survivors"] = [[int(a) for a in st["surv"][g][:max(int(st["r"][g]), 0)]] for g in range(self.G)]
        out["g"] = self.region("gumbel_g").cpu().numpy().view(np.float64).reshape(self.G, self.A)
        out["forced"] = self.region("gumbel_root").cpu().numpy().astype(np.int64)
        return out

    RESIGN_RECORD_DTYPE = np.dtype([("min_stat", np.float64, (2,)), ("result", np.int32), ("plies", np.int32)])

    def resign_log(self, start: int = 0) -> Tuple[np.ndarray, int]:
        """Records [start, cursor) of the playthrough-game log (the ring keeps the last G), oldest first, as a structured
        array of ``RESIGN_RECORD_DTYPE`` (min_stat per player, result from player 0's point of view, plies).  Returns
        (records, cursor)."""
        cursor = self.resign_counters()["logged"]
        start = max(start, cursor - self.G)
        if cursor <= start:
            return np.zeros(0, dtype=self.RESIGN_RECORD_DTYPE), cursor
        raw = self.region("resign_log").cpu().numpy().view(self.RESIGN_RECORD_DTYPE).reshape(-1)
        return raw[np.arange(start, cursor) % self.G].copy(), cursor

    def resign_counters(self) -> Dict[str, int]:
        """{"resigned": games that ended by resignation, "logged": playthrough games logged (= the log cursor)}."""
        c = self.region("resign_counters").cpu().numpy()
        return {"resigned": int(c[0]), "logged": int(c[1])}

    # ------------------------------------------------------------------ read-back
    COUNTER_NAMES = ("leaf_evals", "games", "plies", "wins_p0", "wins_p1", "draws", "descents", "errors")

    def counters(self) -> Dict[str, int]:
        out = (C.c_uint64 * 8)()
        _cabi.check(_cabi.lib().caro_engine_counters(self.handle, C.byref(out), self._stream()))
        return dict(zip(self.COUNTER_NAMES, [int(v) for v in out]))

    def roots(self) -> Tuple[List[int], List[int]]:
        boards = self.region("root_board").cpu().numpy().view(np.uint64)
        return self.game.states_from_boards(boards), [int(p) for p in self.region("root_player").cpu().numpy()]

    def export_tree(self, tree: int) -> Dict[int, dict]:
        """{state_int: {"N","W","Q","P","f32","proof"}} of one arena -- the dict view of lib/mcts.py:29-36, plus the
        solver's edge status ("proof", see ``pool``)."""
        n_nodes = int(self.region("node_count")[tree].item())
        cap = self.cfg.node_capacity
        lo, hi = tree * cap, tree * cap + n_nodes
        A = self.A
        N = self.pool("N", lo, hi)[:, :A].cpu().numpy()
        W = self.pool("W", lo, hi)[:, :A].cpu().numpy()
        Q = self.pool("Q", lo, hi)[:, :A].numpy()
        P = self.pool("P", lo, hi)[:, :A].cpu().numpy()
        F = self.pool("f32", lo, hi)[:, :A].cpu().numpy()
        PF = self.pool("proof", lo, hi)[:, :A].cpu().numpy()
        boards = self.region("node_board")[lo:hi].cpu().numpy().view(np.uint64)
        states = self.game.states_from_boards(boards)
        out = {}
        for i, s in enumerate(states):
            f32 = [bool(F[i, a]) for a in range(A)]
            out[s] = {"N": N[i].tolist(), "W": W[i].copy(), "Q": Q[i].copy(), "P": P[i].copy(), "f32": f32,
                      "proof": PF[i].tolist()}
        return out

    def replay_cursor(self) -> int:
        """Total number of replay entries ever written (one host read)."""
        return int(self.region("replay_cursor").item())

    def replay_live(self) -> int:
        """Entries currently held by the ring = ``len(replay_buffer)`` of train.py:199."""
        return min(self.replay_cursor(), max(0, self.cfg.replay_capacity))

    def replay_sample(self, count: int, rng=None, augment: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """train.py:85-94 without the host round trip: ``random.sample`` draws ``count`` of the live ring entries (the
        reference's sampler, on the entry NUMBERS only), the CUDA gather kernel turns them into the SGD tensors
        (planes float32 [count,2,H,W], pi float32 [count,A], z float32 [count]) straight from the ring.
        ``augment`` (extension, the reference has none): every row goes through a random board symmetry (Connect4: column
        mirror; square m,n,k boards: the eight dihedral symmetries), planes and policy target together."""
        import random as _random
        rng = rng or _random
        cursor = self.replay_cursor()
        live = min(cursor, max(0, self.cfg.replay_capacity))
        assert count <= live, "sample larger than the replay ring's content"
        picks = rng.sample(range(live), count)
        entries = torch.tensor([cursor - live + i for i in picks], dtype=torch.int64).to(self.device, non_blocking=True)
        sym = None
        if augment:
            n_sym = 2 if self.game.game_kind == _cabi.GAME_CONNECT4 else 8
            sym = torch.tensor([rng.randrange(n_sym) for _ in range(count)], dtype=torch.int32).to(self.device, non_blocking=True)
        _, h, w = self.game.obs_shape
        planes = torch.empty((count, 2, h, w), dtype=torch.float32, device=self.device)
        pi = torch.empty((count, self.A), dtype=torch.float32, device=self.device)
        z = torch.empty((count,), dtype=torch.float32, device=self.device)
        _cabi.check(_cabi.lib().caro_engine_replay_gather(self.handle, entries.data_ptr(), sym.data_ptr() if sym is not None else None,
                                                          count, planes.data_ptr(), pi.data_ptr(), z.data_ptr(), self._stream()))
        self._last_symmetry = sym
        return planes, pi, z

    def replay_load(self, entries) -> None:
        """Appends reference tuples (state_int, player, probs, z) to the ring (tests / warm starts)."""
        cap = self.cfg.replay_capacity
        assert cap > 0 and len(entries) <= cap
        cursor = self.replay_cursor()
        idx = (torch.arange(cursor, cursor + len(entries), device=self.device) % cap)
        boards = torch.from_numpy(self.game.boards_from_states([e[0] for e in entries]).view(np.int64)).to(self.device)
        self.region("replay_board")[idx] = boards
        self.region("replay_player")[idx] = torch.tensor([e[1] for e in entries], dtype=torch.uint8, device=self.device)
        self.fregion("replay_pi")[idx] = torch.tensor([list(e[2]) for e in entries], dtype=torch.float32, device=self.device)
        self.fregion("replay_z")[idx] = torch.tensor([float(e[3]) for e in entries], dtype=torch.float32, device=self.device)
        self.region("replay_cursor").fill_(cursor + len(entries))

    def replay_to_pinned(self, start: int, pinned: Dict[str, torch.Tensor]) -> Tuple[int, int]:
        """Copies the ring entries [start, cursor) -- the product of self-play, lib/utils.py:101-106 -- into caller-owned
        PINNED host tensors ``board`` int64 [cap,words], ``player`` uint8 [cap], ``pi`` float32 [cap,A], ``z`` float32 [cap]
        at the same ring slots (at most two contiguous device->host copies per field, asynchronous on the current
        stream after the one synchronous read of the cursor).  Returns (cursor, bytes copied)."""
        cap = self.cfg.replay_capacity
        cursor = self.replay_cursor()
        start = max(start, cursor - cap)
        if cap <= 0 or cursor <= start:
            return cursor, 8
        lo, hi = start % cap, cursor % cap
        spans = [(lo, hi)] if lo < hi else [(lo, cap), (0, hi)]
        nbytes = 8
        for name, view in (("board", self.region("replay_board")), ("player", self.region("replay_player")),
                           ("pi", self.fregion("replay_pi")), ("z", self.fregion("replay_z"))):
            for a, b in spans:
                if b > a:
                    pinned[name][a:b].copy_(view[a:b], non_blocking=True)
                    nbytes += (b - a) * view[0].numel() * view.element_size() if view.dim() > 1 else (b - a) * view.element_size()
        return cursor, nbytes

    def drain_replay(self, start: int = 0):
        """Replay entries [start, cursor) as reference tuples (state_int, player, probs, z)
        (lib/utils.py:101-106).  Returns (entries, cursor).  Host path for the reference-style deque; the trainer
        samples on the device (``replay_sample``)."""
        cursor = self.replay_cursor()
        cap = self.cfg.replay_capacity
        if cap <= 0 or cursor == start:
            return [], cursor
        start = max(start, cursor - cap)
        idx = torch.arange(start, cursor, device=self.device) % cap
        boards = self.region("replay_board")[idx].cpu().numpy().view(np.uint64)
        players = self.region("replay_player")[idx].cpu().numpy()
        pi = self.fregion("replay_pi")[idx].cpu().numpy()
        z = self.fregion("replay_z")[idx].cpu().numpy()
        states = self.game.states_from_boards(boards)
        return [(states[i], int(players[i]), pi[i].tolist(), int(z[i])) for i in range(len(states))], cursor
