"""Drop-in for the reference's ``lib/mcts.py:MCTS`` -- same constructor, methods, argument meaning and the
four dict attributes -- backed by a one-game CUDA engine (``SelfPlayEngine`` with ``games=1``).

It exists for source compatibility (``play_game``, ``Session``, ``evaluate`` style callers that drive ONE
game); the throughput path is ``engine.SelfPlayEngine`` with thousands of games.  Every number comes from the
CUDA kernels; nothing here re-implements search arithmetic on the host.

Differences worth knowing (all documented in DESIGN.md):
  * the tree is keyed per engine (per ``MCTS`` object), exactly like the reference's dicts;
  * Dirichlet noise comes from the engine's Philox streams unless ``noise_fn`` is set (the reference draws from
    the global numpy RNG, which cannot be shared with a GPU);
  * a ``net`` that is a ``caro_ai_b200.model.Net`` / ``DeviceNet`` runs through the fused tensor-core tower with
    EVAL-mode BatchNorm (folded running statistics).  The reference never calls ``.eval()`` and searches with
    train-mode batch statistics that depend on what else is in the leaf batch (SURVEY.md section 0.5); that quirk is
    deliberately not reproduced; any other callable is evaluated as ``net(planes) -> (logits, values)`` + softmax,
    i.e. exactly ``lib/mcts.py:212-218``, on the leaf planes produced by the CUDA encode kernel.
"""
from __future__ import annotations

import weakref
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

from . import _cabi
from .engine import SelfPlayEngine
from .model import DeviceNet, Net

# config.py:26-28
C_PUCT = 1.0
ALPHA = 0.30
EXPLORE = 0.25


class MCTS:
    def __init__(self, game, node_capacity: int = 1 << 16, max_batch: int = 32, seed: int = 0,
                 noise_fn: Optional[Callable[[int, int], np.ndarray]] = None, solver: bool = False, gumbel: bool = False):
        """``noise_fn(batch, actions) -> float64 [batch, actions]`` injects the Dirichlet draws (tests).
        ``solver`` (extension, default off): the MCTS solver (``SelfPlayEngine.set_solver``) for both players of the
        shared tree; ``proof`` then shows which edges it proved.
        ``gumbel`` (extension, default off): every ``search_batch`` searches the root by Gumbel sequential halving
        (``SelfPlayEngine.set_gumbel``, default parameters); ``get_policy_value`` then returns the improved policy for
        tau 1 and a one-hot on the best survivor for tau 0."""
        self.solver = bool(solver)
        self.gumbel = bool(gumbel)
        self.c_puct = C_PUCT
        self.precision = "auto"  # nn.Module nets: one-pass bf16 tower while it holds 1e-3 on probe positions, else bf16x3
        self.game = game
        self.noise_fn = noise_fn
        self._engine: Optional[SelfPlayEngine] = None
        self._cfg = dict(node_capacity=node_capacity, max_batch=max_batch, seed=seed)
        self._device_nets: Dict[int, tuple] = {}
        self._overlay: Optional[Dict[str, dict]] = None  # host-assigned statistics (lib/test_mcts.py:15-21)
        self._minibatches = 0

    # ------------------------------------------------------------------ engine plumbing
    def _eng(self) -> SelfPlayEngine:
        if self._engine is None:
            a = getattr(self.game, "action_space", None)
            assert isinstance(a, int), "a game with an integer action_space is required for device searches"
            self._engine = SelfPlayEngine(self.game, 1, trees_per_game=1, max_batch=self._cfg["max_batch"],
                                          node_capacity=self._cfg["node_capacity"], c_puct=self.c_puct, alpha=ALPHA,
                                          explore=EXPLORE, seed=self._cfg["seed"])
            if self.solver:
                self._engine.set_solver(3)
            if self.gumbel:
                self._engine.set_gumbel(3)
        return self._engine

    @staticmethod
    def _weights_version(net: Net) -> int:
        """Changes whenever a parameter or buffer of ``net`` is written in place (optimizer step, load_state_dict,
        BatchNorm running statistics): torch bumps every tensor's version counter on an in-place write."""
        return sum(t._version for t in net.state_dict(keep_vars=True).values())

    def _device_net(self, net) -> Optional[DeviceNet]:
        """The folded device twin of ``net``.  The reference always searches with the module's LIVE weights, so the twin
        is re-folded whenever the module's tensors have been written since the last search; the cache holds a weak
        reference (a recycled ``id()`` of a collected module can never alias another network)."""
        if isinstance(net, DeviceNet):
            return net
        if isinstance(net, Net):
            key = id(net)
            entry = self._device_nets.get(key)
            version = self._weights_version(net)
            if entry is not None and entry[0]() is net:
                if entry[2] != version:
                    entry[1].update(net)
                    self._device_nets[key] = (entry[0], entry[1], version)
                return entry[1]
            if entry is not None:
                entry[1].close()
            dn = DeviceNet(net, self.game, precision=self.precision)
            self._device_nets[key] = (weakref.ref(net), dn, version)
            return dn
        return None

    def refresh_net(self, net: Net) -> None:
        """Force a re-fold of ``net`` (kept for callers of the first release; the facade now notices weight changes by
        itself through the tensors' version counters)."""
        entry = self._device_nets.get(id(net))
        if entry is not None and entry[0]() is net:
            entry[1].update(net)
            self._device_nets[id(net)] = (entry[0], entry[1], self._weights_version(net))

    def _check_engine(self) -> None:
        """Engine error bits (include/caro_b200.h, counters[7]) become exceptions: a full arena on a long-lived shared
        tree must not pass silently (the reference's dicts simply grow)."""
        err = self._engine.counters()["errors"] if self._engine is not None else 0
        if err & 1:
            raise _cabi.CaroError("MCTS node arena is full (node_capacity=%d): construct MCTS(game, node_capacity=...) larger "
                                  "or clear() the tree" % self._cfg["node_capacity"])

    # ------------------------------------------------------------------ reference surface
    def clear(self) -> None:  # lib/mcts.py:39-43
        self._overlay = None
        if self._engine is not None:
            self._engine.reset(first_player=0)

    def __len__(self) -> int:  # lib/mcts.py:45-46
        if self._overlay is not None:
            return len(self._overlay["value"])
        if self._engine is None:
            return 0
        return int(self._engine.region("node_count")[0].item())

    def is_leaf(self, state_int: int) -> bool:  # lib/mcts.py:150-160
        return state_int not in self.probs

    def _noise(self, batch: int) -> Optional[torch.Tensor]:
        if self.noise_fn is None:
            return None
        z = np.ascontiguousarray(self.noise_fn(batch, self.game.action_space), dtype=np.float64)
        return torch.from_numpy(z.reshape(1, batch, self.game.action_space)).cuda()

    def search_minibatch(self, batch_size: int, state_int: int, player: int, net, device: str = "cpu") -> None:
        """lib/mcts.py:248-287."""
        eng = self._eng()
        assert batch_size <= eng.max_batch, "batch_size exceeds the engine's max_batch"
        eng.set_roots([state_int], [player])
        self._step(eng, batch_size, net)

    def search_batch(self, count: int, batch_size: int, state_int: int, player: int, net, device: str = "cpu") -> None:
        """lib/mcts.py:162-176."""
        eng = self._eng()
        assert batch_size <= eng.max_batch, "batch_size exceeds the engine's max_batch"
        eng.set_roots([state_int], [player])
        dn = self._device_net(net)
        if dn is not None and self.noise_fn is None:
            eng.search(dn, count, batch_size, first_minibatch=self._minibatches & 0x3FFFF)
            self._minibatches += count
            return
        first = self._minibatches & 0x3FFFF
        for i in range(count):
            self._step(eng, batch_size, net, (first, i, count))

    def _step(self, eng: SelfPlayEngine, batch: int, net, search: Tuple[int, int, int] = None) -> None:
        """``search`` = (search index, minibatch, count) of the Gumbel plan; a lone minibatch is a search of its own."""
        first, i, count = search if search is not None else (self._minibatches & 0x3FFFF, 0, 1)
        eng.gumbel_plan(first, i, count, batch)
        eng.select(batch, self._minibatches & 0x3FFFF, self._noise(batch))
        self._minibatches += 1
        eng.plan(batch)
        n = eng.leaf_count()
        if n == 0:
            dummy = torch.zeros(1, dtype=torch.float32, device="cuda")
            eng.expand_backup(batch, dummy, dummy)
            return
        dn = self._device_net(net)
        if dn is not None:
            pri, val = dn.forward_boards(eng.region("leaf_board"), eng.region("leaf_player"), n)
        else:  # lib/mcts.py:212-218 with an arbitrary callable
            planes = eng.leaf_planes(n)
            try:
                dev = next(net.parameters()).device
            except (AttributeError, StopIteration):
                dev = planes.device
            logits, vals = net(planes.to(dev))
            pri = F.softmax(logits, dim=1).detach().to("cuda", torch.float32).contiguous()
            val = vals.detach().to("cuda", torch.float32)[:, 0].contiguous()
        eng.expand_backup(batch, pri, val)

    def find_leaf(self, state_int: int, player: int) -> Tuple[Optional[float], int, int, List[int], List[int]]:
        """lib/mcts.py:97-148: one descent on the current tree (nothing is expanded or backed up)."""
        eng = self._eng()
        eng.set_roots([state_int], [player])
        eng.select(1, self._minibatches & 0x3FFFF, self._noise(1))
        kind = int(eng.region("desc_kind")[0, 0].item())
        depth = int(eng.region("desc_path_len")[0, 0].item())
        nodes = eng.region("desc_path_node")[0, 0, :depth].cpu().numpy()
        actions = [int(a) for a in eng.region("desc_path_action")[0, 0, :depth].cpu().numpy()]
        boards = eng.region("node_board")[torch.from_numpy(nodes.astype(np.int64)).cuda()].cpu().numpy().view(np.uint64)
        states = self.game.states_from_boards(boards) if depth else []
        leaf = self.game.states_from_boards(eng.region("desc_board")[0, 0:1].cpu().numpy().view(np.uint64))[0]
        leaf_player = int(eng.region("desc_player")[0, 0].item())
        value = float(eng.fregion("desc_value")[0, 0].item()) if kind == 1 else None
        return value, leaf, leaf_player, states, actions

    def get_policy_value(self, state_int: int, tau: float = 1) -> Tuple[List[float], List[float]]:
        """lib/mcts.py:289-313."""
        eng = self._eng()
        roots, players = eng.roots()
        if roots[0] != state_int:
            eng.set_roots([state_int], [players[0]])
        pi, q, _ = eng.root_policy(0 if tau == 0 else 1)
        self._check_engine()
        return [float(x) for x in pi[0].cpu().numpy()], [float(x) for x in q[0].cpu().numpy()]

    # ------------------------------------------------------------------ dict views (lib/mcts.py:29-36)
    def _export(self) -> Dict[str, dict]:
        if self._overlay is not None:
            return self._overlay
        out = {"visit_count": {}, "value": {}, "value_avg": {}, "probs": {}, "proof": {}}
        if self._engine is not None:
            for s, n in self._engine.export_tree(0).items():
                out["visit_count"][s] = [int(x) for x in n["N"]]
                out["value"][s] = [float(x) for x in n["W"]]
                out["value_avg"][s] = [float(x) for x in n["Q"]]
                out["probs"][s] = [float(x) for x in n["P"]]
                out["proof"][s] = [int(x) for x in n["proof"]]
        return out

    def _set(self, name: str, value: dict) -> None:
        if self._overlay is None:
            self._overlay = self._export()
        self._overlay[name] = value

    visit_count = property(lambda self: self._export()["visit_count"], lambda self, v: self._set("visit_count", v))
    value = property(lambda self: self._export()["value"], lambda self, v: self._set("value", v))
    value_avg = property(lambda self: self._export()["value_avg"], lambda self, v: self._set("value_avg", v))
    probs = property(lambda self: self._export()["probs"], lambda self, v: self._set("probs", v))
    # solver extension: {state: [edge status]} with 0 unknown, 1 win, 2 loss, 3 draw for the side to move at the state
    proof = property(lambda self: self._export().get("proof", {}))

    def _backup(self, value: float, states: List[int], actions: List[int]) -> None:
        """lib/mcts.py:225-246 on host-assigned statistics (the reference's own unit test drives it this way):
        the rows are flattened, updated by the CUDA ``caro_backup_path`` kernel (float32) and written back."""
        _cabi.require_cuda()
        ov = self._overlay if self._overlay is not None else self._export()
        self._overlay = ov
        keys = list(ov["visit_count"].keys())
        offs, flat_n, flat_w, flat_q = {}, [], [], []
        for k in keys:
            offs[k] = len(flat_n)
            flat_n += [int(x) for x in ov["visit_count"][k]]
            flat_w += [float(x) for x in ov["value"][k]]
            flat_q += [float(x) for x in ov["value_avg"][k]]
        d_n = torch.tensor(flat_n, dtype=torch.int32, device="cuda")
        d_w = torch.tensor(flat_w, dtype=torch.float32, device="cuda")
        d_q = torch.tensor(flat_q, dtype=torch.float32, device="cuda")
        edges = torch.tensor([offs[s] + int(a) for s, a in zip(states, actions)], dtype=torch.int64, device="cuda")
        _cabi.check(_cabi.lib().caro_backup_path(d_n.data_ptr(), d_w.data_ptr(), d_q.data_ptr(), edges.data_ptr(), len(states),
                                                 float(value), torch.cuda.current_stream().cuda_stream))
        n, w, q = d_n.cpu().tolist(), d_w.cpu().tolist(), d_q.cpu().tolist()
        for k in keys:
            a = len(ov["visit_count"][k])
            o = offs[k]
            ov["visit_count"][k] = n[o:o + a]
            ov["value"][k] = w[o:o + a]
            ov["value_avg"][k] = q[o:o + a]
