"""The oracle side of three engine flags (include/caro_b200.h CARO_FLAG_*) that change what a search computes: MASK_PRIORS,
FRESH_TREE and RECYCLE_TREE; the cases tests/test_gpu_flag_matrix.py runs with them; and the kernel instance each case
reaches.  Shared by tests/test_gpu_flag_matrix.py (GPU) and tests/test_host_flag_matrix.py.

Restated from caro-ai_b200/csrc (a change there has to be mirrored here, and the host test then names the case that
moved):
  * expand_backup_body, engine_kernels.cuh:932-954 -- with MASK_PRIORS a new node's row is the network's row with the
    illegal moves zeroed and the legal ones renormalised, in float32, by a GW-lane reduction (masked_priors below);
  * advance_kernel, engine_kernels.cuh:1395-1405 -- after a move of a game that goes on, each of the game's trees is
    cleared with FRESH_TREE, or with RECYCLE_TREE once it holds more than node_cap / 2 nodes (clear_after_move);
  * caro_engine_expand_backup, engine.cu:449-474 -- expand_backup_kernel<R, BK> (32 lanes per game, BK = 8, 16, 32 by
    the batch) or, for Connect4 at batch <= 8 inside the play_multi pipeline of two or more parts (lean_tree) or from
    32,768 games on, expand_backup_group8_kernel (8 lanes per game) (expand_instance below).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence

import numpy as np

from caro_ai_b200._cabi import FLAG_FRESH_TREE, FLAG_MASK_PRIORS, FLAG_RECYCLE_TREE, FLAG_VIRTUAL_LOSS
from harness import StubOracleTree, np_choice
from search_matrix import C4, STUBS, VL_CASES, Case, VirtualLossOracleTree, host_noise, instances, make_roots


# ------------------------------------------------------------------------------------------------ MASK_PRIORS
def legal_part(probs, legal, gw: int) -> np.float32:
    """The legal mass expand_backup_body divides by: lane l adds, in float32 and in increasing a, probs[a] of the legal
    a = l (mod gw); an xor butterfly over the lanes (offsets gw/2 ... 1, float32) then gives every lane the same sum
    (a + b == b + a, so lane l and lane l ^ off compute the same value)."""
    p = np.asarray(probs, dtype=np.float32)
    lanes = [np.float32(0.0)] * gw
    for a in range(len(p)):
        if legal[a]:
            lanes[a % gw] = np.float32(lanes[a % gw] + p[a])
    off = gw // 2
    while off:
        lanes = [np.float32(lanes[lane] + lanes[lane ^ off]) for lane in range(gw)]
        off //= 2
    return lanes[0]


def masked_priors(probs, legal, gw: int) -> np.ndarray:
    """The row expand_backup_body stores for a new node with MASK_PRIORS, for a group of `gw` lanes per game: legal
    moves get f32(p / part) (an IEEE division, __fdiv_rn), or p itself when part is 0; illegal moves get 0."""
    p = np.asarray(probs, dtype=np.float32)
    legal = np.asarray(legal, dtype=bool)
    part = legal_part(p, legal, gw)
    out = np.zeros(len(p), dtype=np.float32)
    out[legal] = p[legal] / (part if part > 0 else np.float32(1.0))
    return out


class MaskedPriorsMixin:
    """For StubOracleTree and VirtualLossOracleTree (and the recorded-tower oracle of the pipeline test): a node is
    created with masked_priors of the network's row, as expand_backup_body does with MASK_PRIORS.  `gw` is the lane
    group of the expand kernel the engine runs: 32 for expand_backup_kernel, 8 for expand_backup_group8_kernel.
    `masked_nodes` counts the created nodes whose row had mass on an illegal move."""

    def __init__(self, game, *args, gw: int = 32, **kwargs):
        super().__init__(game, *args, **kwargs)
        self.gw = gw
        self.masked_nodes = 0

    def _new_node(self, state, prior_row) -> None:
        legal = np.zeros(self.game.action_space, dtype=bool)
        legal[self.game.possible_moves(state)] = True
        row = np.asarray(prior_row, dtype=np.float32)
        self.masked_nodes += int(bool((row[~legal] > 0).any()))
        super()._new_node(state, masked_priors(row, legal, self.gw))


class MaskedStubTree(MaskedPriorsMixin, StubOracleTree):
    pass


class MaskedVirtualLossTree(MaskedPriorsMixin, VirtualLossOracleTree):
    pass


# ------------------------------------------------------------------------------------------------ FRESH / RECYCLE_TREE
def clear_after_move(trees: Sequence, flags: int, node_cap: int) -> List[bool]:
    """advance_kernel's rule for a game that is not over, applied to the game's oracle trees (one or two, each judged on
    its own): clear it with FRESH_TREE, or with RECYCLE_TREE when it holds more than node_cap / 2 nodes (C integer
    division).  Returns which trees were cleared."""
    assert node_cap > 0
    cleared = []
    for t in trees:
        clear = bool(flags & FLAG_FRESH_TREE) or (bool(flags & FLAG_RECYCLE_TREE) and len(t) > node_cap // 2)
        if clear:
            t.clear()
        cleared.append(clear)
    return cleared


# ------------------------------------------------------------------------------------------------ cases
@dataclass(frozen=True)
class FlagCase(Case):
    mask_priors: bool = False
    fresh_tree: bool = False
    recycle_tree: bool = False
    caro: bool = False           # the Caro rule on board (n, k) instead of freestyle m,n,k
    node_capacity: int = 0       # 0: every move's searches fit (count * batch * moves + 8)
    parts: int = 1               # >= 2: SelfPlayEngine.play_multi over that many engines of G games each

    @property
    def flags(self) -> int:
        return ((FLAG_VIRTUAL_LOSS if self.virtual_loss else 0) | (FLAG_MASK_PRIORS if self.mask_priors else 0) |
                (FLAG_FRESH_TREE if self.fresh_tree else 0) | (FLAG_RECYCLE_TREE if self.recycle_tree else 0))

    @property
    def label(self) -> str:
        return "+".join(n for n, on in (("mask", self.mask_priors), ("vl", self.virtual_loss), ("fresh", self.fresh_tree),
                                         ("recycle", self.recycle_tree)) if on)

    @property
    def capacity(self) -> int:
        return self.node_capacity or self.count * self.batch * self.moves + 8

    def product_game(self):
        if self.caro:
            from caro_ai_b200.game import Caro
            return Caro(*self.board)
        return super().product_game()

    def oracle_game(self):
        if self.caro:
            from caro_oracle import CaroOracle
            return CaroOracle(*self.board)
        return super().oracle_game()


def make_flag_tree(case: FlagCase, og, gw: int = 32):
    stub = STUBS[case.stub]
    if case.mask_priors:
        return MaskedVirtualLossTree(og, stub=stub, gw=gw) if case.virtual_loss else MaskedStubTree(og, stub=stub, gw=gw)
    return VirtualLossOracleTree(og, stub=stub) if case.virtual_loss else StubOracleTree(og, stub=stub)


class OracleGames:
    """The oracle half of a flag case: the G games' positions and trees, stepped minibatch by minibatch and move by move
    in the order tests/test_gpu_flag_matrix.py steps the engine, with clear_after_move after every move.  `events`
    counts what the tree flags did at the advances of games that went on: trees kept (non-empty) and cleared, trees
    kept at exactly node_cap / 2 nodes, advances that cleared one of a game's two trees and kept the other, and
    searches after a clear that revisited positions the cleared tree held (those look up keys that had hash slots in
    the tree's previous generation)."""

    def __init__(self, case: FlagCase, roots):
        self.case, self.og = case, case.oracle_game()
        self.states, self.players = [r[0] for r in roots], [r[1] for r in roots]
        self.alive = [True] * case.G
        self.trees = [[make_flag_tree(case, self.og) for _ in range(case.trees_per_game)] for _ in range(case.G)]
        self.ply = 0
        self.largest = 0
        self.events = dict(kept=0, cleared=0, at_half=0, one_of_two=0, revisits=0)
        self._held = {}  # (game, tree) -> positions the tree held when it was last cleared, until its next search

    def tree_index(self, g: int) -> int:
        return self.players[g] if self.case.trees_per_game == 2 else 0

    def minibatch(self, noise) -> None:
        """One minibatch of every live game; noise[g] holds the Dirichlet vectors of game g's descents."""
        for g in range(self.case.G):
            if self.alive[g]:
                self.trees[g][self.tree_index(g)].minibatch(self.case.batch, self.states[g], self.players[g], noise[g])

    def policy(self, g: int):
        tree = self.trees[g][self.tree_index(g)]
        return tree.get_policy_value(self.states[g], tau=1 if self.ply < self.case.tau_plies else 0)

    def advance(self, u) -> List[int]:
        """Every live game plays np.random.choice(A, p=pi) with the uniform u[g]; returns the moves (-1: game over)."""
        actions = []
        for g in range(self.case.G):
            if not self.alive[g]:
                actions.append(-1)
                continue
            t = self.tree_index(g)
            self.largest = max(self.largest, len(self.trees[g][t]))
            held = self._held.pop((g, t), None)
            if held is not None:
                self.events["revisits"] += int(bool(held & set(self.trees[g][t].probs)))
            pi, _ = self.policy(g)
            a = np_choice(pi, u[g])
            actions.append(a)
            self.states[g], won = self.og.move(self.states[g], a, self.players[g])
            self.players[g] = 1 - self.players[g]
            if won or not self.og.possible_moves(self.states[g]):
                self.alive[g] = False
                continue
            sizes = [len(tree) for tree in self.trees[g]]
            held = [set(tree.probs) for tree in self.trees[g]]
            cleared = clear_after_move(self.trees[g], self.case.flags, self.case.capacity)
            for i, (n, c) in enumerate(zip(sizes, cleared)):
                if c and n:
                    self._held[(g, i)] = held[i]
                self.events["cleared"] += int(c and n > 0)
                self.events["kept"] += int(not c and n > 0)
                self.events["at_half"] += int(not c and n == self.case.capacity // 2)
            self.events["one_of_two"] += int(len(cleared) == 2 and cleared[0] != cleared[1])
        self.ply += 1
        return actions

    def masked_nodes(self) -> int:
        return sum(getattr(t, "masked_nodes", 0) for row in self.trees for t in row)


def oracle_run(case: FlagCase) -> OracleGames:
    """A host-noise case played out in the oracle alone, drawing from the seed's stream in the order the GPU runner does
    (roots, then per move the Dirichlet vectors of each minibatch and the move uniforms): the searches, clears and moves
    the engine has to reproduce."""
    assert case.noise == "host"
    og = case.oracle_game()
    rng = np.random.default_rng(case.seed)
    games = OracleGames(case, make_roots(case, og, rng))
    for _ in range(case.moves):
        for _ in range(case.count):
            games.minibatch(host_noise(case, rng))
        games.advance(rng.random(case.G))
    return games


# Masked priors from late random play-outs (most moves illegal), on every select width of the plain search, every
# expand width, one and two trees per game, host and Philox noise.
MASK_CASES: List[FlagCase] = [
    FlagCase("mask_mnk3_3_b8", (3, 3), G=16, count=6, batch=8, max_batch=8, plies=(3, 4, 5, 6, 7), moves=2, seed=501,
             mask_priors=True),
    FlagCase("mask_mnk5_4_b16_tpg2", (5, 4), G=8, count=6, batch=16, max_batch=16, plies=(8, 12, 16), moves=3, seed=502,
             trees_per_game=2, noise="philox", mask_priors=True),
    FlagCase("mask_mnk9_5_b32", (9, 5), G=6, count=5, batch=32, max_batch=32, plies=(20, 35, 50), moves=2, seed=503,
             noise="philox", mask_priors=True),
    FlagCase("mask_mnk15_5_b8_tpg2", (15, 5), G=4, count=6, batch=8, max_batch=8, plies=(40, 70, 100), moves=2, seed=504,
             trees_per_game=2, mask_priors=True),
    FlagCase("mask_caro9_5_b16", (9, 5), G=6, count=6, batch=16, max_batch=16, plies=(20, 30, 45), moves=2, seed=505,
             mask_priors=True, caro=True),
    FlagCase("mask_c4_b8", C4, G=16, count=6, batch=8, max_batch=8, plies=(12, 24, 34), moves=3, seed=506,
             noise="philox", mask_priors=True),
    FlagCase("mask_c4_b16_tpg2", C4, G=8, count=6, batch=16, max_batch=16, plies=(10, 20, 30), moves=3, seed=507,
             trees_per_game=2, mask_priors=True),
    FlagCase("mask_c4_b32", C4, G=8, count=5, batch=32, max_batch=32, plies=(18, 30, 36), moves=2, seed=508,
             noise="philox", mask_priors=True),
]

# Masked priors under virtual loss: the boards and widths of the virtual-loss matrix (select_vl_kernel on m,n,k,
# select_vl_group_kernel on Connect4).
MASK_VL_CASES: List[FlagCase] = [
    FlagCase("mask_" + c.name, c.board, G=c.G, count=c.count, batch=c.batch, max_batch=c.max_batch, plies=c.plies,
             moves=c.moves, seed=c.seed, noise=c.noise, virtual_loss=True, mask_priors=True)
    for c in VL_CASES
]

# A tree emptied after every move; node_capacity is one move's searches (the tree kept would overflow it).
FRESH_CASES: List[FlagCase] = [
    FlagCase("fresh_mnk3_3", (3, 3), G=16, count=4, batch=8, max_batch=8, plies=(0, 1, 2), moves=4, seed=601,
             fresh_tree=True, node_capacity=32),
    FlagCase("fresh_mnk9_5_tpg2", (9, 5), G=4, count=5, batch=16, max_batch=16, plies=(0, 10), moves=5, seed=602,
             trees_per_game=2, noise="philox", fresh_tree=True, node_capacity=80),
    FlagCase("fresh_c4", C4, G=8, count=5, batch=8, max_batch=8, plies=(0, 6, 12), moves=6, seed=603,
             fresh_tree=True, node_capacity=40),
    FlagCase("fresh_c4_tpg2", C4, G=8, count=4, batch=32, max_batch=32, plies=(0, 8), moves=4, seed=604,
             trees_per_game=2, noise="philox", fresh_tree=True, node_capacity=128),
]

# A tree kept until it holds more than half of the arena.  Host noise: tests/test_host_flag_matrix.py replays these
# cases in the oracle and asserts what the capacities were chosen for -- trees kept and cleared, a tree kept at exactly
# node_cap / 2 nodes, one of a game's two trees cleared and the other kept, and searches after a clear that look up
# positions the cleared tree held.
RECYCLE_CASES: List[FlagCase] = [
    # batch 1 on an open board: every descent adds one node, so the tree holds 12, 24, 12, ... nodes at the advances
    FlagCase("recycle_mnk9_5_b1", (9, 5), G=4, count=12, batch=1, max_batch=8, plies=(0, 4, 8), moves=5, seed=701,
             recycle_tree=True, node_capacity=24),
    FlagCase("recycle_c4_tpg2_odd", C4, G=8, count=5, batch=8, max_batch=8, plies=(0, 4, 8), moves=6, seed=702,
             trees_per_game=2, recycle_tree=True, node_capacity=25),
    FlagCase("recycle_mnk5_4_b16", (5, 4), G=6, count=4, batch=16, max_batch=16, plies=(0, 3), moves=5, seed=703,
             recycle_tree=True, node_capacity=61),
]

# The benchmark's virtual-loss row through its own path: Connect4, two play_multi parts, batch 8, the bf16 tower,
# virtual loss and masked priors, Philox noise; lean_tree puts its expand + back-up on the eight-lane kernel.
PIPELINE_CASE = FlagCase("pipeline_vl_mask_c4", C4, G=64, count=40, batch=8, max_batch=8, plies=(0,), moves=2, seed=800,
                         noise="philox", virtual_loss=True, mask_priors=True, parts=2, node_capacity=1024)

FLAG_CASES: List[FlagCase] = MASK_CASES + MASK_VL_CASES + FRESH_CASES + RECYCLE_CASES


# ------------------------------------------------------------------------------------------------ dispatch
def apad(A: int) -> int:
    return (A + 7) & ~7  # Dims::Apad, engine.cu fill_dims


def expand_instance(case: Case, lean_tree: bool) -> str:
    """caro_engine_expand_backup, engine.cu:463-471 (CARO_EXPAND_GROUP8 unset: "auto")."""
    if case.batch <= 8 and apad(case.A) <= 8 and case.connect4 and (lean_tree or case.G >= 32768):
        return "expand_backup_group8_kernel<C4Rules>"
    width = 8 if case.batch <= 8 else 16 if case.batch <= 16 else 32
    return "expand_backup_kernel<%s,%d>" % ("C4Rules" if case.connect4 else "MnkRules", width)


def flag_instances(case: FlagCase) -> dict:
    """search_matrix.instances with the expand instance of the path the case runs: launch by launch through the C ABI
    (lean_tree off), or play_multi over `parts` engines (lean_tree on from two parts); "expand_stepped" is the twin
    engines' instance of a pipeline case."""
    inst = dict(instances(case))
    inst["expand"] = expand_instance(case, lean_tree=case.parts >= 2)
    if case.parts >= 2:
        inst["expand_stepped"] = expand_instance(case, lean_tree=False)
    inst["advance"] = "advance_kernel<%s>" % ("C4Rules" if case.connect4 else "MnkRules")
    return inst
