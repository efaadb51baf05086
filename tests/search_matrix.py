"""The search-kernel matrix: which positions, batch widths, noise sources and tree layouts the bit-exact parity tests
run, which template instance of the tree kernels each case reaches (restated from csrc/engine.cu), and the oracle side
of the virtual-loss extension.  Shared by tests/test_gpu_search_matrix.py (GPU) and tests/test_host_search_matrix.py.

Dispatch restated from caro-ai_b200/csrc/engine.cu (a change there has to be mirrored here, and the host test then
says which instance lost its case):
  * launch_select, engine.cu:188-234 -- Philox noise_kernel<GW, APL> by the action count A; select by A: <= 8 the
    thread-per-descent kernel (ROWV 2; its dense twin only above 128 * 5 * 148 descents per launch), <= 16 the
    thread-per-descent kernel (ROWV 4, m,n,k only), then select_kernel<R, 32, APL> with APL = 1, 2, 4, 8 up to 32, 64,
    128 and beyond; with CARO_FLAG_VIRTUAL_LOSS select_vl_group_kernel for A <= 8 and select_vl_kernel above;
  * caro_engine_plan, engine.cu:407-423 -- plan_kernel<Board, GP> with GP = 8, 16, 32 by the minibatch's batch;
  * caro_engine_expand_backup, engine.cu:425-446 -- expand_backup_kernel<R, BK> with BK = 8, 16, 32 by the batch
    (Connect4 at batch <= 8 takes the eight-lane kernel inside the parts pipeline or from 32,768 games on).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Tuple

import numpy as np

from harness import StubOracleTree, oracle_for, random_position
from oracle.stubs import chain_priors, stub_priors

STUBS = {"hash": stub_priors, "chain": chain_priors}


@dataclass(frozen=True)
class Case:
    name: str
    board: Tuple[int, int]       # (n, k) of an m,n,k game, or (0, 0) for Connect4
    G: int
    count: int                   # minibatches per move
    batch: int
    max_batch: int
    plies: Tuple[int, ...]       # random plies of the root positions (game g gets plies[g % len])
    moves: int
    seed: int
    trees_per_game: int = 1
    noise: str = "host"          # "host": np.random.dirichlet injected; "philox": the device's own stream
    tau_plies: int = 1
    stub: str = "hash"
    virtual_loss: bool = False
    min_path: int = 0            # the longest back-up path must exceed this (chain cases)

    @property
    def connect4(self) -> bool:
        return self.board == (0, 0)

    @property
    def A(self) -> int:
        return 7 if self.connect4 else self.board[0] ** 2

    def product_game(self):
        from caro_ai_b200.game import ConnectFour, TicTacToe
        return ConnectFour() if self.connect4 else TicTacToe(*self.board)

    def oracle_game(self):
        from oracle.games import ConnectFourOracle, MNKOracle
        return ConnectFourOracle() if self.connect4 else MNKOracle(*self.board)


C4 = (0, 0)
# Root plies mix empty boards, mid-game positions and (on boards small enough to fill at random without a finished
# line) positions with one to three legal moves left, so that wins and draws occur inside the searches.
PARITY_CASES: List[Case] = [
    Case("mnk2_2", (2, 2), G=16, count=6, batch=8, max_batch=8, plies=(0, 1, 2), moves=3, seed=101, noise="philox"),
    Case("mnk3_3_b1", (3, 3), G=24, count=12, batch=1, max_batch=8, plies=(0, 2, 4, 6, 7, 8), moves=3, seed=102),
    Case("mnk3_3_b32", (3, 3), G=16, count=5, batch=32, max_batch=32, plies=(0, 1, 3, 5, 6, 7), moves=3, seed=103,
         noise="philox", tau_plies=2),
    Case("mnk4_4", (4, 4), G=16, count=8, batch=16, max_batch=32, plies=(0, 3, 8, 13, 14, 15), moves=3, seed=104,
         noise="philox"),
    Case("mnk5_4_tpg2", (5, 4), G=8, count=8, batch=9, max_batch=16, plies=(0, 6, 12, 18), moves=3, seed=105,
         trees_per_game=2, noise="philox"),
    Case("mnk6_5", (6, 5), G=8, count=6, batch=31, max_batch=32, plies=(0, 10, 20), moves=2, seed=106, noise="philox"),
    Case("mnk8_5", (8, 5), G=8, count=10, batch=3, max_batch=8, plies=(0, 16, 32), moves=2, seed=107),
    Case("mnk9_5_tpg2", (9, 5), G=6, count=6, batch=17, max_batch=32, plies=(0, 20, 40), moves=3, seed=108,
         trees_per_game=2, noise="philox"),
    Case("mnk11_5", (11, 5), G=6, count=10, batch=8, max_batch=8, plies=(0, 30, 60), moves=3, seed=109, tau_plies=2),
    Case("mnk12_5", (12, 5), G=4, count=5, batch=32, max_batch=32, plies=(0, 40, 80), moves=2, seed=110, noise="philox"),
    Case("mnk15_5", (15, 5), G=4, count=6, batch=16, max_batch=16, plies=(0, 50, 100), moves=2, seed=111),
    Case("c4_b32", C4, G=16, count=5, batch=32, max_batch=32, plies=(0, 10, 24, 36, 38), moves=3, seed=112, noise="philox"),
    Case("c4_b17_tpg2", C4, G=8, count=6, batch=17, max_batch=32, plies=(0, 20, 36), moves=4, seed=113, trees_per_game=2,
         tau_plies=2),
]

# Deep paths: the chain stub on boards where no line can end the game early (k = n) and on Connect4 from the empty
# board.  The counts are what the CPU oracle needs to pass the depths (tests/test_host_search_matrix.py).
CHAIN_CASES: List[Case] = [
    Case("chain_mnk9_9", (9, 9), G=2, count=140, batch=8, max_batch=8, plies=(0,), moves=1, seed=201, stub="chain",
         min_path=64),
    Case("chain_mnk12_12", (12, 12), G=2, count=80, batch=32, max_batch=32, plies=(0,), moves=1, seed=202,
         stub="chain", min_path=32),
    Case("chain_c4", C4, G=4, count=80, batch=16, max_batch=16, plies=(0,), moves=1, seed=203, stub="chain",
         min_path=32),
]

# Virtual loss (extension): select_vl_kernel on m,n,k boards, select_vl_group_kernel on Connect4, batch 8 and 32.
VL_CASES: List[Case] = [
    Case("vl_%s_b%d" % (tag, b), board, G=G, count=count, batch=b, max_batch=b, plies=plies, moves=2, seed=300 + i,
         virtual_loss=True, noise="philox" if b == 32 else "host")
    for i, (tag, board, G, count, plies) in enumerate([("mnk3_3", (3, 3), 16, 8, (0, 2, 5, 7)),
                                                        ("mnk5_4", (5, 4), 8, 8, (0, 6, 14)),
                                                        ("mnk9_5", (9, 5), 4, 6, (0, 20, 40)),
                                                        ("c4", C4, 12, 6, (0, 12, 30))])
    for b in (8, 32)
]

ALL_CASES = PARITY_CASES + CHAIN_CASES + VL_CASES

# Philox noise for every noise-kernel width (part of tests/test_gpu_search_matrix.py): board side for each action count
NOISE_BOARDS = [2, 3, 4, 5, 6, 8, 9, 11, 12, 15]


# ------------------------------------------------------------------------------------------------ dispatch
def noise_instance(A: int) -> str:
    """launch_select's Philox branch (engine.cu:200-206)."""
    gw, apl = (8, 1) if A <= 8 else (16, 1) if A <= 16 else (32, 1) if A <= 32 else (32, 2) if A <= 64 else \
        (32, 4) if A <= 128 else (32, 8)
    return "noise_kernel<%d,%d>" % (gw, apl)


def instances(case: Case) -> dict:
    """The kernel instance each launch of `case` reaches."""
    A, R = case.A, ("C4Rules" if case.connect4 else "MnkRules")
    descents = case.G * case.batch
    assert descents <= 128 * 5 * 148, "would take the dense thread-per-descent select kernel"
    if case.virtual_loss:
        select = "select_vl_group_kernel<%s>" % R if A <= 8 else "select_vl_kernel<%s>" % R  # engine.cu:213-218
    elif A <= 8:
        select = "select_thread_kernel<%s,2>" % R                                            # engine.cu:224
    elif A <= 16:
        select = "select_thread_kernel<%s,4>" % R                                            # engine.cu:226
    else:
        select = "select_kernel<%s,32,%d>" % (R, 1 if A <= 32 else 2 if A <= 64 else 4 if A <= 128 else 8)
    width = 8 if case.batch <= 8 else 16 if case.batch <= 16 else 32                           # engine.cu:418-420, 441-443
    assert not (case.connect4 and case.batch <= 8 and case.G >= 32768), "would take the eight-lane expand kernel"
    board = "C4Board" if case.connect4 else "MnkBoard"
    return {"select": select, "noise": noise_instance(A) if case.noise == "philox" else None,
            "plan": "plan_kernel<%s,%d>" % (board, width), "expand": "expand_backup_kernel<%s,%d>" % (R, width)}


# ------------------------------------------------------------------------------------------------ oracle side
def make_tree(case: Case, og):
    stub = STUBS[case.stub]
    return VirtualLossOracleTree(og, stub=stub) if case.virtual_loss else StubOracleTree(og, stub=stub)


def make_roots(case: Case, og, rng):
    return [random_position(og, rng, int(case.plies[i % len(case.plies)])) for i in range(case.G)]


def host_noise(case: Case, rng):
    return rng.dirichlet([0.3] * case.A, size=(case.G, case.batch))


def oracle_first_move(case: Case):
    """The oracle half of the first move of `case` with host noise, consuming the seed's stream in the order the GPU
    runner does.  Returns (trees, longest path in edges)."""
    assert case.noise == "host"
    og = case.oracle_game()
    rng = np.random.default_rng(case.seed)
    roots = make_roots(case, og, rng)
    trees = [[make_tree(case, og) for _ in range(case.trees_per_game)] for _ in range(case.G)]
    longest = 0
    for t in (t for row in trees for t in row):
        t.trace = []
    for _ in range(case.count):
        noise = host_noise(case, rng)
        for g in range(case.G):
            (state, who) = roots[g]
            trees[g][who if case.trees_per_game == 2 else 0].minibatch(case.batch, state, who, noise[g])
    for t in (t for row in trees for t in row):
        for mb in t.trace:
            longest = max([longest] + [len(d[4]) for d in mb["descents"]])
    return trees, longest


class VirtualLossOracleTree(StubOracleTree):
    """Restates select_vl_kernel (csrc/engine_kernels.cuh:455-550), the virtual-loss extension: the descents of a
    minibatch are made one after the other, and descent j scores an edge (s, a) at depth d that k earlier descents
    of the minibatch took at depth d as if it had k more visits that all lost: n = N + k, w = f32(W - k), and sum N
    includes the k's.  The root keeps float64 P' and U, but its Q is f32(w / n) for every visited edge (there is no
    python-float branch); interior scores are float32; ties go to the lowest action.  Plan, expansion and back-up are
    the reference's (OracleMCTS.search_minibatch)."""

    def search_minibatch(self, batch_size, state_int, player, net, device="cpu"):
        self._paths = []
        super().search_minibatch(batch_size, state_int, player, net, device)

    def virtual_visits(self, s, depth):
        k = [0] * self.game.action_space
        for states, actions in self._paths:
            if len(states) > depth and states[depth] == s:
                k[actions[depth]] += 1
        return k

    def vl_scores(self, s, depth, k, z=None):
        """PUCT scores of every action of node `s` with virtual visits `k` (-inf for illegal moves); `z` is the
        descent's Dirichlet vector at the root (depth 0)."""
        n_row, w_row, p_row = self.visit_count[s], self.value[s], self.probs[s]
        sum_n = sum(n_row) + sum(k)
        illegal = set(self.game.invalid_moves(s))
        c_f, keep_f = np.float32(self.c_puct), np.float32(1.0 - self.explore)
        sq64, sq32 = math.sqrt(sum_n), np.sqrt(np.float32(sum_n))
        out = []
        for a in range(self.game.action_space):
            if a in illegal:
                out.append(-math.inf)
                continue
            n = n_row[a] + k[a]
            w = np.float32(w_row[a]) - np.float32(k[a])
            p = np.float32(p_row[a])
            q = w / np.float32(n) if n > 0 else np.float32(0.0)
            if depth == 0:
                pn = float(keep_f * p) + self.explore * float(z[a])
                out.append(float(q) + self.c_puct * pn * sq64 / (1 + n))
            else:
                t = (c_f * p * sq32) / np.float32(1 + n)
                out.append(float(q + t))
        return out

    def find_leaf(self, state_int, player):
        path_states, path_actions = [], []
        s, who, value = state_int, player, None
        while s in self.probs:
            depth = len(path_states)
            path_states.append(s)
            z = self.dirichlet([self.alpha] * self.game.action_space) if depth == 0 else None
            scores = self.vl_scores(s, depth, self.virtual_visits(s, depth), z)
            a = int(np.argmax(scores))  # first maximum
            path_actions.append(a)
            s, won = self.game.move(s, a, who)
            if won:
                value = -1.0
            who = 1 - who
            if value is None and len(self.game.possible_moves(s)) == 0:
                value = 0.0
            if value is not None:
                break
        self._paths.append((path_states, path_actions))
        return value, s, who, path_states, path_actions
