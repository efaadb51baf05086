"""Caro test material shared by tests/test_host_caro.py (CPU) and tests/test_gpu_caro.py (B200): a table of hand-built
positions, root positions constructed so that a search meets both a both-ends-blocked run and a win, and the search
cases (tests/search_matrix.py's Case on the Caro rule)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, NamedTuple, Tuple

import numpy as np

from caro_oracle import CaroOracle
from harness import random_position
from oracle.games import MNKOracle
from search_matrix import Case

EMPTY = 2


# ------------------------------------------------------------------------------------------------ hand-built table
class Position(NamedTuple):
    name: str
    n: int
    k: int
    lines: Tuple[Tuple[int, int, int, int, str], ...]  # (row, col, dr, dc, pattern): pattern from (row, col) on
    caro_wins: bool
    freestyle_wins: bool


def build(pos: Position, mover: int):
    """(state int, move, mover) of `pos`.  Pattern characters: 'x' mover, 'o' opponent, '.' empty, '*' the move
    (empty before it); every cell no pattern names is empty."""
    n = pos.n
    d = [EMPTY] * (n * n)
    move = None
    for r, c, dr, dc, pattern in pos.lines:
        for i, ch in enumerate(pattern):
            rr, cc = r + i * dr, c + i * dc
            assert 0 <= rr < n and 0 <= cc < n, (pos.name, rr, cc)
            cell = {"x": mover, "o": 1 - mover, ".": EMPTY, "*": EMPTY}[ch]
            assert d[rr * n + cc] in (EMPTY, cell), (pos.name, rr, cc)
            d[rr * n + cc] = cell
            if ch == "*":
                move = rr * n + cc
    assert move is not None, pos.name
    return MNKOracle._from_digits(d), move, mover


H, V, D, AD = (0, 1), (1, 0), (1, 1), (-1, 1)  # row, column, diagonal, anti-diagonal
TABLE: List[Position] = [
    Position("open_five", 15, 5, ((7, 3) + H + (".xx*xx.",),), True, True),
    Position("five_blocked_one_end", 15, 5, ((7, 3) + H + ("oxx*xx.",),), True, True),
    Position("five_blocked_both_ends", 15, 5, ((7, 3) + H + ("oxx*xxo",),), False, True),
    Position("five_blocked_both_ends_column", 15, 5, ((2, 9) + V + ("oxxxx*o",),), False, True),
    Position("five_blocked_both_ends_diagonal", 15, 5, ((4, 4) + D + ("ox*xxxo",),), False, True),
    Position("five_blocked_both_ends_anti_diagonal", 15, 5, ((12, 1) + AD + ("o*xxxxo",),), False, True),
    Position("edge_and_opponent", 15, 5, ((4, 0) + H + ("xx*xxo",),), True, True),
    Position("edge_and_opponent_diagonal", 15, 5, ((10, 10) + D + ("xx*xx",), (9, 9) + D + ("o",)), True, True),
    Position("edge_at_both_ends_k_eq_n", 5, 5, ((2, 0) + H + ("xx*xx",),), True, True),
    Position("edge_at_both_ends_k_eq_n_anti_diagonal", 7, 7, ((6, 0) + AD + ("xxx*xxx",),), True, True),
    Position("overline_blocked_both_ends", 15, 5, ((7, 2) + H + ("oxxx*xxxo",),), False, True),
    Position("overline_blocked_one_end", 15, 5, ((7, 2) + H + ("oxxx*xxx.",),), True, True),
    Position("join_into_blocked_nine", 15, 5, ((6, 2) + H + ("oxxxx*xxxxo",),), False, True),
    # unreachable in play (a run of k already on the board) but accepted by caro_boards_apply: a ray walk capped at
    # k - 1 cells stops inside the six and misses the blocker
    Position("join_into_blocked_nine_long_side", 15, 5, ((6, 1) + H + ("oxx*xxxxxxo",),), False, True),
    Position("join_into_open_nine_long_side", 15, 5, ((6, 1) + H + ("oxx*xxxxxx.",),), True, True),
    Position("blocked_row_winning_column", 15, 5, ((7, 3) + H + ("oxx*xxo",), (5, 6) + V + ("xx",), (8, 6) + V + ("xx.",)),
             True, True),
    Position("blocked_row_winning_anti_diagonal", 15, 5,
             ((7, 3) + H + ("oxx*xxo",), (9, 4) + AD + ("xx",), (6, 7) + AD + ("xx",)), True, True),
    Position("blocked_row_and_column", 15, 5, ((7, 3) + H + ("oxx*xxo",), (2, 6) + V + ("oxxxx",), (8, 6) + V + ("o",)),
             False, True),
    Position("empty_gap_is_no_block", 15, 5, ((7, 3) + H + ("oxx*xx.o",),), True, True),
    Position("four_blocked_both_ends_no_run", 15, 5, ((7, 3) + H + ("ox*xxo",),), False, False),
    Position("k2_blocked_both_ends", 4, 2, ((1, 0) + H + ("o*xo",),), False, True),
    Position("k2_edge_and_opponent", 4, 2, ((1, 0) + H + ("*xo.",),), True, True),
    Position("k2_diagonal_blocked_both_ends", 4, 2, ((0, 0) + D + ("ox*o",),), False, True),
    Position("k2_board_2", 2, 2, ((0, 0) + H + ("*x",),), True, True),
    Position("k_eq_n_15", 15, 15, ((14, 0) + H + ("xxxxxxx*xxxxxxx",),), True, True),
    Position("k3_blocked_both_ends", 5, 3, ((4, 0) + H + ("ox*xo",),), False, True),
    Position("k3_blocked_both_ends_one_direction_open_other", 5, 3, ((4, 0) + H + ("ox*xo",), (2, 2) + V + ("xx",)),
             True, True),
]


# ------------------------------------------------------------------------------------------------ constructed roots
DIRECTIONS = (H, V, D, AD)


def _segment(n, rng, length):
    """Cells of a random straight segment of `length` cells that fits an n x n board, or None."""
    for _ in range(50):
        dr, dc = DIRECTIONS[int(rng.integers(4))]
        r, c = int(rng.integers(n)), int(rng.integers(n))
        cells = [(r + i * dr, c + i * dc) for i in range(length)]
        if all(0 <= rr < n and 0 <= cc < n for rr, cc in cells):
            return [rr * n + cc for rr, cc in cells]
    return None


def blocked_and_winning_root(og: CaroOracle, rng, empties: int):
    """(state, mover, blocked_move, winning_move): a random dense board with `empties` empty cells on which the mover
    has a move that completes a run of k with opponent stones past both ends (it does not win under Caro, it would
    under freestyle) and a move that wins under Caro."""
    n, k = og.board_len, og.k_to_win
    assert n >= k + 2, "no run of k fits between two opponent stones"
    free = MNKOracle(n, k)
    while True:
        who = int(rng.integers(2))
        d = [int(v) for v in rng.integers(0, 2, n * n)]
        blocked = _segment(n, rng, k + 2)
        win = _segment(n, rng, k)
        if blocked is None or win is None or set(blocked) & set(win):
            continue
        for cell, v in zip(blocked, [1 - who] + [who] * k + [1 - who]):
            d[cell] = v
        for cell in win:
            d[cell] = who
        b_move, w_move = blocked[1 + int(rng.integers(k))], win[int(rng.integers(k))]
        d[b_move] = d[w_move] = EMPTY
        others = [i for i in range(n * n) if d[i] != EMPTY and i not in blocked and i not in win]
        for i in rng.choice(others, size=max(0, empties - 2), replace=False):
            d[int(i)] = EMPTY
        s = MNKOracle._from_digits(d)
        if og.move(s, b_move, who)[1] or not free.move(s, b_move, who)[1] or not og.move(s, w_move, who)[1]:
            continue
        return s, who, b_move, w_move


def blocked_gap_opening(og: CaroOracle, rng, segments: int):
    """A sparse opening with `segments` lines "o x..x _ x..x o" (k - 1 stones of one side around an empty gap, an
    opponent stone past both ends; the sides alternate), every gap a move that completes a run of k blocked at both
    ends.  Self-play from it goes through such moves often, which play from the empty board rarely does."""
    n, k = og.board_len, og.k_to_win
    free = MNKOracle(n, k)
    while True:
        d = [EMPTY] * (n * n)
        gaps = []
        for i in range(segments):
            who = i % 2
            cells = _segment(n, rng, k + 2)
            if cells is None or any(d[c] != EMPTY for c in cells):
                break
            gap = cells[1 + int(rng.integers(k))]
            for cell, v in zip(cells, [1 - who] + [who] * k + [1 - who]):
                d[cell] = v
            d[gap] = EMPTY
            gaps.append((gap, who))
        if len(gaps) < segments:
            continue
        s = MNKOracle._from_digits(d)
        if all(not og.move(s, g, who)[1] and free.move(s, g, who)[1] for g, who in gaps):
            return s


# ------------------------------------------------------------------------------------------------ search cases
@dataclass(frozen=True)
class CaroCase(Case):
    """A search-matrix case on the Caro rule.  Root positions are constructed (blocked_and_winning_root) with
    `plies[g % len]` empty cells, except on boards where no run of k fits between two opponent stones (n < k + 2:
    every line of the board is at most k + 1 cells long, so the rule cannot differ from freestyle); those take
    random positions after `plies` random moves like the freestyle matrix."""

    @property
    def blocks_possible(self) -> bool:
        return self.board[0] >= self.board[1] + 2

    def product_game(self):
        from caro_ai_b200.game import Caro
        return Caro(*self.board)

    def oracle_game(self):
        return CaroOracle(*self.board)


def make_caro_roots(case: CaroCase, og, rng):
    """[(state, mover)] of the case's games, drawn from `rng` (the GPU runner and the host check draw them alike)."""
    roots = []
    for g in range(case.G):
        p = int(case.plies[g % len(case.plies)])
        if case.blocks_possible:
            s, who, _, _ = blocked_and_winning_root(og, rng, p)
            roots.append((s, who))
        else:
            roots.append(random_position(og, rng, p))
    return roots


CARO_CASES: List[CaroCase] = [
    CaroCase("caro2_2", (2, 2), G=16, count=6, batch=8, max_batch=8, plies=(0, 1, 2), moves=3, seed=401, noise="philox"),
    CaroCase("caro3_3_b1", (3, 3), G=16, count=12, batch=1, max_batch=8, plies=(2, 4, 6, 7), moves=3, seed=402),
    CaroCase("caro4_2_b16", (4, 2), G=16, count=8, batch=16, max_batch=32, plies=(3, 4, 6), moves=3, seed=403,
             noise="philox"),
    CaroCase("caro5_3_tpg2", (5, 3), G=8, count=8, batch=9, max_batch=16, plies=(4, 6, 8), moves=3, seed=404,
             trees_per_game=2, noise="philox"),
    CaroCase("caro7_5_b31", (7, 5), G=8, count=6, batch=31, max_batch=32, plies=(5, 8), moves=2, seed=405, noise="philox"),
    CaroCase("caro8_5_b3", (8, 5), G=8, count=12, batch=3, max_batch=8, plies=(4, 6), moves=2, seed=406),
    CaroCase("caro9_5_tpg2", (9, 5), G=6, count=6, batch=17, max_batch=32, plies=(5, 7), moves=3, seed=407,
             trees_per_game=2),
    CaroCase("caro11_5_b8", (11, 5), G=6, count=10, batch=8, max_batch=8, plies=(4, 6), moves=2, seed=408,
             noise="philox", tau_plies=2),
    CaroCase("caro12_5_tpg2", (12, 5), G=4, count=6, batch=16, max_batch=16, plies=(5, 7), moves=2, seed=409,
             trees_per_game=2, noise="philox"),
    CaroCase("caro15_5_b32", (15, 5), G=4, count=5, batch=32, max_batch=32, plies=(6, 8), moves=2, seed=410),
    CaroCase("vl_caro6_4_b8", (6, 4), G=8, count=8, batch=8, max_batch=8, plies=(4, 6), moves=2, seed=411,
             virtual_loss=True),
]


# ------------------------------------------------------------------------------------------------ what a search met
def rule_events(og: CaroOracle, trees_and_roots):
    """(blocked, blocked_next_to_win) over oracle trees that recorded their descents (tree.trace = []):
    `blocked` counts descent steps that played a move completing a run of k blocked at both ends (the game went on);
    `blocked_next_to_win` counts tree nodes where one visited edge is such a move and another visited edge wins."""
    free = MNKOracle(og.board_len, og.k_to_win)
    blocked_steps = 0
    node_kinds = {}
    for tree, _ in trees_and_roots:
        for mb in tree.trace:
            for _value, _leaf, _leaf_player, states, actions in mb["descents"]:
                leaf_who = _leaf_player
                depth = len(states)
                for i, (s, a) in enumerate(zip(states, actions)):
                    who = leaf_who if (depth - i) % 2 == 0 else 1 - leaf_who
                    won = og.move(s, a, who)[1]
                    is_blocked = not won and free.move(s, a, who)[1]
                    blocked_steps += is_blocked
                    kinds = node_kinds.setdefault((id(tree), s), set())
                    kinds.add("win" if won else "blocked" if is_blocked else "other")
    both = sum(1 for kinds in node_kinds.values() if {"win", "blocked"} <= kinds)
    return blocked_steps, both
