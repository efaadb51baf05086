"""Oracle (CPU, test-only) of Caro: the m,n,k board where a run blocked at both ends does not win.

Caro (Vietnamese gomoku) keeps MNKOracle's board, state integers, planes, actions, render and draw rule; only the win
test of `move` differs.  A move of player p into cell c wins iff in at least one of the four full lines through c (row,
column, diagonal, anti-diagonal, as MNKOracle._lines_through collects them)

  1. the maximal run of p's stones that contains c is at least k long (overlines count), and
  2. that run is not blocked at both ends: an end is blocked when the cell just past it is on the board and holds an
     opponent stone.  The board edge never blocks (Caro is played on an unbounded grid).

The rule is restated here from the full lines, not from the kernel's ray walk (csrc/rules.cuh).
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

from oracle.games import MNKOracle


class CaroOracle(MNKOracle):
    """Caro(n, k): MNKOracle with the both-ends-blocked rule."""

    def _positions_in_lines(self, row: int, col: int) -> List[int]:
        """Index of (row, col) inside each of the four lines of _lines_through, in the same order."""
        n = self.board_len
        return [col, row, min(row, col), min(n - 1 - row, col)]

    def _line_wins(self, line: Sequence[int], at: int, player: int) -> bool:
        """Does the maximal run of `player` through line[at] reach k without an opponent stone at both ends?"""
        lo = at
        while lo > 0 and line[lo - 1] == player:
            lo -= 1
        hi = at
        while hi < len(line) - 1 and line[hi + 1] == player:
            hi += 1
        if hi - lo + 1 < self.k_to_win:
            return False
        opponent = 1 - player
        blocked_lo = lo > 0 and line[lo - 1] == opponent
        blocked_hi = hi < len(line) - 1 and line[hi + 1] == opponent
        return not (blocked_lo and blocked_hi)

    def move(self, state: int, move: int, player: int) -> Tuple[int, bool]:
        """MNKOracle.move with the Caro win test; the target cell is overwritten without an emptiness check."""
        assert player == self.player_white or player == self.player_black
        assert 0 <= move < self.action_space
        d = self._digits(state)
        row, col = divmod(int(move), self.board_len)
        d[row * self.board_len + col] = int(player)
        lines = self._lines_through(d, row, col)
        won = any(self._line_wins(line, at, player) for line, at in zip(lines, self._positions_in_lines(row, col)))
        return self._from_digits(d), won
