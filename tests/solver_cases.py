"""Search roots for the solver's parity tests: the matrix cases of tests/search_matrix.py, with late-game roots on the
boards where random play rarely leaves a position close to its end without a finished line."""
from __future__ import annotations

import dataclasses

import numpy as np

from search_matrix import CHAIN_CASES, PARITY_CASES, make_roots

LATE_EMPTIES = (2, 3, 4, 5)


def late_position(og, rng, empties, threat):
    """An n x n board tiled so that no line is longer than two stones, with `empties` random cells left empty.
    threat 0: nothing else (every game from it is a draw at full board); 1 / 2: the first k - 1 cells of the top row hold
    the stones of the player not to move / to move and the k-th is empty, so the mover must block there / wins there."""
    n, k = og.board_len, og.k_to_win
    digits = [((c // 2) + r) % 2 for r in range(n) for c in range(n)]
    for cell in rng.choice(n * n, size=empties, replace=False):
        digits[int(cell)] = og.empty
    who = int(rng.integers(2))
    if threat:
        owner = 1 - who if threat == 1 else who
        for c in range(k - 1):
            digits[c] = owner
        digits[k - 1] = og.empty
    return og._from_digits(digits), who


def solver_roots(case, og, rng):
    """The matrix case's roots (Connect4 and boards up to 4 x 4 already end inside the searches), late roots on larger
    boards."""
    if case.connect4 or case.A <= 16 or case.stub == "chain":
        return make_roots(case, og, rng)
    return [late_position(og, rng, LATE_EMPTIES[g % len(LATE_EMPTIES)], g % 3) for g in range(case.G)]


SOLVER_PARITY_CASES = [dataclasses.replace(c, name="solver_" + c.name) for c in PARITY_CASES]
SOLVER_CHAIN_CASES = [dataclasses.replace(c, name="solver_" + c.name) for c in CHAIN_CASES]
