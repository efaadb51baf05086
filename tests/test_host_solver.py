"""The MCTS solver extension without a GPU: the host restatement's proofs are exact game values, and the C ABI, header
and CLI surfaces agree."""
import ctypes as C
import os
import re
import zlib

import numpy as np
import pytest

from caro_oracle import CaroOracle
from conftest import ROOT
from harness import random_position
from oracle.games import ConnectFourOracle, MNKOracle
from solver_reference import DRAW, LOSS, UNKNOWN, WIN, Negamax, SolverOracleTree, node_status, pi_weights


def solve_from(og, state, who, rng, batch=8, max_minibatches=400):
    """Searches one root with the solver until the root is proven or the budget is spent; returns the tree."""
    tree = SolverOracleTree(og)
    for _ in range(max_minibatches):
        tree.minibatch(batch, state, who, rng.dirichlet([0.3] * og.action_space, size=batch))
        if tree.status(state) != UNKNOWN:
            break
    return tree


def check_proofs(og, tree, who_of):
    """Every proven edge of `tree` equals exact negamax; returns the number of proven edges."""
    nm = Negamax(og)
    proven = 0
    for s, row in tree.proof.items():
        who = who_of[s]
        for a, st in enumerate(row):
            if st != UNKNOWN:
                assert st == nm.edge_status(s, a, who), (s, a, st)
                proven += 1
    return proven


def movers(tree, og, state, who):
    """Side to move at every node of the tree, found by walking it from the root."""
    out, todo = {state: who}, [(state, who)]
    while todo:
        s, w = todo.pop()
        for a in og.possible_moves(s):
            c, won = og.move(s, a, w)
            if c in tree.proof and c not in out and not won:
                out[c] = 1 - w
                todo.append((c, 1 - w))
    return out


CASES = [("mnk3_3", lambda: MNKOracle(3, 3), (2, 3, 4, 5, 6), 6),
         ("c4", ConnectFourOracle, (28, 30, 32), 4),
         ("mnk5_4", lambda: MNKOracle(5, 4), (13, 15), 4),
         ("caro7_5", lambda: CaroOracle(7, 5), (37, 39), 3)]


@pytest.mark.parametrize("name,make,plies,roots", CASES, ids=[c[0] for c in CASES])
def test_oracle_proofs_are_exact(name, make, plies, roots):
    og = make()
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    total = 0
    for i in range(roots):
        state, who = random_position(og, rng, plies[i % len(plies)])
        tree = solve_from(og, state, who, rng, max_minibatches=60)
        total += check_proofs(og, tree, movers(tree, og, state, who))
    assert total > 0, "%s: nothing proven" % name


def test_proofs_from_the_empty_3x3_board_are_exact():
    """From the empty board the solver proves many edges, every one of them exact, but 1,600 descents do not prove the
    root a draw: a DRAW root needs every edge proven, and PUCT leaves low-prior edges unvisited."""
    og = MNKOracle(3, 3)
    tree = solve_from(og, og.initial_state, 0, np.random.default_rng(7), batch=8, max_minibatches=200)
    assert check_proofs(og, tree, movers(tree, og, og.initial_state, 0)) > 20
    assert tree.stopped > 0
    pi, _ = tree.get_policy_value(og.initial_state, tau=1)
    assert abs(sum(pi) - 1.0) < 1e-12


def test_node_status_and_policy_rules():
    assert node_status([WIN, LOSS, UNKNOWN], [0, 1, 2]) == WIN
    assert node_status([LOSS, LOSS, WIN], [0, 1]) == LOSS
    assert node_status([LOSS, DRAW, UNKNOWN], [0, 1]) == DRAW
    assert node_status([LOSS, DRAW, UNKNOWN], [0, 1, 2]) == UNKNOWN
    assert node_status([LOSS, LOSS], [0, 1]) == LOSS
    assert node_status([UNKNOWN, UNKNOWN], [0, 1]) == UNKNOWN
    assert pi_weights([5, 3, 2], [LOSS, UNKNOWN, DRAW]) == [0, 3, 2]
    assert pi_weights([5, 0, 0], [LOSS, UNKNOWN, UNKNOWN]) == [5, 0, 0]  # nothing left: the counts stay


def test_header_and_ctypes_agree_on_set_solver():
    from caro_ai_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "caro_b200.h")).read()
    assert re.search(r"int caro_engine_set_solver\(caro_engine\* e, int players, void\* stream\);", header)
    for region in ("solver_params", "solver_counters"):
        assert '"%s"' % region in header
    res, args = _cabi._SIGNATURES["caro_engine_set_solver"]
    assert res is C.c_int and args == [C.c_void_p, C.c_int, C.c_void_p]
    lib = _cabi.lib()
    assert lib.caro_engine_set_solver(None, 3, None) == -1 and b"null engine" in lib.caro_last_error()
    assert "CARO_FLAG_SOLVER" not in header


def test_cli_solver_option_is_off_by_default():
    from caro_ai_b200 import train
    assert train.parse_args(["-n", "x", "-g", "0"]).solver is False
    assert train.parse_args(["-n", "x", "-g", "0", "--solver"]).solver is True
    import argparse
    import caro_ai_b200.play as play
    seen = {}

    def fake_parse(self, argv=None, namespace=None):
        seen["actions"] = {a.dest: a.default for a in self._actions}
        raise SystemExit(0)
    orig = argparse.ArgumentParser.parse_args
    argparse.ArgumentParser.parse_args = fake_parse
    try:
        with pytest.raises(SystemExit):
            play.main(["a", "b", "-g", "0"])
    finally:
        argparse.ArgumentParser.parse_args = orig
    assert seen["actions"]["solver"] is False
