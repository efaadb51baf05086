"""Host restatement of the MCTS solver extension (include/caro_b200.h caro_engine_set_solver) and an exact negamax to
check its proofs against.

Edge status, for the side to move at the edge's node: UNKNOWN 0, WIN 1, LOSS 2, DRAW 3 (bits 29-30 of the engine's N
word).  A node's status is a pure function of its row and legality: WIN if a legal edge is WIN, LOSS if every legal edge
is LOSS, DRAW if every legal edge is proven, none WIN and one DRAW, else UNKNOWN.

SolverOracleTree is StubOracleTree with the solver on:
  * select: a descent that reaches a proven non-root node stops there as a terminal with value +1 / -1 / 0 for the
    node's mover; at a node with a WIN edge the lowest WIN edge is taken; LOSS edges are left out of the argmax unless
    every legal edge is LOSS; descents from a proven root are skipped (their noise vector is still consumed);
  * back-up: values as the reference's, then, in queue order, each terminal entry proves its last edge (leaf value -1:
    WIN, 0: DRAW, +1: LOSS) and walks up its path while the node above is proven, setting the next edge to the
    negated node status;
  * policy: a proven-WIN root gives pi one-hot on its lowest WIN edge whatever tau is; otherwise LOSS edges are zeroed
    in the visit counts before the reference's pi (renormalised; tau = 0: argmax over the rest), unless that leaves no
    visit at all, then the counts stay as they are.
"""
from __future__ import annotations

from typing import Dict, List

import numpy as np

from harness import StubOracleTree
from oracle.stubs import stub_priors

UNKNOWN, WIN, LOSS, DRAW = 0, 1, 2, 3
NEGATE = {WIN: LOSS, LOSS: WIN, DRAW: DRAW}
VALUE_OF = {WIN: 1.0, LOSS: -1.0, DRAW: 0.0}  # value of a proven node for its mover


def node_status(row, legal) -> int:
    st = [row[a] for a in legal]
    if any(x == WIN for x in st):
        return WIN
    if st and all(x == LOSS for x in st):
        return LOSS
    if st and all(x != UNKNOWN for x in st) and any(x == DRAW for x in st):
        return DRAW
    return UNKNOWN


def pi_weights(n_row, proof_row):
    """Visit counts the move and pi are drawn from at an unproven-WIN root: LOSS edges zeroed unless nothing is left."""
    w = [0 if proof_row[a] == LOSS else int(n) for a, n in enumerate(n_row)]
    return w if sum(w) > 0 else [int(n) for n in n_row]


class SolverOracleTree(StubOracleTree):
    def __init__(self, game, solver: bool = True, stub=stub_priors, **kw):
        super().__init__(game, stub=stub, **kw)
        self.solver = solver
        self.proof: Dict[int, List[int]] = {}
        self.stopped = 0        # descents stopped at a proven node
        self.proven_edges = 0   # edges that went from UNKNOWN to proven

    def clear(self):
        super().clear()
        self.proof.clear()

    def _new_node(self, state, prior_row):
        super()._new_node(state, prior_row)
        self.proof[state] = [UNKNOWN] * self.game.action_space

    def status(self, s) -> int:
        return node_status(self.proof[s], self.game.possible_moves(s)) if s in self.proof else UNKNOWN

    def find_leaf(self, state_int, player):
        if not self.solver:
            return super().find_leaf(state_int, player)
        path_states, path_actions = [], []
        s, who, value = state_int, player, None
        while s in self.probs:
            st = self.status(s)
            if st != UNKNOWN:
                if not path_states:  # proven root: the descent is skipped
                    self.dirichlet([self.alpha] * self.game.action_space)
                    return "skip", s, who, [], []
                self.stopped += 1
                return VALUE_OF[st], s, who, path_states, path_actions
            path_states.append(s)
            pri = self.probs[s]
            if s == state_int:
                pri = self._noisy(pri)
            scores = self._ucb(self.value_avg[s], pri, self.visit_count[s])
            legal = self.game.possible_moves(s)
            for a in self.game.invalid_moves(s):
                scores[a] = -np.inf
            row = self.proof[s]
            wins = [a for a in legal if row[a] == WIN]
            if wins:
                a = wins[0]
            else:
                if not all(row[a] == LOSS for a in legal):
                    for a in legal:
                        if row[a] == LOSS:
                            scores[a] = -np.inf
                a = int(np.argmax(scores))
            path_actions.append(a)
            s, won = self.game.move(s, a, who)
            if won:
                value = -1.0
            who = 1 - who
            if value is None and len(self.game.possible_moves(s)) == 0:
                value = 0.0
            if value is not None:
                break
        return value, s, who, path_states, path_actions

    def search_minibatch(self, batch_size, state_int, player, net, device="cpu"):
        """OracleMCTS.search_minibatch plus skipped descents and the proof pass."""
        backups, terminals = [], []
        todo_states, todo_players, todo_paths = [], [], []
        seen = set()
        leaves_dbg = []
        for _ in range(batch_size):
            value, leaf, leaf_player, states, actions = self.find_leaf(state_int, player)
            if self.trace is not None:
                leaves_dbg.append((value, leaf, leaf_player, list(states), list(actions)))
            if value == "skip":
                continue
            if value is not None:
                backups.append((value, states, actions))
                terminals.append((value, states, actions))
            elif leaf not in seen:
                seen.add(leaf)
                todo_states.append(leaf)
                todo_players.append(leaf_player)
                todo_paths.append((states, actions))
        if todo_states:
            pri, vals = self.evaluate(todo_states, todo_players, net, device)
            for leaf, (states, actions), v, p in zip(todo_states, todo_paths, vals, pri):
                self._new_node(leaf, p)
                backups.append((v, states, actions))
        for v, states, actions in backups:
            self._backup(v, states, actions)
        if self.solver:
            for v, states, actions in terminals:
                self.prove(v, states, actions)
        if self.trace is not None:
            self.trace.append({"descents": leaves_dbg, "expanded": list(todo_states)})

    def prove(self, value, states, actions):
        st = WIN if value < 0 else (LOSS if value > 0 else DRAW)
        for s, a in zip(reversed(states), reversed(actions)):
            row = self.proof[s]
            if row[a] == UNKNOWN:
                self.proven_edges += 1
            row[a] = st
            ns = self.status(s)
            if ns == UNKNOWN:
                break
            st = NEGATE[ns]

    def get_policy_value(self, state_int, tau=1):
        if not self.solver:
            return super().get_policy_value(state_int, tau)
        A = self.game.action_space
        row = self.proof[state_int]
        legal = self.game.possible_moves(state_int)
        wins = [a for a in legal if row[a] == WIN]
        if wins:
            pi = [0.0] * A
            pi[wins[0]] = 1.0
            return pi, self.value_avg[state_int]
        w = pi_weights(self.visit_count[state_int], row)
        if tau == 0:
            pi = [0.0] * A
            pi[int(np.argmax(w))] = 1.0
        else:
            z = sum(w)
            pi = [c / z for c in w]
        return pi, self.value_avg[state_int]


class Negamax:
    """Exact game value by negamax with a memo: +1 / -1 / 0 for the side to move (the games are impartial in the
    sense that the value depends on the position and the mover only)."""

    def __init__(self, game):
        self.game = game
        self.memo: Dict[tuple, int] = {}

    def value(self, s, who) -> int:
        key = (s, who)
        v = self.memo.get(key)
        if v is not None:
            return v
        best = -2
        for a in self.game.possible_moves(s):
            best = max(best, self.edge_value(s, a, who))
            if best == 1:
                break
        v = 0 if best == -2 else best
        self.memo[key] = v
        return v

    def edge_value(self, s, a, who) -> int:
        child, won = self.game.move(s, a, who)
        if won:
            return 1
        if not self.game.possible_moves(child):
            return 0
        return -self.value(child, 1 - who)

    def edge_status(self, s, a, who) -> int:
        return {1: WIN, -1: LOSS, 0: DRAW}[self.edge_value(s, a, who)]
