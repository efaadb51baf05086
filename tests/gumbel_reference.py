"""Host restatement of the Gumbel root search extension (include/caro_b200.h caro_engine_set_gumbel), step by step:

  1. draws g(a): read from the engine's "gumbel_g" export (the device's Philox + double log); `host_draws` recomputes them
     through the host compile of csrc/rng.cuh (tests/native/gumbel_check.cpp);
  2. q(a) = value_avg of a visited edge (a python float or an np.float32, exactly the Q the root branch of select uses);
     an unvisited edge gets sum P q / sum P over the visited legal edges in action order (0 when none is visited or their
     prior mass is 0); sigma = ((c_visit + max N) * c_scale) * ((q + 1) * 0.5); base = scale * g + log P;
     score = base + sigma; logit = log P + sigma; ties to the lowest action;
  3. schedule: m = min(m_param, legal), H = ceil(log2 m), r_p = min(m, max(2, ceil(m / 2^p))), phase floor(k H / C') of
     local minibatch k = i - i0, top m by base at k = 0, top r_p of the survivors by score when the phase changes,
     descent j forced onto survivor ((k - k_phase_start) b + j) mod r_p;
  4. pi' = softmax of logit over the legal moves (exp(l - max) summed in action order, quotients stored as float32),
     uniform when every legal logit is -inf;
  5. move = argmax score over the survivors (over every legal move when no phase ran).
All in numpy float64.  GumbelOracleTree is StubOracleTree with steps 3-5 at the root of its searches.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence

import numpy as np

from harness import StubOracleTree
from oracle.stubs import stub_priors

DEFAULTS = dict(m=16, c_visit=50.0, c_scale=0.1, scale=1.0)


# ------------------------------------------------------------------------------------------------ schedule
def phases(m: int) -> int:
    """H = ceil(log2 m)."""
    h = 0
    while (1 << h) < m:
        h += 1
    return h


def survivors(m: int, p: int) -> int:
    """r_p = min(m, max(2, ceil(m / 2^p)))."""
    return min(m, max(2, -(-m // (1 << p))))


def phase_of(k: int, m: int, cp: int) -> int:
    return (k * phases(m)) // cp


def schedule(m: int, cp: int, batch: int):
    """[(phase, r, k_phase_start, [survivor slot of each descent])] for the C' = cp local minibatches of a search."""
    out, phase, kstart = [], -1, 0
    for k in range(cp):
        p = phase_of(k, m, cp)
        if p != phase:
            phase, kstart = p, k
        r = survivors(m, phase)
        out.append((phase, r, kstart, [((k - kstart) * batch + j) % r for j in range(batch)]))
    return out


# ------------------------------------------------------------------------------------------------ scores
def _log(p) -> float:
    with np.errstate(divide="ignore"):
        return float(np.log(np.float64(p)))


def completed_q(n_row: Sequence[int], q_row: Sequence[float], p_row: Sequence[float], legal: Sequence[int]) -> List[float]:
    """q(a) of every action: the edge's Q when visited, else the prior-weighted mean Q of the visited legal edges."""
    sp = spq = 0.0
    for a in legal:
        if n_row[a] > 0:
            p = float(np.float32(p_row[a]))
            sp += p
            spq += p * float(q_row[a])
    qbar = spq / sp if sp > 0.0 else 0.0
    return [float(q_row[a]) if n_row[a] > 0 else qbar for a in range(len(n_row))]


def sigmas(n_row, q_row, p_row, legal, c_visit: float, c_scale: float) -> List[float]:
    scale = (c_visit + float(max([int(n_row[a]) for a in legal] + [0]))) * c_scale
    return [scale * ((q + 1.0) * 0.5) for q in completed_q(n_row, q_row, p_row, legal)]


def improved_policy(n_row, q_row, p_row, legal, c_visit: float, c_scale: float) -> np.ndarray:
    """pi' as float32 [A]."""
    A = len(n_row)
    sig = sigmas(n_row, q_row, p_row, legal, c_visit, c_scale)
    logit = {a: _log(np.float32(p_row[a])) + sig[a] for a in legal}
    pi = np.zeros(A, dtype=np.float32)
    lmax = max(logit.values())
    if lmax == -math.inf:
        for a in legal:
            pi[a] = np.float32(1.0 / len(legal))
        return pi
    ex = {a: float(np.exp(logit[a] - lmax)) for a in legal}
    s = 0.0
    for a in sorted(legal):
        s += ex[a]
    for a in legal:
        pi[a] = np.float32(ex[a] / s)
    return pi


def top(actions: Sequence[int], key: dict, count: int) -> List[int]:
    """The `count` best actions by `key`, ties to the lowest action."""
    return sorted(actions, key=lambda a: (-key[a], a))[:count]


def ulp_diff(a, b) -> int:
    """Largest distance in float32 units in the last place between two float32 arrays of the same sign pattern."""
    ia = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    ib = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    return int(np.abs(ia - ib).max()) if ia.size else 0


# ------------------------------------------------------------------------------------------------ oracle tree
class GumbelOracleTree(StubOracleTree):
    def __init__(self, game, gumbel: bool = True, m: int = 16, c_visit: float = 50.0, c_scale: float = 0.1,
                 scale: float = 1.0, stub=stub_priors, **kw):
        super().__init__(game, stub=stub, **kw)
        self.gumbel = gumbel
        self.m_param, self.c_visit, self.c_scale, self.scale = m, c_visit, c_scale, scale
        self.g: Optional[np.ndarray] = None
        self.forced: Optional[List[int]] = None
        self._reset_search()

    def _reset_search(self):
        self.i0, self.phase, self.kstart, self.m, self.surv = -1, -1, 0, 0, []

    # ---- step 3: one minibatch of the schedule
    def plan(self, g_row, mb: int, count: int, batch: int, state: int) -> List[int]:
        """The forced root actions of minibatch `mb` (-1 = PUCT); `g_row` = the search's draws (used at mb 0)."""
        if not self.gumbel:
            self.forced = None
            return [-1] * batch
        if mb == 0:
            self._reset_search()
            self.g = np.asarray(g_row, dtype=np.float64).copy()
        if state not in self.probs:
            self.forced = None
            return [-1] * batch
        if self.i0 < 0:
            self.i0 = mb
        k, cp = mb - self.i0, count - self.i0
        legal = self.game.possible_moves(state)
        if self.phase < 0:
            self.m = min(self.m_param, len(legal))
            self.surv = top(legal, self.bases(state), self.m)
            self.phase, self.kstart = 0, 0
        p = phase_of(k, self.m, cp)
        if p != self.phase:
            self.surv = top(self.surv, self.scores(state), survivors(self.m, p))
            self.phase, self.kstart = p, k
        r = len(self.surv)
        self.forced = [self.surv[((k - self.kstart) * batch + j) % r] for j in range(batch)]
        return list(self.forced)

    def bases(self, s) -> dict:
        return {a: self.scale * float(self.g[a]) + _log(np.float32(self.probs[s][a])) for a in self.game.possible_moves(s)}

    def sigma_row(self, s) -> List[float]:
        legal = self.game.possible_moves(s)
        return sigmas(self.visit_count[s], self.value_avg[s], self.probs[s], legal, self.c_visit, self.c_scale)

    def scores(self, s) -> dict:
        sig, base = self.sigma_row(s), self.bases(s)
        return {a: base[a] + sig[a] for a in base}

    # ---- the root step of a descent
    def find_leaf(self, state_int, player):
        if not self.forced:
            return super().find_leaf(state_int, player)
        # OracleMCTS.find_leaf with the root action taken from the plan; the device still draws this descent's noise
        # vector, so it is consumed here too
        path_states, path_actions = [], []
        s, who, value = state_int, player, None
        while s in self.probs:
            path_states.append(s)
            if s == state_int:
                a = self.forced[self._j]
                self._j += 1
            else:
                scores = self._ucb(self.value_avg[s], self.probs[s], self.visit_count[s])
                for b in self.game.invalid_moves(s):
                    scores[b] = -np.inf
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

    # ---- steps 4 and 5
    def improved(self, s) -> np.ndarray:
        return improved_policy(self.visit_count[s], self.value_avg[s], self.probs[s], self.game.possible_moves(s),
                               self.c_visit, self.c_scale)

    def move(self, s) -> int:
        sc = self.scores(s)
        cands = self.surv if self.phase >= 0 and self.surv else self.game.possible_moves(s)
        return top(cands, sc, 1)[0]

    def get_policy_value(self, state_int, tau=1):
        if not self.gumbel:
            return super().get_policy_value(state_int, tau)
        if tau == 0:
            pi = [0.0] * self.game.action_space
            pi[self.move(state_int)] = 1.0
        else:
            pi = [float(x) for x in self.improved(state_int)]
        return pi, self.value_avg[state_int]
