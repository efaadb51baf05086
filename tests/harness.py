"""Parity harness: drives the CUDA engine and the oracle with IDENTICAL network outputs
(oracle.stubs.stub_priors, a per-board pure function) and IDENTICAL random numbers (injected
Dirichlet noise / uniforms), then diffs trees, policies and moves.  Used by tests/ and
__graft_entry__.smoke() only."""
import numpy as np

from oracle.games import ConnectFourOracle, MNKOracle
from oracle.mcts import OracleMCTS
from oracle.stubs import stub_priors


def oracle_for(game):
    """Oracle twin of a caro_ai_b200 game object."""
    if game.game_kind == 0:
        return ConnectFourOracle()
    return MNKOracle(game.board_len, game.k_to_win)


class StubOracleTree(OracleMCTS):
    """OracleMCTS whose network is the integer stub and whose Dirichlet draws are replayed from
    `noise[minibatch][descent]`.  `stub` is the network: stub_priors, or any other pure function of the planes with
    the same signature (oracle.stubs.chain_priors)."""

    def __init__(self, game, c_puct=1.0, alpha=0.3, explore=0.25, stub=stub_priors):
        super().__init__(game, c_puct, alpha, explore, dirichlet=self._next_noise)
        self._noise = None
        self._j = 0
        self._stub = stub

    def _next_noise(self, alpha):
        z = self._noise[self._j]
        self._j += 1
        return z

    def evaluate(self, states, players, net, device="cpu"):
        planes = self.game.states_to_training_batch(states, players)
        return self._stub(planes, self.game.action_space)

    def minibatch(self, batch, state, player, noise_bj):
        self._noise, self._j = noise_bj, 0
        self.search_minibatch(batch, state, player, None)


def random_position(ogame, rng, plies):
    while True:
        s, who, ok = ogame.initial_state, int(rng.integers(2)), True
        for _ in range(plies):
            legal = ogame.possible_moves(s)
            if not legal:
                ok = False
                break
            s, won = ogame.move(s, int(rng.choice(legal)), who)
            who = 1 - who
            if won:
                ok = False
                break
        if ok and ogame.possible_moves(s):
            return s, who


def f32_bits(x):
    return np.asarray(x, dtype=np.float32).view(np.uint32)


def diff_tree(engine_tree, oracle_tree, A):
    """List of human-readable differences between an exported engine arena and an OracleMCTS."""
    errs = []
    keys_e, keys_o = set(engine_tree), set(oracle_tree.probs)
    if keys_e != keys_o:
        errs.append("node sets differ: engine-only %d, oracle-only %d" % (len(keys_e - keys_o), len(keys_o - keys_e)))
    for s in keys_e & keys_o:
        n = engine_tree[s]
        if list(n["N"]) != [int(x) for x in oracle_tree.visit_count[s]]:
            errs.append("N differs at %d: %s vs %s" % (s, n["N"], oracle_tree.visit_count[s]))
            continue
        if not np.array_equal(f32_bits(n["P"]), f32_bits(oracle_tree.probs[s])):
            errs.append("P differs at %d" % s)
        ow = oracle_tree.value[s]
        oq = oracle_tree.value_avg[s]
        if not np.array_equal(f32_bits(n["W"]), f32_bits([float(w) for w in ow])):
            errs.append("W differs at %d: %s vs %s" % (s, n["W"], ow))
        if not np.array_equal(f32_bits(n["Q"]), f32_bits([np.float32(q) for q in oq])):
            errs.append("Q differs at %d: %s vs %s" % (s, n["Q"], oq))
        for a in range(A):  # numpy promotion state of W(s,a): float32 once a net value arrived
            if n["N"][a] > 0 and n["f32"][a] != isinstance(ow[a], np.floating):
                errs.append("W type flag differs at %d action %d" % (s, a))
    return errs


def np_choice(p, u):
    """np.random.choice(len(p), p=p) given its one uniform draw u (numpy/random/mtrand.pyx)."""
    cdf = np.cumsum(np.asarray(p, dtype=np.float64))
    cdf /= cdf[-1]
    return int(np.searchsorted(cdf, u, side="right"))
