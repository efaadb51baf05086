"""Caro without a GPU: the rule on hand-built positions (CaroOracle next to the freestyle MNKOracle), the constructed
search roots, that every Caro search case would grow different trees under the freestyle rule, and the Python surface
(get_game, the CLIs' -g 2)."""
import numpy as np
import pytest

from caro_cases import CARO_CASES, TABLE, blocked_and_winning_root, blocked_gap_opening, build, make_caro_roots, rule_events
from caro_oracle import CaroOracle
from harness import StubOracleTree
from oracle.games import MNKOracle
from search_matrix import host_noise


@pytest.mark.parametrize("pos", TABLE, ids=[p.name for p in TABLE])
@pytest.mark.parametrize("mover", [0, 1])
def test_table_caro_against_freestyle(pos, mover):
    state, move, who = build(pos, mover)
    caro_state, caro_won = CaroOracle(pos.n, pos.k).move(state, move, who)
    free_state, free_won = MNKOracle(pos.n, pos.k).move(state, move, who)
    assert caro_won == pos.caro_wins, pos.name
    assert free_won == pos.freestyle_wins, pos.name
    assert caro_state == free_state  # the board is the same; only the win test differs


def test_table_covers_the_rule():
    differ = [p for p in TABLE if p.caro_wins != p.freestyle_wins]
    assert differ and all(p.freestyle_wins and not p.caro_wins for p in differ)  # Caro only ever refuses a win
    assert {p.k for p in TABLE} >= {2, 3, 5, 15} and any(p.n == p.k for p in TABLE) and any(p.n == 2 for p in TABLE)


def test_caro_oracle_keeps_the_mnk_surface():
    og, ref = CaroOracle(9, 5), MNKOracle(9, 5)
    rng = np.random.default_rng(5)
    for _ in range(20):
        s = int(ref._from_digits([int(v) for v in rng.integers(0, 3, 81)]))
        assert og.possible_moves(s) == ref.possible_moves(s)
        assert og.render(s) == ref.render(s)
        np.testing.assert_array_equal(og.states_to_training_batch([s], [1]), ref.states_to_training_batch([s], [1]))


@pytest.mark.parametrize("n,k", [(4, 2), (5, 3), (7, 5), (9, 5), (15, 5)])
def test_constructed_roots(n, k):
    og, free = CaroOracle(n, k), MNKOracle(n, k)
    rng = np.random.default_rng(n * 100 + k)
    for empties in (2, 4, 7):
        s, who, b, w = blocked_and_winning_root(og, rng, empties)
        assert len(og.possible_moves(s)) == empties and {b, w} <= set(og.possible_moves(s))
        assert not og.move(s, b, who)[1] and free.move(s, b, who)[1]
        assert og.move(s, w, who)[1]


@pytest.mark.parametrize("n,segments", [(9, 3), (15, 6)])
def test_blocked_gap_openings(n, segments):
    og, free = CaroOracle(n, 5), MNKOracle(n, 5)
    rng = np.random.default_rng(n)
    s = blocked_gap_opening(og, rng, segments)
    refused = [(a, p) for a in og.possible_moves(s) for p in (0, 1) if free.move(s, a, p)[1] and not og.move(s, a, p)[1]]
    assert len(refused) >= segments and len(og.possible_moves(s)) == n * n - segments * 6


def _first_move_trees(case, og):
    """The oracle trees of the case's first move with host Dirichlet noise drawn from the case's seed."""
    rng = np.random.default_rng(case.seed)
    roots = make_caro_roots(case, CaroOracle(*case.board), rng)
    trees = [[StubOracleTree(og) for _ in range(case.trees_per_game)] for _ in range(case.G)]
    for row in trees:
        for t in row:
            t.trace = []
    for _ in range(case.count):
        noise = host_noise(case, rng)
        for g, (state, who) in enumerate(roots):
            trees[g][who if case.trees_per_game == 2 else 0].minibatch(case.batch, state, who, noise[g])
    return trees, roots


def _tree_key(tree):
    return {s: list(tree.visit_count[s]) for s in tree.probs}


@pytest.mark.parametrize("case", [c for c in CARO_CASES if not c.virtual_loss], ids=lambda c: c.name)
def test_search_cases_differ_from_freestyle(case):
    """Under the freestyle rule the same roots and noise grow different trees: a search kernel that ignored the rule
    could not match the Caro oracle.  Cases with device (Philox) noise are checked here with host noise from their
    seed; the GPU test checks the device's own draws met both a blocked run and a win.  On boards with n < k + 2 no
    run fits between two opponent stones, so there the two rules must agree."""
    caro, _ = _first_move_trees(case, CaroOracle(*case.board))
    free, _ = _first_move_trees(case, MNKOracle(*case.board))
    same = all(_tree_key(a) == _tree_key(b) for ra, rb in zip(caro, free) for a, b in zip(ra, rb))
    if case.blocks_possible:
        assert not same, case.name
        blocked, both = rule_events(CaroOracle(*case.board), [(t, None) for row in caro for t in row])
        assert blocked > 0 and both > 0, (case.name, blocked, both)
    else:
        assert same, case.name


def test_caro_cases_reach_every_select_family():
    from search_matrix import instances
    selects = {instances(c)["select"].replace("MnkRules", "R") for c in CARO_CASES}
    assert selects >= {"select_thread_kernel<R,2>", "select_thread_kernel<R,4>", "select_kernel<R,32,1>",
                       "select_kernel<R,32,2>", "select_kernel<R,32,4>", "select_kernel<R,32,8>", "select_vl_kernel<R>"}
    widths = {instances(c)["expand"] for c in CARO_CASES}
    assert len(widths) == 3  # batches below and at 8, 16 and 32
    assert any(c.batch < 8 for c in CARO_CASES) and {8, 16, 32} <= {c.batch for c in CARO_CASES}
    assert {c.noise for c in CARO_CASES} == {"host", "philox"} and {c.trees_per_game for c in CARO_CASES} == {1, 2}


def test_get_game_and_cli_accept_caro(tmp_path):
    from caro_ai_b200 import _cabi
    from caro_ai_b200 import play as play_cli, train as train_cli
    from caro_ai_b200.game import Caro, ConnectFour, TicTacToe, get_game
    g = get_game("2")
    assert type(g) is Caro and isinstance(g, TicTacToe) and (g.n, g.k) == (15, 5) and g.game_kind == _cabi.GAME_CARO == 2
    assert g.obs_shape == (2, 15, 15) and g.action_space == 225 and g.board_words == 8
    assert type(get_game("0")) is ConnectFour and type(get_game("1")) is TicTacToe and get_game("1").n == 3
    c = Caro(9, 4)
    assert (c.n, c.k, c.board_len, c.k_to_win) == (9, 4, 9, 4)
    s = c.initial_state
    assert c.words_to_state(c.state_to_words(s)) == s and c.render(s) == TicTacToe(9, 4).render(s)
    with pytest.raises(AssertionError):
        Caro(16, 5)
    assert train_cli.parse_args(["-g", "2", "-n", "x"]).game == "2"
    with pytest.raises(SystemExit):
        train_cli.parse_args(["-g", "3", "-n", "x"])
    missing = [str(tmp_path / "a.dat"), str(tmp_path / "b.dat")]
    with pytest.raises(FileNotFoundError):  # -g 2 parses; the run stops at the missing checkpoint, before any device work
        play_cli.main(["-g", "2"] + missing)
    with pytest.raises(SystemExit):
        play_cli.main(["-g", "3"] + missing)
