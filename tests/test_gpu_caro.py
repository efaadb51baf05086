"""Caro on the B200 (run with -m gpu): the board kernels, the search kernels, whole self-play games and the CLIs, each
against CaroOracle (tests/caro_oracle.py)."""
import collections
import os

import numpy as np
import pytest

import test_gpu_search_matrix as matrix
from caro_cases import CARO_CASES, TABLE, blocked_gap_opening, build, make_caro_roots, rule_events
from caro_oracle import CaroOracle
from harness import random_position
from oracle.games import MNKOracle
from search_matrix import make_tree

pytestmark = pytest.mark.gpu

BOARDS = sorted({(n, min(n, 5)) for n in range(2, 16)} | {(n, n) for n in (3, 6, 9, 15)} | {(n, 3) for n in (4, 8, 13)})


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _check_apply(n, k, states, actions, players):
    """caro_boards_apply and caro_boards_legal_mask of game 2 against CaroOracle, one batch."""
    from caro_ai_b200.game import Caro
    game, og = Caro(n, k), CaroOracle(n, k)
    new, won, draw = game.apply_batch(states, actions, players)
    for i, (s, a, p) in enumerate(zip(states, actions, players)):
        want, w = og.move(s, a, p)
        assert new[i] == want and bool(won[i]) == w, (n, k, s, a, p)
        assert bool(draw[i]) == (not w and not og.possible_moves(want)), (n, k, s, a, p)
    masks = game.legal_masks(sorted(set(states)))
    for s, m in zip(sorted(set(states)), masks):
        assert list(np.nonzero(m)[0]) == og.possible_moves(s)
    return won


def test_board_kernels_hand_built_table(torch_cuda):
    by_board = collections.defaultdict(list)
    for pos in TABLE:
        for mover in (0, 1):
            by_board[(pos.n, pos.k)].append((pos,) + build(pos, mover))
    for (n, k), rows in by_board.items():
        won = _check_apply(n, k, [r[1] for r in rows], [r[2] for r in rows], [r[3] for r in rows])
        assert [bool(w) for w in won] == [r[0].caro_wins for r in rows]


@pytest.mark.parametrize("n,k", BOARDS)
def test_board_kernels_reachable_positions(torch_cuda, n, k):
    """Positions of random Caro play (blocked runs included), every legal move of the side to move."""
    og = CaroOracle(n, k)
    rng = np.random.default_rng(1000 * n + k)
    states, actions, players = [], [], []
    for i in range(24):
        s, who = random_position(og, rng, int(rng.integers(0, min(n * n - 1, 3 * n))))  # 2x2 has no 3-ply open position
        for a in og.possible_moves(s):
            states.append(s)
            actions.append(a)
            players.append(who)
    _check_apply(n, k, states, actions, players)


@pytest.mark.parametrize("n,k", BOARDS)
def test_board_kernels_dense_boards_with_long_runs(torch_cuda, n, k):
    """Dense random boards (not reachable in play) with a planted run of up to the whole line, longer than 2k - 1
    where the board allows, and random flanks; the move is any cell of the run or next to it, occupied or not (the
    target cell is overwritten)."""
    og, free = CaroOracle(n, k), MNKOracle(n, k)
    rng = np.random.default_rng(7 * n + k)
    dirs = ((0, 1), (1, 0), (1, 1), (-1, 1))
    states, actions, players = [], [], []
    longest = 0
    for _ in range(400):
        who = int(rng.integers(2))
        d = [int(v) for v in rng.choice([0, 1, 2], size=n * n, p=[0.4, 0.4, 0.2])]
        dr, dc = dirs[int(rng.integers(4))]
        r0, c0 = (0, int(rng.integers(n))) if dr == 1 else (int(rng.integers(n)), 0)
        line = []
        r, c = r0, c0
        while 0 <= r < n and 0 <= c < n:
            line.append(r * n + c)
            r, c = r + dr, c + dc
        length = int(rng.integers(1, len(line) + 1))
        start = int(rng.integers(0, len(line) - length + 1))
        for cell in line[start:start + length]:
            d[cell] = who
        for j in (start - 1, start + length):  # flanks: mostly the opponent, so that blocks are common
            if 0 <= j < len(line):
                d[line[j]] = 1 - who if rng.random() < 0.8 else int(rng.integers(3))
        longest = max(longest, length)
        move = line[int(rng.integers(max(0, start - 1), min(len(line), start + length + 1)))]
        states.append(MNKOracle._from_digits(d))
        actions.append(move)
        players.append(who)
    won = _check_apply(n, k, states, actions, players)
    refused = sum(1 for i, w in enumerate(won) if not w and free.move(states[i], actions[i], players[i])[1])
    if n >= k + 2:
        assert refused > 0, "no blocked run among the dense boards"
    assert longest >= min(n, 2 * k)


# ------------------------------------------------------------------------------------------------ search parity
@pytest.mark.parametrize("case", CARO_CASES, ids=[c.name for c in CARO_CASES])
def test_caro_search_parity(torch_cuda, case, monkeypatch):
    """tests/test_gpu_search_matrix.run_case on the Caro rule: trees, policies, sampled moves, roots and status bit for
    bit against StubOracleTree on CaroOracle.  The runner takes its roots and oracle trees from module helpers; here
    the roots are constructed (caro_cases.make_caro_roots) and the trees record their descents, so that the test can
    say from the oracle that the searches played a move completing a run blocked at both ends (and went on) next to
    a winning move."""
    trees = []

    def recording_tree(c, og):
        t = make_tree(c, og)
        t.trace = []
        trees.append(t)
        return t

    monkeypatch.setattr(matrix, "make_roots", make_caro_roots)
    monkeypatch.setattr(matrix, "make_tree", recording_tree)
    terminal, _ = matrix.run_case(torch_cuda, case)
    blocked, both = rule_events(case.oracle_game(), [(t, None) for t in trees])
    if case.blocks_possible:
        assert blocked > 0 and both > 0, (case.name, blocked, both)
    assert terminal > 0, "%s: no terminal descent" % case.name


# ------------------------------------------------------------------------------------------------ whole games
@pytest.mark.parametrize("n,games", [(9, 256), (15, 192)])
def test_caro_self_play_games_match_the_oracle(torch_cuda, n, games):
    """Self-play to the end with the real 5 x 64 tower, Philox noise and tree compaction, one ply at a time through
    caro_engine_search and caro_engine_advance; every finished game replayed through CaroOracle.  Half of the games
    start from the empty board, half from openings with blocked gaps (caro_cases.blocked_gap_opening): from the
    empty board the search finds open fives long before a blocked one forms."""
    torch = torch_cuda
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import Caro
    from caro_ai_b200.model import DeviceNet, Net
    game, og, free = Caro(n, 5), CaroOracle(n, 5), MNKOracle(n, 5)
    A = game.action_space
    torch.manual_seed(n)
    dn = DeviceNet(Net(game.obs_shape, A).eval(), game)
    eng = SelfPlayEngine(game, games, max_batch=8, node_capacity=8 * 80 + 8, replay_capacity=games * A, seed=31 + n,
                         compact_tree=True)
    eng.reset(first_player=-1)
    roots, first = eng.roots()
    rng = np.random.default_rng(n)
    roots = [roots[g] if g % 2 == 0 else blocked_gap_opening(og, rng, 3 if n == 9 else 6) for g in range(games)]
    eng.set_roots(roots, first)
    moves = [[] for _ in range(games)]
    for _ in range(A):
        eng.search(dn, 10, 8)
        acts = eng.advance(10, None, auto_restart=False).cpu().numpy()
        for g in range(games):
            if acts[g] >= 0:
                moves[g].append(int(acts[g]))
        if int((eng.region("status") == 0).sum().item()) == 0:
            break
    c = eng.counters()
    assert c["errors"] == 0 and c["games"] == games and c["plies"] == sum(len(m) for m in moves)
    result = eng.region("result").cpu().numpy()
    entries, _ = eng.drain_replay()
    want = collections.Counter()
    tally = collections.Counter()
    blocked = 0
    for g in range(games):
        s, who = roots[g], first[g]
        history = []
        won = False
        for i, a in enumerate(moves[g]):
            assert not won and a in og.possible_moves(s), (g, i)
            history.append((s, who))
            nxt, won = og.move(s, a, who)
            blocked += (not won) and free.move(s, a, who)[1]
            s, who = nxt, 1 - who
        assert won or not og.possible_moves(s), "game %d stopped before its end" % g
        res = 0 if not won else (1 if history[-1][1] == 0 else -1)
        assert result[g] == res, (g, result[g], res)
        tally["wins_p0" if res == 1 else "wins_p1" if res == -1 else "draws"] += 1
        last = 1 if won else 0
        for t, (st, p) in enumerate(history):
            back = len(history) - 1 - t
            want[(st, p, -last if back & 1 else last)] += 1
    assert collections.Counter((s, p, z) for s, p, _, z in entries) == want
    assert all(c[key] == tally[key] for key in ("wins_p0", "wins_p1", "draws"))
    assert blocked > 0, "no game went through a run of five blocked at both ends"
    eng.close()
    dn.close()


# ------------------------------------------------------------------------------------------------ CLIs and Session
def test_caro_train_play_and_session(torch_cuda, tmp_path, capsys):
    """train.py -g 2 for two steps (the ring passes MIN_REPLAY_TO_TRAIN, so SGD rounds and the arena run), play.py -g 2
    on the promoted checkpoint (a fresh 15 x 15 net when the arena promoted none), and Session on Caro: a user move that
    completes a five blocked at both ends does not end the game, the bot answers."""
    torch = torch_cuda
    import random
    from caro_ai_b200 import play as play_cli, train as train_cli
    from caro_ai_b200.game import Caro
    from caro_ai_b200.model import Net, load_checkpoint, save_checkpoint
    from caro_ai_b200.play_session import Session
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        random.seed(0)
        torch.manual_seed(0)
        assert train_cli.main(["-g", "2", "-n", "caro", "--games", "48", "--max-steps", "2", "--evaluate-every", "2",
                               "--compact-tree"]) == 0
    finally:
        os.chdir(cwd)
    out = capsys.readouterr().out
    assert "Step 2, steps" in out and "Net evaluated, win ratio = " in out
    ratio = float(out.split("Net evaluated, win ratio = ")[1].split()[0])
    saved = os.path.join(tmp_path, "saves", "caro", "best_001_00002.dat")
    assert os.path.exists(saved) == (ratio > 0.60)
    game = Caro()
    if not os.path.exists(saved):
        save_checkpoint(Net(game.obs_shape, game.action_space), saved)
    load_checkpoint(saved, game)
    assert play_cli.main(["-g", "2", "-r", "2", saved, saved]) == 0
    out = capsys.readouterr()
    lines = [l for l in out.out.splitlines() if " vs " in l]
    assert len(lines) == 2 and "Leaderboard:" in out.out
    for l in lines:
        w, lo, d = [int(x.split("=")[1].rstrip(",")) for x in l.split("->")[1].split()]
        assert w + lo + d == 2

    s = Session(game, saved, player_moves_first=True)
    pos = next(p for p in TABLE if p.name == "five_blocked_both_ends")
    state, move, _ = build(pos, s.USER_PLAYER)
    s.state = state
    assert s.is_valid_move(move) and s.move_player(move) is False and not s.is_draw()
    assert s.move_bot() in (False, True) and len(s.moves) == 2 and s.value is not None
    assert s.moves[1] in CaroOracle(15, 5).possible_moves(MNKOracle(15, 5).move(state, move, s.USER_PLAYER)[0])
    assert s.render().startswith("Position evaluation: ") and "<pre>|" in s.render()
