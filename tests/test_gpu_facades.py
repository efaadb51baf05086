"""GPU tests of the drop-in facades (lib/mcts.py:MCTS, lib/utils.py:play_game, lib/play_session.py:Session,
play.py, train.py) and the size-independent properties of the engine at BASELINE.json's full configuration."""
import collections
import os

import numpy as np
import pytest

from conftest import GOLDEN
from harness import StubOracleTree, diff_tree, oracle_for, random_position
from oracle.mcts import OracleMCTS, play_game as oracle_play_game
from oracle.stubs import stub_forward

pytestmark = pytest.mark.gpu


def keyed_noise(seed, A):
    """Dirichlet vectors addressed by (minibatch, descent) so that the facade (which draws a vector for every
    descent) and the oracle (which draws only at an expanded root) consume identical numbers."""
    def vec(mb, j):
        return np.random.default_rng([seed, mb, j]).dirichlet([0.3] * A)
    return vec


class FacadeOracle(OracleMCTS):
    """Oracle tree driven with the same keyed noise and the torch stub network the facade gets."""

    def __init__(self, game, vec):
        super().__init__(game, dirichlet=lambda alpha: self._draw())
        self.vec, self.mb, self.j = vec, 0, 0

    def _draw(self):
        z = self.vec(self.mb, self.j)
        self.j += 1
        return z

    def search_minibatch(self, batch_size, state_int, player, net, device="cpu"):
        self.j = 0
        super().search_minibatch(batch_size, state_int, player, net, device)
        self.mb += 1


def facade_tree(game, vec, seed=0):
    from caro_ai_b200.mcts import MCTS
    t = MCTS(game, node_capacity=4096, max_batch=16)
    counter = {"mb": 0}

    def noise_fn(batch, A):
        z = np.stack([vec(counter["mb"], j) for j in range(batch)])
        counter["mb"] += 1
        return z
    t.noise_fn = noise_fn
    return t


@pytest.mark.parametrize("which", ["connect4", "tictactoe"])
def test_mcts_facade_matches_oracle(which):
    """search_batch / get_policy_value / dict views / find_leaf of the facade vs the oracle, bit-exact, with an
    arbitrary callable network evaluated exactly like lib/mcts.py:212-218 (planes -> net -> softmax)."""
    from caro_ai_b200.game import ConnectFour, TicTacToe
    game = ConnectFour() if which == "connect4" else TicTacToe(3, 3)
    og = oracle_for(game)
    A = game.action_space
    rng = np.random.default_rng(5)
    net = lambda x: stub_forward(x, A)
    for trial in range(3):
        root, who = random_position(og, rng, int(rng.integers(0, 5)))
        vec = keyed_noise(100 + trial, A)
        ft, ot = facade_tree(game, vec), FacadeOracle(og, vec)
        ft.search_batch(6, 8, root, who, net)
        ot.search_batch(6, 8, root, who, net)
        assert len(ft) == len(ot)
        assert ft.visit_count == {s: list(v) for s, v in ot.visit_count.items()}
        for s in ot.probs:
            np.testing.assert_array_equal(np.float32(ft.probs[s]), np.float32(ot.probs[s]))
            np.testing.assert_array_equal(np.float32(ft.value[s]), np.float32([float(w) for w in ot.value[s]]))
            np.testing.assert_array_equal(np.float32(ft.value_avg[s]), np.float32([np.float32(q) for q in ot.value_avg[s]]))
        for tau in (1, 0):
            pf, qf = ft.get_policy_value(root, tau=tau)
            po, qo = ot.get_policy_value(root, tau=tau)
            assert pf == [float(x) for x in po]
            np.testing.assert_allclose(qf, [float(x) for x in qo], atol=1e-6)
        assert ft.is_leaf(root) is False and ft.is_leaf(123456789 if which == "connect4" else 111111111) is True
        # one more descent on the frozen tree, same noise on both sides
        ot.j = 0
        vo = ot.find_leaf(root, who)
        vf = ft.find_leaf(root, who)
        assert vf == (vo[0], vo[1], vo[2], list(vo[3]), list(vo[4]))
        ft.clear()
        assert len(ft) == 0


def test_reference_backup_unit_test_through_facade():
    """lib/test_mcts.py:9-38 driven against the facade (dict assignment + _backup); float32 arithmetic."""
    from unittest.mock import MagicMock
    from caro_ai_b200.mcts import MCTS
    tree = MCTS(MagicMock())
    tree.visit_count = {1: [0, 1], 2: [1, 0], 3: [0, 0]}
    tree.value = {1: [0.0, 0.5], 2: [0.6, 0.0], 3: [0.0, 0.0]}
    tree.value_avg = {1: [0.0, 0.5], 2: [0.6, 0.0], 3: [0.0, 0.0]}
    tree.probs = {1: [0.1, 0.9], 2: [0.8, 0.2], 3: [0.7, 0.3]}
    tree._backup(0.2, [1, 2, 3], [1, 0, 0])
    assert tree.visit_count == {1: [0, 2], 2: [2, 0], 3: [1, 0]}
    for got, want in [(tree.value, {1: [0.0, 0.3], 2: [0.8, 0.0], 3: [-0.2, 0.0]}),
                      (tree.value_avg, {1: [0.0, 0.15], 2: [0.4, 0.0], 3: [-0.2, 0.0]})]:
        assert got.keys() == want.keys()
        for k in want:
            np.testing.assert_allclose(got[k], want[k], atol=1e-6)


def test_play_game_facade_matches_oracle():
    """lib/utils.py:play_game through the facade vs the oracle: same np.random stream for the moves, same keyed
    noise, same stub network -> identical results, step counts and replay buffers (one shared tree, train.py:185)."""
    import torch
    from caro_ai_b200 import mcts as fm, utils as fu
    from caro_ai_b200.game import TicTacToe
    from caro_ai_b200.model import Net
    game = TicTacToe(3, 3)
    og = oracle_for(game)
    A = game.action_space

    class StubNet(Net):  # passes play_game's isinstance check; forward = integer stub
        def forward(self, x):
            lg, v = stub_forward(x, A)
            return lg.to(x.device), v.to(x.device)

    net = StubNet(game.obs_shape, A)
    for seed in (3, 4):
        vec = keyed_noise(seed, A)
        ft = facade_tree(game, vec)
        ft._device_net = lambda n: None  # force the generic-callable path (the stub is not a real tower)
        ot = FacadeOracle(og, vec)
        rb_f, rb_o = collections.deque(maxlen=1000), collections.deque(maxlen=1000)
        np.random.seed(seed)
        res_f = fu.play_game(game, ft, rb_f, net, net, 3, 5, 8)
        np.random.seed(seed)
        res_o = oracle_play_game(og, ot, rb_o, net, net, 3, 5, 8)
        assert res_f == res_o
        assert [(s, p, z) for s, p, _, z in rb_f] == [(s, p, z) for s, p, _, z in rb_o]
        for (_, _, pf, _), (_, _, po, _) in zip(rb_f, rb_o):
            assert list(pf) == [float(x) for x in po]


def test_session_and_cli_smoke(tmp_path, capsys):
    """play_session.Session on a shipped checkpoint; play.py and train.py mains end to end (tiny sizes)."""
    import torch
    from caro_ai_b200 import play as play_cli, train as train_cli
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import Net, save_checkpoint
    from caro_ai_b200.play_session import Session
    ck = os.path.join(GOLDEN, "checkpoints", "connect4_best_026_12000.dat")
    s = Session(ConnectFour(), ck, player_moves_first=True)
    assert s.is_valid_move(3) and not s.is_draw()
    s.move_player(3)
    won = s.move_bot()
    assert won is False and len(s.moves) == 2 and s.value is not None
    assert s.render().startswith("Position evaluation: ") and "<pre>0123456" in s.render()
    # tournament: two TicTacToe nets, 6 rounds per ordered pair, reference output format (play.py:59-76)
    g = TicTacToe(3, 3)
    paths = []
    for i in range(2):
        torch.manual_seed(i)
        p = str(tmp_path / ("m%d.dat" % i))
        save_checkpoint(Net(g.obs_shape, g.action_space), p)
        paths.append(p)
    assert play_cli.main(["-g", "1", "-r", "6"] + paths) == 0
    out = capsys.readouterr()
    lines = [l for l in out.out.splitlines() if " vs " in l]
    assert len(lines) == 2 and "Leaderboard:" in out.out and "games/s" in out.err
    for l in lines:
        w, lo, d = [int(x.split("=")[1].rstrip(",")) for x in l.split("->")[1].split()]
        assert w + lo + d == 6
    # training loop: 2 steps of 32 TicTacToe games, replay grows, no crash (replay < MIN_REPLAY_TO_TRAIN: no SGD)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        assert train_cli.main(["-g", "1", "-n", "smoke", "--games", "32", "--max-steps", "2"]) == 0
    finally:
        os.chdir(cwd)


def test_train_step_and_evaluate():
    """train.py:62-149 pieces on real self-play data: SGD rounds reduce the loss, evaluate returns a ratio."""
    import torch
    import torch.optim as optim
    from caro_ai_b200 import config as cfg, train as T
    from caro_ai_b200.game import TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    from caro_ai_b200.utils import TBMeanTracker, play_games_batched
    game = TicTacToe(3, 3)
    torch.manual_seed(0)
    net = Net(game.obs_shape, game.action_space).cuda()
    best = DeviceNet(net, game)
    replay = collections.deque(maxlen=5000)
    stats = play_games_batched(game, 128, best, best, 10, 10, 8, replay_buffer=replay, trees_per_game=1, seed=1)
    assert stats["games"] == 128 and stats["wins"] + stats["losses"] + stats["draws"] == 128
    assert len(replay) == stats["plies"] >= 128 * 5
    for s, p, pi, z in list(replay)[:50]:
        assert p in (0, 1) and z in (-1, 0, 1) and abs(sum(pi) - 1.0) < 1e-5 and len(pi) == 9

    class W:
        def add_scalar(self, *a):
            pass

        def close(self):
            pass
    opt = optim.SGD(net.parameters(), lr=cfg.LEARNING_RATE, momentum=0.9)
    with TBMeanTracker(W(), 10) as tb:
        first = T.train_neural_net(game, net, replay, opt, tb, 1, torch.device("cuda"))
        for i in range(3):
            last = T.train_neural_net(game, net, replay, opt, tb, 2 + i, torch.device("cuda"))
    assert last[0] < first[0]
    ratio = T.evaluate(game, net, best, 8, seed=3, device=torch.device("cuda"))
    assert 0.0 <= ratio <= 1.0


def test_full_size_properties():
    """BASELINE.json configs[1] shape (4096 games, 100 x 8 descents per move) for a few plies: invariants that do
    not need the oracle."""
    import torch
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.model import DeviceNet, Net
    game = ConnectFour()
    torch.manual_seed(0)
    dn = DeviceNet(Net(game.obs_shape, game.action_space).eval(), game)
    G, C_, B = 4096, 100, 8
    eng = SelfPlayEngine(game, G, max_batch=B, node_capacity=4096, replay_capacity=1 << 16, seed=9)
    plies = 3
    eng.play(dn, dn, moves=plies, count=C_, batch=B, tau_plies=10, auto_restart=True)
    c = eng.counters()
    assert c["errors"] == 0
    assert c["descents"] == G * B * C_ * plies and c["plies"] == G * plies
    nodes = eng.region("node_count").cpu().numpy()
    assert int(nodes.sum()) == c["leaf_evals"]          # every evaluated leaf became exactly one node
    assert nodes.min() > C_ and nodes.max() <= C_ * B * plies
    # per-node algebra on a sample of arenas: Q == f32(W / N), N >= 0, priors form a distribution
    cap = eng.cfg.node_capacity
    for g in (0, 17, 4095):
        n_nodes = int(nodes[g])
        lo, hi = g * cap, g * cap + n_nodes
        n, w, q, p = (eng.pool(name, lo, hi)[:, :7].cpu().numpy() for name in ("N", "W", "Q", "P"))
        assert (n >= 0).all()
        np.testing.assert_array_equal(q[n > 0], (w[n > 0] / n[n > 0].astype(np.float32)).astype(np.float32))
        assert (q[n == 0] == 0).all() and (w[n == 0] == 0).all()
        np.testing.assert_allclose(p.sum(axis=1), 1.0, atol=1e-5)
        assert (np.abs(q) <= 1.0 + 1e-6).all()
    # root statistics: visits at the root never exceed the descents of the plies searched from it
    pi, q, n = eng.root_policy(1)
    assert int(n.sum(dim=1).max().item()) <= C_ * B * plies
    # two engines with the same seed produce identical games (Philox streams are addressed, not consumed)
    eng2 = SelfPlayEngine(game, 64, max_batch=B, node_capacity=2048, seed=9)
    eng3 = SelfPlayEngine(game, 64, max_batch=B, node_capacity=2048, seed=9)
    for e in (eng2, eng3):
        e.play(dn, dn, moves=4, count=12, batch=B, tau_plies=10, auto_restart=True)
    assert eng2.roots() == eng3.roots()
    assert torch.equal(eng2.region("nodes")[: 64 * 2048], eng3.region("nodes")[: 64 * 2048])


def test_finished_games_replay_and_restart():
    """Games played to the end: W/L/D add up, replay z alternates back from the last mover (lib/utils.py:101-106),
    re-seated slots start from the initial position with a cleared tree."""
    import torch
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    game = TicTacToe(3, 3)
    torch.manual_seed(0)
    dn = DeviceNet(Net(game.obs_shape, game.action_space).eval(), game)
    eng = SelfPlayEngine(game, 256, max_batch=8, node_capacity=1024, replay_capacity=1 << 14, seed=2)
    eng.play(dn, dn, moves=9, count=6, batch=8, tau_plies=2, auto_restart=False)
    c = eng.counters()
    assert c["errors"] == 0 and c["games"] == 256 == c["wins_p0"] + c["wins_p1"] + c["draws"]
    entries, cursor = eng.drain_replay()
    assert cursor == c["plies"] == len(entries)
    og = oracle_for(game)
    # split the ring into games: every game starts from the initial state
    starts = [i for i, e in enumerate(entries) if e[0] == game.initial_state] + [len(entries)]
    assert len(starts) - 1 == 256
    for a, b in zip(starts[:-1], starts[1:]):
        chunk = entries[a:b]
        zs = [e[3] for e in chunk]
        assert zs[-1] in (0, 1) and all(zs[i] == -zs[i + 1] for i in range(len(zs) - 1))
        for (s, p, pi, z), (s2, p2, _, _) in zip(chunk[:-1], chunk[1:]):
            assert p2 == 1 - p
            legal = og.possible_moves(s)
            nxt = [og.move(s, a_, p)[0] for a_ in legal]
            assert s2 in nxt                      # consecutive replay states are one legal move apart
            assert all(pi[a_] == 0 for a_ in range(9) if a_ not in legal)
    assert (eng.region("status") == 1).all()
    eng.reset()
    assert eng.roots()[0] == [game.initial_state] * 256 and int(eng.region("node_count").sum().item()) == 0


def test_caro_pipeline_parts_do_not_share_head_scratch():
    """Caro 15x15 runs its FC heads in a separate kernel from exported features; two pipeline parts have tower launches
    in flight at the same time, so the scratch is slotted per launch: a 2-part run must reproduce the two single-engine
    runs bit for bit (same seeds, Philox streams are addressed by game id)."""
    import torch
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    game = TicTacToe(15, 5)
    torch.manual_seed(0)
    dn = DeviceNet(Net(game.obs_shape, game.action_space).eval(), game)

    def engines():
        return [SelfPlayEngine(game, 48, max_batch=8, node_capacity=2048, seed=31 + h) for h in range(2)]

    solo = engines()
    for e in solo:
        e.play(dn, dn, moves=2, count=12, batch=8, tau_plies=10, auto_restart=True)
    pair = engines()
    SelfPlayEngine.play_multi(pair, dn, moves=2, count=12, batch=8, tau_plies=10, auto_restart=True)
    torch.cuda.synchronize()
    for a, b in zip(solo, pair):
        assert a.counters() == b.counters() and a.counters()["errors"] == 0
        assert a.roots() == b.roots()
        assert torch.equal(a.region("nodes"), b.region("nodes"))  # every record: N (+ float32 bit), W, P, child links
    dn.close()


def test_bench_engine_arm_prints_the_contract_line():
    """`python bench.py` on a small batch: ONE JSON line with the contract's keys, a roofline and an e2e object whose
    byte counts match the host buffers that are copied per step, launches counted, no engine errors."""
    import json
    import subprocess
    import sys
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--games", "512", "--steps", "4", "--warmup", "3",
                          "--preroll", "40", "--no-cpu-baseline", "--node-capacity", "8192", "--extra-small"],
                         capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks"):
        assert key in d, key
    assert d["metric"] == "connect4_mcts_leaf_evals_per_sec" and d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 4
    assert d["engine_errors"] == 0 and d["gpu_launches"] >= 4 * 100 * 2 * 5  # noise, select, plan, tower, expand+backup per minibatch and part
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 512 * 17 <= d["e2e"]["d2h_bytes_per_step"]
    assert d["net_precision"]["selected"] == "fp16" and d["net_precision"]["calibration"]["max_abs_prior_diff"] < 1e-3
    assert d["bf16_same_workload"]["precision"] == "bf16" and d["bf16_same_workload"]["value"] > 0
    tr = d["extra"]["train"]
    assert tr["rounds"] == 20 and tr["sgd_ms_per_round"] > 0 and tr["gradient_bytes"] == 188301 * 4 and tr["allreduce_us"] is None
    for tag in ("connect4_4096_games", "connect4_4096_games_virtual_loss", "caro_15x15_1600_sims", "caro_15x15_1600_sims_deep10"):
        assert d["extra"]["configs"][tag]["leaf_evals_per_sec"] > 0 and d["extra"]["configs"][tag]["errors"] == 0
    r = d["roofline"]
    assert r["bound"] == "tensor" and 0 < r["frac"] < 1.5 and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert "workload" in d["config"] and d["dtype"] == "f16" and d["scaling"] == "weak"


def test_bench_dumps_the_same_outputs_of_its_last_step_on_every_run(tmp_path):
    """`bench.py --dump-outputs DIR`: float32 / float64 arrays within 64 MB, identical from run to run with the same
    arguments; one position, side, ply and policy per game, and exactly one replay block (opened by the empty board)
    per game that ended in the last ply."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    G = 512
    runs = []
    for i in range(2):
        d = tmp_path / ("run%d" % i)
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--games", str(G), "--steps", "3", "--warmup", "1",
                              "--preroll", "20", "--no-cpu-baseline", "--no-extra", "--node-capacity", "8192", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900, cwd=root)
        assert out.returncode == 0, out.stderr[-3000:]
        runs.append({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = runs
    assert set(a) == {"move_pi", "replay_board", "replay_pi", "replay_player", "replay_z", "root_board", "root_ply", "root_player"}
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        np.testing.assert_array_equal(a[name], b[name], err_msg=name)
    assert a["root_board"].shape == (G, 2) and a["move_pi"].shape == (G, 7) and a["root_ply"].shape == a["root_player"].shape == (G,)
    going_on = a["root_ply"] > 0
    np.testing.assert_allclose(a["move_pi"][going_on].sum(axis=1), 1.0, atol=1e-5)
    assert (a["move_pi"][~going_on] == 0).all()
    assert int((a["replay_board"][:, 0] == 0).sum()) == int((~going_on).sum())
    assert set(np.unique(a["replay_z"])) <= {-1.0, 0.0, 1.0}
    np.testing.assert_allclose(a["replay_pi"].sum(axis=1), 1.0, atol=1e-5)


def test_connect4_pipeline_matches_single_engine_play():
    """The parts pipeline (CUDA graph per ply, expand+backup with eight lanes per game, noise prefetched under the network
    pass) vs a single engine's play() (separate launches, expand+backup with one warp per game): same seeds => the same
    games and bit-identical trees (N, W, Q, P), also with numbers of games that are not multiples of a block's share, and
    over ply boundaries with re-seated games, for even and odd numbers of minibatches per ply."""
    import torch
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.model import DeviceNet, Net
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    game = ConnectFour()
    torch.manual_seed(0)
    dn = DeviceNet(Net(game.obs_shape, game.action_space).eval(), game)

    def engines():
        return [SelfPlayEngine(game, g, max_batch=8, node_capacity=4096, seed=77 + h) for h, g in enumerate((200, 131))]

    for count in (12, 7):
        solo = engines()
        for e in solo:
            e.play(dn, dn, moves=9, count=count, batch=8, tau_plies=3, auto_restart=True)
        pair = engines()
        SelfPlayEngine.play_multi(pair, dn, moves=9, count=count, batch=8, tau_plies=3, auto_restart=True)
        torch.cuda.synchronize()
        for a, b in zip(solo, pair):
            ca, cb = a.counters(), b.counters()
            assert ca == cb and ca["errors"] == 0 and ca["leaf_evals"] > 0, (count, ca, cb)
            assert a.roots() == b.roots()
            for name in ("nodes", "node_count"):
                assert torch.equal(a.region(name), b.region(name)), (count, name)
        for e in solo + pair:
            e.close()
    dn.close()
