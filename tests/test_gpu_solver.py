"""The MCTS solver extension on the B200 (run with -m gpu): bit-exact parity with its host restatement on every select
family, exact proofs with the real network, the switch off being the parent's search, graph replays that follow the
switch, the per-player mask and its refusals, and the CLIs end to end."""
import os
import random

import numpy as np
import pytest

from conftest import GOLDEN
from harness import diff_tree, np_choice, random_position
from search_matrix import STUBS, host_noise, instances
from solver_cases import SOLVER_CHAIN_CASES, SOLVER_PARITY_CASES, solver_roots
from solver_reference import UNKNOWN, Negamax, SolverOracleTree

pytestmark = pytest.mark.gpu

C4_CKPT = os.path.join(GOLDEN, "checkpoints", "connect4_best_026_12000.dat")
_PROVEN_BY_FAMILY = {}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def run_solver_case(torch, case):
    """run_case of tests/test_gpu_search_matrix.py with the solver on for both players: trees (with their proofs),
    policies, moves, roots and the solver counters against SolverOracleTree.  Returns the edges proven."""
    from caro_ai_b200.engine import SelfPlayEngine
    game, og = case.product_game(), case.oracle_game()
    G, A, batch, tpg = case.G, case.A, case.batch, case.trees_per_game
    rng = np.random.default_rng(case.seed)
    roots = solver_roots(case, og, rng)
    eng = SelfPlayEngine(game, G, trees_per_game=tpg, max_batch=case.max_batch,
                         node_capacity=case.count * batch * case.moves + 8, seed=case.seed)
    eng.set_solver(3)
    eng.set_roots([r[0] for r in roots], [r[1] for r in roots])
    trees = [[SolverOracleTree(og, stub=STUBS[case.stub]) for _ in range(tpg)] for _ in range(G)]
    stub = STUBS[case.stub]
    states, players = [r[0] for r in roots], [r[1] for r in roots]
    alive = [True] * G
    for move in range(case.moves):
        for i in range(case.count):
            if case.noise == "philox":
                buf = torch.full((G, batch, A), float("nan"), dtype=torch.float64, device="cuda")
                eng.select(batch, i, None, noise_out=buf)
                noise = buf.cpu().numpy()
            else:
                noise = host_noise(case, rng)
                eng.select(batch, i, torch.from_numpy(noise).cuda())
            eng.plan(batch)
            n = eng.leaf_count()
            planes = eng.leaf_planes(n).cpu().numpy()
            pri, val = stub(planes, A) if n else (np.zeros((1, A), np.float32), np.zeros(1, np.float32))
            eng.expand_backup(batch, torch.from_numpy(np.ascontiguousarray(pri)).cuda(),
                              torch.from_numpy(np.ascontiguousarray(val)).cuda())
            for g in range(G):
                if alive[g]:
                    trees[g][players[g] if tpg == 2 else 0].minibatch(batch, states[g], players[g], noise[g])
        for g in range(G):
            if not alive[g]:
                continue
            for t in range(tpg):
                exported = eng.export_tree(g * tpg + t)
                errs = diff_tree(exported, trees[g][t], A)
                errs += ["proof differs at %d: %s vs %s" % (s, exported[s]["proof"], trees[g][t].proof[s])
                         for s in exported if s in trees[g][t].proof and exported[s]["proof"] != trees[g][t].proof[s]]
                assert not errs, "%s: game %d move %d tree %d: %s" % (case.name, g, move, t, errs[:5])
        pi_d, q_d, _ = eng.root_policy(2, case.tau_plies)
        pi_d = pi_d.cpu().numpy()
        plies_dev = eng.region("ply").cpu().numpy()
        u = rng.random(G)
        actions = eng.advance(case.tau_plies, torch.from_numpy(u).cuda()).cpu().numpy()
        hist = eng.fregion("hist_pi").cpu().numpy()
        for g in range(G):
            if not alive[g]:
                assert actions[g] == -1
                continue
            tree = trees[g][players[g] if tpg == 2 else 0]
            pi, _ = tree.get_policy_value(states[g], tau=1 if plies_dev[g] < case.tau_plies else 0)
            assert [float(x) for x in pi] == pi_d[g].tolist(), "%s: policy differs, game %d move %d" % (case.name, g, move)
            np.testing.assert_array_equal(hist[g, min(plies_dev[g], hist.shape[1] - 1)], np.asarray(pi, dtype=np.float32))
            a = np_choice(pi, u[g])
            assert a == actions[g], "%s: move differs, game %d move %d" % (case.name, g, move)
            states[g], won = og.move(states[g], a, players[g])
            players[g] = 1 - players[g]
            if won or not og.possible_moves(states[g]):
                alive[g] = False
        st_dev, _ = eng.roots()
        assert st_dev == states
    oracle_trees = [t for row in trees for t in row]
    sc = eng.solver_counters()
    assert sc == {"stopped": sum(t.stopped for t in oracle_trees), "proven": sum(t.proven_edges for t in oracle_trees)}
    assert eng.counters()["errors"] == 0
    eng.close()
    return sc["proven"]


@pytest.mark.parametrize("case", SOLVER_PARITY_CASES + SOLVER_CHAIN_CASES,
                         ids=[c.name for c in SOLVER_PARITY_CASES + SOLVER_CHAIN_CASES])
def test_solver_parity_matrix(torch_cuda, case):
    proven = run_solver_case(torch_cuda, case)
    family = instances(case)["select"]
    _PROVEN_BY_FAMILY[family] = _PROVEN_BY_FAMILY.get(family, 0) + proven


def test_every_select_family_proved_edges(torch_cuda):
    """Not vacuous: every select instance the parity cases reach proved edges (runs after the parity cases)."""
    families = {instances(c)["select"] for c in SOLVER_PARITY_CASES}
    missing = [f for f in families if _PROVEN_BY_FAMILY.get(f, 0) == 0]
    assert len(_PROVEN_BY_FAMILY) >= len(families) and not missing, (missing, _PROVEN_BY_FAMILY)


# ------------------------------------------------------------------------------------------------ real network
def _c4_net(torch, trained):
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.model import DeviceNet, Net, load_checkpoint
    game = ConnectFour()
    torch.manual_seed(5)
    net = load_checkpoint(C4_CKPT, game) if trained else Net(game.obs_shape, game.action_space)
    return game, DeviceNet(net.eval(), game)


def _late_c4_roots(G, seed, plies=28):
    from oracle.games import ConnectFourOracle
    og = ConnectFourOracle()
    rng = np.random.default_rng(seed)
    return og, [random_position(og, rng, plies) for _ in range(G)]


def _check_tree_proofs(eng, og, nm, tree):
    """Every proven edge of arena `tree` against exact negamax; returns the number checked."""
    cap = eng.cfg.node_capacity
    n_nodes = int(eng.region("node_count")[tree].item())
    lo, hi = tree * cap, tree * cap + n_nodes
    proof = eng.pool("proof", lo, hi)[:, :eng.A].cpu().numpy()
    players = eng.region("node_player")[lo:hi].cpu().numpy()
    states = eng.game.states_from_boards(eng.region("node_board")[lo:hi].cpu().numpy().view(np.uint64))
    checked = 0
    for i in np.nonzero(proof.any(axis=1))[0]:
        for a in np.nonzero(proof[i])[0]:
            assert proof[i, a] == nm.edge_status(states[i], int(a), int(players[i])), (tree, states[i], int(a))
            checked += 1
    return checked


@pytest.mark.parametrize("trained", [False, True], ids=["random_init", "connect4_best_026"])
@pytest.mark.parametrize("compact", [False, True], ids=["keep", "compact"])
def test_proofs_are_exact_with_the_real_network(torch_cuda, trained, compact):
    from caro_ai_b200.engine import SelfPlayEngine
    game, dn = _c4_net(torch_cuda, trained)
    og, roots = _late_c4_roots(16, 11 + trained)
    nm = Negamax(og)
    eng = SelfPlayEngine(game, 16, trees_per_game=2, max_batch=8, node_capacity=2048 if compact else 4096, seed=3,
                         compact_tree=compact)
    eng.set_solver(3)
    eng.set_roots([r[0] for r in roots], [r[1] for r in roots])
    checked = 0
    for _ in range(14):
        SelfPlayEngine.play_multi([eng], dn, moves=1, count=10, batch=8, tau_plies=2, auto_restart=False)
        for tree in range(32):
            checked += _check_tree_proofs(eng, og, nm, tree)
        if int((eng.region("status") == 0).sum().item()) == 0:
            break
    assert checked > 100 and eng.solver_counters()["proven"] > 0
    assert eng.counters()["errors"] == 0
    eng.close()
    dn.close()


# ------------------------------------------------------------------------------------------------ switch and graphs
def _state(eng):
    out = {name: eng.region(name).cpu().numpy().copy() for name in ("nodes", "node_count", "root_board", "status", "ply", "result")}
    n = eng.replay_cursor()  # games finishing in the same ply take ring slots in any order: compare the rows as a set
    bd, pi, z = (eng.region("replay_board")[:n].cpu().numpy(), eng.fregion("replay_pi")[:n].cpu().numpy(),
                 eng.fregion("replay_z")[:n].cpu().numpy())
    out["replay"] = sorted((bd[i].tobytes(), pi[i].tobytes(), float(z[i])) for i in range(n))
    out["counters"] = eng.counters()
    out["solver"] = eng.solver_counters()
    return out


def _same(a, b):
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert a[k].tobytes() == b[k].tobytes(), k
        else:
            assert a[k] == b[k], k


@pytest.mark.parametrize("name", ["c4", "ttt3"])
def test_solver_off_is_the_parent(torch_cuda, name):
    """set_solver(0) leaves every tree, counter and replay row bit-identical to an engine that never heard of it."""
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    game = ConnectFour() if name == "c4" else TicTacToe()
    torch_cuda.manual_seed(1)
    dn = DeviceNet(Net(game.obs_shape, game.action_space).eval(), game)
    snaps = []
    for arm in range(2):
        eng = SelfPlayEngine(game, 64, trees_per_game=1, max_batch=8, node_capacity=16384, replay_capacity=64 * 42, seed=9)
        if arm:
            eng.set_solver(3)
            eng.set_solver(0)
        eng.reset(first_player=-1)
        eng.play(dn, dn, moves=10, count=4, batch=8, tau_plies=3, auto_restart=True)
        SelfPlayEngine.play_multi([eng], dn, moves=6, count=4, batch=8, tau_plies=3, auto_restart=True)
        snaps.append(_state(eng))
        eng.close()
    _same(snaps[0], snaps[1])
    assert snaps[1]["solver"] == {"stopped": 0, "proven": 0}


def test_graph_replays_follow_the_switch(torch_cuda):
    """A ply graph captured with the solver off runs it after set_solver(3), and stops after set_solver(0): the same
    sequence without graphs gives bit-identical trees and counters."""
    from caro_ai_b200.engine import SelfPlayEngine
    game, dn = _c4_net(torch_cuda, False)
    og, roots = _late_c4_roots(32, 21, plies=24)
    snaps = []
    for graph in (True, False):
        if not graph:
            os.environ["CARO_NO_GRAPH"] = "1"
        try:
            eng = SelfPlayEngine(game, 32, trees_per_game=2, max_batch=8, node_capacity=4096, seed=4)
            eng.set_roots([r[0] for r in roots], [r[1] for r in roots])
            ply = lambda: SelfPlayEngine.play_multi([eng], dn, moves=1, count=8, batch=8, tau_plies=2, auto_restart=False)
            for _ in range(2):
                ply()
            assert eng.solver_counters() == {"stopped": 0, "proven": 0}
            assert int(eng.pool("proof").sum().item()) == 0
            eng.set_solver(3)
            for _ in range(3):
                ply()
            on = eng.solver_counters()
            assert on["proven"] > 0
            eng.set_solver(0)
            for _ in range(2):
                ply()
            assert eng.solver_counters() == on
            snaps.append(_state(eng))
            eng.close()
        finally:
            os.environ.pop("CARO_NO_GRAPH", None)
    _same(snaps[0], snaps[1])
    dn.close()


@pytest.mark.parametrize("mask", [1, 2])
def test_per_player_mask_proves_only_that_players_tree(torch_cuda, mask):
    from caro_ai_b200.engine import SelfPlayEngine
    game, dn = _c4_net(torch_cuda, False)
    og, roots = _late_c4_roots(32, 31, plies=28)
    eng = SelfPlayEngine(game, 32, trees_per_game=2, max_batch=8, node_capacity=4096, seed=5)
    eng.set_solver(mask)
    eng.set_roots([r[0] for r in roots], [r[1] for r in roots])
    SelfPlayEngine.play_multi([eng], dn, moves=4, count=8, batch=8, tau_plies=0, auto_restart=False)
    cap = eng.cfg.node_capacity
    proof = eng.pool("proof").reshape(32, 2, cap, -1)
    on, off = (0, 1) if mask == 1 else (1, 0)
    assert int((proof[:, on] != 0).sum().item()) > 0
    assert int((proof[:, off] != 0).sum().item()) == 0
    eng.close()
    dn.close()


def test_refusals(torch_cuda):
    from caro_ai_b200 import _cabi
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour
    game = ConnectFour()
    one = SelfPlayEngine(game, 4, trees_per_game=1, node_capacity=64)
    two = SelfPlayEngine(game, 4, trees_per_game=2, node_capacity=64)
    vl = SelfPlayEngine(game, 4, trees_per_game=2, node_capacity=64, virtual_loss=True)
    for eng, mask in ((one, 1), (one, 2), (two, 4), (two, -1), (vl, 3), (vl, 1)):
        with pytest.raises(_cabi.CaroError):
            eng.set_solver(mask)
    one.set_solver(3)
    one.set_solver(0)
    for m in range(4):
        two.set_solver(m)
    vl.set_solver(0)
    assert int(two.region("solver_params")[0].item()) == 3
    for e in (one, two, vl):
        e.close()


# ------------------------------------------------------------------------------------------------ end to end
def test_session_with_solver(torch_cuda):
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.play_session import Session
    game = ConnectFour()
    og, roots = _late_c4_roots(1, 41, plies=30)
    sess = Session(game, C4_CKPT, player_moves_first=False, solver=True)
    sess.state = roots[0][0]
    np.random.seed(0)
    state = sess.state
    sess.move_bot()
    proof = sess.mcts_store.proof
    assert any(any(row) for row in proof.values())
    row = proof[state]
    nm = Negamax(og)
    assert all(st == UNKNOWN or st == nm.edge_status(state, a, game.player_black) for a, st in enumerate(row))
    if any(st == 1 for st in row):
        assert sess.moves[-1] == row.index(1)


def test_play_cli_with_solver(torch_cuda, capsys):
    from caro_ai_b200 import play
    assert play.main(["-g", "0", C4_CKPT, os.path.join(GOLDEN, "checkpoints", "connect4_best_025_10600.dat"), "-r", "8",
                      "--solver"]) == 0
    assert "Leaderboard:" in capsys.readouterr().out


def test_train_cli_with_solver(torch_cuda, tmp_path, capsys):
    from caro_ai_b200 import train as train_cli
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        random.seed(0)
        torch_cuda.manual_seed(0)
        assert train_cli.main(["-g", "1", "-n", "sv", "--games", "256", "--max-steps", "2", "--evaluate-every", "100",
                               "--solver"]) == 0
    finally:
        os.chdir(cwd)
    assert "Step 2, steps" in capsys.readouterr().out
