"""The engine flags that change the search (MASK_PRIORS, FRESH_TREE, RECYCLE_TREE) against their oracle statement
(tests/flag_reference.py), bit for bit, on the B200 (run with -m gpu).

Each case is the parity run of tests/test_gpu_search_matrix.py with the flags on: after every minibatch the searched trees
(N, W, Q, P and the node sets), after every move pi, Q, the sampled moves, roots and status, and every tree once the
advance has cleared or kept it.  tests/test_host_flag_matrix.py proves which kernel instance each case reaches.  The
last test runs the benchmark's virtual-loss row (virtual loss + masked priors, two play_multi parts, the bf16 tower)
through its own pipeline against twin engines stepped launch by launch and against the oracle."""
import os
import subprocess

import numpy as np
import pytest

from flag_reference import FRESH_CASES, MASK_CASES, MASK_VL_CASES, PIPELINE_CASE, RECYCLE_CASES, MaskedVirtualLossTree, \
    OracleGames, flag_instances
from harness import diff_tree, np_choice, random_position
from search_matrix import STUBS, host_noise, make_roots

pytestmark = pytest.mark.gpu

STREAM_CHOICE = 0x43484F49  # kStreamChoice, csrc/rng.cuh


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def run_flag_case(torch, case):
    """Engine and oracle side by side through `case.moves` moves of `case.count` minibatches; returns the OracleGames,
    whose counters say what the flags did."""
    from caro_ai_b200.engine import SelfPlayEngine
    game = case.product_game()
    G, A, batch, tpg = case.G, case.A, case.batch, case.trees_per_game
    rng = np.random.default_rng(case.seed)
    roots = make_roots(case, case.oracle_game(), rng)
    eng = SelfPlayEngine(game, G, trees_per_game=tpg, max_batch=case.max_batch, node_capacity=case.capacity,
                         seed=case.seed, virtual_loss=case.virtual_loss, mask_priors=case.mask_priors,
                         fresh_tree=case.fresh_tree, recycle_tree=case.recycle_tree)
    eng.set_roots([r[0] for r in roots], [r[1] for r in roots])
    games = OracleGames(case, roots)
    stub = STUBS[case.stub]

    def check_trees(where, searched_only):
        for g in range(G):
            if not games.alive[g]:
                continue
            for t in ([games.tree_index(g)] if searched_only else range(tpg)):
                errs = diff_tree(eng.export_tree(g * tpg + t), games.trees[g][t], A)
                assert not errs, "%s: %s, game %d tree %d: %s" % (case.name, where, g, t, errs[:5])

    for move in range(case.moves):
        if case.fresh_tree:
            counts = eng.region("node_count").cpu().numpy()
            for g in range(G):
                for t in range(tpg):
                    if games.alive[g]:
                        assert counts[g * tpg + t] == 0 and len(games.trees[g][t]) == 0, (case.name, move, g, t)
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
            games.minibatch(noise)
            check_trees("move %d minibatch %d" % (move, i), searched_only=True)
        pi_d, q_d, _ = eng.root_policy(2, case.tau_plies)
        pi_d, q_d = pi_d.cpu().numpy(), q_d.cpu().numpy()
        assert (eng.region("ply").cpu().numpy()[games.alive] == games.ply).all()
        alive = list(games.alive)
        policies = {g: games.policy(g) for g in range(G) if alive[g]}
        u = rng.random(G)
        actions = eng.advance(case.tau_plies, torch.from_numpy(u).cuda()).cpu().numpy()
        want = games.advance(u)
        for g in range(G):
            if not alive[g]:
                assert actions[g] == -1
                continue
            pi, q = policies[g]
            assert [float(x) for x in pi] == pi_d[g].tolist(), "%s: policy differs, game %d move %d" % (case.name, g, move)
            np.testing.assert_allclose(np.array([float(x) for x in q]), q_d[g], atol=1e-6)
            assert actions[g] == want[g], "%s: sampled move differs, game %d move %d" % (case.name, g, move)
        check_trees("after move %d" % move, searched_only=False)
        st_dev, pl_dev = eng.roots()
        status = eng.region("status").cpu().numpy()
        for g in range(G):
            assert st_dev[g] == games.states[g] and (status[g] == 0) == games.alive[g], (case.name, g, move)
            if games.alive[g]:
                assert pl_dev[g] == games.players[g]
    assert eng.counters()["errors"] == 0
    eng.close()
    return games


@pytest.mark.parametrize("case", MASK_CASES + MASK_VL_CASES, ids=[c.name for c in MASK_CASES + MASK_VL_CASES])
def test_masked_priors_match_the_oracle(torch_cuda, case):
    games = run_flag_case(torch_cuda, case)
    assert games.masked_nodes() > 0, "%s: no created node had illegal mass to remove" % case.name


@pytest.mark.parametrize("case", FRESH_CASES, ids=[c.name for c in FRESH_CASES])
def test_fresh_tree_matches_the_oracle(torch_cuda, case):
    """Every advance of a game that goes on empties its trees; the next search starts from nothing and meets positions
    the emptied tree held (their hash slots belong to the previous generation)."""
    ev = run_flag_case(torch_cuda, case).events
    assert ev["cleared"] > 0 and ev["kept"] == 0 and ev["revisits"] > 0, (case.name, ev)


@pytest.mark.parametrize("case", RECYCLE_CASES, ids=[c.name for c in RECYCLE_CASES])
def test_recycle_tree_matches_the_oracle(torch_cuda, case):
    """Trees kept and trees cleared, and searches after a clear that revisit positions the cleared tree held; the
    exact-threshold and one-of-two events are asserted on the host (tests/test_host_flag_matrix.py)."""
    ev = run_flag_case(torch_cuda, case).events
    assert ev["kept"] > 0 and ev["cleared"] > 0 and ev["revisits"] > 0, (case.name, ev)


# ------------------------------------------------------------------------------------------------ benchmark's VL row
class RecordedMaskedVirtualLossTree(MaskedVirtualLossTree):
    """The virtual-loss oracle with masked priors over eight lanes (expand_backup_group8_kernel), fed the Dirichlet
    vectors the engine's Philox sampler produced and the tower's rows for the very leaves it asks about."""

    def __init__(self, game):
        super().__init__(game, gw=8)
        self.rows = {}

    def evaluate(self, states, players, net, device="cpu"):
        pri = np.stack([self.rows[s][0] for s in states]).astype(np.float32)
        val = np.array([self.rows[s][1] for s in states], dtype=np.float32)
        return pri, val


def _philox():
    from conftest import ROOT
    from resign_reference import HOSTCHECK, philox
    if not os.path.exists(HOSTCHECK):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC",
                               os.path.join(ROOT, "tests", "native", "hostcheck.cpp"), "-o", HOSTCHECK])
    return philox


def test_benchmark_virtual_loss_row_through_its_pipeline(torch_cuda):
    """bench.py's connect4_4096_games_virtual_loss configuration at a small game count: virtual loss + masked priors,
    two play_multi parts (one CUDA graph per ply; lean_tree puts expand + back-up on the eight-lane kernel), batch 8,
    Philox noise, the bf16 tcgen05 tower, roots from random play-outs so that full columns occur.  (1) Twin engines
    stepped launch by launch through the C ABI (the 32-lane expand kernel) equal the pipelined engines bit for bit;
    (2) sampled games replayed in the virtual-loss oracle with masked priors over eight lanes, the recorded noise and
    tower rows give identical trees after every minibatch, policies, and moves drawn with the engine's Philox uniform."""
    torch = torch_cuda
    from resign_reference import u01d
    from caro_ai_b200 import _cabi
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.model import DeviceNet, Net
    philox = _philox()
    case = PIPELINE_CASE
    inst = flag_instances(case)
    assert inst["expand"] == "expand_backup_group8_kernel<C4Rules>" and inst["expand_stepped"] != inst["expand"]
    game, og = case.product_game(), case.oracle_game()
    A, Bt, Cn, Gp, parts = case.A, case.batch, case.count, case.G, case.parts
    torch.manual_seed(0)
    dn = DeviceNet(Net(game.obs_shape, game.action_space).eval(), game, precision="bf16")
    rng = np.random.default_rng(case.seed)
    roots = [[random_position(og, rng, (0, 14, 24, 32)[g % 4]) for g in range(Gp)] for _ in range(parts)]

    def engines():
        es = [SelfPlayEngine(game, Gp, max_batch=Bt, node_capacity=case.capacity, seed=case.seed + h,
                             virtual_loss=True, mask_priors=True) for h in range(parts)]
        for e, r in zip(es, roots):
            e.set_roots([s for s, _ in r], [p for _, p in r])
        return es

    fast = engines()
    SelfPlayEngine.play_multi(fast, dn, moves=case.moves, count=Cn, batch=Bt, tau_plies=10, auto_restart=True)
    twins = engines()
    sample = [0, 1, 2, 3, 21, 42, 63]
    trees = {(h, g): RecordedMaskedVirtualLossTree(og) for h in range(parts) for g in sample}
    tracked = set(trees)  # sampled games still in their first game (a finished game restarts from an empty board)
    lib = _cabi.lib()
    stream = torch.cuda.current_stream().cuda_stream
    noise_buf = torch.empty((Gp, Bt, A), dtype=torch.float64, device="cuda")
    probs = torch.empty((Gp * Bt, A), dtype=torch.float32, device="cuda")
    values = torch.empty((Gp * Bt,), dtype=torch.float32, device="cuda")
    gidx = torch.tensor(sample, device="cuda")
    leaf_evals = 0
    for ply in range(case.moves):
        root = {}
        for h, e in enumerate(twins):
            st, pl = e.roots()
            for g in sample:
                root[(h, g)] = (st[g], pl[g])
        for mb in range(Cn):
            for h, e in enumerate(twins):
                e.select(Bt, mb, None, noise_out=noise_buf)
                e.plan(Bt)
                _cabi.check(lib.caro_net_forward(dn.handle, game.game_kind, 0, 0, e.region("leaf_board").data_ptr(),
                                                 e.region("leaf_player").data_ptr(), e.region("leaf_count").data_ptr(),
                                                 Gp * Bt, probs.data_ptr(), values.data_ptr(), dn.impl, stream))
                kind = e.region("desc_kind")[gidx].cpu().numpy()
                slot = e.region("desc_slot")[gidx].cpu().numpy()
                boards = e.region("desc_board")[gidx].cpu().numpy().view(np.uint64)
                nz = noise_buf[gidx].cpu().numpy()
                sl = torch.from_numpy(np.maximum(slot, 0).reshape(-1).astype(np.int64)).cuda()
                prow = probs[sl].cpu().numpy().reshape(len(sample), Bt, A)
                vrow = values[sl].cpu().numpy().reshape(len(sample), Bt)
                e.expand_backup(Bt, probs, values)
                for i, g in enumerate(sample):
                    if (h, g) not in tracked:
                        continue
                    states = game.states_from_boards(boards[i])
                    t = trees[(h, g)]
                    t.rows = {}
                    for j in range(Bt):
                        if kind[i, j] == 2 and slot[i, j] >= 0:
                            t.rows[states[j]] = (prow[i, j], vrow[i, j])
                            leaf_evals += 1
                    s, p = root[(h, g)]
                    t.minibatch(Bt, s, p, nz[i])
                    errs = diff_tree(e.export_tree(g), t, A)
                    assert not errs, "part %d game %d ply %d minibatch %d: %s" % (h, g, ply, mb, errs[:5])
        for h, e in enumerate(twins):
            pi_d = e.root_policy(2, 10)[0][gidx].cpu().numpy()
            uid = e.region("uid").cpu().numpy().astype(np.uint64)
            dev_ply = e.region("ply").cpu().numpy()
            actions = e.advance(10, None, auto_restart=True).cpu().numpy()
            st, pl = e.roots()
            for i, g in enumerate(sample):
                if (h, g) not in tracked:
                    continue
                s, p = root[(h, g)]
                pi, _ = trees[(h, g)].get_policy_value(s, tau=1)
                assert [float(x) for x in pi] == pi_d[i].tolist(), "part %d game %d ply %d: policy" % (h, g, ply)
                seed = case.seed + h
                r = philox(int(uid[g]) & 0xFFFFFFFF, int(uid[g]) >> 32, int(dev_ply[g]), 0,
                           (seed & 0xFFFFFFFF) ^ STREAM_CHOICE, seed >> 32)
                assert actions[g] == np_choice(pi, u01d(r[0], r[1])), "part %d game %d ply %d: move" % (h, g, ply)
                s2, won = og.move(s, int(actions[g]), p)
                if won or not og.possible_moves(s2):
                    tracked.discard((h, g))
                else:
                    assert st[g] == s2 and pl[g] == 1 - p
    assert len(tracked) >= len(trees) // 2, "too few sampled games lasted both plies"
    assert leaf_evals > len(trees) * case.moves * Cn
    assert sum(t.masked_nodes for t in trees.values()) > 0, "no created node had illegal mass to remove"
    torch.cuda.synchronize()
    for a, b in zip(fast, twins):
        ca, cb = a.counters(), b.counters()
        assert ca == cb and ca["errors"] == 0 and ca["descents"] == Gp * Bt * Cn * case.moves
        assert a.roots() == b.roots()
        for name in ("nodes", "node_count", "ply", "status"):
            assert torch.equal(a.region(name), b.region(name)), name
    for e in fast + twins:
        e.close()
    dn.close()
