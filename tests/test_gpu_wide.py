"""128-filter networks on the GPU: the SIMT tower and the wide tcgen05 tower (csrc/net_wide.cu, fp16 and bf16 operands)
against PyTorch fp32, precision "auto", invariance of a leaf's outputs, routing, the self-play pipeline, and the
training / tournament / session entry points with wide checkpoints."""
import os
import random

import numpy as np
import pytest

from harness import oracle_for, random_position

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _wide_net(torch, game, blocks, seed, randomise_bn=True):
    from caro_ai_b200.model import Net
    torch.manual_seed(seed)
    net = Net(game.obs_shape, game.action_space, blocks=blocks, filters=128)
    if randomise_bn:
        with torch.no_grad():
            for m in net.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.running_mean.uniform_(-0.2, 0.2)
                    m.running_var.uniform_(0.7, 1.3)
                    m.weight.uniform_(0.6, 1.0)
                    m.bias.uniform_(-0.1, 0.1)
    return net.eval()


def _reference(torch, game, net, states, players):
    og = oracle_for(game)
    planes = torch.tensor(og.states_to_training_batch(states, players))
    with torch.no_grad():
        logits, val = net(planes)
    return torch.softmax(logits, dim=1).numpy(), val.numpy()[:, 0]


def _positions(game, rng, count):
    og = oracle_for(game)
    cells = game.obs_shape[1] * game.obs_shape[2]
    top = 30 if game.game_kind == 0 else min(40, max(1, cells - 4))
    return [random_position(og, rng, int(rng.integers(0, top))) for _ in range(count)]


def _games():
    from caro_ai_b200.game import ConnectFour, TicTacToe
    return [(ConnectFour(), 160), (TicTacToe(3, 3), 100), (TicTacToe(9, 5), 60), (TicTacToe(15, 5), 40)]


def test_wide_towers_match_pytorch_fp32(torch_cuda):
    """SIMT (impl 1) within 2e-4, the wide tower with fp16 operands (impl 7) within 1e-3 and with bf16 operands (impl 0)
    within 2e-3 of PyTorch fp32 at 1, 5 and 10 blocks on every board family."""
    torch = torch_cuda
    from caro_ai_b200.model import DeviceNet
    rng = np.random.default_rng(128)
    for game, count in _games():
        pos = _positions(game, rng, count)
        states, players = [p[0] for p in pos], [p[1] for p in pos]
        for blocks in (1, 5, 10):
            net = _wide_net(torch, game, blocks, 100 + blocks)
            ref_p, ref_v = _reference(torch, game, net, states, players)
            dn = DeviceNet(net, game, precision="fp32-simt")
            assert dn.filters == 128 and dn.blocks == blocks
            for impl, tol in ((1, 2e-4), (7, 1e-3), (0, 2e-3)):
                p, v = dn.forward_states(states, players, impl=impl)
                dp = float(np.abs(p.cpu().numpy() - ref_p).max())
                dv = float(np.abs(v.cpu().numpy() - ref_v).max())
                assert dp <= tol and dv <= tol, (type(game).__name__, game.obs_shape, blocks, impl, dp, dv)
            p3, v3 = dn.forward_states(states, players, impl=3)  # impl 3 is the bf16 wide tower as well
            p0, v0 = dn.forward_states(states, players, impl=0)
            assert torch.equal(p3, p0) and torch.equal(v3, v0)
            dn.close()


def test_auto_selects_a_tensor_core_tower_for_random_init_wide_nets(torch_cuda):
    torch = torch_cuda
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet
    rng = np.random.default_rng(5)
    for game, blocks, count in ((ConnectFour(), 5, 200), (TicTacToe(15, 5), 10, 40)):
        net = _wide_net(torch, game, blocks, 7, randomise_bn=False)
        dn = DeviceNet(net, game)
        cal = dn.calibration
        assert cal["filters"] == 128 and cal["selected"] in ("fp16", "bf16"), cal
        assert dn.precision == cal["selected"]
        pos = _positions(game, rng, count)  # not the probe set (random play-outs of another generator)
        states, players = [p[0] for p in pos], [p[1] for p in pos]
        ref_p, ref_v = _reference(torch, game, net, states, players)
        p, v = dn.forward_states(states, players)
        assert float(np.abs(p.cpu().numpy() - ref_p).max()) <= 1e-3 and float(np.abs(v.cpu().numpy() - ref_v).max()) <= 1e-3
        dn.close()


def test_wide_tower_outputs_do_not_depend_on_grid_batch_or_count(torch_cuda):
    """777 leaves: bit-identical at grid limits 0, 1 and 13, after a shuffle of the batch, and under a device-side count
    below max_count (rows past it keep their sentinel) -- for the in-kernel heads (Connect4, fp16) and the exported
    heads of large boards (15 x 15, bf16)."""
    torch = torch_cuda
    from caro_ai_b200 import _cabi
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet
    rng = np.random.default_rng(77)
    for game, impl in ((ConnectFour(), 7), (TicTacToe(15, 5), 0)):
        net = _wide_net(torch, game, 3, 9)
        dn = DeviceNet(net, game, precision="fp32-simt")
        base = _positions(game, rng, 97)
        pos = [base[i % len(base)] for i in range(777)]
        d_boards = torch.from_numpy(game.boards_from_states([p[0] for p in pos]).view(np.int64)).cuda()
        d_who = torch.tensor([p[1] for p in pos], dtype=torch.uint8, device="cuda")
        p_ref, v_ref = dn.forward_boards(d_boards, d_who, 777, impl)
        for lim in (1, 13, 0):
            dn.set_grid_limit(lim)
            p, v = dn.forward_boards(d_boards, d_who, 777, impl)
            assert torch.equal(p, p_ref) and torch.equal(v, v_ref), lim
        perm = torch.randperm(777, generator=torch.Generator().manual_seed(3)).cuda()
        p, v = dn.forward_boards(d_boards[perm].contiguous(), d_who[perm].contiguous(), 777, impl)
        assert torch.equal(p, p_ref[perm]) and torch.equal(v, v_ref[perm])
        A = game.action_space
        probs = torch.full((777, A), -7.0, dtype=torch.float32, device="cuda")
        values = torch.full((777,), -7.0, dtype=torch.float32, device="cuda")
        d_count = torch.tensor([301], dtype=torch.int32, device="cuda")
        _cabi.check(_cabi.lib().caro_net_forward(dn.handle, game.game_kind, game.n, game.k, d_boards.data_ptr(), d_who.data_ptr(),
                                                 d_count.data_ptr(), 777, probs.data_ptr(), values.data_ptr(), impl,
                                                 torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert torch.equal(probs[:301], p_ref[:301]) and torch.equal(values[:301], v_ref[:301])
        assert bool((probs[301:] == -7.0).all()) and bool((values[301:] == -7.0).all())
        dn.close()


def test_wide_handles_refuse_the_64_only_towers(torch_cuda):
    torch = torch_cuda
    from caro_ai_b200 import _cabi
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.model import DeviceNet
    game = ConnectFour()
    net = _wide_net(torch, game, 2, 1)
    with pytest.raises(ValueError, match="128"):
        DeviceNet(net, game, precision="bf16x3")
    dn = DeviceNet(net, game, precision="bf16")
    pos = _positions(game, np.random.default_rng(1), 8)
    for impl in (2, 4, 5, 6):
        with pytest.raises(_cabi.CaroError, match="128"):
            dn.forward_states([p[0] for p in pos], [p[1] for p in pos], impl=impl)
    dn.close()


def test_wide_pipeline_parts_reproduce_solo_runs(torch_cuda):
    """A 2-part play_multi with a wide network equals the two engines run alone (counters, roots, every node record):
    Connect4, and 15 x 15 with tree compaction (exported heads, slotted per launch), on the tower "auto" selects and on
    the SIMT tower (the parts' network passes overlap on their side streams)."""
    torch = torch_cuda
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet
    cases = [(game, games, cap, compact, precision) for precision in ("auto", "fp32-simt")
             for game, games, cap, compact in ((ConnectFour(), 64, 2048, False), (TicTacToe(15, 5), 48, 2048, True))]
    for game, games, cap, compact, precision in cases:
        dn = DeviceNet(_wide_net(torch, game, 3, 21, randomise_bn=False), game, precision=precision)
        assert dn.precision != "fp32-simt" if precision == "auto" else dn.precision == "fp32-simt"

        def engines():
            return [SelfPlayEngine(game, games, max_batch=8, node_capacity=cap, seed=41 + h, compact_tree=compact) for h in range(2)]

        solo = engines()
        for e in solo:
            e.play(dn, dn, moves=2, count=12, batch=8, tau_plies=10, auto_restart=True)
        pair = engines()
        SelfPlayEngine.play_multi(pair, dn, moves=2, count=12, batch=8, tau_plies=10, auto_restart=True)
        torch.cuda.synchronize()
        for a, b in zip(solo, pair):
            assert a.counters() == b.counters() and a.counters()["errors"] == 0
            assert a.roots() == b.roots()
            assert torch.equal(a.region("nodes"), b.region("nodes")), (type(game).__name__, precision)
        for e in solo + pair:
            e.close()
        dn.close()


def test_wide_training_tournament_and_session(torch_cuda, tmp_path, capsys):
    torch = torch_cuda
    from caro_ai_b200 import play as play_cli
    from caro_ai_b200 import train as train_cli
    from caro_ai_b200.game import TicTacToe
    from caro_ai_b200.model import load_checkpoint, save_checkpoint
    from caro_ai_b200.play_session import Session
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        random.seed(0)
        torch.manual_seed(0)
        assert train_cli.main(["-g", "1", "-n", "wide", "--games", "512", "--filters", "128", "--blocks", "2",
                               "--max-steps", "2", "--evaluate-every", "2"]) == 0
    finally:
        os.chdir(cwd)
    out = capsys.readouterr().out
    assert "Step 2, steps" in out and "Net evaluated, win ratio = " in out
    assert "(conv_2)" in out and "Conv2d(128, 128" in out  # the printed network is 2 x 128
    game = TicTacToe(3, 3)
    paths = []
    for seed in (1, 2):
        path = os.path.join(str(tmp_path), "wide_%d.dat" % seed)
        save_checkpoint(_wide_net(torch, game, 2, seed, randomise_bn=False), path)
        paths.append(path)
    assert load_checkpoint(paths[0], game).filters == 128
    assert play_cli.main(["-g", "1", paths[0], paths[1], "-r", "4"]) == 0
    out = capsys.readouterr().out
    assert "%s vs %s -> w=" % (paths[0], paths[1]) in out and "Leaderboard:" in out
    s = Session(game, paths[0], True)
    assert s.model.filters == 128 and s.model.blocks == 2
    s.move_bot()
    assert len(s.moves) == 1 and 0 <= s.moves[0] < 9
