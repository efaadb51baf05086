"""The split-precision wide tower (impl 8: csrc/net_wide.cu with bf16 hi + lo operands) on the GPU: every board size and
depth against the float64 reference, invariance of a leaf's outputs, exact homogeneity under a power-of-two rescaling,
precision "auto" on the "trained-like" test net of wide_split_net.py, DeviceNet.update(), the two-part self-play
pipeline, and play.py / Session with a checkpoint of the test net."""
import os

import numpy as np
import pytest

import net_reference as R
import wide_split_net as S
from test_gpu_net_matrix import _check, _device, _forward_repeated, _take, leaf_counts

pytestmark = pytest.mark.gpu

X3 = S.IMPL_WIDE_X3

# (max |p - p_ref|, max |v - v_ref|, max |log p - log p_ref|) of impl 8 on the matrix nets, per board class ("small": up
# to 64 cells, FC heads in the tower; "large": the heads GEMM follows) and depth (True: more than 10 residual blocks).
# 3x the largest deviation measured over this matrix on an NVIDIA B200 (1,000 W power limit; none reached the SIMT tower's
# 2e-4 ceiling), raised to net_reference.FLOOR.
BOUNDS_X3 = {("small", False): (2.1e-07, 5.0e-06, 4.2e-06), ("small", True): (8.5e-06, 2.6e-06, 1.7e-04),
             ("large", False): (1.9e-07, 1.7e-06, 1.3e-05), ("large", True): (2.1e-05, 1.8e-06, 6.4e-04)}


def bound_x3(game, blocks):
    b = BOUNDS_X3[(R.board_class(game), blocks > 10)]
    return tuple(max(x, f) for x, f in zip(b, R.FLOOR))


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _matrix_cases():
    return [(g, b) for g in R.matrix_games() for b in R.matrix_depths(g)]


@pytest.mark.parametrize("case", _matrix_cases(), ids=lambda c: "%s-b%d" % (R.game_label(c[0]), c[1]))
def test_split_wide_tower_matches_the_float64_reference(torch_cuda, case):
    """Impl 8 on the matrix net of every board and depth: empty, random and dense positions, at leaf counts around its
    group size, every repeated leaf bit-identical to its first copy."""
    torch = torch_cuda
    from caro_ai_b200.model import DeviceNet, fold_state_dict
    game, blocks = case
    net = R.matrix_net(game, 128, blocks)
    shape = R.shape_of(game, 128, blocks)
    pos = R.base_positions(game, 2)
    ref = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, R.planes_of(game, pos), device="cuda")
    dn = DeviceNet(net, game, precision="fp32-simt")
    d_boards, d_who = _device(torch, game, pos)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    bound = bound_x3(game, blocks)
    what = (R.game_label(game), blocks, X3)
    p, v = dn.forward_boards(d_boards, d_who, len(pos), X3)
    devs = [_check(p, v, ref, bound, what)]
    for count in leaf_counts(R.group_boards("wide_bf16", game), sms):  # the split tower's group is the wide tower's
        p, v, idx = _forward_repeated(torch, dn, d_boards, d_who, count, X3)
        devs.append(_check(p, v, _take(ref, idx), bound, what + (count,)))
    print("deviation", what, tuple(max(d[m] for d in devs) for m in range(3)))
    dn.close()


def _cases_both_heads():
    from caro_ai_b200.game import ConnectFour, TicTacToe
    return [ConnectFour(), TicTacToe(15, 5)]


@pytest.mark.parametrize("game", _cases_both_heads(), ids=R.game_label)
def test_split_wide_outputs_do_not_depend_on_grid_batch_or_count(torch_cuda, game):
    """777 leaves of the test net: bit-identical at grid limits 0, 1 and 13, after a shuffle, under a device-side count
    below max_count (rows past it keep their sentinel), and for every repeated leaf -- in-kernel heads (Connect4) and
    exported heads (15 x 15)."""
    torch = torch_cuda
    from caro_ai_b200 import _cabi
    from caro_ai_b200.model import DeviceNet
    _, sd = S.trained_like_net(game, 3)
    dn = DeviceNet(sd, game, precision="bf16x3-wide")
    assert dn.impl == X3
    base = R.base_positions(game, 7)
    n = 777
    pos = [base[i % len(base)] for i in range(n)]
    d_boards, d_who = _device(torch, game, pos)
    p_ref, v_ref, _ = _forward_repeated(torch, dn, d_boards[:len(base)], d_who[:len(base)], n, X3)
    for lim in (1, 13, 0):
        dn.set_grid_limit(lim)
        p, v = dn.forward_boards(d_boards, d_who, n, X3)
        assert torch.equal(p, p_ref) and torch.equal(v, v_ref), lim
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(3)).cuda()
    p, v = dn.forward_boards(d_boards[perm].contiguous(), d_who[perm].contiguous(), n, X3)
    assert torch.equal(p, p_ref[perm]) and torch.equal(v, v_ref[perm])
    A = game.action_space
    probs = torch.full((n, A), -7.0, dtype=torch.float32, device="cuda")
    values = torch.full((n,), -7.0, dtype=torch.float32, device="cuda")
    d_count = torch.tensor([301], dtype=torch.int32, device="cuda")
    _cabi.check(_cabi.lib().caro_net_forward(dn.handle, game.game_kind, game.n, game.k, d_boards.data_ptr(), d_who.data_ptr(),
                                             d_count.data_ptr(), n, probs.data_ptr(), values.data_ptr(), X3,
                                             torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert torch.equal(probs[:301], p_ref[:301]) and torch.equal(values[:301], v_ref[:301])
    assert bool((probs[301:] == -7.0).all()) and bool((values[301:] == -7.0).all())
    dn.close()


def _rescale_games():
    from caro_ai_b200.game import ConnectFour, TicTacToe
    return [ConnectFour(), TicTacToe(9, 5), TicTacToe(15, 5)]


@pytest.mark.parametrize("game", _rescale_games(), ids=R.game_label)
def test_split_wide_tower_is_exactly_homogeneous(torch_cuda, game):
    """The test net and its 2^17-rescaled state dict give bit-identical outputs on impl 8 (bf16 hi + lo keep fp32's
    exponent range); both are within the matrix bound of the float64 reference."""
    torch = torch_cuda
    from caro_ai_b200.model import DeviceNet, fold_state_dict
    net, sd = S.trained_like_net(game, 5)
    shape = R.shape_of(game, 128, 5)
    pos = R.base_positions(game, 2)
    ref = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, R.planes_of(game, pos), device="cuda")
    d_boards, d_who = _device(torch, game, pos)
    dn = DeviceNet(net, game, precision="bf16x3-wide")
    ds = DeviceNet(sd, game, precision="bf16x3-wide")
    p0, v0 = dn.forward_boards(d_boards, d_who, len(pos))
    p1, v1 = ds.forward_boards(d_boards, d_who, len(pos))
    assert torch.equal(p0, p1) and torch.equal(v0, v1)
    dev = _check(p1, v1, ref, None, (R.game_label(game), "rescaled"))
    assert dev[0] <= 1e-4 and dev[1] <= 1e-4, dev
    dn.close()
    ds.close()


@pytest.mark.parametrize("game", _cases_both_heads(), ids=R.game_label)
def test_auto_selects_the_split_wide_tower_for_the_trained_like_net(torch_cuda, game, monkeypatch):
    """On the test net "auto" rejects fp16 (range) and bf16 (precision), selects "bf16x3-wide" (impl 8) with its measured
    deviation recorded, and the selected tower holds 1e-3 on held-out positions; with a margin no tower can meet, the
    SIMT tower is still selected."""
    torch = torch_cuda
    from caro_ai_b200 import model
    from caro_ai_b200.model import DeviceNet, fold_state_dict
    net, sd = S.trained_like_net(game, 5)
    limit = model.CALIBRATION_MARGIN * model.PRIOR_TOLERANCE
    dn = DeviceNet(sd, game)
    cal = dn.calibration
    assert cal["filters"] == 128, cal
    fp16_fails = not (cal["fp16_max_abs_prior_diff"] <= limit and cal["fp16_max_abs_value_diff"] <= limit)
    bf16_fails = cal["bf16_max_abs_prior_diff"] > limit or cal["bf16_max_abs_value_diff"] > limit
    assert fp16_fails and bf16_fails, cal  # the premise: both one-pass towers miss the check
    assert cal["selected"] == "bf16x3-wide" and dn.precision == "bf16x3-wide" and dn.impl == X3, cal
    assert cal["split_max_abs_prior_diff"] <= 1e-4 and cal["split_max_abs_value_diff"] <= 1e-4, cal
    shape = R.shape_of(game, 128, 5)
    held = R.base_positions(game, 5)
    ref = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, R.planes_of(game, held), device="cuda")
    p, v = dn.forward_states([q[0] for q in held], [q[1] for q in held])
    dev = _check(p, v, ref, None, (R.game_label(game), "auto", dn.precision))
    assert dev[0] <= 1e-3 and dev[1] <= 1e-3, (dev, cal)
    dn.close()
    monkeypatch.setattr(model, "CALIBRATION_MARGIN", 1e-9)
    ds = DeviceNet(sd, game)
    assert ds.precision == "fp32-simt" and ds.impl == model.IMPL_SIMT, ds.calibration
    assert "split_max_abs_prior_diff" in ds.calibration
    ds.close()


def _comparable(calibration):
    return {k: ("nan" if isinstance(v, float) and v != v else v) for k, v in calibration.items()}


@pytest.mark.parametrize("game", _cases_both_heads(), ids=R.game_label)
def test_update_repacks_the_split_images(torch_cuda, game):
    """After update(test net) a wide handle gives what a fresh DeviceNet(test net) gives, bit for bit, on impl 8 (the lo
    weight image is repacked, and on 15 x 15 the heads GEMM image) and selects the split tower again."""
    torch = torch_cuda
    from caro_ai_b200.model import DeviceNet, Net
    torch.manual_seed(3)
    net_a = Net(game.obs_shape, game.action_space, blocks=5, filters=128)
    R.randomise_bn(torch, net_a)
    net_a.eval()
    _, sd = S.trained_like_net(game, 5)
    pos = R.base_positions(game, 6)
    d_boards, d_who = _device(torch, game, pos)
    dn = DeviceNet(net_a, game)
    assert dn.precision in ("fp16", "bf16"), dn.calibration
    p_a, _ = dn.forward_boards(d_boards, d_who, len(pos), X3)
    dn.update(sd)
    fresh = DeviceNet(sd, game)
    assert dn.precision == fresh.precision == "bf16x3-wide"
    assert _comparable(dn.calibration) == _comparable(fresh.calibration)  # the fp16 deviations are NaN (overflow)
    p0, v0 = dn.forward_boards(d_boards, d_who, len(pos), X3)
    p1, v1 = fresh.forward_boards(d_boards, d_who, len(pos), X3)
    assert torch.equal(p0, p1) and torch.equal(v0, v1)
    assert not torch.equal(p0, p_a)
    fresh.close()
    dn.close()


def test_split_wide_pipeline_parts_reproduce_solo_runs(torch_cuda):
    """A 2-part play_multi on impl 8 equals the two engines run alone (counters, roots, every node record): Connect4,
    and 15 x 15 with tree compaction (exported heads, slotted per launch)."""
    torch = torch_cuda
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet
    for game, games, cap, compact in ((ConnectFour(), 64, 2048, False), (TicTacToe(15, 5), 48, 2048, True)):
        _, sd = S.trained_like_net(game, 3)
        dn = DeviceNet(sd, game)
        assert dn.impl == X3, dn.calibration

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
            assert torch.equal(a.region("nodes"), b.region("nodes")), R.game_label(game)
        for e in solo + pair:
            e.close()
        dn.close()


def test_checkpoint_of_the_test_net_runs_the_split_tower_in_play_and_session(torch_cuda, tmp_path, capsys, monkeypatch):
    torch = torch_cuda
    from caro_ai_b200 import play as play_cli
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.model import DeviceNet, Net
    from caro_ai_b200.play_session import Session
    game = ConnectFour()
    _, sd = S.trained_like_net(game, 5)
    path = os.path.join(str(tmp_path), "wide_split.dat")
    torch.save(sd, path)
    made = []

    class Recording(DeviceNet):
        def __init__(self, *a, **kw):
            super().__init__(*a, **kw)
            made.append(self)

    monkeypatch.setattr(play_cli, "DeviceNet", Recording)
    assert play_cli.main(["-g", "0", path, path, "-r", "2"]) == 0
    assert "%s vs %s -> w=" % (path, path) in capsys.readouterr().out
    assert len(made) == 2 and all(d.impl == X3 for d in made), [d.calibration for d in made]
    s = Session(game, path, True)
    assert s.model.filters == 128 and s.model.blocks == 5
    s.move_bot()
    assert len(s.moves) == 1 and 0 <= s.moves[0] < 7
    (dn,) = [entry[1] for entry in s.mcts_store._device_nets.values()]
    assert dn.impl == X3, dn.calibration
    # the split wide tower exists for 128 filters only
    net64 = Net(game.obs_shape, game.action_space).eval()
    with pytest.raises(ValueError):
        DeviceNet(net64, game, precision="bf16x3-wide")
    d64 = DeviceNet(net64, game, precision="bf16")
    from caro_ai_b200 import _cabi
    with pytest.raises(_cabi.CaroError, match="128"):
        d64.forward_states([game.initial_state], [0], impl=X3)
    d64.close()
