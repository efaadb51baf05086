"""Every network tower on every board size against the float64 reference of tests/net_reference.py.

Matrix: Connect4 and TicTacToe(n, min(n, 5)) for n = 2 .. 15, 64 and 128 filters, 1 and 5 residual blocks (20 on Connect4,
8 x 8 and 15 x 15), every impl of caro_net_forward.  Positions: the empty board with each side to move, random play-outs and
dense boards.  Per tower: finite outputs, priors summing to 1, max |p - p_ref|, |v - v_ref| and |log p - log p_ref| within
the tower's bound (net_reference.BOUNDS), at leaf counts around each tower's group size, with every repeated leaf
bit-identical to its first copy.  Also: the in-kernel FC heads past the head-feature slot (32,769 leaves), exact
homogeneity under a power-of-two rescaling of the residual stream, precision "auto" on the rescaled nets, DeviceNet.update()
on 128-filter handles, and the combinations the library refuses."""
import numpy as np
import pytest

import net_reference as R

pytestmark = pytest.mark.gpu

HEADFEAT_SLOT = 32768  # leaves of one head-feature slot (net_tc.cu / net_wide.cu); larger launches run the FC heads in the tower


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def refused(game, filters, impl):
    """Combinations caro_net_forward refuses: the row-tiled-only impls 5 and 7 of 64-filter handles on boards larger than
    6 x 7, and the split-precision and CTA-pair impls 2, 4, 5 and 6 of 128-filter handles."""
    _, h, w = game.obs_shape
    if filters == 128:
        return impl in (2, 4, 5, 6)
    return impl in (5, 7) and not (h <= 6 and w <= 7)


def _device(torch, game, positions):
    d_boards = torch.from_numpy(game.boards_from_states([p[0] for p in positions]).view(np.int64)).cuda()
    d_who = torch.tensor([p[1] for p in positions], dtype=torch.uint8, device="cuda")
    return d_boards, d_who


def _take(ref, idx):
    return tuple(r[idx] for r in ref)


def _check(p, v, ref, bound, what):
    """Finite, normalised, within ``bound`` of ``ref``; returns the deviations.  ``bound`` None checks all but the bound."""
    p, v = p.cpu().numpy(), v.cpu().numpy()
    assert np.isfinite(p).all() and np.isfinite(v).all(), what
    assert float(np.abs(p.astype(np.float64).sum(axis=1) - 1.0).max()) <= 1e-5, what
    dev = R.deviations(p, v, ref)
    if bound is not None:
        assert all(dev[m] <= bound[m] for m in range(3)), (what, dev, bound)
    return dev


def leaf_counts(nb, sms):
    """Around a tower's group of nb boards: one leaf, a group short of one, one group, one over, one group per SM, and one
    group more than there are SMs."""
    return sorted({c for c in (1, nb - 1, nb, nb + 1, sms * nb, sms * nb + 1) if c >= 1})


def _forward_repeated(torch, dn, d_boards, d_who, count, impl):
    """``count`` leaves cycling through the base positions; every copy of a position must equal its first one bitwise."""
    nbase = d_who.numel()
    idx = np.arange(count) % nbase
    t = torch.from_numpy(idx).cuda()
    p, v = dn.forward_boards(d_boards[t].contiguous(), d_who[t].contiguous(), count, impl)
    if count > nbase:
        assert torch.equal(p, p[t]) and torch.equal(v, v[t]), ("copies differ", impl, count)
    return p, v, idx


def run_case(torch, game, filters, blocks, check_bounds=True):
    """The matrix for one (board, width, depth): {tower: worst deviations}."""
    from caro_ai_b200 import _cabi
    from caro_ai_b200.model import DeviceNet, fold_state_dict
    net = R.matrix_net(game, filters, blocks)
    shape = R.shape_of(game, filters, blocks)
    pos = R.base_positions(game, 2)
    ref = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, R.planes_of(game, pos), device="cuda")
    dn = DeviceNet(net, game, precision="fp32-simt")
    d_boards, d_who = _device(torch, game, pos)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    worst = {}
    for impl in R.impls_of(filters):
        tower = R.tower_of(game, filters, impl)
        what = (R.game_label(game), filters, blocks, impl, tower)
        assert (tower is None) == refused(game, filters, impl), what
        if tower is None:
            with pytest.raises(_cabi.CaroError):
                dn.forward_boards(d_boards, d_who, len(pos), impl)
            continue
        bound = R.bound_of(tower, game, blocks) if check_bounds else None
        p, v = dn.forward_boards(d_boards, d_who, len(pos), impl)
        devs = [_check(p, v, ref, bound, what)]
        for count in leaf_counts(R.group_boards(tower, game), sms):
            p, v, idx = _forward_repeated(torch, dn, d_boards, d_who, count, impl)
            devs.append(_check(p, v, _take(ref, idx), bound, what + (count,)))
        worst[tower] = tuple(max(d[m] for d in devs) for m in range(3))
    dn.close()
    return worst


@pytest.mark.parametrize("case", R.matrix_cases(), ids=lambda c: "%s-f%d-b%d" % (R.game_label(c[0]), c[1], c[2]))
def test_every_tower_matches_the_float64_reference(torch_cuda, case):
    run_case(torch_cuda, *case)


def _large_count_cases():
    from caro_ai_b200.game import TicTacToe
    return [(TicTacToe(n, 5), f) for n in (9, 15) for f in (64, 128)]


@pytest.mark.parametrize("case", _large_count_cases(), ids=lambda c: "%s-f%d" % (R.game_label(c[0]), c[1]))
def test_head_feature_slot_boundary(torch_cuda, case):
    """32,768 leaves fill one head-feature slot (FC heads in the heads GEMM); 32,769 make the tower run them itself.  Both
    against the reference, on every tensor-core tower of boards with more than 64 cells."""
    torch = torch_cuda
    from caro_ai_b200.model import DeviceNet, fold_state_dict
    game, filters = case
    net = R.matrix_net(game, filters, 1)
    shape = R.shape_of(game, filters, 1)
    pos = R.base_positions(game, 2)
    ref = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, R.planes_of(game, pos), device="cuda")
    dn = DeviceNet(net, game, precision="fp32-simt")
    d_boards, d_who = _device(torch, game, pos)
    for impl in ((0, 7) if filters == 128 else (3, 4)):
        tower = R.tower_of(game, filters, impl)
        for count in (HEADFEAT_SLOT, HEADFEAT_SLOT + 1):
            p, v, idx = _forward_repeated(torch, dn, d_boards, d_who, count, impl)
            _check(p, v, _take(ref, idx), R.bound_of(tower, game, 1), (R.game_label(game), filters, impl, count))
    dn.close()


RESCALE = 2.0 ** 17


def _rescale_cases():
    from caro_ai_b200.game import ConnectFour, TicTacToe
    return [(g, f) for g in (ConnectFour(), TicTacToe(9, 5), TicTacToe(15, 5)) for f in (64, 128)]


def exact_under_rescaling(game, filters):
    """Impls whose every stage is exactly homogeneous in the residual stream: bf16 or fp32 operands, fp32 accumulation,
    LeakyReLU, and head convolutions whose products (w / s)(s v) equal w v.  The SIMT tower at both widths, the wide bf16
    tower, and on boards past 8 x 8 the one-pass and split tap-per-MMA towers followed by the heads GEMM.  Not in this
    list: the fp16 towers (s v leaves fp16's range) and the row-tiled bf16 tower, whose residual stream carries an e5m2
    tail (net_rt.cu) of a narrower range."""
    _, h, w = game.obs_shape
    if filters == 128:
        return (1, 0, 3)
    return (1, 3, 4) if h * w > 64 else (1,)


@pytest.mark.parametrize("case", _rescale_cases(), ids=lambda c: "%s-f%d" % (R.game_label(c[0]), c[1]))
def test_power_of_two_rescaling(torch_cuda, case):
    """Multiplying the residual stream by 2^17 through the BatchNorm parameters leaves the exactly homogeneous towers
    bit-identical and the row-tiled bf16 tower within its bound; precision "auto" then never picks fp16, keeps 1e-3 on
    held-out positions, and picks bf16 for 128 filters."""
    torch = torch_cuda
    from caro_ai_b200.model import DeviceNet, fold_state_dict
    game, filters = case
    blocks = 5
    net = R.matrix_net(game, filters, blocks)
    scaled = R.rescaled_state_dict(net.state_dict(), RESCALE)
    shape = R.shape_of(game, filters, blocks)
    pos = R.base_positions(game, 2)
    ref = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, R.planes_of(game, pos), device="cuda")
    d_boards, d_who = _device(torch, game, pos)
    dn = DeviceNet(net, game, precision="fp32-simt")
    ds = DeviceNet(scaled, game, precision="fp32-simt")
    exact = exact_under_rescaling(game, filters)
    for impl in exact:
        p0, v0 = dn.forward_boards(d_boards, d_who, len(pos), impl)
        p1, v1 = ds.forward_boards(d_boards, d_who, len(pos), impl)
        assert torch.equal(p0, p1) and torch.equal(v0, v1), (R.game_label(game), filters, impl)
    if filters == 64 and game.game_kind == 0:  # the row-tiled bf16 tower
        p, v = ds.forward_boards(d_boards, d_who, len(pos), 0)
        _check(p, v, ref, R.bound_of("rt_bf16", game, blocks), (R.game_label(game), filters, "rescaled", 0))
    dn.close()
    ds.close()
    da = DeviceNet(scaled, game)
    assert da.precision != "fp16", da.calibration
    if filters == 128:
        assert da.precision == "bf16", da.calibration
    held = R.base_positions(game, 5)
    ref_h = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, R.planes_of(game, held), device="cuda")
    p, v = da.forward_states([q[0] for q in held], [q[1] for q in held])
    dev = _check(p, v, ref_h, None, (R.game_label(game), filters, "auto", da.precision))
    assert dev[0] <= 1e-3 and dev[1] <= 1e-3, (dev, da.calibration)
    da.close()


@pytest.mark.parametrize("n", [None, 15], ids=["connect4", "mnk15x5"])
def test_update_on_wide_handles(torch_cuda, n):
    """After update(net_b) a 128-filter handle gives what a fresh DeviceNet(net_b) gives, bit for bit, on impls 0, 1 and 7
    (on 15 x 15 the heads GEMM image is repacked too); the precision check runs again; a blob of another depth is refused."""
    torch = torch_cuda
    from caro_ai_b200 import _cabi
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    game = ConnectFour() if n is None else TicTacToe(n, 5)
    torch.manual_seed(3)
    net_a = Net(game.obs_shape, game.action_space, blocks=5, filters=128)
    R.randomise_bn(torch, net_a)
    net_a.eval()
    net_b = R.matrix_net(game, 128, 5)
    pos = R.base_positions(game, 6)
    d_boards, d_who = _device(torch, game, pos)
    dn = DeviceNet(net_a, game)
    before = dn.calibration
    dn.update(net_b)
    assert dn.calibration is not before
    fresh = DeviceNet(net_b, game)
    assert dn.calibration == fresh.calibration and dn.precision == fresh.precision
    for impl in (0, 1, 7):
        p0, v0 = dn.forward_boards(d_boards, d_who, len(pos), impl)
        p1, v1 = fresh.forward_boards(d_boards, d_who, len(pos), impl)
        assert torch.equal(p0, p1) and torch.equal(v0, v1), impl
    with pytest.raises(_cabi.CaroError):
        dn.update(R.matrix_net(game, 128, 4))
    fresh.close()
    dn.close()


@pytest.mark.parametrize("filters", [64, 128])
def test_auto_precision_on_2x2_boards(torch_cuda, filters):
    """A 2 x 2 board calibrates and runs a tensor-core tower at both widths."""
    torch = torch_cuda
    from caro_ai_b200.game import TicTacToe
    from caro_ai_b200.model import DeviceNet
    game = TicTacToe(2, 2)
    dn = DeviceNet(R.matrix_net(game, filters, 5), game)
    assert dn.precision in ("fp16", "bf16", "bf16x3"), dn.calibration
    dn.close()
