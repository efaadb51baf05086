"""The premise of the split-precision wide tower (impl 8), on the host: on the "trained-like" 128-filter test net of
wide_split_net.py, a float64 emulation of the wide tower's operand schemes shows that one fp16 pass (range) and one bf16
pass (precision) both miss the 0.8e-3 calibration margin, while bf16 hi + lo pairs stay below 1e-4.  No GPU needed."""
import numpy as np
import pytest

import net_reference as R
import wide_split_net as S

MARGIN = 0.8e-3   # DeviceNet's calibration: CALIBRATION_MARGIN x PRIOR_TOLERANCE


def _cases():
    from caro_ai_b200.game import ConnectFour, TicTacToe
    return [(ConnectFour(), 5), (TicTacToe(9, 5), 10)]


@pytest.mark.parametrize("case", _cases(), ids=lambda c: "%s-b%d" % (R.game_label(c[0]), c[1]))
def test_one_pass_towers_miss_the_check_and_the_split_tower_keeps_it(case):
    from caro_ai_b200.model import fold_state_dict
    game, blocks = case
    _, sd = S.trained_like_net(game, blocks)
    shape = R.shape_of(game, 128, blocks)
    blob = fold_state_dict(sd, *shape[:3])
    planes = R.planes_of(game, R.base_positions(game, 3))
    ref_p, ref_v, _ = R.reference(blob, shape, planes)
    dev = {}
    for scheme in ("fp64", "fp16", "bf16", "split"):
        p, v = S.emulate(blob, shape, planes, scheme)
        finite = bool(np.isfinite(p).all() and np.isfinite(v).all())
        dev[scheme] = (float(np.abs(p - ref_p).max()), float(np.abs(v - ref_v).max())) if finite else None
    assert dev["fp64"] is not None and max(dev["fp64"]) <= 1e-12, dev  # the emulation is the reference's function
    assert dev["fp16"] is None or max(dev["fp16"]) > MARGIN, dev
    assert dev["bf16"] is not None and max(dev["bf16"]) > MARGIN, dev
    assert dev["split"] is not None and dev["split"][0] < 1e-4 and dev["split"][1] < 1e-4, dev


def test_the_rescaling_is_exact_and_the_unscaled_net_has_the_same_function():
    """The rescaled state dict folds to a blob whose float64 reference equals the unscaled net's to rounding, so the GPU
    tests may compare the split tower's output on either."""
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.model import fold_state_dict
    game = ConnectFour()
    net, sd = S.trained_like_net(game, 2)
    shape = R.shape_of(game, 128, 2)
    planes = R.planes_of(game, R.base_positions(game, 4))
    a = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, planes)
    b = R.reference(fold_state_dict(sd, *shape[:3]), shape, planes)
    for x, y in zip(a[:2], b[:2]):
        assert float(np.abs(x - y).max()) <= 1e-9
