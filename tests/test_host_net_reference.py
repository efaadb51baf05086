"""The float64 network reference of tests/net_reference.py on the host (no GPU): it agrees with PyTorch's fp32 ``Net``
through the weight fold and the blob layout, a power-of-two rescaling of the residual stream is exact in the blob and in
the reference, and every blob mutation that stands for a kernel bug moves the outputs well past the GPU tests' bounds."""
import numpy as np
import pytest
import torch

import net_reference as R

# A mutant must move some output by this many times the case's largest bound.  The largest bounds are the bf16 towers';
# on 59 of the 66 cases every mutant clears 5x them, on the other seven the weakest (two policy channels swapped, or one
# K-step dropped) clears 1.9x to 5x.
MUTATION_MARGIN = 1.5


def _games():
    from caro_ai_b200.game import ConnectFour, TicTacToe
    return [ConnectFour(), TicTacToe(2, 2), TicTacToe(3, 3), TicTacToe(8, 5), TicTacToe(9, 5), TicTacToe(15, 5)]


@pytest.mark.parametrize("filters", [64, 128])
@pytest.mark.parametrize("blocks", [1, 5, 20])
def test_reference_matches_the_fp32_net(filters, blocks):
    from caro_ai_b200.model import fold_state_dict
    for game in _games():
        net = R.matrix_net(game, filters, blocks)
        shape = R.shape_of(game, filters, blocks)
        planes = R.planes_of(game, R.base_positions(game, 2))
        ref = R.reference(fold_state_dict(net.state_dict(), *shape[:3]), shape, planes)
        with torch.no_grad():
            logits, value = net(torch.from_numpy(planes))
        dev = R.deviations(torch.softmax(logits, dim=1).numpy(), value.numpy()[:, 0], ref)
        assert dev[0] <= 1e-5 and dev[1] <= 1e-5 and dev[2] <= 1e-4, (R.game_label(game), dev)


@pytest.mark.parametrize("filters", [64, 128])
def test_power_of_two_rescaling_is_exact_in_the_blob_and_the_reference(filters):
    """In the float32 blob, conv_in's weights and every conv bias of the tower are multiplied by s exactly, the head
    convolutions' weights divided by s, and nothing else changes; the float64 reference gives bit-identical outputs."""
    from caro_ai_b200.model import fold_state_dict
    s = 2.0 ** 17
    for game in _games():
        blocks = 5
        net = R.matrix_net(game, filters, blocks)
        shape = R.shape_of(game, filters, blocks)
        blob = fold_state_dict(net.state_dict(), *shape[:3])
        scaled = fold_state_dict(R.rescaled_state_dict(net.state_dict(), s), *shape[:3])
        w, ws = R.unpack_blob(blob, *shape), R.unpack_blob(scaled, *shape)
        for name in w:
            scaled_up = name.startswith("conv_in") or name.startswith("conv_b")
            scaled_down = name in ("val_conv_w", "pol_conv_w")
            expect = w[name] * s if scaled_up else w[name] / s if scaled_down else w[name]
            assert torch.equal(ws[name], expect), (R.game_label(game), name)
        planes = R.planes_of(game, R.base_positions(game, 2))
        for a, b in zip(R.reference(blob, shape, planes), R.reference(scaled, shape, planes)):
            assert np.array_equal(a, b), R.game_label(game)


@pytest.mark.parametrize("case", R.matrix_cases(), ids=lambda c: "%s-f%d-b%d" % (R.game_label(c[0]), c[1], c[2]))
def test_every_mutation_is_caught_by_the_gpu_bounds(case):
    """On the GPU matrix's net and positions, each mutant moves p, v or log p by at least MUTATION_MARGIN times the largest
    bound the GPU test applies to that metric on the case, so that the bug it stands for cannot pass there."""
    from caro_ai_b200.model import fold_state_dict
    game, filters, blocks = case
    net = R.matrix_net(game, filters, blocks)
    shape = R.shape_of(game, filters, blocks)
    blob = fold_state_dict(net.state_dict(), *shape[:3])
    planes = R.planes_of(game, R.base_positions(game, 2))
    ref = R.reference(blob, shape, planes)
    bound = R.case_bound(game, filters, blocks)
    for name in R.MUTATIONS:
        dev = R.deviations(*R.reference(blob, shape, planes, mutation=name)[:2], ref)
        ratio = max(dev[m] / bound[m] for m in range(3))
        assert ratio >= MUTATION_MARGIN, (name, dev, bound, ratio)
