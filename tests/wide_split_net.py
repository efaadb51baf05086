"""The "trained-like" 128-filter test network of the split-precision wide tower (impl 8), and a float64 emulation of the
wide tower's three operand schemes.

The test net is ``net_reference.matrix_net`` with two changes that make both one-pass wide towers miss the 1e-3 check:
* its policy FC is multiplied by POLICY_GAIN, so that the policy logits span as widely as a trained network's do and one
  bf16 pass (8 mantissa bits) loses the priors' precision;
* the residual stream is rescaled by RESCALE (``net_reference.rescaled_state_dict``), so that the activations leave
  fp16's range (|x| < 65,504).  bf16 hi + lo pairs keep fp32's exponent range, so the split tower is exactly homogeneous
  under this power-of-two scaling: its outputs equal those of the unscaled net bit for bit.

The emulation rounds the convolution operands the way each scheme does (activations and weights to fp16, to bf16, or to
bf16 hi + lo pairs with hi*hi + lo*hi + hi*lo per product) and computes everything else in float64, from the folded blob
alone (``net_reference.unpack_blob``)."""
import torch
import torch.nn.functional as Fn

import net_reference as R

IMPL_WIDE_X3 = 8   # caro_net_forward: the wide tower in split precision
POLICY_GAIN = 100.0
RESCALE = 2.0 ** 17


def trained_like_net(game, blocks):
    """(net, state dict): the matrix net with its policy FC x POLICY_GAIN, and its state dict rescaled by RESCALE."""
    net = R.matrix_net(game, 128, blocks)
    with torch.no_grad():
        net.policy[0].weight.mul_(POLICY_GAIN)
        net.policy[0].bias.mul_(POLICY_GAIN)
    return net, R.rescaled_state_dict(net.state_dict(), RESCALE)


def _bf16(x):
    return x.to(torch.bfloat16).to(torch.float64)


def _f16(x):
    return x.to(torch.float16).to(torch.float64)


def _conv(x, w, scheme):
    """3x3 convolution (padding 1, no bias) with the operands rounded as ``scheme`` rounds them."""
    if scheme == "fp64":
        return Fn.conv2d(x, w, padding=1)
    if scheme in ("fp16", "bf16"):
        r = _f16 if scheme == "fp16" else _bf16
        return Fn.conv2d(r(x), r(w), padding=1)
    assert scheme == "split"
    xh, wh = _bf16(x), _bf16(w)
    xl, wl = _bf16(x - xh), _bf16(w - wh)
    return Fn.conv2d(xh, wh, padding=1) + Fn.conv2d(xl, wh, padding=1) + Fn.conv2d(xh, wl, padding=1)


def emulate(blob, shape, planes, scheme):
    """(priors [B, A], values [B]) float64 numpy arrays of the tower evaluated with ``scheme`` ("fp64", "fp16", "bf16"
    or "split") on the convolutions of the residual stream; heads in float64, as the kernels run them on the fp32 stream
    (fp32 in the tower or the bf16 hi + lo heads GEMM)."""
    rows, cols, actions, blocks, filters = shape
    w = R.unpack_blob(blob, *shape)
    lrelu = lambda t: torch.where(t > 0, t, R.LEAKY * t)  # noqa: E731
    with torch.no_grad():
        x = torch.as_tensor(planes, dtype=torch.float64)
        b = x.shape[0]
        v = lrelu(_conv(x, w["conv_in_w"], scheme) + w["conv_in_b"].view(1, -1, 1, 1))
        for i in range(blocks):
            v = v + lrelu(_conv(v, w["conv_w%d" % i], scheme) + w["conv_b%d" % i].view(1, -1, 1, 1))
        val = lrelu(Fn.conv2d(v, w["val_conv_w"], w["val_conv_b"])).reshape(b, -1)
        hid = lrelu(val @ w["val_fc1_w"].T + w["val_fc1_b"])
        u = hid @ w["val_fc2_w"] + w["val_fc2_b"]
        pol = lrelu(Fn.conv2d(v, w["pol_conv_w"], w["pol_conv_b"])).reshape(b, -1)
        logits = pol @ w["pol_fc_w"].T + w["pol_fc_b"]
        return torch.softmax(logits, dim=1).numpy(), torch.tanh(u).numpy()
