"""Float64 reference of the policy/value network, computed from the folded weight blob alone.

The blob layout is the one documented in include/caro_b200.h:
    conv_in  w[F][2][3][3] b[F] | blocks x ( w[F][F][3][3] b[F] ) |
    conv_val w[F] b[1] | value.0 w[20][HW] b[20] | value.2 w[20] b[1] |
    conv_policy w[2][F] b[2] | policy.0 w[A][2*HW] b[A]
and the function is lib/model.py's forward with eval-mode BatchNorm folded in:
    v = lrelu(conv_in(x)); blocks x { v = v + lrelu(conv_i(v)) }
    value = tanh(fc2(lrelu(fc1(lrelu(conv_val(v))))))
    policy = softmax(fc(flatten_channel_major(lrelu(conv_policy(v)))))  over all A actions
with lrelu slope 0.01.  Nothing here uses the package's ``Net`` or its kernels, so a wrong fold, a wrong layout or a wrong
kernel cannot hide behind a shared mistake.

Also here, because both the host and the GPU tests need them: the networks of the GPU test matrix (``matrix_net``), the
blob mutations that stand for plausible kernel bugs (``MUTATIONS``), the tower each impl runs (``tower_of``), each tower's
group geometry (``group_boards``) and its error bounds (``bound_of``)."""
import numpy as np
import torch
import torch.nn.functional as Fn

LEAKY = 0.01


def blob_layout(rows, cols, actions, blocks, filters):
    """[(name, shape)] in blob order."""
    F, hw = filters, rows * cols
    parts = [("conv_in_w", (F, 2, 3, 3)), ("conv_in_b", (F,))]
    for i in range(blocks):
        parts += [("conv_w%d" % i, (F, F, 3, 3)), ("conv_b%d" % i, (F,))]
    parts += [("val_conv_w", (1, F, 1, 1)), ("val_conv_b", (1,)), ("val_fc1_w", (20, hw)), ("val_fc1_b", (20,)),
              ("val_fc2_w", (20,)), ("val_fc2_b", (1,)),
              ("pol_conv_w", (2, F, 1, 1)), ("pol_conv_b", (2,)), ("pol_fc_w", (actions, 2 * hw)), ("pol_fc_b", (actions,))]
    return parts


def unpack_blob(blob, rows, cols, actions, blocks, filters):
    """Dict of float64 CPU tensors, one per layout entry; the blob's size must match the shape exactly."""
    flat = torch.from_numpy(np.asarray(blob, dtype=np.float32).astype(np.float64))
    out, o = {}, 0
    for name, shape in blob_layout(rows, cols, actions, blocks, filters):
        n = int(np.prod(shape))
        out[name] = flat[o:o + n].reshape(shape).clone()
        o += n
    assert o == flat.numel(), "blob of %d floats, layout wants %d" % (flat.numel(), o)
    return out


def _lrelu(x):
    return torch.where(x > 0, x, LEAKY * x)


def forward64(w, blocks, planes, device="cpu"):
    """(policy logits [B, A], value pre-activation [B]) in float64 from unpacked weights and [B, 2, H, W] planes."""
    w = {k: v.to(device) for k, v in w.items()}
    x = torch.as_tensor(np.asarray(planes), dtype=torch.float64, device=device)
    b = x.shape[0]
    v = _lrelu(Fn.conv2d(x, w["conv_in_w"], w["conv_in_b"], padding=1))
    for i in range(blocks):
        v = v + _lrelu(Fn.conv2d(v, w["conv_w%d" % i], w["conv_b%d" % i], padding=1))
    val = _lrelu(Fn.conv2d(v, w["val_conv_w"], w["val_conv_b"])).reshape(b, -1)
    hid = _lrelu(val @ w["val_fc1_w"].T + w["val_fc1_b"])
    u = hid @ w["val_fc2_w"] + w["val_fc2_b"]
    pol = _lrelu(Fn.conv2d(v, w["pol_conv_w"], w["pol_conv_b"])).reshape(b, -1)  # channel-major flatten
    logits = pol @ w["pol_fc_w"].T + w["pol_fc_b"]
    return logits, u


def reference(blob, shape, planes, mutation=None, device="cpu"):
    """(priors [B, A], values [B], log-priors [B, A]) as float64 numpy arrays.  ``shape`` = (rows, cols, actions, blocks,
    filters); ``mutation`` names an entry of MUTATIONS, applied to the weights before the forward pass."""
    rows, cols, actions, blocks, filters = shape
    w = unpack_blob(blob, *shape)
    if mutation is not None:
        MUTATIONS[mutation](w, shape)
    with torch.no_grad():
        logits, u = forward64(w, blocks, planes, device)
        logp = torch.log_softmax(logits, dim=1)
        return torch.exp(logp).cpu().numpy(), torch.tanh(u).cpu().numpy(), logp.cpu().numpy()


# ------------------------------------------------------------------------------------------- mutations
# Each stands for a bug a kernel could plausibly have; the host tests check that every one of them moves the outputs far
# beyond the bounds the GPU tests allow, so that such a bug could not pass them.  Layer-local bugs are placed in the last
# residual layer, whose error the deeper layers cannot damp.
def _mirror_taps(w, shape):  # a tap-shift sign error: the 3x3 taps of the last residual layer mirrored left-right
    last = "conv_w%d" % (shape[3] - 1)
    w[last] = w[last].flip(-1)


def _swap_inputs(w, shape):  # side to move confused: the two input planes swapped
    w["conv_in_w"] = w["conv_in_w"][:, [1, 0]]


def _drop_k_step(w, shape):  # a missed K-step: the last 16 input channels of the last residual layer dropped
    w["conv_w%d" % (shape[3] - 1)][:, -16:] = 0.0


def _swap_policy(w, shape):  # the two policy 1x1 channels swapped
    w["pol_conv_w"] = w["pol_conv_w"][[1, 0]]
    w["pol_conv_b"] = w["pol_conv_b"][[1, 0]]


def _skip_last_block(w, shape):  # the last residual block skipped
    last = shape[3] - 1
    w["conv_w%d" % last][:] = 0.0
    w["conv_b%d" % last][:] = 0.0


def _fc1_transposed(w, shape):  # value FC1 read in the transposed [HW][20] layout
    hw = shape[0] * shape[1]
    w["val_fc1_w"] = w["val_fc1_w"].reshape(-1).reshape(hw, 20).T.contiguous()


MUTATIONS = {"mirror_taps": _mirror_taps, "swap_inputs": _swap_inputs, "drop_k_step": _drop_k_step,
             "swap_policy": _swap_policy, "skip_last_block": _skip_last_block, "fc1_transposed": _fc1_transposed}


# ------------------------------------------------------------------------------------------- the test matrix
def matrix_games():
    """Connect4 and TicTacToe(n, min(n, 5)) for every board size the device boards hold."""
    from caro_ai_b200.game import ConnectFour, TicTacToe
    return [ConnectFour()] + [TicTacToe(n, min(n, 5)) for n in range(2, 16)]


def matrix_depths(game):
    """1 and 5 residual blocks everywhere; 20 on Connect4, 8 x 8 (the last board with in-kernel FC heads) and 15 x 15."""
    _, h, w = game.obs_shape
    return (1, 5, 20) if game.game_kind == 0 or h in (8, 15) else (1, 5)


def matrix_cases():
    """[(game, filters, blocks)] of the GPU matrix."""
    return [(g, f, b) for g in matrix_games() for f in (64, 128) for b in matrix_depths(g)]


def game_label(game):
    return "connect4" if game.game_kind == 0 else "mnk%dx%d" % (game.n, game.k)


def shape_of(game, filters, blocks):
    _, h, w = game.obs_shape
    return (h, w, game.action_space, blocks, filters)


def random_positions(game, rng, count):
    """Random legal play-outs: non-terminal positions with a move left."""
    from harness import oracle_for, random_position
    og = oracle_for(game)
    cells = game.obs_shape[1] * game.obs_shape[2]
    top = 30 if game.game_kind == 0 else min(40, max(1, cells // 2))
    return [random_position(og, rng, int(rng.integers(0, top + 1))) for _ in range(count)]


def dense_positions(game, rng, count):
    """Boards no game reaches: m,n,k boards with every cell, or all but one, filled at random (the decimal state
    encoding takes any digits; on 15 x 15 these reach the last bitboard word, cells 192 and above), Connect4 columns
    filled to random heights (full ones included) through the field-list encoding."""
    out = []
    for i in range(count):
        who = int(rng.integers(2))
        if game.game_kind == 0:
            heights = rng.integers(0, 7, 7)
            heights[i % 7] = 6
            cols = [[int(t) for t in rng.integers(0, 2, int(hgt))] for hgt in heights]
            out.append((game.encode_lists(cols), who))
        else:
            cells = game.n * game.n
            digits = [str(int(d)) for d in rng.integers(0, 2, cells)]
            if i % 2:
                digits[int(rng.integers(cells))] = "2"
            out.append((int("".join(digits)), who))
    return out


def base_positions(game, seed):
    """The empty board with each side to move, random play-outs and dense boards."""
    rng = np.random.default_rng(seed)
    return [(game.initial_state, 0), (game.initial_state, 1)] + random_positions(game, rng, 20) + dense_positions(game, rng, 6)


def planes_of(game, positions):
    from harness import oracle_for
    return oracle_for(game).states_to_training_batch([p[0] for p in positions], [p[1] for p in positions])


def randomise_bn(torch_mod, net):
    """BatchNorm statistics and affine parameters away from their initial values, as in the other network tests."""
    with torch_mod.no_grad():
        for m in net.modules():
            if isinstance(m, torch_mod.nn.BatchNorm2d):
                m.running_mean.uniform_(-0.2, 0.2)
                m.running_var.uniform_(0.7, 1.3)
                m.weight.uniform_(0.6, 1.0)
                m.bias.uniform_(-0.1, 0.1)


VALUE_STD = 0.005  # spread of the matrix nets' value head output over the base positions, centred on 0


def matrix_net(game, filters, blocks):
    """Seeded ``Net`` (eval) with randomised BatchNorm and a re-centred value head.  A random-init value head is all bias:
    its output barely depends on the position, so a wrong value-FC layout would move it by no more than rounding does.
    Value FC2 is scaled so that its output spreads over the base positions with a standard deviation of VALUE_STD around
    0 (its bias re-centres it), measured with the float64 reference.  The spread is kept small because the error of the
    bf16 towers grows with it, while the bugs of MUTATIONS move the value in proportion to it."""
    from caro_ai_b200.model import Net, fold_state_dict
    torch.manual_seed(1000 * blocks + filters + 7 * game.action_space + game.game_kind)
    net = Net(game.obs_shape, game.action_space, blocks=blocks, filters=filters)
    randomise_bn(torch, net)
    net.eval()
    shape = shape_of(game, filters, blocks)
    w = unpack_blob(fold_state_dict(net.state_dict(), *shape[:3]), *shape)
    with torch.no_grad():
        _, u = forward64(w, blocks, planes_of(game, base_positions(game, 1)))
        c = VALUE_STD / float(u.std())
        net.value[2].weight.mul_(c)
        net.value[2].bias.fill_(-c * (float(u.mean()) - float(w["val_fc2_b"][0])))
    return net


def rescaled_state_dict(sd, s):
    """The same function with the residual stream multiplied by ``s`` (a power of two) through the BatchNorm parameters:
    conv_in's gamma and beta x s; every residual block's beta, conv bias and running mean x s; both head convolutions'
    gamma / s with conv bias and running mean x s.  Exact in float64 and float32."""
    out = {k: v.clone() for k, v in sd.items()}
    out["conv_in.1.weight"] *= s
    out["conv_in.1.bias"] *= s
    i = 1
    while "conv_%d.0.weight" % i in out:
        for key in ("conv_%d.1.bias", "conv_%d.0.bias", "conv_%d.1.running_mean"):
            out[key % i] *= s
        i += 1
    for head in ("conv_val", "conv_policy"):
        out[head + ".1.weight"] /= s
        out[head + ".0.bias"] *= s
        out[head + ".1.running_mean"] *= s
    return out


# ------------------------------------------------------------------------------------------- towers, geometry, bounds
def tower_of(game, filters, impl):
    """The kernel caro_net_forward runs for ``impl`` (csrc/net.cu), or None where it refuses the combination.
    Row-tiled towers (net_rt.cu, net_rx.cu) take boards up to 6 x 7; the heads GEMM (net_heads.cu) follows the
    tap-per-MMA and wide towers on boards with more than 64 cells."""
    _, h, w = game.obs_shape
    if impl == 1:
        return "simt128" if filters == 128 else "simt"
    if filters == 128:
        return {0: "wide_bf16", 3: "wide_bf16", 7: "wide_f16"}.get(impl)
    row_tiled = h <= 6 and w <= 7
    if row_tiled:
        return {0: "rt_bf16", 2: "rx", 3: "tc_bf16", 4: "tc_x3", 5: "rt_bf16", 6: "tc_bf16", 7: "rt_f16"}.get(impl)
    return {0: "tc_bf16", 2: "tc_x3", 3: "tc_bf16", 4: "tc_x3", 6: "tc_bf16"}.get(impl)


def group_boards(tower, game):
    """Boards per group (one CTA's unit of work) of a tower, mirroring its launcher:
    * tap-per-MMA (net_tc.cu) and wide (net_wide.cu) towers lay a board out with row pitch W + 1 and one zero row after it,
      (H + 1)(W + 1) rows, in a group of 512 rows (one-pass 64-filter tower, 4 M-tiles) or 256 rows (split-precision and
      wide towers, 2 M-tiles); the group holds at most 32 boards and nb x (20 + A) FC floats of scratch, 2 floats per row;
    * row-tiled towers (net_rt.cu, net_rx.cu) put one board row of 128 / pitch boards in an M-tile, pitch 4 for boards
      narrower than 4 columns and 8 otherwise;
    * the SIMT tower runs one leaf per thread block."""
    _, h, w = game.obs_shape
    a = game.action_space
    if tower.startswith("simt"):
        return 1
    if tower in ("rt_bf16", "rt_f16", "rx"):
        return 128 // (4 if w < 4 else 8)
    rows = 512 if tower == "tc_bf16" else 256
    return min(rows // ((h + 1) * (w + 1)), 32, rows * 2 // (20 + a))


# (max |p - p_ref|, max |v - v_ref|, max |log p - log p_ref|) per tower, board class ("small": up to 64 cells, FC heads in
# the tower; "large": the heads GEMM follows) and depth (True: more than 10 residual blocks).  Set at 3x the largest
# deviation measured over the matrix on an NVIDIA B200 (1,000 W power limit), capped for p and v at the ceilings the other
# network tests use (SIMT 2e-4, one-pass towers 1e-3 and 2e-3 past 10 blocks), and raised to FLOOR, about fp32 rounding.
# The v deviations were measured with a value spread of 4 x VALUE_STD and divided by 4 (tanh is linear near 0).
BOUNDS = {
    "simt": {("small", False): (1.2e-07, 1.8e-05, 8.2e-07), ("small", True): (4.0e-07, 6.1e-07, 4.9e-06),
             ("large", False): (1.9e-08, 3.3e-06, 1.8e-06), ("large", True): (2.8e-07, 4.3e-07, 8.4e-06)},
    "simt128": {("small", False): (1.3e-07, 2.0e-06, 7.7e-07), ("small", True): (1.2e-06, 6.1e-07, 9.1e-06),
                ("large", False): (1.1e-08, 2.4e-06, 1.5e-06), ("large", True): (3.2e-06, 1.1e-07, 4.0e-05)},
    "rx": {("small", False): (2.6e-07, 1.7e-05, 1.5e-06), ("small", True): (2.7e-07, 2.3e-06, 1.8e-06)},
    "tc_x3": {("small", False): (3.5e-07, 1.5e-05, 3.1e-06), ("small", True): (3.5e-06, 8.6e-06, 9.5e-05),
              ("large", False): (1.7e-07, 1.6e-06, 1.5e-05), ("large", True): (5.1e-06, 2.9e-06, 1.0e-04)},
    "rt_f16": {("small", False): (9.2e-05, 3.6e-04, 3.9e-04), ("small", True): (2.2e-04, 6.4e-04, 1.5e-03)},
    "wide_f16": {("small", False): (1.4e-05, 2.2e-04, 2.2e-04), ("small", True): (2.8e-04, 1.0e-04, 4.0e-03),
                 ("large", False): (2.4e-06, 1.4e-04, 1.9e-04), ("large", True): (1.8e-04, 2.3e-05, 1.9e-03)},
    "rt_bf16": {("small", False): (2.4e-04, 6.0e-04, 1.3e-03), ("small", True): (5.5e-04, 2.0e-03, 3.8e-03)},
    "tc_bf16": {("small", False): (2.3e-04, 7.9e-04, 1.7e-03), ("small", True): (1.7e-03, 2.0e-03, 2.0e-02),
                ("large", False): (2.1e-05, 4.0e-04, 2.4e-03), ("large", True): (1.8e-03, 7.9e-04, 3.6e-02)},
    "wide_bf16": {("small", False): (1.8e-04, 5.0e-04, 1.5e-03), ("small", True): (2.0e-03, 1.2e-03, 3.2e-02),
                  ("large", False): (1.5e-05, 7.7e-04, 2.1e-03), ("large", True): (9.2e-04, 1.9e-04, 1.6e-02)},
}
FLOOR = (1e-6, 1e-6, 1e-5)


def board_class(game):
    _, h, w = game.obs_shape
    return "small" if h * w <= 64 else "large"


def bound_of(tower, game, blocks):
    b = BOUNDS[tower][(board_class(game), blocks > 10)]
    return tuple(max(x, f) for x, f in zip(b, FLOOR))


def impls_of(filters):
    return (0, 1, 2, 3, 4, 5, 6, 7) if filters == 64 else (0, 1, 3, 7)


def case_bound(game, filters, blocks):
    """The largest bound, per metric, that the GPU matrix applies to any tower of the case."""
    bounds = [bound_of(t, game, blocks) for t in (tower_of(game, filters, i) for i in impls_of(filters)) if t is not None]
    return tuple(max(b[m] for b in bounds) for m in range(3))


def deviations(p, v, ref):
    """(max |p - p_ref|, max |v - v_ref|, max |log p - log p_ref|) of float arrays against reference()'s output."""
    ref_p, ref_v, ref_logp = ref
    p = np.asarray(p, dtype=np.float64)
    with np.errstate(divide="ignore"):
        logp = np.log(p)
    return (float(np.abs(p - ref_p).max()), float(np.abs(np.asarray(v, dtype=np.float64) - ref_v).max()),
            float(np.abs(logp - ref_logp).max()))
