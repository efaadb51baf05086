"""Policy/value network: the reference's ``Net`` surface (lib/model.py:10-107) and its device twin.

* ``Net`` is a plain ``nn.Module`` with the reference's ``state_dict`` key set / shapes, so the
  shipped ``saves/*/best_*.dat`` checkpoints load unchanged and new ones are written in the same
  format.  It is what the SGD step trains (autograd, plain PyTorch -- out of scope for hand kernels).
* ``fold_state_dict`` merges eval-mode BatchNorm into the convolutions (SURVEY.md A.6) and lays the
  result out as the float32 blob ``caro_net_create`` expects (include/caro_b200.h).
* ``DeviceNet`` owns a ``caro_net`` handle: the fused bf16 tcgen05 tower used on the search path.
"""
from __future__ import annotations

import copy
import ctypes as C
from typing import Dict, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import _cabi

NUM_FILTERS = 64  # lib/model.py:7
WIDTHS = (64, 128)  # filters of the towers the CUDA kernels evaluate
BN_EPS = 1e-5


def _block(cin: int, cout: int, ksize: int) -> nn.Sequential:
    return nn.Sequential(nn.Conv2d(cin, cout, kernel_size=ksize, padding=ksize // 2), nn.BatchNorm2d(cout),
                         nn.LeakyReLU())


class Net(nn.Module):
    """lib/model.py:10-94.  ``forward`` returns (policy logits [B,A], value [B,1]).

    ``blocks`` (extension): number of residual blocks ``conv_1 .. conv_<blocks>``.  The reference has exactly five
    (lib/model.py:21-45) and that is the default -- same ``state_dict`` keys, same initialisation order; BASELINE.json
    configs[3] asks for a "deep residual net", which the reference does not define: here it is a deeper tower of the same
    blocks (1..20), evaluated by the same CUDA kernels (the depth is read off the weight blob).

    ``filters`` (extension): the width of every convolution, 64 (the reference's NUM_FILTERS) or 128.  The key names are
    the same at both widths, only the shapes scale."""

    def __init__(self, input_shape, actions_n, blocks: int = 5, filters: int = NUM_FILTERS):
        super().__init__()
        if not 1 <= blocks <= 20:
            raise ValueError("blocks must be 1 .. 20, got %r" % (blocks,))
        if filters not in WIDTHS:
            raise ValueError("filters must be one of %s, got %r" % (WIDTHS, filters))
        self.input_shape = tuple(input_shape)
        self.actions_n = int(actions_n)
        self.blocks = int(blocks)
        self.filters = int(filters)
        nf = self.filters
        _, h, w = self.input_shape
        self.conv_in = _block(self.input_shape[0], nf, 3)
        for i in range(1, self.blocks + 1):
            setattr(self, "conv_%d" % i, _block(nf, nf, 3))
        self.conv_val = _block(nf, 1, 1)
        # the reference sizes its heads by pushing zeros through them in train mode
        # (lib/model.py:55,69,74-80), leaving one BatchNorm running-stat update behind; kept so that
        # a fresh Net() here equals a fresh reference Net() under the same seed.
        probe = torch.zeros(1, nf, h, w)
        val_size = int(np.prod(self.conv_val(probe).size()))
        self.value = nn.Sequential(nn.Linear(val_size, 20), nn.LeakyReLU(), nn.Linear(20, 1), nn.Tanh())
        self.conv_policy = _block(nf, 2, 1)
        pol_size = int(np.prod(self.conv_policy(probe).size()))
        self.policy = nn.Sequential(nn.Linear(pol_size, self.actions_n))

    def forward(self, x):
        b = x.size()[0]
        v = self.conv_in(x)
        for i in range(1, self.blocks + 1):
            v = v + getattr(self, "conv_%d" % i)(v)
        val = self.value(self.conv_val(v).view(b, -1))
        pol = self.policy(self.conv_policy(v).view(b, -1))
        return pol, val


class NetWrapper:
    """lib/model.py:97-107."""

    def __init__(self, model):
        self.model = model
        self.target_model = copy.deepcopy(model)

    def sync(self):
        self.target_model.load_state_dict(self.model.state_dict())


def _fold(conv_w, conv_b, bn_w, bn_b, mean, var):
    scale = bn_w / torch.sqrt(var + BN_EPS)
    return conv_w * scale.view(-1, 1, 1, 1), (conv_b - mean) * scale + bn_b


def state_dict_shape(sd: Dict[str, torch.Tensor]) -> Tuple[int, int]:
    """(blocks, filters) of a ``Net`` state dict: the number of ``conv_N`` groups and the output channels of conv_in."""
    blocks = 0
    while "conv_%d.0.weight" % (blocks + 1) in sd:
        blocks += 1
    return blocks, int(sd["conv_in.0.weight"].shape[0])


def fold_state_dict(sd: Dict[str, torch.Tensor], rows: int, cols: int, actions: int) -> np.ndarray:
    """Eval-mode BN folding + flattening into the blob layout of include/caro_b200.h.  The depth and the width are read
    off the state dict."""
    sd = {k: v.detach().double().cpu() for k, v in sd.items() if v.dtype.is_floating_point}
    parts = []

    def folded(name):
        return _fold(sd[name + ".0.weight"], sd[name + ".0.bias"], sd[name + ".1.weight"], sd[name + ".1.bias"],
                     sd[name + ".1.running_mean"], sd[name + ".1.running_var"])

    blocks, filters = state_dict_shape(sd)
    for name in ["conv_in"] + ["conv_%d" % i for i in range(1, blocks + 1)]:
        w, b = folded(name)
        parts += [w.reshape(-1), b.reshape(-1)]
    w, b = folded("conv_val")
    parts += [w.reshape(-1), b.reshape(-1), sd["value.0.weight"].reshape(-1), sd["value.0.bias"].reshape(-1),
              sd["value.2.weight"].reshape(-1), sd["value.2.bias"].reshape(-1)]
    w, b = folded("conv_policy")
    parts += [w.reshape(-1), b.reshape(-1), sd["policy.0.weight"].reshape(-1), sd["policy.0.bias"].reshape(-1)]
    blob = torch.cat(parts).float().numpy()
    expect = _cabi.lib().caro_net_blob_floats_shape(rows, cols, actions, blocks, filters)
    if blob.size != expect:
        raise ValueError("state dict of %d blocks x %d filters folds to %d floats, the %dx%d board's blob layout wants %d"
                         % (blocks, filters, blob.size, rows, cols, expect))
    return np.ascontiguousarray(blob)


IMPL_TCGEN05, IMPL_SIMT, IMPL_TCGEN05_X3, IMPL_TCGEN05_F16, IMPL_WIDE_X3 = 0, 1, 2, 7, 8
PRIOR_TOLERANCE = 1e-3      # BASELINE.json north_star: priors / values within 1e-3 of the fp32 reference
CALIBRATION_MARGIN = 0.8    # the probe set is a sample: switch to the split mode at 0.8 x the tolerance
_PROBE_BOARDS: Dict[tuple, tuple] = {}


def probe_positions(game, count: int = 256, seed: int = 2026):
    """(d_boards, d_who): ``count`` positions reached by random legal play-outs of 0 .. ~2/3 of the longest game, played
    with the CUDA board kernels (no host rules).  Cached per game shape; used to pick the tower's precision."""
    key = (game.game_kind, game.n, game.k, count, seed, torch.cuda.current_device())
    if key not in _PROBE_BOARDS:
        rng = np.random.default_rng(seed)
        A = game.action_space
        max_plies = 42 if game.game_kind == _cabi.GAME_CONNECT4 else A
        states = [game.initial_state] * count
        players = [int(x) for x in rng.integers(0, 2, count)]
        target = rng.integers(0, max(1, min(60, (2 * max_plies) // 3)), count)
        for ply in range(int(target.max())):
            masks = game.legal_masks(states)
            acts, idx = [], []
            for i in range(count):
                legal = np.nonzero(masks[i])[0]
                if ply < target[i] and legal.size:
                    idx.append(i)
                    acts.append(int(rng.choice(legal)))
            if not idx:
                break
            new_states, won, draw = game.apply_batch([states[i] for i in idx], acts, [players[i] for i in idx])
            for j, i in enumerate(idx):
                if won[j] or draw[j]:
                    target[i] = 0  # keep the last non-terminal position
                else:
                    states[i], players[i] = new_states[j], 1 - players[i]
        d_boards = torch.from_numpy(game.boards_from_states(states).view(np.int64)).cuda()
        d_who = torch.tensor(players, dtype=torch.uint8, device="cuda")
        _PROBE_BOARDS[key] = (d_boards, d_who)
    return _PROBE_BOARDS[key]


class DeviceNet:
    """Folded network resident on the GPU (``caro_net`` handle)."""

    def __init__(self, net_or_state_dict, game, precision: str = "auto"):
        """``precision``:
        "auto"   (default) -- after every weight upload 256 probe positions run through the fp32 SIMT tower and the
                 one-pass tensor-core towers, fastest first: "fp16" (boards up to 6 x 7), then "bf16"; a one-pass tower is
                 used only while BOTH priors and values agree with fp32 within CALIBRATION_MARGIN x 1e-3 (lib/mcts.py:212-218
                 contract), otherwise the split-precision tower is selected.  Random-init networks (the benchmark) run
                 "fp16" (3.7e-5 / 8.1e-5 off fp32 on Connect4; "bf16": 1.1e-4 / 5.0e-4); trained checkpoints whose policy
                 logits span +-100 (the shipped Connect4 nets) switch to "bf16x3" (DESIGN.md section 2).
        "fp16"   one fp16 tensor-core pass (activations and weights fp16, fp32 accumulate; boards up to 6 x 7): 11 mantissa
                 bits on both MMA operands and no separate residual tail -- more accurate AND 8 % faster than "bf16", but
                 fp16's range (|x| < 65,504): forced use leaves the range check to the caller,
        "bf16"   one bf16 tensor-core pass, fp32 accumulate (forced; the caller vouches for the tolerance),
        "bf16x3" hi/lo split of activations and weights, three MMAs per product: fp32-class accuracy (boards up to 6 x 7:
                 fp16 hi + lo, row-tiled; larger boards: bf16 hi + lo, tap-per-MMA),
        "bf16x3-wide" the split-precision form of the wide tower (128 filters only): bf16 hi + lo activations and weights,
                 three MMAs per product, fp32 residual stream,
        "fp32-simt" the SIMT numerics-reference kernel.
        128-filter networks (``Net(filters=128)``) run the wide tensor-core tower (csrc/net_wide.cu) with fp16, bf16 or bf16
        hi + lo operands on every board size, or the SIMT tower; "auto" tries "fp16", then "bf16", then "bf16x3-wide", and
        falls back to "fp32-simt" only when all three miss the check.  "bf16x3" (the 64-filter split towers) is not
        available for them."""
        _cabi.require_cuda()
        assert precision in ("auto", "fp16", "bf16", "bf16x3", "bf16x3-wide", "fp32-simt")
        sd = net_or_state_dict.state_dict() if isinstance(net_or_state_dict, nn.Module) else net_or_state_dict
        self.blocks, self.filters = state_dict_shape(sd)
        if precision == "bf16x3" and self.filters != NUM_FILTERS:
            raise ValueError("precision 'bf16x3' is not available for %d-filter networks (64 only); their split-precision "
                             "tower is 'bf16x3-wide'" % self.filters)
        if precision == "bf16x3-wide" and self.filters != WIDTHS[1]:
            raise ValueError("precision 'bf16x3-wide' is the split tower of 128-filter networks, not of %d-filter ones "
                             "(use 'bf16x3')" % self.filters)
        self.requested = precision
        _, self.rows, self.cols = game.obs_shape
        self.actions = game.action_space
        self.game = game
        blob = fold_state_dict(sd, self.rows, self.cols, self.actions)
        handle = C.c_void_p()
        if self.filters == NUM_FILTERS:
            _cabi.check(_cabi.lib().caro_net_create(self.rows, self.cols, self.actions, blob.ctypes.data, blob.size,
                                                    C.byref(handle)))
        else:
            _cabi.check(_cabi.lib().caro_net_create_shape(self.rows, self.cols, self.actions, self.blocks, self.filters,
                                                          blob.ctypes.data, blob.size, C.byref(handle)))
        self.handle = handle
        self.calibration = None
        self._select(precision)

    def _select(self, precision: str) -> None:
        if precision == "auto":
            precision = self.calibrate()
        self.precision = precision
        self.impl = {"fp16": IMPL_TCGEN05_F16, "bf16": IMPL_TCGEN05, "bf16x3": IMPL_TCGEN05_X3, "bf16x3-wide": IMPL_WIDE_X3,
                     "fp32-simt": IMPL_SIMT}[precision]

    def calibrate(self, d_boards=None, d_who=None) -> str:
        """Max |prior| / |value| deviation of the one-pass towers (fp16 where it applies, then bf16) from the fp32 SIMT
        tower on probe positions (``d_boards`` / ``d_who``: caller-supplied device boards, e.g. replay positions; default:
        cached random play-outs).  If neither keeps the margin, the split-precision tower of the width ("bf16x3" at 64
        filters, "bf16x3-wide" at 128) is measured too (``split_max_abs_*``) and selected if it keeps it; "fp32-simt" is
        the last resort.  Returns the precision that keeps the 1e-3 contract and records the measurement in
        ``self.calibration``."""
        if d_boards is None:
            d_boards, d_who = probe_positions(self.game)
        n = int(d_who.numel())
        p32, v32 = self.forward_boards(d_boards, d_who, n, IMPL_SIMT)
        limit = CALIBRATION_MARGIN * PRIOR_TOLERANCE
        ok = False
        self.calibration = {"positions": n, "filters": self.filters}
        if self.filters != NUM_FILTERS:  # the wide tower: fp16 on every board, then bf16, then its split mode
            candidates = [("fp16", IMPL_TCGEN05_F16)]
        else:
            candidates = [("fp16", IMPL_TCGEN05_F16)] if self.rows <= 6 and self.cols <= 7 else []  # the row-tiled towers' boards
        for name, impl in candidates + [("bf16", IMPL_TCGEN05)]:  # both are measured (and recorded), the first that passes is used
            p16, v16 = self.forward_boards(d_boards, d_who, n, impl)
            dp = float((p16 - p32).abs().max().item())
            dv = float((v16 - v32).abs().max().item())
            finite = bool(torch.isfinite(p16).all().item() and torch.isfinite(v16).all().item())
            self.calibration.update({name + "_max_abs_prior_diff": dp, name + "_max_abs_value_diff": dv})
            if not ok:  # max_abs_*: the selected one-pass tower's deviation (the last one tried if none passes)
                self.calibration.update(max_abs_prior_diff=dp, max_abs_value_diff=dv)
            if not ok and finite and dp <= limit and dv <= limit:
                ok = True
                self.calibration["selected"] = name
        if ok:
            return self.calibration["selected"]
        # the split mode is checked too (the 64-filter row-tiled one is fp16 hi + lo, of a finite range): the SIMT tower is
        # the last resort
        split, split_impl = ("bf16x3", IMPL_TCGEN05_X3) if self.filters == NUM_FILTERS else ("bf16x3-wide", IMPL_WIDE_X3)
        self.calibration["selected"] = split
        px, vx = self.forward_boards(d_boards, d_who, n, split_impl)
        dpx, dvx = float((px - p32).abs().max().item()), float((vx - v32).abs().max().item())
        self.calibration.update(split_max_abs_prior_diff=dpx, split_max_abs_value_diff=dvx)
        if not (dpx <= limit and dvx <= limit):
            self.calibration["selected"] = "fp32-simt"
        return self.calibration["selected"]

    def update(self, net_or_state_dict):
        """NetWrapper.sync() on the device side: re-fold, re-upload and (precision "auto") re-check the tolerance."""
        sd = net_or_state_dict.state_dict() if isinstance(net_or_state_dict, nn.Module) else net_or_state_dict
        blob = fold_state_dict(sd, self.rows, self.cols, self.actions)
        _cabi.check(_cabi.lib().caro_net_update(self.handle, blob.ctypes.data, blob.size))
        self._select(self.requested)

    def forward_boards(self, d_boards, d_who, count: int, impl: int = None):
        """(priors [count,A], values [count]) float32 CUDA tensors for device boards."""
        impl = self.impl if impl is None else impl
        probs = torch.empty((count, self.actions), dtype=torch.float32, device="cuda")
        values = torch.empty((count,), dtype=torch.float32, device="cuda")
        if count:
            g = self.game
            _cabi.check(_cabi.lib().caro_net_forward(self.handle, g.game_kind, g.n, g.k, d_boards.data_ptr(),
                                                     d_who.data_ptr(), None, count, probs.data_ptr(), values.data_ptr(),
                                                     impl, torch.cuda.current_stream().cuda_stream))
        return probs, values

    def set_grid_limit(self, ctas: int) -> None:
        """Limit the persistent tower to ``ctas`` SMs (0 = all), leaving the rest to concurrent tree kernels."""
        _cabi.check(_cabi.lib().caro_net_set_grid_limit(self.handle, int(ctas)))

    def forward_states(self, states, players, impl: int = None):
        d_boards = torch.from_numpy(self.game.boards_from_states(states).view(np.int64)).cuda()
        d_who = torch.tensor(list(players), dtype=torch.uint8, device="cuda")
        return self.forward_boards(d_boards, d_who, len(states), impl)

    def close(self):
        if self.handle:
            _cabi.lib().caro_net_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def load_checkpoint(path: str, game) -> Net:
    """play.py:29-35 / play_session.py:13-16: ``torch.load`` of a reference ``.dat`` state_dict.  The ``Net`` is built
    with the depth and width found in the file, so deeper and 128-filter checkpoints load as well as the reference's."""
    sd = torch.load(path, map_location=lambda storage, loc: storage)
    blocks, filters = state_dict_shape(sd)
    net = Net(game.obs_shape, game.action_space, blocks=blocks, filters=filters)
    net.load_state_dict(sd)
    return net


def save_checkpoint(net: Net, path: str) -> None:
    """train.py:214-216."""
    torch.save(net.state_dict(), path)
