"""128-filter networks on the host side: the Net's shapes, the blob layout of include/caro_b200.h at both widths, the
argument checks of caro_net_create_shape, checkpoints of any shape and the train.py switches.  No GPU needed."""
import ctypes as C
import glob
import os

import pytest
import torch

from conftest import GOLDEN


def _lib():
    from caro_ai_b200 import _cabi
    return _cabi.lib()


def test_wide_net_keys_shapes_and_forward():
    from caro_ai_b200.model import Net
    base, wide = Net((2, 6, 7), 7), Net((2, 6, 7), 7, filters=128)
    sd_base, sd_wide = base.state_dict(), wide.state_dict()
    assert set(sd_base) == set(sd_wide)
    assert tuple(sd_wide["conv_in.0.weight"].shape) == (128, 2, 3, 3)
    assert tuple(sd_wide["conv_3.0.weight"].shape) == (128, 128, 3, 3)
    assert tuple(sd_wide["conv_5.1.running_mean"].shape) == (128,)
    assert tuple(sd_wide["conv_val.0.weight"].shape) == (1, 128, 1, 1)
    assert tuple(sd_wide["conv_policy.0.weight"].shape) == (2, 128, 1, 1)
    assert tuple(sd_wide["value.0.weight"].shape) == tuple(sd_base["value.0.weight"].shape) == (20, 42)
    assert tuple(sd_wide["policy.0.weight"].shape) == tuple(sd_base["policy.0.weight"].shape) == (7, 84)
    logits, value = wide.eval()(torch.rand(3, 2, 6, 7))
    assert tuple(logits.shape) == (3, 7) and tuple(value.shape) == (3, 1)
    for bad in (96, 256, 32):
        with pytest.raises(ValueError):
            Net((2, 6, 7), 7, filters=bad)


def test_default_width_keeps_the_seeded_initialisation():
    from caro_ai_b200.model import Net
    torch.manual_seed(11)
    a = Net((2, 3, 3), 9).state_dict()
    torch.manual_seed(11)
    b = Net((2, 3, 3), 9, filters=64).state_dict()
    assert list(a) == list(b)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_blob_sizes_of_both_widths():
    from caro_ai_b200.model import Net, fold_state_dict
    lib = _lib()
    for (h, w, a) in ((6, 7, 7), (3, 3, 9), (15, 15, 225)):
        for blocks in (1, 5, 20):
            assert lib.caro_net_blob_floats_shape(h, w, a, blocks, 64) == lib.caro_net_blob_floats_deep(h, w, a, blocks)
        hw = h * w
        expect = 128 * 2 * 9 + 128 + 3 * (128 * 128 * 9 + 128) + 128 + 1 + 20 * hw + 20 + 20 + 1 + 2 * 128 + 2 + a * 2 * hw + a
        assert lib.caro_net_blob_floats_shape(h, w, a, 3, 128) == expect
    for blocks in (1, 4):
        net = Net((2, 6, 7), 7, blocks=blocks, filters=128)
        assert fold_state_dict(net.state_dict(), 6, 7, 7).size == lib.caro_net_blob_floats_shape(6, 7, 7, blocks, 128)
    for bad in (32, 96, 256, 0):
        assert lib.caro_net_blob_floats_shape(6, 7, 7, 5, bad) == 0
    for bad in (0, 21):
        assert lib.caro_net_blob_floats_shape(6, 7, 7, bad, 128) == 0


def test_create_shape_rejects_bad_arguments_before_looking_for_a_device():
    from caro_ai_b200 import _cabi
    from caro_ai_b200.model import Net, fold_state_dict
    lib = _lib()
    blob64 = fold_state_dict(Net((2, 6, 7), 7, blocks=2).state_dict(), 6, 7, 7)
    blob128 = fold_state_dict(Net((2, 6, 7), 7, blocks=2, filters=128).state_dict(), 6, 7, 7)
    handle = C.c_void_p()
    cases = [
        (2, 96, blob128),    # unsupported width
        (2, 256, blob128),
        (0, 128, blob128),   # unsupported depth
        (21, 128, blob128),
        (2, 128, blob64),    # a 64-wide blob stated as 128 wide
        (3, 128, blob128),   # the wrong depth for the blob
        (2, 64, blob128),
    ]
    for blocks, filters, blob in cases:
        rc = lib.caro_net_create_shape(6, 7, 7, blocks, filters, blob.ctypes.data, blob.size, C.byref(handle))
        assert rc == -1, (blocks, filters, blob.size, rc)  # CARO_E_ARG
        assert not handle.value
    rc = lib.caro_net_create_shape(1, 7, 7, 2, 128, blob128.ctypes.data, blob128.size, C.byref(handle))
    assert rc == -1
    with pytest.raises(_cabi.CaroError):
        _cabi.check(lib.caro_net_create_shape(6, 7, 7, 2, 96, blob128.ctypes.data, blob128.size, C.byref(handle)))


def test_load_checkpoint_builds_the_shape_in_the_file(tmp_path):
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import Net, load_checkpoint, save_checkpoint
    game = ConnectFour()
    torch.manual_seed(5)
    net = Net((2, 6, 7), 7, blocks=3, filters=128)
    path = os.path.join(str(tmp_path), "wide.dat")
    save_checkpoint(net, path)
    back = load_checkpoint(path, game)
    assert back.blocks == 3 and back.filters == 128
    sd, sb = net.state_dict(), back.state_dict()
    assert set(sd) == set(sb)
    for k in sd:
        assert torch.equal(sd[k], sb[k]), k
    shipped = sorted(glob.glob(os.path.join(GOLDEN, "checkpoints", "*.dat")))
    assert len(shipped) == 4
    for f in shipped:
        g = ConnectFour() if "connect4" in os.path.basename(f) else TicTacToe(3, 3)
        m = load_checkpoint(f, g)
        assert m.blocks == 5 and m.filters == 64


def test_train_cli_shape_switches():
    from caro_ai_b200 import train
    args = train.parse_args(["-g", "0", "-n", "x"])
    assert args.blocks == 5 and args.filters == 64
    args = train.parse_args(["-g", "1", "-n", "x", "--blocks", "10", "--filters", "128"])
    assert args.blocks == 10 and args.filters == 128
    for bad in (["--filters", "96"], ["--blocks", "0"], ["--blocks", "21"]):
        with pytest.raises(SystemExit):
            train.parse_args(["-g", "0", "-n", "x"] + bad)
