"""CPU tests of the product's host logic: C-ABI surface, loud failure without a GPU, checkpoint/fold algebra,
small helpers.  No CUDA compute is invoked (there is no CPU fallback to invoke)."""
import collections
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT


def test_library_exports_every_declared_symbol():
    from caro_ai_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "caro_b200.h")).read()
    code = re.sub(r"/\*.*?\*/", "", header, flags=re.S)  # prototypes only, not the prose
    declared = set(re.findall(r"\b(caro_[a-z0-9_]+)\s*\(", code))
    lib = _cabi.lib()
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing
    assert set(_cabi.exported_symbols()) <= declared, set(_cabi.exported_symbols()) - declared
    assert lib.caro_abi_version() == 2


def test_flag_constants_match_the_header_and_are_validated():
    """The CARO_FLAG_* values of include/caro_b200.h are the ones the Python mirror passes; unknown bits and a compaction
    request whose index map cannot fit shared memory are refused by the (CPU-side) configuration check."""
    from caro_ai_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "caro_b200.h")).read()
    values = {k: int(v) for k, v in re.findall(r"CARO_FLAG_([A-Z_]+)\s*=\s*(\d+)", header)}
    assert values == {"VIRTUAL_LOSS": _cabi.FLAG_VIRTUAL_LOSS, "MASK_PRIORS": _cabi.FLAG_MASK_PRIORS, "FRESH_TREE": _cabi.FLAG_FRESH_TREE,
                      "RECYCLE_TREE": _cabi.FLAG_RECYCLE_TREE, "COMPACT_TREE": _cabi.FLAG_COMPACT_TREE}
    lib = _cabi.lib()
    ok = _cabi.EngineConfig(0, 0, 0, 64, 1, 8, 8192, 0, 1.0, 0.3, 0.25, 0, _cabi.FLAG_COMPACT_TREE, 0)
    assert lib.caro_engine_workspace_bytes(C.byref(ok)) > 0
    unknown = _cabi.EngineConfig(0, 0, 0, 64, 1, 8, 8192, 0, 1.0, 0.3, 0.25, 0, 32, 0)
    assert lib.caro_engine_workspace_bytes(C.byref(unknown)) == 0 and b"flags" in lib.caro_last_error()
    too_big = _cabi.EngineConfig(0, 0, 0, 4, 1, 8, 70000, 0, 1.0, 0.3, 0.25, 0, _cabi.FLAG_COMPACT_TREE, 0)
    assert lib.caro_engine_workspace_bytes(C.byref(too_big)) == 0 and b"COMPACT_TREE" in lib.caro_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_compute_entry_points_fail_loudly_without_a_gpu():
    from caro_ai_b200 import _cabi
    from caro_ai_b200.game import ConnectFour
    lib = _cabi.lib()
    assert lib.caro_device_count() == 0
    buf = (C.c_uint64 * 4)()
    rc = lib.caro_boards_apply(0, 0, 0, buf, buf, buf, 1, buf, None, None, None)
    assert rc == -2 and b"no CPU fallback" in lib.caro_last_error()
    cfg = _cabi.EngineConfig(0, 0, 0, 4, 1, 8, 64, 0, 1.0, 0.3, 0.25, 0)
    assert lib.caro_engine_workspace_bytes(C.byref(cfg)) > 0  # pure arithmetic, allowed
    handle = C.c_void_p()
    assert lib.caro_engine_create(C.byref(cfg), buf, 1 << 40, C.byref(handle), None) == -2
    with pytest.raises(_cabi.CaroError):
        ConnectFour().move(ConnectFour().initial_state, 3, 1)  # the facade raises instead of computing on the CPU
    with pytest.raises(_cabi.CaroError):
        from caro_ai_b200.engine import SelfPlayEngine
        SelfPlayEngine(ConnectFour(), 4)


def test_engine_config_validation():
    from caro_ai_b200 import _cabi
    lib = _cabi.lib()
    bad = [_cabi.EngineConfig(7, 0, 0, 4, 1, 8, 64, 0, 1.0, 0.3, 0.25, 0),      # unknown game
           _cabi.EngineConfig(1, 16, 5, 4, 1, 8, 64, 0, 1.0, 0.3, 0.25, 0),     # n > 15
           _cabi.EngineConfig(0, 0, 0, 4, 3, 8, 64, 0, 1.0, 0.3, 0.25, 0),      # trees_per_game
           _cabi.EngineConfig(0, 0, 0, 4, 1, 33, 64, 0, 1.0, 0.3, 0.25, 0),     # max_batch
           _cabi.EngineConfig(0, 0, 0, 0, 1, 8, 64, 0, 1.0, 0.3, 0.25, 0)]      # no games
    for cfg in bad:
        assert lib.caro_engine_workspace_bytes(C.byref(cfg)) == 0
    ok = _cabi.EngineConfig(0, 0, 0, 4096, 1, 8, 24576, 0, 1.0, 0.3, 0.25, 0)
    gb = lib.caro_engine_workspace_bytes(C.byref(ok)) / 1e9
    assert 15 < gb < 40  # DESIGN.md section 3 byte budget


def test_net_state_dict_layout_and_fold(golden_net):
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import Net, fold_state_dict
    import torch.nn.functional as F
    for case in golden_net:
        game = ConnectFour() if case["game"] == "connect4" else TicTacToe(3, 3)
        torch.manual_seed(case["seed"])
        net = Net(game.obs_shape, game.action_space)
        assert {k: list(v.shape) for k, v in net.state_dict().items()} == case["keys"]
        if case["checkpoint"]:
            ck = "connect4_best_026_12000.dat" if case["game"] == "connect4" else "tictactoe_best_005_00900.dat"
            net.load_state_dict(torch.load(os.path.join(GOLDEN, "checkpoints", ck), map_location="cpu"))
        net.eval()
        _, H, W = game.obs_shape
        A = game.action_space
        blob = torch.from_numpy(fold_state_dict(net.state_dict(), H, W, A))
        assert blob.numel() == __import__("caro_ai_b200._cabi", fromlist=["x"]).lib().caro_net_blob_floats(H, W, A)
        # evaluate the folded blob with plain torch ops and compare with the module (BN folding algebra)
        x = torch.rand(5, 2, H, W).round()
        o = [0]

        def take(n):
            r = blob[o[0]:o[0] + n]
            o[0] += n
            return r
        v = F.leaky_relu(F.conv2d(x, take(64 * 2 * 9).view(64, 2, 3, 3), take(64), padding=1), 0.01)
        for _ in range(5):
            v = v + F.leaky_relu(F.conv2d(v, take(64 * 64 * 9).view(64, 64, 3, 3), take(64), padding=1), 0.01)
        hw = H * W
        val = F.leaky_relu(F.conv2d(v, take(64).view(1, 64, 1, 1), take(1)), 0.01).view(-1, hw)
        val = torch.tanh(F.linear(F.leaky_relu(F.linear(val, take(20 * hw).view(20, hw), take(20)), 0.01), take(20).view(1, 20), take(1)))
        pol = F.leaky_relu(F.conv2d(v, take(2 * 64).view(2, 64, 1, 1), take(2)), 0.01).view(-1, 2 * hw)
        pol = F.linear(pol, take(A * 2 * hw).view(A, 2 * hw), take(A))
        with torch.no_grad():
            rp, rv = net(x)
        scale = max(1.0, float(rp.abs().max()))
        assert float((pol - rp).abs().max()) < 2e-4 * scale and float((val - rv).abs().max()) < 1e-4


def test_small_helpers():
    from caro_ai_b200.distributed import shard_games
    from caro_ai_b200.utils import TBMeanTracker, update_counts
    d = {}
    update_counts(d, "a", (1, 2, 3))
    update_counts(d, "a", (1, 0, 0))
    update_counts(d, ("a", "b"), (0, 1, 0))
    assert d == {"a": (2, 2, 3), ("a", "b"): (0, 1, 0)}

    class W:
        def __init__(self):
            self.rows, self.closed = [], False

        def add_scalar(self, *a):
            self.rows.append(a)

        def close(self):
            self.closed = True
    w = W()
    with TBMeanTracker(w, batch_size=2) as tb:
        tb.track("x", 1.0, 0)
        tb.track("x", torch.tensor([3.0, 5.0]), 1)
        tb.track("x", np.float32(9.0), 2)
    assert w.rows == [("x", 2.5, 1)] and w.closed
    for total, ws in [(4096, 8), (20, 8), (7, 2), (1, 4)]:
        parts = [shard_games(total, r, ws) for r in range(ws)]
        assert sum(c for _, c in parts) == total
        assert all(parts[i][0] + parts[i][1] == parts[i + 1][0] for i in range(ws - 1))
        assert max(c for _, c in parts) - min(c for _, c in parts) <= 1


def test_config_matches_reference_values():
    from caro_ai_b200 import config as cfg
    assert (cfg.MCTS_SEARCHES, cfg.MCTS_BATCH_SIZE, cfg.STEPS_BEFORE_TAU_0) == (10, 8, 10)   # config.py:3-4,14
    assert (cfg.C_PUCT, cfg.ALPHA, cfg.EXPLORE) == (1.0, 0.30, 0.25)                         # config.py:26-28
    assert (cfg.REPLAY_BUFFER, cfg.BATCH_SIZE, cfg.TRAIN_ROUNDS, cfg.MIN_REPLAY_TO_TRAIN) == (5000, 256, 10, 2000)
    assert (cfg.PLAY_MCTS_SEARCHES, cfg.PLAY_MCTS_BATCH_SIZE, cfg.BEST_NET_WIN_RATIO) == (40, 8, 0.60)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the oracle port on the host cores) prints ONE JSON line with the keys of the
    bench contract, `impl: reference`, a cpu_baseline describing the run and an e2e object without copies."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "e2e", "cpu_baseline", "impl"):
        assert key in d, key
    assert d["impl"] == "reference" and d["metric"] == "connect4_mcts_leaf_evals_per_sec" and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    vendored = os.path.exists(os.path.join(ROOT, "baseline", "_ref", "lib", "mcts.py"))  # build() copies the unmodified reference
    assert d["cpu_baseline"]["kind"] == ("reference" if vendored else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]
    # ranks other than 0 stay silent under torchrun
    env["RANK"] = "1"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_refuses_zero_steps_and_a_dump_of_the_cpu_arm(tmp_path):
    import subprocess
    import sys
    for extra in (["--steps", "0"], ["--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path / "d")]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120,
                             cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr)
    assert not os.path.exists(tmp_path / "d")


def test_render_strings_match_the_reference(golden_render):
    """game.render (connect_four.py:267-281, tictactoe.py:237-259) and Session.render (play_session.py:38-49) byte for
    byte against strings produced by the unmodified reference (tests/golden/make_golden2.py)."""
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.play_session import Session

    def game_of(tag):
        if tag == "connect4":
            return ConnectFour()
        _, n, k = tag.split(":")
        return TicTacToe(int(n), int(k))
    total = 0
    for block in golden_render["games"]:
        g = game_of(block["game"])
        for row in block["positions"]:
            assert g.render(row["state"]) == row["render"], (block["game"], row["state"])
            total += 1
    assert total >= 60
    for row in golden_render["sessions"]:
        s = Session.__new__(Session)  # the string needs no checkpoint, tree or GPU
        s.game, s.state, s.value = game_of(row["game"]), row["state"], row["value"]
        assert s.render() == row["render"]


def test_sgd_losses_match_the_reference_train_step(golden_train):
    """train.py:95-106 (MSE + soft-target cross-entropy) on the first batch the reference's train_neural_net drew from the
    fixture's replay buffer (same `random` seed, same Net seed): value / policy loss to 1e-5.  CPU, like the reference ran
    it; the planes come from the oracle's encoder here (the CUDA encoder's parity is a -m gpu test)."""
    import random
    from caro_ai_b200 import config as cfg
    from caro_ai_b200.model import Net
    from caro_ai_b200.train import sgd_losses
    from helpers import oracle_game
    for case in golden_train:
        og = oracle_game(case["game"])
        replay = collections.deque([(s, p, pi, z) for s, p, pi, z in case["replay"]], maxlen=cfg.REPLAY_BUFFER)
        random.seed(case["sample_seed"])
        batch = random.sample(replay, cfg.BATCH_SIZE)
        assert [b[0] for b in batch[:8]] == case["first_batch_states"]
        torch.manual_seed(case["net_seed"])
        net = Net(og.obs_shape, og.action_space)
        for k, v in net.state_dict().items():
            if v.dtype.is_floating_point:
                assert abs(float(v.double().sum()) - case["init_sum"][k]) < 1e-9, k  # same initial weights as the reference's Net
        net.train()
        planes = torch.tensor(og.states_to_training_batch([b[0] for b in batch], [b[1] for b in batch]))
        total, lv, lp = sgd_losses(net, planes, torch.FloatTensor([b[2] for b in batch]), torch.FloatTensor([b[3] for b in batch]))
        assert abs(lv.item() - case["round0"]["loss_value"]) < 1e-5
        assert abs(lp.item() - case["round0"]["loss_policy"]) < 1e-5
        assert abs(total.item() - (lv.item() + lp.item())) < 1e-6


def test_single_rank_collective_helpers_are_identities():
    from caro_ai_b200 import distributed as D
    assert D.all_min(1234) == 1234
    t = (torch.ones(3, 2), torch.zeros(3))
    out = D.all_gather_rows(t)
    assert out[0] is t[0] and out[1] is t[1]
    assert D.reduce_tallies(1, 2, 3) == (1, 2, 3)


def test_deep_tower_blob_sizes():
    """The number of residual blocks is a property of the weight blob: 5 (the reference) by default, 1..20 accepted."""
    from caro_ai_b200 import _cabi
    from caro_ai_b200.model import Net, fold_state_dict
    lib = _cabi.lib()
    per_block = 64 * 64 * 9 + 64
    assert lib.caro_net_blob_floats_deep(6, 7, 7, 5) == lib.caro_net_blob_floats(6, 7, 7)
    assert lib.caro_net_blob_floats_deep(6, 7, 7, 10) == lib.caro_net_blob_floats(6, 7, 7) + 5 * per_block
    assert lib.caro_net_blob_floats_deep(6, 7, 7, 0) == 0 and lib.caro_net_blob_floats_deep(6, 7, 7, 21) == 0
    net = Net((2, 3, 3), 9, blocks=7)
    assert fold_state_dict(net.state_dict(), 3, 3, 9).size == lib.caro_net_blob_floats_deep(3, 3, 9, 7)
    x = torch.rand(4, 2, 3, 3)
    logits, value = net(x)
    assert tuple(logits.shape) == (4, 9) and tuple(value.shape) == (4, 1)
