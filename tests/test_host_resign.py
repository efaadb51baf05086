"""CPU tests of the resignation extension: the calibration functions of utils.py, the host restatement of the kernel's
statistic, the C ABI's argument checks, the header against the ctypes mirror, the train.py options and the rank
reduction of the calibration (world size 2, gloo)."""
import ctypes as C
import math
import os
import re
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT
from resign_reference import false_positive, root_stat


def _records(rows):
    from caro_ai_b200.engine import SelfPlayEngine
    return np.array([((m0, m1), r, p) for m0, m1, r, p in rows], dtype=SelfPlayEngine.RESIGN_RECORD_DTYPE)


def test_grid_is_fixed():
    from caro_ai_b200 import utils
    assert len(utils.RESIGN_GRID) == 50 and utils.RESIGN_GRID[0] == -0.99 and utils.RESIGN_GRID[-1] == -0.50
    assert all(round(b - a, 2) == 0.01 for a, b in zip(utils.RESIGN_GRID, utils.RESIGN_GRID[1:]))


def test_tallies_count_draws_and_wins_but_not_losses_and_compare_strictly():
    from caro_ai_b200 import utils
    i90, i80 = utils.RESIGN_GRID.index(-0.9), utils.RESIGN_GRID.index(-0.8)
    # player 0 dipped to -0.85: a loss for player 0 is never a false positive, a draw or a win is
    for result, fp in ((-1, 0), (0, 1), (1, 1)):
        t = utils.resign_tallies(_records([(-0.85, 0.3, result, 20)]))
        assert t[i90].tolist() == [0, 1] and t[i80].tolist() == [fp, 1], result
    # the same for player 1 (a loss for player 1 is result +1)
    for result, fp in ((1, 0), (0, 1), (-1, 1)):
        t = utils.resign_tallies(_records([(0.3, -0.85, result, 20)]))
        assert t[i80].tolist() == [fp, 1], result
    # min == t does not count (stat < t resigns), the next grid point up does
    t = utils.resign_tallies(_records([(-0.9, 0.5, 0, 9)]))
    assert t[i90, 0] == 0 and t[i90 + 1, 0] == 1
    # +inf minima (a player who never had a statistic) never count
    t = utils.resign_tallies(_records([(math.inf, math.inf, 0, 1)]))
    assert t[:, 0].sum() == 0 and (t[:, 1] == 1).all()
    # every row agrees with the per-record definition
    rng = np.random.default_rng(3)
    rows = [(float(rng.uniform(-1, 0)), float(rng.uniform(-1, 0)), int(rng.integers(-1, 2)), 10) for _ in range(300)]
    t = utils.resign_tallies(_records(rows))
    for i, th in enumerate(utils.RESIGN_GRID):
        assert t[i].tolist() == [sum(false_positive((r[0], r[1]), r[2], th) for r in rows), 300]
    assert utils.resign_tallies(_records([])).sum() == 0


def test_choose_threshold_takes_the_largest_within_target_and_waits_for_records():
    from caro_ai_b200 import utils
    # 200 games: 190 clean losses for player 0 at -0.95, 10 draws where player 0 dipped to -0.7
    rows = [(-0.95, 0.5, -1, 30)] * 190 + [(-0.7, 0.2, 0, 40)] * 10
    t = utils.resign_tallies(_records(rows))
    assert utils.choose_resign_threshold(t) == -0.5  # 10 / 200 = 5 % <= 5 % everywhere
    assert utils.choose_resign_threshold(t, target=0.04) == -0.7  # above -0.7 the draws count
    assert utils.choose_resign_threshold(t, min_records=201) is None
    assert utils.choose_resign_threshold(utils.resign_tallies(_records(rows[:199]))) is None
    bad = utils.resign_tallies(_records([(-0.995, -0.995, 0, 5)] * 300))
    assert utils.choose_resign_threshold(bad) is None  # no threshold qualifies
    # tallies add element-wise
    a, b = _records(rows[:120]), _records(rows[120:])
    assert (utils.resign_tallies(a) + utils.resign_tallies(b) == t).all()


def test_host_statistic_sums_in_action_order():
    """A 3x3 root row where numpy's pairwise sum rounds differently from the kernel's sequential __dadd_rn chain."""
    tiny = float(np.float32(2.0 ** -53))
    w = np.array([1.0] + [tiny] * 8, dtype=np.float32)
    n = [1] * 9
    seq = 1.0
    for v in w[1:]:
        seq = seq + float(v)
    assert seq == 1.0 and float(np.sum(w.astype(np.float64))) != seq
    assert root_stat(n, w) == max(seq / 9.0, 1.0)
    # v_best: the most visited edge, lowest action on ties, float32 division
    w2 = np.array([-3.0, -2.0, -2.0], dtype=np.float32)
    assert root_stat([3, 3, 1], w2) == max((-7.0) / 7.0, float(np.float32(-3.0) / np.float32(3.0)))
    w3 = np.array([-1.0, 0.2, -0.9], dtype=np.float32)
    assert root_stat([1, 2, 7], w3) == float(np.float32(-0.9) / np.float32(7.0))
    assert root_stat([0, 0, 0], w3) is None


def test_set_resign_refuses_bad_arguments_before_touching_the_device():
    from caro_ai_b200 import _cabi
    lib = _cabi.lib()
    assert lib.caro_engine_set_resign(None, 1, -0.9, 0.1, None) == -1  # CARO_E_ARG
    assert b"null" in lib.caro_last_error()
    bogus = C.c_void_p(16)  # never dereferenced: every argument below is refused first
    for th, share in ((float("nan"), 0.1), (1.5, 0.1), (-1.0001, 0.1), (-0.9, -0.01), (-0.9, 1.01), (-0.9, float("nan"))):
        assert lib.caro_engine_set_resign(bogus, 1, th, share, None) == -1, (th, share)
        assert (b"threshold" if not -1 <= th <= 1 else b"playthrough") in lib.caro_last_error()


def test_header_and_ctypes_mirror_agree():
    from caro_ai_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "caro_b200.h")).read()
    code = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    m = re.search(r"int\s+caro_engine_set_resign\s*\(([^)]*)\)", code)
    assert m, "caro_engine_set_resign is not declared"
    params = [p.strip() for p in m.group(1).split(",")]
    assert [re.sub(r"\s*\w+$", "", p) for p in params] == ["caro_engine*", "int", "double", "double", "void*"]
    res, args = _cabi._SIGNATURES["caro_engine_set_resign"]
    assert res is C.c_int and args == [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p]
    for region in ("resign_params", "resign_playthrough", "resign_min", "resign_log", "resign_counters"):
        assert '"%s"' % region in header, region
    assert "#define CARO_ABI_VERSION 2" in header
    assert "CARO_FLAG_RESIGN" not in header


def test_engine_regions_follow_every_existing_region():
    """Workspace sizes grow by the resignation regions only; a config's existing bytes stay where they were."""
    from caro_ai_b200 import _cabi
    lib = _cabi.lib()
    for game, n, k, G in ((0, 0, 0, 64), (1, 9, 5, 100), (2, 15, 5, 7)):
        cfg = _cabi.EngineConfig(game, n, k, G, 2, 8, 512, 64, 1.0, 0.3, 0.25, 0, 0, 0)
        total = lib.caro_engine_workspace_bytes(C.byref(cfg))
        assert total > 0
        # params 24 B, playthrough G B, minima 16 G B, log 24 G B, counters 16 B, each 256-aligned
        tail = 0
        for nbytes in (24, G, 16 * G, 24 * G, 16):
            tail = ((tail + 255) & ~255) + nbytes
        assert total >= tail


def test_train_options_parse_with_off_as_default():
    from caro_ai_b200 import train
    a = train.parse_args(["-g", "1", "-n", "x"])
    assert a.resign is None and a.resign_playthrough == 0.1
    assert train.parse_args(["-g", "1", "-n", "x", "--resign", "off"]).resign is None
    assert train.parse_args(["-g", "1", "-n", "x", "--resign", "auto"]).resign == "auto"
    b = train.parse_args(["-g", "0", "-n", "x", "--resign", "-0.9", "--resign-playthrough", "0.25"])
    assert b.resign == -0.9 and b.resign_playthrough == 0.25
    for bad in (["--resign", "1.5"], ["--resign", "sometimes"], ["--resign-playthrough", "1.2"]):
        with pytest.raises(SystemExit):
            train.parse_args(["-g", "0", "-n", "x"] + bad)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_rows(rank):
    # rank 0 alone: 150 clean games (too few to calibrate); rank 1 alone: 100 games, 10 % draws that dipped to -0.8
    if rank == 0:
        return [(-0.95, 0.4, -1, 30)] * 150
    return [(0.4, -0.95, 1, 30)] * 90 + [(-0.8, 0.1, 0, 40)] * 10


def _worker(rank, world_size, port, results):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    import sys
    sys.path.insert(0, ROOT)
    from caro_ai_b200 import utils
    local = utils.choose_resign_threshold(utils.resign_tallies(_records(_rank_rows(rank))))
    t, tallies = utils.resign_threshold_over_ranks(_records(_rank_rows(rank)))
    results[rank] = (local, t, tallies.tolist())
    dist.destroy_process_group()


def test_two_ranks_pick_the_same_threshold_from_unequal_logs():
    from caro_ai_b200 import utils
    port = _free_port()
    with mp.Manager() as mgr:
        results = mgr.dict()
        mp.spawn(_worker, args=(2, port, results), nprocs=2, join=True)
        r0, r1 = results[0], results[1]
    both = _records(_rank_rows(0) + _rank_rows(1))
    want = utils.choose_resign_threshold(utils.resign_tallies(both))
    assert r0[0] is None and r1[0] is None  # neither rank holds 200 games
    assert want == -0.5 and r0[1] == r1[1] == want  # 10 / 250 = 4 %
    assert r0[2] == r1[2] == utils.resign_tallies(both).tolist()
