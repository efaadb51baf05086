"""The Gumbel root search extension without a GPU: the phase tables, sigma / completed Q / pi' on hand-built rows, the
host compile of the Gumbel draw, the oracle's forced descents, and the C ABI, header and CLI surfaces."""
import argparse
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from gumbel_native import gumbel_lib, host_draws
from gumbel_reference import (GumbelOracleTree, completed_q, improved_policy, phase_of, phases, schedule, sigmas,
                              survivors, top)
from oracle.games import MNKOracle


# ------------------------------------------------------------------------------------------------ schedule
@pytest.mark.parametrize("m", [1, 2, 3, 5, 7, 16, 32])
def test_phase_tables(m):
    H = phases(m)
    assert (1 << H) >= m and (H == 0 or (1 << (H - 1)) < m)
    assert survivors(m, 0) == m and (m < 2 or survivors(m, max(H - 1, 0)) == 2)
    for cp in range(1, 13):
        for batch in (1, 3, 8):
            rows = schedule(m, cp, batch)
            assert len(rows) == cp and rows[0][0] == 0 and rows[0][1] == m
            seen = [r[0] for r in rows]
            assert seen == sorted(seen) and max(seen) <= max(H - 1, 0)
            if cp >= H:  # with enough minibatches every phase runs
                assert sorted(set(seen)) == list(range(max(H, 1)))
            for phase, r, kstart, slots in rows:
                assert r == survivors(m, phase) and 1 <= r <= m
                assert all(0 <= s < r for s in slots) and len(slots) == batch
                assert phase_of(kstart, m, cp) == phase and (kstart == 0 or phase_of(kstart - 1, m, cp) < phase)
            # every descent of a phase cycles through its survivors in order
            for phase in set(seen):
                flat = [s for p, r, _, slots in rows if p == phase for s in slots]
                r = survivors(m, phase)
                assert flat == [i % r for i in range(len(flat))]


def test_skipped_phases():
    # m = 32 (H = 5) over C' = 2 minibatches: phase 0 (32 survivors) then phase 2 (8), phases 1, 3, 4 skipped
    rows = schedule(32, 2, 8)
    assert [(p, r) for p, r, _, _ in rows] == [(0, 32), (2, 8)]
    assert [p for p, _, _, _ in schedule(16, 3, 1)] == [0, 1, 2]
    assert [p for p, _, _, _ in schedule(3, 1, 4)] == [0]
    assert schedule(1, 5, 4) == [(0, 1, 0, [0, 0, 0, 0])] * 5


# ------------------------------------------------------------------------------------------------ scores
def test_sigma_and_completed_q_by_hand():
    n = [4, 0, 2, 0, 0]
    q = [0.5, 0.0, -0.25, 0.0, 0.0]
    p = [0.4, 0.3, 0.2, 0.1, 0.0]
    legal = [0, 1, 2, 4]                      # action 3 is illegal
    p32 = [float(np.float32(x)) for x in p]
    qbar = (p32[0] * 0.5 + p32[2] * -0.25) / (p32[0] + p32[2])
    cq = completed_q(n, q, p, legal)
    assert cq[0] == 0.5 and cq[2] == -0.25 and cq[1] == qbar and cq[4] == qbar
    sig = sigmas(n, q, p, legal, 50.0, 0.1)
    scale = (50.0 + 4.0) * 0.1
    assert sig[0] == scale * ((0.5 + 1.0) * 0.5) and sig[1] == scale * ((qbar + 1.0) * 0.5)
    # no visit: every q is 0, sigma = c_visit * c_scale * 0.5
    assert sigmas([0] * 5, [0.0] * 5, p, legal, 50.0, 0.1) == [50.0 * 0.1 * 0.5] * 5


def test_improved_policy_by_hand():
    n = [4, 0, 2, 0, 0]
    q = [0.5, 0.0, -0.25, 0.0, 0.0]
    p = [0.4, 0.3, 0.2, 0.1, 0.0]
    legal = [0, 1, 2, 4]
    pi = improved_policy(n, q, p, legal, 50.0, 0.1)
    sig = sigmas(n, q, p, legal, 50.0, 0.1)
    logit = np.array([math.log(float(np.float32(p[a]))) + sig[a] for a in (0, 1, 2)])
    ref = np.exp(logit - logit.max()) / np.exp(logit - logit.max()).sum()
    np.testing.assert_allclose(pi[[0, 1, 2]], ref, rtol=1e-6)
    assert pi[3] == 0.0 and pi[4] == 0.0        # illegal, and P = 0 (log P = -inf)
    assert pi.dtype == np.float32 and abs(float(pi.sum()) - 1.0) < 1e-6
    assert pi[0] > pi[1] > pi[2]                # the visited winning edge gains, the losing one drops below its prior
    # every legal logit -inf: uniform over the legal moves
    u = improved_policy([0, 0, 0], [0.0] * 3, [0.0, 0.0, 1.0], [0, 1], 50.0, 0.1)
    assert u.tolist() == [0.5, 0.5, 0.0]


def test_ties_go_to_the_lowest_action():
    key = {0: 1.0, 1: 2.0, 2: 2.0, 3: -math.inf, 4: -math.inf}
    assert top([4, 3, 2, 1, 0], key, 5) == [1, 2, 0, 3, 4]
    tree = GumbelOracleTree(MNKOracle(2, 2), m=4)
    s = tree.game.initial_state
    tree._new_node(s, np.full(4, 0.25, dtype=np.float32))
    tree.plan(np.zeros(4), 0, 4, 2, s)  # equal draws and priors: the survivors are in action order
    assert tree.surv == [0, 1, 2, 3] and tree.forced == [0, 1] and tree.move(s) == 0


# ------------------------------------------------------------------------------------------------ the draw
def test_host_draw_interval_and_moments():
    lib = gumbel_lib()
    rng = np.random.default_rng(7)
    seeds = rng.integers(0, 2 ** 63, size=4)
    g = []
    for i in range(100000):
        s = int(seeds[i % 4])
        g.append(lib.gc_gumbel(s & 0xFFFFFFFF, s >> 32, i // 225, i % 7, (i // 7) % 50, i % 225))
    g = np.array(g)
    assert np.isfinite(g).all()
    euler = 0.5772156649015329
    assert abs(g.mean() - euler) < 0.02          # sd 1.28 / sqrt(1e5) = 0.004
    assert abs(g.var() - math.pi ** 2 / 6) < 0.05
    u = np.array([lib.gc_uniform(1, 2, i, 0, 0, i % 225) for i in range(2000)])
    assert (u > 0).all() and (u < 1).all()
    # distinct addresses give distinct draws; the same address the same draw
    assert host_draws(5, 3, 0, 1, 9) == host_draws(5, 3, 0, 1, 9)
    assert host_draws(5, 3, 0, 1, 9) != host_draws(5, 3, 1, 1, 9) != host_draws(5, 3, 0, 2, 9)


# ------------------------------------------------------------------------------------------------ the oracle's descents
def test_oracle_forces_the_planned_root_actions():
    og = MNKOracle(3, 3)
    tree = GumbelOracleTree(og, m=4)
    s = og.initial_state
    rng = np.random.default_rng(3)
    g = rng.gumbel(size=9)
    count, batch = 6, 4
    for i in range(count):
        forced = tree.plan(g, i, count, batch, s)
        if i == 0:
            assert forced == [-1] * batch and tree.i0 == -1  # the root is not in the tree yet
        else:
            assert tree.i0 == 1 and len(set(forced)) <= 4 and set(forced) <= set(tree.surv)
        tree.trace = []
        tree.minibatch(batch, s, 0, rng.dirichlet([0.3] * 9, size=batch))
        if forced[0] >= 0:
            assert [d[4][0] for d in tree.trace[-1]["descents"]] == forced
    assert tree.phase == phases(4) - 1 and len(tree.surv) == 2
    pi, _ = tree.get_policy_value(s, tau=1)
    assert abs(sum(pi) - 1.0) < 1e-6 and tree.get_policy_value(s, tau=0)[0][tree.move(s)] == 1.0
    assert tree.move(s) in tree.surv


# ------------------------------------------------------------------------------------------------ surfaces
def test_header_and_ctypes_agree_on_gumbel():
    from caro_ai_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "caro_b200.h")).read()
    assert re.search(r"int caro_engine_set_gumbel\(caro_engine\* e, int players, int m, double c_visit, double c_scale, "
                     r"double gumbel_scale,\s+void\* stream\);", header)
    assert re.search(r"int caro_engine_gumbel_plan\(caro_engine\* e, int search_index, int minibatch, int count, int batch, "
                     r"void\* stream\);", header)
    for region in ("gumbel_params", "gumbel_g", "gumbel_state", "gumbel_root"):
        assert '"%s"' % region in header
    assert "#define CARO_ABI_VERSION 2" in header
    res, args = _cabi._SIGNATURES["caro_engine_set_gumbel"]
    assert res is C.c_int and args == [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p]
    res, args = _cabi._SIGNATURES["caro_engine_gumbel_plan"]
    assert res is C.c_int and args == [C.c_void_p] + [C.c_int] * 4 + [C.c_void_p]
    lib = _cabi.lib()
    assert lib.caro_engine_set_gumbel(None, 3, 16, 50.0, 0.1, 1.0, None) == -1 and b"null engine" in lib.caro_last_error()
    assert lib.caro_engine_gumbel_plan(None, 0, 0, 1, 8, None) == -1 and b"null engine" in lib.caro_last_error()
    from caro_ai_b200.engine import SelfPlayEngine
    assert SelfPlayEngine.GUMBEL_STATE_DTYPE.itemsize == 80


def test_cli_gumbel_options():
    from caro_ai_b200 import train
    a = train.parse_args(["-n", "x", "-g", "0"])
    assert a.gumbel is False and a.gumbel_m == 16
    a = train.parse_args(["-n", "x", "-g", "0", "--gumbel", "--gumbel-m", "8"])
    assert a.gumbel is True and a.gumbel_m == 8
    for bad in ("0", "33"):
        with pytest.raises(SystemExit):
            train.parse_args(["-n", "x", "-g", "0", "--gumbel-m", bad])
    import caro_ai_b200.play as play
    seen = {}

    def fake_parse(self, argv=None, namespace=None):
        seen["actions"] = {a.dest: a.default for a in self._actions}
        raise SystemExit(0)
    orig = argparse.ArgumentParser.parse_args
    argparse.ArgumentParser.parse_args = fake_parse
    try:
        with pytest.raises(SystemExit):
            play.main(["a", "b", "-g", "0"])
    finally:
        argparse.ArgumentParser.parse_args = orig
    assert seen["actions"]["gumbel"] is False
