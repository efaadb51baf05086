"""Host-side half of the search-kernel matrix (no GPU): every case of tests/test_gpu_search_matrix.py maps to the kernel
instances engine.cu launches for it, together the cases reach every instance, the chain stub drives the oracle past
the depths the deep-path cases assert, and the virtual-loss oracle scores a hand-built tree as worked out by hand."""
import math

import numpy as np

from oracle.games import MNKOracle
from oracle.stubs import chain_priors
from search_matrix import ALL_CASES, CHAIN_CASES, PARITY_CASES, VL_CASES, VirtualLossOracleTree, instances, \
    noise_instance, oracle_first_move, NOISE_BOARDS

SELECT_MNK = ["select_thread_kernel<MnkRules,2>", "select_thread_kernel<MnkRules,4>"] + \
    ["select_kernel<MnkRules,32,%d>" % apl for apl in (1, 2, 4, 8)]
NOISE = ["noise_kernel<%d,%d>" % gw_apl for gw_apl in ((8, 1), (16, 1), (32, 1), (32, 2), (32, 4), (32, 8))]


def test_cases_map_to_the_engine_dispatch():
    by_name = {c.name: instances(c) for c in ALL_CASES}
    assert len(by_name) == len(ALL_CASES), "case names must be unique"
    assert by_name["mnk2_2"]["select"] == "select_thread_kernel<MnkRules,2>"
    assert by_name["mnk4_4"]["select"] == "select_thread_kernel<MnkRules,4>"
    assert by_name["mnk8_5"]["select"] == "select_kernel<MnkRules,32,2>"  # A = 64, the upper edge of APL 2
    assert by_name["mnk11_5"]["select"] == "select_kernel<MnkRules,32,4>"
    assert by_name["mnk12_5"]["select"] == "select_kernel<MnkRules,32,8>"
    assert by_name["c4_b32"]["plan"] == "plan_kernel<C4Board,32>" and by_name["c4_b32"]["expand"] == "expand_backup_kernel<C4Rules,32>"
    assert by_name["vl_mnk9_5_b8"]["select"] == "select_vl_kernel<MnkRules>"
    assert by_name["vl_c4_b32"]["select"] == "select_vl_group_kernel<C4Rules>"
    assert [noise_instance(n * n) for n in (2, 4, 5, 8, 11, 15)] == [NOISE[0], NOISE[1], NOISE[2], NOISE[3], NOISE[4], NOISE[5]]
    assert [noise_instance(n * n + 1) for n in (4, 8)] == [NOISE[2], NOISE[4]]  # 17 and 65 actions: one width up


def test_matrix_covers_every_instance():
    plain = [c for c in PARITY_CASES + CHAIN_CASES]
    got = {k: {instances(c)[k] for c in plain} for k in ("select", "noise", "plan", "expand")}
    assert set(SELECT_MNK) <= got["select"], set(SELECT_MNK) - got["select"]
    assert "select_thread_kernel<C4Rules,2>" in got["select"]
    assert set(NOISE[1:]) <= got["noise"], set(NOISE[1:]) - got["noise"]  # <8,1> is also in test_gpu_round2
    assert {noise_instance(n * n) for n in NOISE_BOARDS} == set(NOISE)   # the stand-alone noise test: every width
    for width in (8, 16, 32):
        cases = [c for c in plain if instances(c)["plan"].endswith(",%d>" % width)]
        batches = {c.batch for c in cases}
        # each plan / expand width with a batch equal to and one below it, on boards of at least two select widths
        assert width in batches and min(batches) < width, (width, batches)
        assert len({instances(c)["select"] for c in cases}) >= 2, width
        for board in ("MnkBoard", "C4Board"):
            assert "plan_kernel<%s,%d>" % (board, width) in got["plan"] or width != 32, (board, width)
        assert "expand_backup_kernel<MnkRules,%d>" % width in got["expand"]
    assert "expand_backup_kernel<C4Rules,32>" in got["expand"]
    # a batch below max_batch ([G][batch][A] noise, [G][B] descents), with both noise sources
    assert {c.noise for c in plain if c.batch < c.max_batch} == {"host", "philox"}
    # two trees per game on m,n,k boards, and on Connect4
    assert any(c.trees_per_game == 2 and not c.connect4 for c in plain) and any(c.trees_per_game == 2 and c.connect4 for c in plain)
    # the tau = 1 and the tau = 0 move of root_policy / advance at every select width
    for sel in got["select"]:
        assert any(0 < c.tau_plies < c.moves for c in plain if instances(c)["select"] == sel), sel
    # Philox noise on a board of every noise width the parity cases reach
    assert {noise_instance(c.A) for c in plain if c.noise == "philox"} >= set(NOISE[1:])
    # batch widths used across the matrix
    assert {1, 3, 8, 9, 16, 17, 31, 32} <= {c.batch for c in plain}
    # back-up paths past one and two passes of the 32-lane depth loop, on both rule sets, and at batch 32
    assert max(c.min_path for c in CHAIN_CASES if not c.connect4) >= 64 and any(c.min_path >= 32 and c.connect4 for c in CHAIN_CASES)
    assert any(c.batch == 32 and c.min_path >= 32 for c in CHAIN_CASES)
    # virtual loss: the one-thread-per-game kernel on three m,n,k boards, the group kernel on Connect4, batch 8 and 32
    vl = {(c.board, c.batch): instances(c)["select"] for c in VL_CASES}
    assert {b for (b, _), s in vl.items() if s == "select_vl_kernel<MnkRules>"} == {(3, 3), (5, 4), (9, 5)}
    assert {bt for (_, bt) in vl} == {8, 32} and "select_vl_group_kernel<C4Rules>" in vl.values()


def test_chain_stub_reaches_the_asserted_depth():
    """The deep-path cases use host noise from their seed, so this CPU run IS the search the engine must reproduce:
    its longest path is the one the GPU test asserts on."""
    for case in CHAIN_CASES:
        _, longest = oracle_first_move(case)
        assert longest > case.min_path, (case.name, longest, case.min_path)


def test_chain_stub_is_a_pure_function_of_the_planes():
    og = MNKOracle(9, 9)
    s = og.initial_state
    for a in (40, 3, 77):
        s, _ = og.move(s, a, 0)
    planes = og.states_to_training_batch([s, s, og.initial_state], [1, 1, 0])
    p, v = chain_priors(planes, 81)
    assert p.dtype == np.float32 and v.dtype == np.float32 and not v.any()
    assert np.array_equal(p[0], p[1]) and abs(float(p[0].sum()) - 1.0) < 1e-5
    top = int(np.argmax(p[0]))
    assert p[0, top] == np.float32(0.99) and top not in (40, 3, 77)
    assert np.all(p[0][np.arange(81) != top] == np.float32(0.01 / 80))


def _tree():
    """Empty 3x3 root, player 0, with two visited edges: (0) N = 1, W = f32(0.25); (1) N = 3, W = -1.0, a python float
    (three back-ups of terminal values, which the plain select would divide in float64)."""
    og = MNKOracle(3, 3)
    t = VirtualLossOracleTree(og)
    root = og.initial_state
    p = np.array([0.4, 0.3, 0.1, 0.05, 0.05, 0.05, 0.02, 0.02, 0.01], dtype=np.float32)
    t._new_node(root, p)
    t.visit_count[root][0], t.value[root][0] = 1, np.float32(0.25)
    t.visit_count[root][1], t.value[root][1] = 3, -1.0
    return og, t, root, p


def test_virtual_loss_oracle_scores_by_hand():
    og, t, root, p = _tree()
    z = np.full(9, 1 / 9)
    f = np.float32

    def root_score(q, pa, sum_n, n):  # Q + c * (f64(f32(0.75 * P)) + 0.25 * z) * sqrt(sum N) / (1 + n)
        return q + 1.0 * (float(f(0.75) * pa) + 0.25 / 9) * math.sqrt(sum_n) / (1 + n)

    # descent 0: no virtual visits; sum N = 4
    s0 = t.vl_scores(root, 0, [0] * 9, z)
    assert s0[0] == root_score(0.25, p[0], 4, 1)
    assert s0[1] == root_score(float(f(-1.0) / f(3.0)), p[1], 4, 3)  # f32(-1/3), not the float64 quotient
    assert s0[1] != root_score(-1.0 / 3.0, p[1], 4, 3)
    assert s0[2] == root_score(0.0, p[2], 4, 0)
    assert int(np.argmax(s0)) == 0
    # descent 1: one virtual visit on (root, 0): n = 2, w = f32(0.25 - 1) = -0.75, q = -0.375; sum N = 5
    s1 = t.vl_scores(root, 0, [1] + [0] * 8, z)
    assert s1[0] == root_score(-0.375, p[0], 5, 2)
    assert s1[2] == root_score(0.0, p[2], 5, 0)
    assert int(np.argmax(s1)) == 2
    # descent 2: virtual visits on 0 and 2; actions 3, 4 and 5 tie and the lowest wins
    s2 = t.vl_scores(root, 0, [1, 0, 1] + [0] * 6, z)
    assert s2[2] == root_score(-1.0, p[2], 6, 1) and s2[3] == s2[4] == s2[5] == root_score(0.0, p[3], 6, 0)
    assert int(np.argmax(s2)) == 3
    # interior (float32): t = f32(f32(f32(c * P) * f32(sqrt(sum N))) / (1 + n)), score = f32(Q + t)
    child = og.move(root, 4, 0)[0]
    t._new_node(child, p)
    t.visit_count[child][0], t.value[child][0] = 2, np.float32(0.3)
    si = t.vl_scores(child, 1, [1] + [0] * 8)
    n0 = 3
    want0 = f(f(0.3) - f(1.0)) / f(n0) + (f(1.0) * p[0] * np.sqrt(f(3))) / f(1 + n0)
    assert si[0] == float(want0) and isinstance(want0, np.float32)
    assert si[4] == -math.inf  # occupied cell
    assert si[8] == float(f(1.0) * p[8] * np.sqrt(f(3)) / f(1))


def test_virtual_loss_oracle_spreads_one_minibatch():
    """Three descents of one minibatch on the hand-built tree: without virtual loss all three would take action 0;
    here they take 0, 2 and 3 (the scores above), expand three distinct leaves and back each up once."""
    og, t, root, _ = _tree()
    t._noise, t._j = np.full((3, 9), 1 / 9), 0
    t.search_minibatch(3, root, 0, None)
    assert [acts for _, acts in t._paths] == [[0], [2], [3]]
    assert t.visit_count[root][:4] == [2, 3, 1, 1] and len(t.probs) == 4
