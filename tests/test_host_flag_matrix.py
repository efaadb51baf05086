"""Host-side half of the flag matrix (no GPU): the restated MASK_PRIORS renormalisation against float64, the restated
tree clear of FRESH_TREE / RECYCLE_TREE worked by hand, every case of tests/test_gpu_flag_matrix.py mapped to the kernel
instances engine.cu launches for it, the cases together reaching every (flags, select, expand) cell, and the recycle
cases doing in the oracle what their capacities were chosen for."""
import numpy as np
import pytest

from flag_reference import FLAG_CASES, FLAG_FRESH_TREE, FLAG_MASK_PRIORS, FLAG_RECYCLE_TREE, FRESH_CASES, MASK_CASES, \
    MASK_VL_CASES, PIPELINE_CASE, RECYCLE_CASES, clear_after_move, flag_instances, legal_part, masked_priors, \
    oracle_run
from search_matrix import VL_CASES, instances
from oracle.stubs import stub_priors

f32 = np.float32


def _gamma(d):
    """Higham's gamma_d for float32: a sum of non-negative terms, each of which goes through at most d roundings, is
    within gamma_d of the exact sum (relative)."""
    u = 2.0 ** -24
    return d * u / (1 - d * u)


def _depth(legal, gw):
    """Roundings a term of legal_part goes through at most: the adds of its lane after the first, then the butterfly."""
    per_lane = np.bincount(np.flatnonzero(legal) % gw, minlength=gw)
    return max(int(per_lane.max()) - 1, 0) + int(np.log2(gw))


def _rows(A, rng, count):
    """Rows of the kind the engine masks: the hash stub's priors of random boards, Dirichlet draws rounded to float32,
    and rows with a few large entries over many tiny ones."""
    planes = rng.integers(0, 2, size=(count, 2, A)).astype(np.float32)
    rows = list(stub_priors(planes, A)[0])
    rows += list(rng.dirichlet([0.3] * A, size=count).astype(np.float32))
    for _ in range(count):
        r = (rng.random(A) * 1e-4).astype(np.float32)
        r[rng.choice(A, size=min(3, A), replace=False)] = f32(0.3)
        rows.append(r)
    return rows


# ------------------------------------------------------------------------------------------------ MASK_PRIORS
@pytest.mark.parametrize("A", [7, 9, 25, 81, 225])
def test_masked_priors_against_float64(A):
    """One and several actions per lane (A = 7 .. 225 over 32 lanes; 8 lanes where the eight-lane kernel runs), against
    the float64 q = p / sum(legal p): the float32 legal mass is within gamma_d of the float64 sum, d the roundings a
    term goes through; every legal prior is the correctly rounded p / part (float64 quotient rounded once more, which
    for float32 operands is the IEEE float32 quotient); so it is within half an ulp plus q * gamma_d / (1 - gamma_d) of
    q; the row sums to one within 1e-6; illegal moves are exactly zero.  (A flat 2-ulp bound does not hold for a float32
    sum: rows here reach 3.5 ulp at A = 225, all of it from the sum.)"""
    rng = np.random.default_rng(A)
    for gw in ((8, 32) if A <= 8 else (32,)):
        for row in _rows(A, rng, 40):
            for density in (1.0, 0.6, 0.2):
                legal = rng.random(A) < density
                legal[rng.integers(A)] = True
                out = masked_priors(row, legal, gw)
                assert out.dtype == np.float32 and (out[~legal] == 0).all()
                p64 = row.astype(np.float64)
                total = p64[legal].sum()
                part = legal_part(row, legal, gw)
                g = _gamma(_depth(legal, gw))
                assert abs(float(part) - total) <= g * total, (A, gw, density)
                assert np.array_equal(out[legal], (p64[legal] / np.float64(part)).astype(np.float32)), (A, gw, density)
                q = p64[legal] / total
                err = np.abs(out[legal].astype(np.float64) - q)
                assert (err <= 0.5 * np.spacing(out[legal]).astype(np.float64) + q * g / (1 - g)).all(), (A, gw, density)
                assert abs(out.astype(np.float64).sum() - 1.0) < 1e-6


def test_masked_priors_all_legal_is_the_row_renormalised():
    """Every move legal: a row whose float32 sum is exactly 1 comes back unchanged, one that sums to exactly 2 comes back
    halved (both exact in float32), and any row comes back as the correctly rounded row / part."""
    for A in (7, 9, 81):
        legal = np.ones(A, dtype=bool)
        row = np.full(A, f32(2.0 ** -7), dtype=np.float32)
        row[0] = f32(1.0 - (A - 1) * 2.0 ** -7)  # dyadic: every partial sum is exact
        for gw in (8, 32):
            assert np.array_equal(masked_priors(row, legal, gw), row)
            assert np.array_equal(masked_priors(2 * row, legal, gw), row)
    rng = np.random.default_rng(1)
    row = rng.random(25).astype(np.float32)
    legal = np.ones(25, dtype=bool)
    part = legal_part(row, legal, 32)
    assert np.array_equal(masked_priors(row, legal, 32), (row.astype(np.float64) / np.float64(part)).astype(np.float32))


def test_masked_priors_zero_legal_mass_keeps_the_raw_zeros():
    """No mass on any legal move: part = 0, no division, the legal priors stay at their raw 0 and the illegal ones are
    zeroed (no NaN from 0 / 0)."""
    row = np.array([0.0, 0.5, 0.0, 0.25, 0.0, 0.25, 0.0], dtype=np.float32)
    legal = row == 0
    for gw in (8, 32):
        out = masked_priors(row, legal, gw)
        assert np.isfinite(out).all() and not out.any()


@pytest.mark.parametrize("A", [7, 81])
def test_masked_priors_single_legal_move_is_exactly_one(A):
    """One legal move: its prior is exactly 1.0, whatever the network gave it, including values p for which
    p * f32(1 / p) rounds to 0.99999994."""
    rng = np.random.default_rng(7)
    values = list(rng.random(200).astype(np.float32)) + [f32(0.543625), f32(0.9350724), f32(3e-8), f32(1.0)]
    for p in values:
        for a in (0, A - 1, A // 2):
            row = np.full(A, f32(0.1), dtype=np.float32)
            row[a] = p
            legal = np.arange(A) == a
            for gw in ((8, 32) if A <= 8 else (32,)):
                out = masked_priors(row, legal, gw)
                assert out[a] == f32(1.0) and out.sum() == f32(1.0), (p, a, gw, out[a])


def test_masked_priors_lane_groups():
    """Eight and 32 lanes give the same bits while A <= 8 (one action per lane either way; the wider butterfly only adds
    zeros), and different bits on a row over more than 32 actions: lane 0 of eight lanes adds p[0], p[8], .., p[32]
    into 1.0 one tiny term at a time (each rounds away), while 32 lanes pair the tiny terms up before they meet 1.0."""
    rng = np.random.default_rng(3)
    for A in range(1, 9):
        for row in _rows(A, rng, 10):
            for mask in range(1, 1 << A):
                legal = np.array([(mask >> a) & 1 for a in range(A)], dtype=bool)
                assert np.array_equal(masked_priors(row, legal, 8).view(np.uint32),
                                      masked_priors(row, legal, 32).view(np.uint32))
    row = np.zeros(33, dtype=np.float32)
    row[0] = f32(1.0)
    row[[8, 16, 24, 32]] = f32(2.0 ** -24)
    legal = np.ones(33, dtype=bool)
    out8, out32 = masked_priors(row, legal, 8), masked_priors(row, legal, 32)
    assert out8[0] == f32(1.0)  # part = 1.0
    assert out32[0] == f32(1.0) / f32(1.0 + 2.0 ** -23)  # part = 1 + 2^-23
    assert not np.array_equal(out8, out32)


# ------------------------------------------------------------------------------------------------ FRESH / RECYCLE_TREE
class _Tree:
    def __init__(self, n):
        self.n, self.cleared = n, False

    def __len__(self):
        return self.n

    def clear(self):
        self.n, self.cleared = 0, True


def test_clear_after_move_by_hand():
    R, F = FLAG_RECYCLE_TREE, FLAG_FRESH_TREE
    assert clear_after_move([_Tree(12)], R, 24) == [False]           # exactly node_cap / 2: kept
    assert clear_after_move([_Tree(13)], R, 24) == [True]            # node_cap / 2 + 1: cleared
    assert clear_after_move([_Tree(12)], R, 25) == [False]           # odd capacity: 25 / 2 = 12 in C
    assert clear_after_move([_Tree(13)], R, 25) == [True]
    assert clear_after_move([_Tree(0)], R, 1) == [False] and clear_after_move([_Tree(1)], R, 1) == [True]
    two = [_Tree(13), _Tree(12)]
    assert clear_after_move(two, R, 24) == [True, False] and [len(t) for t in two] == [0, 12]  # each tree on its own
    assert clear_after_move([_Tree(0), _Tree(30)], F, 24) == [True, True]  # fresh: every tree, the empty one too
    assert clear_after_move([_Tree(3)], F | R, 24) == [True]
    assert clear_after_move([_Tree(500)], FLAG_MASK_PRIORS, 24) == [False]  # neither tree flag: the tree is kept


def test_recycle_cases_clear_keep_and_revisit():
    """The recycle cases use host noise, so this oracle run IS what the engine must reproduce: trees are kept and
    cleared, one keeps exactly node_cap / 2 nodes (where `>=` would clear it), a game clears one of its two trees and
    keeps the other, searches after a clear look up positions the cleared tree held, and no tree outgrows its arena."""
    total = dict(kept=0, cleared=0, at_half=0, one_of_two=0, revisits=0)
    for case in RECYCLE_CASES:
        games = oracle_run(case)
        assert games.largest <= case.capacity, (case.name, games.largest)
        assert games.events["kept"] and games.events["cleared"] and games.events["revisits"], (case.name, games.events)
        for k, v in games.events.items():
            total[k] += v
    assert all(total.values()), total
    assert any(c.capacity % 2 for c in RECYCLE_CASES) and any(c.trees_per_game == 2 for c in RECYCLE_CASES)


def test_fresh_and_mask_cases_in_the_oracle():
    """Fresh cases: one move's searches fit the arena they are given (the kept tree would not), every advance of a game
    that goes on clears, and the next search revisits positions.  Mask cases: created nodes had illegal mass to drop."""
    for case in FRESH_CASES:
        assert case.count * case.batch <= case.capacity < case.count * case.batch * case.moves, case.name
        if case.noise == "host":
            games = oracle_run(case)
            assert not games.events["kept"] and games.events["cleared"] and games.events["revisits"], case.name
    for case in MASK_CASES + MASK_VL_CASES:
        if case.noise == "host":
            assert oracle_run(case).masked_nodes() > 0, case.name


# ------------------------------------------------------------------------------------------------ dispatch
SELECT_C4 = "select_thread_kernel<C4Rules,2>"
VL_MNK, VL_C4 = "select_vl_kernel<MnkRules>", "select_vl_group_kernel<C4Rules>"


def _eb(R, w):
    return "expand_backup_kernel<%s,%d>" % (R, w)


GROUP8 = "expand_backup_group8_kernel<C4Rules>"


def test_flag_cases_map_to_the_engine_dispatch():
    by_name = {c.name: flag_instances(c) for c in FLAG_CASES + [PIPELINE_CASE]}
    assert len(by_name) == len(FLAG_CASES) + 1, "case names must be unique"
    for c in FLAG_CASES:  # launch by launch: the stand-alone dispatch of the search matrix
        assert by_name[c.name]["expand"] == instances(c)["expand"], c.name
    assert by_name["mask_mnk3_3_b8"]["select"] == "select_thread_kernel<MnkRules,4>"
    assert by_name["mask_mnk5_4_b16_tpg2"]["select"] == "select_kernel<MnkRules,32,1>"
    assert by_name["mask_mnk9_5_b32"]["select"] == "select_kernel<MnkRules,32,4>"
    assert by_name["mask_mnk15_5_b8_tpg2"]["select"] == "select_kernel<MnkRules,32,8>"  # A = 225: 8 actions per lane
    assert by_name["mask_caro9_5_b16"]["expand"] == _eb("MnkRules", 16)
    assert by_name["mask_c4_b32"]["expand"] == _eb("C4Rules", 32)
    assert by_name["mask_vl_mnk9_5_b32"]["select"] == VL_MNK and by_name["mask_vl_c4_b8"]["select"] == VL_C4
    assert by_name["recycle_mnk9_5_b1"]["plan"] == "plan_kernel<MnkBoard,8>"
    pipe = by_name[PIPELINE_CASE.name]
    assert pipe["select"] == VL_C4 and pipe["expand"] == GROUP8 and pipe["expand_stepped"] == _eb("C4Rules", 8)
    assert pipe["noise"] == "noise_kernel<8,1>" and pipe["advance"] == "advance_kernel<C4Rules>"


def test_flag_matrix_covers_every_cell():
    cells = {(c.label, flag_instances(c)["select"], flag_instances(c)["expand"]) for c in FLAG_CASES + [PIPELINE_CASE]}
    required = {
        # masked priors: every select width of the plain search on the listed boards, every expand width on both rules
        ("mask", "select_thread_kernel<MnkRules,4>", _eb("MnkRules", 8)),
        ("mask", "select_kernel<MnkRules,32,1>", _eb("MnkRules", 16)),
        ("mask", "select_kernel<MnkRules,32,4>", _eb("MnkRules", 32)),
        ("mask", "select_kernel<MnkRules,32,8>", _eb("MnkRules", 8)),
        ("mask", "select_kernel<MnkRules,32,4>", _eb("MnkRules", 16)),  # Caro 9 x 9
        ("mask", SELECT_C4, _eb("C4Rules", 8)), ("mask", SELECT_C4, _eb("C4Rules", 16)), ("mask", SELECT_C4, _eb("C4Rules", 32)),
        # masked priors under virtual loss: both virtual-loss select kernels at both batch widths, and the pipeline
        ("mask+vl", VL_MNK, _eb("MnkRules", 8)), ("mask+vl", VL_MNK, _eb("MnkRules", 32)),
        ("mask+vl", VL_C4, _eb("C4Rules", 8)), ("mask+vl", VL_C4, _eb("C4Rules", 32)), ("mask+vl", VL_C4, GROUP8),
        # tree clears on m,n,k and Connect4
        ("fresh", "select_thread_kernel<MnkRules,4>", _eb("MnkRules", 8)),
        ("fresh", "select_kernel<MnkRules,32,4>", _eb("MnkRules", 16)),
        ("fresh", SELECT_C4, _eb("C4Rules", 8)), ("fresh", SELECT_C4, _eb("C4Rules", 32)),
        ("recycle", "select_kernel<MnkRules,32,4>", _eb("MnkRules", 8)),
        ("recycle", "select_kernel<MnkRules,32,1>", _eb("MnkRules", 16)),
        ("recycle", SELECT_C4, _eb("C4Rules", 8)),
    }
    assert required <= cells, sorted(required - cells)
    mask = [c for c in MASK_CASES]
    assert {c.batch for c in mask} == {8, 16, 32} and {c.trees_per_game for c in mask} == {1, 2}
    assert {c.noise for c in mask} == {"host", "philox"} and any(c.caro for c in mask)
    assert {c.board for c in mask} == {(3, 3), (5, 4), (9, 5), (15, 5), (0, 0)}
    assert {(c.board, c.batch, c.plies) for c in MASK_VL_CASES} == {(c.board, c.batch, c.plies) for c in VL_CASES}
    assert all(c.mask_priors and c.virtual_loss for c in MASK_VL_CASES)
    assert {c.board for c in FRESH_CASES} == {(3, 3), (9, 5), (0, 0)} and {c.trees_per_game for c in FRESH_CASES} == {1, 2}
    assert all(4 <= c.moves <= 6 for c in FRESH_CASES)
    assert PIPELINE_CASE.parts == 2 and PIPELINE_CASE.batch == 8 and PIPELINE_CASE.moves == 2
    assert PIPELINE_CASE.connect4 and PIPELINE_CASE.virtual_loss and PIPELINE_CASE.mask_priors
