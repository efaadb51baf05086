"""Resignation on the B200 (run with -m gpu): off is the parent bit for bit, the kernel applies the rule exactly as the host
restates it (tests/resign_reference.py), playthrough games are the Philox draw and log what they saw, parameters reach a
captured ply graph on the next ply, and the worker / train.py calibrate end to end."""
import os
import random

import numpy as np
import pytest

from conftest import GOLDEN
from resign_reference import is_playthrough, root_stat

pytestmark = pytest.mark.gpu

# (game, trees per game, tree compaction)
CASES = [("c4", 1, False), ("c4", 2, True), ("ttt", 1, True), ("ttt", 2, False), ("caro9", 1, True), ("caro9", 2, False)]
SEED = 0x1234567890AB


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


_NETS = {}


def _game_net(torch, name):
    from caro_ai_b200.game import Caro, ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    if name not in _NETS:
        game = {"c4": ConnectFour, "ttt": lambda: TicTacToe(3, 3), "caro9": lambda: Caro(9, 5)}[name]()
        torch.manual_seed(11)
        _NETS[name] = (game, DeviceNet(Net(game.obs_shape, game.action_space).eval(), game))
    return _NETS[name]


def _engine(game, G, tpg, compact, seed=SEED):
    from caro_ai_b200.engine import SelfPlayEngine
    plies = 42 if game.game_kind == 0 else game.action_space
    # a ply writes at most one replay row per game: the ring never wraps within the 32 plies a test plays at most
    return SelfPlayEngine(game, G, trees_per_game=tpg, max_batch=8, node_capacity=2048 if compact else 24 * plies + 64,
                          replay_capacity=G * max(plies, 32), seed=seed, compact_tree=compact)


def _replay_rows(eng):
    n = eng.replay_cursor()
    assert n <= eng.cfg.replay_capacity
    bd = eng.region("replay_board")[:n].cpu().numpy()
    pl = eng.region("replay_player")[:n].cpu().numpy()
    pi = eng.fregion("replay_pi")[:n].cpu().numpy()
    z = eng.fregion("replay_z")[:n].cpu().numpy()
    return bd, pl, pi, z


def _snapshot(eng):
    bd, pl, pi, z = _replay_rows(eng)
    rows = sorted((tuple(bd[i].tolist()), int(pl[i]), pi[i].tobytes(), float(z[i])) for i in range(len(z)))
    p, q, n = eng.root_policy(1, 0)
    out = {name: eng.region(name).cpu().numpy().copy() for name in ("root_board", "root_player", "status", "ply", "result", "uid")}
    out.update(counters=eng.counters(), replay=rows, pi=p.cpu().numpy(), q=q.cpu().numpy(), n=n.cpu().numpy())
    return out


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], np.ndarray):  # bit for bit (a root without visits has a NaN policy in both)
            assert a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes(), k
        else:
            assert a[k] == b[k], k


def _segments(eng):
    """Replay rows split into games (every game starts from the empty board): (boards, players, z) per game."""
    bd, pl, _, z = _replay_rows(eng)
    starts = [i for i in range(len(z)) if not bd[i].any()] + [len(z)]
    return [(bd[a:b], pl[a:b], z[a:b]) for a, b in zip(starts, starts[1:])]


def _alternating(z):
    last = z[-1]
    return all(z[len(z) - 1 - i] == (last if i % 2 == 0 else -last) for i in range(len(z)))


def _root_rows(torch, eng):
    """N (masked) and W of every game's root node in the mover's tree, as numpy [G, A] (None rows: root not found)."""
    G, tpg, cap, A = eng.G, eng.cfg.trees_per_game, eng.cfg.node_capacity, eng.A
    rb = eng.region("root_board")
    rp = eng.region("root_player").long()
    tree = torch.arange(G, device=rb.device) * tpg + (rp if tpg == 2 else 0)
    nb = eng.region("node_board").view(G * tpg, cap, -1)[tree]
    cnt = eng.region("node_count")[tree].long()
    hit = (nb == rb[:, None, :]).all(-1) & (torch.arange(cap, device=rb.device)[None, :] < cnt[:, None])
    found = hit.any(-1).cpu().numpy()
    idx = tree * cap + hit.int().argmax(-1)
    rec = eng.region("nodes")[idx]
    n = (rec[:, 0, :A] & 0x7FFFFFFF).cpu().numpy()
    w = rec[:, 1, :A].contiguous().view(torch.float32).cpu().numpy()
    return [(n[g], w[g]) if found[g] else None for g in range(G)]


# ------------------------------------------------------------------------------------------- 1. off is the parent
@pytest.mark.parametrize("name,tpg,compact", CASES)
def test_resign_off_and_never_firing_are_the_parent(torch_cuda, name, tpg, compact):
    torch = torch_cuda
    game, dn = _game_net(torch, name)
    G = 48
    # advance, ply by ply, with the actions
    engs = [_engine(game, G, tpg, compact) for _ in range(2)]
    engs[1].set_resign(-1.0, 0.0)
    for e in engs:
        e.reset(first_player=-1)
    acts = [[], []]
    for ply in range(10):
        for i, e in enumerate(engs):
            e.search(dn, 3, 8)
            acts[i].append(e.advance(4, auto_restart=True).cpu().numpy())
    assert all(np.array_equal(x, y) for x, y in zip(*acts))
    _assert_same(_snapshot(engs[0]), _snapshot(engs[1]))
    # play(), to the end of most games and past it with auto-restart
    for e in engs:
        e.play(dn, dn, moves=12, count=3, batch=8, tau_plies=4, auto_restart=True)
    _assert_same(_snapshot(engs[0]), _snapshot(engs[1]))
    assert engs[1].resign_counters() == {"resigned": 0, "logged": 0}
    for e in engs:
        e.close()
    # play_multi (the captured ply graph), two parts per arm
    arms = []
    for arm in range(2):
        parts = [_engine(game, G // 2, tpg, compact, seed=SEED + 7 * h) for h in range(2)]
        if arm:
            for e in parts:
                e.set_resign(-1.0, 0.0)
        for e in parts:
            e.reset(first_player=-1)
        from caro_ai_b200.engine import SelfPlayEngine
        SelfPlayEngine.play_multi(parts, dn, moves=14, count=3, batch=8, tau_plies=4, auto_restart=True)
        arms.append(parts)
    for a, b in zip(*arms):
        _assert_same(_snapshot(a), _snapshot(b))
        assert b.resign_counters()["resigned"] == 0
    for e in arms[0] + arms[1]:
        e.close()


# ------------------------------------------------------------------------------------------- 2. the rule, 3. playthrough
@pytest.mark.parametrize("name,tpg,compact", CASES)
def test_rule_and_playthrough_log_match_the_host(torch_cuda, name, tpg, compact):
    """Ply by ply: the host reads the mover's root row, computes stat, and predicts which games resign; on plies 1 and 3 the
    threshold is the median of that ply's statistics of the games that may resign, so both outcomes occur by construction.
    A quarter of the games are playthrough games: the host keeps their minima and checks the log records."""
    torch = torch_cuda
    game, dn = _game_net(torch, name)
    G, share = 64, 0.25
    eng = _engine(game, G, tpg, compact)
    eng.set_resign(-1.0, share)
    eng.reset(first_player=-1)
    uid = eng.region("uid").cpu().numpy().astype(np.uint64)
    play = np.array([is_playthrough(int(u), SEED, share) for u in uid])
    assert np.array_equal(eng.region("resign_playthrough").cpu().numpy() == 1, play)
    assert 0 < play.sum() < G
    mins = np.full((G, 2), np.inf)
    finished_pt, resigned_total, games_total = [], 0, 0
    max_plies = 42 if game.game_kind == 0 else game.action_space
    for ply in range(max_plies):
        active = eng.region("status").cpu().numpy() == 0
        if not active.any():
            break
        eng.search(dn, 3, 8)
        rows = _root_rows(torch, eng)
        who = eng.region("root_player").cpu().numpy().astype(int)
        plies_before = eng.region("ply").cpu().numpy().copy()
        stat = [root_stat(*r) if (r is not None and active[g]) else None for g, r in enumerate(rows)]
        eligible = [stat[g] for g in range(G) if active[g] and not play[g] and stat[g] is not None]
        t = float(np.median(eligible)) if ply in (1, 3) and eligible else -1.0
        eng.set_resign(t, share)
        want = np.array([active[g] and not play[g] and stat[g] is not None and stat[g] < t for g in range(G)])
        if ply in (1, 3) and eligible:
            assert want.any() and (active & ~play & ~want).any()
        for g in range(G):
            if active[g] and play[g] and stat[g] is not None:
                mins[g, who[g]] = min(mins[g, who[g]], stat[g])
        before = eng.counters()
        rc0 = eng.resign_counters()
        act = eng.advance(4, auto_restart=False).cpu().numpy()
        after = eng.counters()
        status = eng.region("status").cpu().numpy()
        result = eng.region("result").cpu().numpy()
        assert np.array_equal(act == -1, want | ~active)
        assert after["plies"] - before["plies"] == int(active.sum())
        assert eng.resign_counters()["resigned"] - rc0["resigned"] == int(want.sum())
        for g in np.nonzero(want)[0]:
            assert status[g] == 1 and result[g] == (-1 if who[g] == 0 else 1)
        ended = active & (status == 1)
        games_total += int(ended.sum())
        resigned_total += int(want.sum())
        for g in np.nonzero(ended & play)[0]:
            finished_pt.append((mins[g, 0], mins[g, 1], int(result[g]), int(plies_before[g]) + 1))
        assert after["games"] - before["games"] == int(ended.sum())
        wins0 = int((ended & (result == 1)).sum())
        assert after["wins_p0"] - before["wins_p0"] == wins0
    assert resigned_total > 0 and games_total == G
    assert eng.counters()["errors"] == 0
    # the log: one record per finished playthrough game, with the host's minima, result and plies
    recs, cursor = eng.resign_log()
    assert cursor == len(finished_pt) == int(play.sum())
    got = sorted((float(r["min_stat"][0]), float(r["min_stat"][1]), int(r["result"]), int(r["plies"])) for r in recs)
    assert got == sorted(finished_pt)
    # replay rows: every game is one segment with alternating z; resigned games end in z = -1 on the resigner's position
    segs = _segments(eng)
    assert len(segs) == G and all(_alternating(z) for _, _, z in segs)
    assert sum(1 for _, _, z in segs if z[-1] == -1) == resigned_total
    eng.close()


def test_playthrough_draw_and_full_logging(torch_cuda):
    torch = torch_cuda
    game, dn = _game_net(torch, "ttt")
    eng = _engine(game, 256, 1, False)
    eng.set_resign(0.5, 0.5)
    eng.reset(first_player=-1)
    uid = eng.region("uid").cpu().numpy().astype(np.uint64)
    want = [is_playthrough(int(u), SEED, 0.5) for u in uid]
    assert (eng.region("resign_playthrough").cpu().numpy() == 1).tolist() == want
    assert 64 < sum(want) < 192
    # playthrough 1.0 logs every game, and at the largest threshold none of them resigns
    eng.set_resign(1.0, 1.0)
    eng.reset(first_player=-1)
    assert bool((eng.region("resign_playthrough") == 1).all())
    mins = eng.region("resign_min").view(torch.float64)
    assert bool(torch.isinf(mins).all())
    eng.play(dn, dn, moves=9, count=3, batch=8, tau_plies=4, auto_restart=False)
    assert bool((eng.region("status") == 1).all())
    rc = eng.resign_counters()
    assert rc == {"resigned": 0, "logged": 256} and eng.counters()["games"] == 256
    recs, _ = eng.resign_log()
    assert len(recs) == 256 and (recs["plies"] >= 5).all() and np.isfinite(recs["min_stat"]).any(axis=1).all()
    eng.close()


# ------------------------------------------------------------------------------------------- 4. parameters reach the graph
def test_play_multi_threshold_change_takes_effect_and_restart_reseats(torch_cuda):
    """The parameters live in device memory, so the captured ply graph of play_multi sees every change on its next replay;
    auto-restart clears a re-seated slot's minima and draws its playthrough flag anew."""
    torch = torch_cuda
    from caro_ai_b200.engine import SelfPlayEngine
    game, dn = _game_net(torch, "ttt")
    seeds = [SEED + h for h in range(2)]
    parts = [_engine(game, 64, 1, True, seed=s) for s in seeds]

    def ply():
        SelfPlayEngine.play_multi(parts, dn, moves=1, count=3, batch=8, tau_plies=4, auto_restart=True)

    # log only, every game played through: slots re-seated by a ply start over at +inf, running games have both minima
    for e in parts:
        e.set_resign(-1.0, 1.0)
        e.reset(first_player=-1)
    restarts = 0
    for _ in range(9):
        ply()
        for e in parts:
            plies = e.region("ply").cpu().numpy()
            m = e.region("resign_min").view(torch.float64).cpu().numpy()
            assert np.isinf(m[plies == 0]).all() and np.isfinite(m[plies >= 2]).all()
            assert (e.region("resign_playthrough").cpu().numpy() == 1).all()
            restarts += int((plies == 0).sum())
    assert restarts > 0
    assert all(e.resign_counters()["resigned"] == 0 for e in parts)
    assert all(e.resign_counters()["logged"] == e.counters()["games"] > 0 for e in parts)
    # threshold 1.0 and no playthrough, set between two replays of the same graph: the next ply resigns (nearly) every game
    for e in parts:
        e.set_resign(1.0, 0.0)
        e.reset(first_player=-1)
    played0 = [e.region("played").cpu().numpy().copy() for e in parts]
    ply()
    for e, p0, seed in zip(parts, played0, seeds):
        rs = e.resign_counters()["resigned"]
        assert rs >= 0.9 * e.G, rs
        again = e.region("played").cpu().numpy() != p0
        assert int(again.sum()) == rs  # a game cannot end otherwise on its first ply
        assert bool((e.region("status") == 0).all())
        assert (e.region("ply").cpu().numpy()[again] == 0).all()
        assert (e.region("root_board").cpu().numpy()[again] == 0).all()
        assert (e.region("resign_playthrough").cpu().numpy() == 0).all()
    # never firing again: nothing resigns on the next plies
    for e in parts:
        e.set_resign(-1.0, 0.0)
    before = [e.resign_counters()["resigned"] for e in parts]
    for _ in range(2):
        ply()
    assert [e.resign_counters()["resigned"] for e in parts] == before
    for e in parts:
        e.close()


# ------------------------------------------------------------------------------------------- 5. worker and train.py
def test_worker_calibrates_and_trained_net_resigns_at_the_logged_threshold(torch_cuda):
    torch = torch_cuda
    from caro_ai_b200 import config as cfg
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.model import DeviceNet, load_checkpoint
    from caro_ai_b200.utils import SelfPlayWorker, choose_resign_threshold, resign_tallies
    game = ConnectFour()
    dn = DeviceNet(load_checkpoint(os.path.join(GOLDEN, "checkpoints", "connect4_best_026_12000.dat"), game).eval(), game)
    G = 256
    args = (game, G, cfg.MCTS_SEARCHES, cfg.MCTS_BATCH_SIZE, cfg.STEPS_BEFORE_TAU_0)
    # "auto": the first step logs every game and resigns none
    w = SelfPlayWorker(*args, replay_steps=1, min_replay=100, seed=21, resign="auto", resign_playthrough=0.1)
    s1 = w.play_step(dn)
    r1 = w.resign_stats()
    assert r1["logged"] == G == s1["games"] and r1["resigned"] == 0 and r1["window"] == G
    s2 = w.play_step(dn)
    r2 = w.resign_stats()
    assert s2["games"] == G and r2["resigned"] + r2["logged"] <= G
    if r1["threshold"] is None:
        assert r2["resigned"] == 0 and r2["logged"] == G
    w.close()
    # a log-only run of seeded games gives the threshold; the same games with that threshold and no playthrough resign
    # exactly where the log says a player's statistic first fell below it
    log_only = SelfPlayWorker(*args, replay_steps=1, min_replay=100, seed=33, resign=-1.0, resign_playthrough=1.0)
    log_only.play_step(dn)
    recs, _ = log_only.engine.resign_log()
    assert len(recs) == G
    t = choose_resign_threshold(resign_tallies(recs), min_records=G)
    assert t is not None
    predicted = int((recs["min_stat"].min(axis=1) < t).sum())
    log_only.close()
    w2 = SelfPlayWorker(*args, replay_steps=1, min_replay=100, seed=33, resign=t, resign_playthrough=0.0)
    s = w2.play_step(dn)
    rs = w2.resign_stats()
    assert rs["resigned"] == predicted >= 1 and rs["logged"] == 0 and s["games"] == G
    segs = _segments(w2.engine)
    assert len(segs) == G and all(_alternating(z) for _, _, z in segs)
    assert sum(1 for _, _, z in segs if z[-1] == -1) == predicted
    w2.close()
    dn.close()


def test_train_main_with_auto_resignation(torch_cuda, tmp_path, capsys):
    torch = torch_cuda
    from caro_ai_b200 import train as train_cli
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        random.seed(0)
        torch.manual_seed(0)
        assert train_cli.main(["-g", "1", "-n", "rs", "--games", "512", "--max-steps", "2", "--evaluate-every", "100",
                               "--resign", "auto"]) == 0
    finally:
        os.chdir(cwd)
    out = capsys.readouterr().out
    assert "Step 2, steps" in out and ", resign " in out
