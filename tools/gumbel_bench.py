"""What does the Gumbel root search buy in play strength, and what does it cost in self-play?

  * Strength: the trained Connect4 checkpoint with Gumbel at its roots against itself without it (per-player mask, two
    trees per game), 2 x `--games` games with the colours swapped, at equal budgets search_batch (2, 8), (4, 8), (10, 8),
    (40, 8), gumbel_scale 1 and 0, the paper's m = 16, c_visit = 50, c_scale = 0.1; tau = 0 like play.py for the plain side.
    Score = (wins + draws / 2) / games for the Gumbel side, with a 95 % normal interval.
  * Cost: auto-restart self-play (`play_multi`, one part), Gumbel on both sides against off, alternated per round:
    games/s, plies/s, descents and leaf evaluations per ply (their ratio is what the duplicate drop leaves), and the time
    of gumbel_plan_kernel per minibatch (CUDA events around 200 launches on the engine as self-play left it).  Connect4
    with the trained checkpoint and a random-init net (10 x 8 searches, tau for 10 plies), Caro 15x15 random-init
    (compaction on).
Prints one JSON line per measurement, each with the card's name and power limit.

    python tools/gumbel_bench.py [--games 1000] [--rounds 2] [--c4-games 2048] [--caro-games 256] [--plies 60]
"""
import argparse
import json
import math
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from solver_bench import CKPT, card  # noqa: E402


def strength(game, dn, games, searches, batch, scale):
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.utils import run_to_completion
    w = l = d = 0
    for first in (0, 1):  # the Gumbel side (player 0) moves first, then second
        eng = SelfPlayEngine(game, games, trees_per_game=2, max_batch=batch, node_capacity=searches * batch * 42 + 8,
                             seed=77 + first)
        eng.set_gumbel(1, m=16, c_visit=50.0, c_scale=0.1, scale=scale)
        eng.reset(first_player=first)
        run_to_completion(eng, dn, dn, 0, searches, batch, first)
        c = eng.counters()
        assert c["errors"] == 0
        w, l, d = w + c["wins_p0"], l + c["wins_p1"], d + c["draws"]
        eng.close()
    n = w + l + d
    score = (w + 0.5 * d) / n
    var = (w * (1 - score) ** 2 + l * score ** 2 + d * (0.5 - score) ** 2) / n
    half = 1.96 * math.sqrt(var / n)
    return {"wins": w, "losses": l, "draws": d, "score": round(score, 4), "ci95": [round(score - half, 4), round(score + half, 4)]}


def plan_kernel_ms(eng, count, batch, launches=200):
    import torch
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(launches):
        eng.gumbel_plan(0, i % count, count, batch)
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / launches


def self_play(game, dn, G, plies, gumbel, compact, seed):
    import torch
    from caro_ai_b200 import config as cfg
    from caro_ai_b200.engine import SelfPlayEngine
    plies_max = 42 if game.game_kind == 0 else game.action_space
    cap = 4000 if compact else cfg.MCTS_SEARCHES * cfg.MCTS_BATCH_SIZE * plies_max + 8
    eng = SelfPlayEngine(game, G, trees_per_game=1, max_batch=cfg.MCTS_BATCH_SIZE, node_capacity=cap, seed=seed,
                         compact_tree=compact)
    if gumbel:
        eng.set_gumbel(3)
    eng.reset(first_player=-1)
    run = lambda n: SelfPlayEngine.play_multi([eng], dn, moves=n, count=cfg.MCTS_SEARCHES, batch=cfg.MCTS_BATCH_SIZE,
                                              tau_plies=cfg.STEPS_BEFORE_TAU_0, auto_restart=True)
    run(4)  # warm-up: graph capture
    torch.cuda.synchronize()
    c0 = eng.counters()
    t = time.time()
    run(plies)
    torch.cuda.synchronize()
    dt = time.time() - t
    c1 = eng.counters()
    assert c1["errors"] == 0
    plan_ms = plan_kernel_ms(eng, cfg.MCTS_SEARCHES, cfg.MCTS_BATCH_SIZE) if gumbel else 0.0
    eng.close()
    games, np_ = c1["games"] - c0["games"], max(1, c1["plies"] - c0["plies"])
    return {"games_per_s": round(games / dt, 1), "plies_per_s": round((c1["plies"] - c0["plies"]) / dt, 1),
            "descents_per_ply": round((c1["descents"] - c0["descents"]) / np_, 2),
            "leaf_evals_per_ply": round((c1["leaf_evals"] - c0["leaf_evals"]) / np_, 3),
            "plies_per_game": round((c1["plies"] - c0["plies"]) / max(1, games), 3), "games": games, "seconds": round(dt, 3),
            "gumbel_plan_ms_per_minibatch": round(plan_ms, 4)}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=1000, help="strength games per colour and setting (0 = skip)")
    ap.add_argument("--rounds", type=int, default=2, help="alternated off / on rounds of the cost measurement")
    ap.add_argument("--c4-games", type=int, default=2048)
    ap.add_argument("--caro-games", type=int, default=256, help="0 = skip")
    ap.add_argument("--plies", type=int, default=60, help="timed auto-restart plies per arm and round")
    args = ap.parse_args(argv)
    import torch
    from caro_ai_b200.game import Caro, ConnectFour
    from caro_ai_b200.model import DeviceNet, Net, load_checkpoint
    who = card()
    c4 = ConnectFour()
    trained = DeviceNet(load_checkpoint(CKPT, c4).eval(), c4)
    torch.manual_seed(0)
    rand_c4 = DeviceNet(Net(c4.obs_shape, c4.action_space).eval(), c4)
    if args.games:
        for scale in (1.0, 0.0):
            for searches, batch in ((2, 8), (4, 8), (10, 8), (40, 8)):
                r = strength(c4, trained, args.games, searches, batch, scale)
                print(json.dumps({"kind": "strength", "game": "connect4", "net": "connect4_best_026", "searches": searches,
                                  "batch": batch, "gumbel_scale": scale, "m": 16, "c_visit": 50.0, "c_scale": 0.1, **r,
                                  "card": who}), flush=True)
    workloads = [("connect4", "connect4_best_026", c4, trained, args.c4_games, False),
                 ("connect4", "random_init", c4, rand_c4, args.c4_games, False)]
    if args.caro_games:
        caro = Caro()
        torch.manual_seed(0)
        workloads.append(("caro15", "random_init", caro, DeviceNet(Net(caro.obs_shape, caro.action_space).eval(), caro),
                          args.caro_games, True))
    for name, net, game, dn, G, compact in workloads:
        for rnd in range(args.rounds):
            for gumbel in (False, True):
                r = self_play(game, dn, G, args.plies, gumbel, compact, seed=100 + rnd)
                print(json.dumps({"kind": "cost", "game": name, "net": net, "gumbel": gumbel, "round": rnd, "G": G, **r,
                                  "card": who}), flush=True)


if __name__ == "__main__":
    main()
