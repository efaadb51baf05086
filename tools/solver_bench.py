"""What does the MCTS solver buy in play strength, and what does it cost in self-play?

  * Strength: the trained Connect4 checkpoint with the solver against itself without it (per-player mask, two trees per
    game), 2 x `--games` games with the colours swapped, at search_batch (10, 8), (40, 8) and (20, 16), tau = 0 like
    play.py.  Score = (wins + draws / 2) / games for the solver side, with a 95 % normal interval.
  * Cost: auto-restart self-play (`play_multi`, one part) with the solver on both sides against off, alternated per round:
    games/s, plies and leaf evaluations per finished game, descents stopped at proven nodes and edges proven (and the same
    per ply, for Caro, where few games end inside the timed window).  Connect4
    with the trained checkpoint and with a random-init net (10 x 8 searches, tau for 10 plies), Caro 15x15 with a
    random-init net (tree compaction).
Prints one JSON line per measurement, each with the card's name and power limit.

    python tools/solver_bench.py [--games 1000] [--rounds 2] [--c4-games 2048] [--caro-games 256] [--plies 60]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CKPT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "checkpoints",
                    "connect4_best_026_12000.dat")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def strength(game, dn, games, searches, batch):
    from caro_ai_b200.utils import play_games_batched
    w = l = d = 0
    for first in (True, False):  # the solver side (player 0) moves first, then second
        s = play_games_batched(game, games, dn, dn, 0, searches, batch, net1_plays_first=first, trees_per_game=2,
                               seed=77 + first, solver=(True, False))
        w, l, d = w + s["wins"], l + s["losses"], d + s["draws"]
    n = w + l + d
    score = (w + 0.5 * d) / n
    var = (w * (1 - score) ** 2 + l * score ** 2 + d * (0.5 - score) ** 2) / n
    half = 1.96 * math.sqrt(var / n)
    return {"wins": w, "losses": l, "draws": d, "score": round(score, 4), "ci95": [round(score - half, 4), round(score + half, 4)]}


def self_play(game, dn, G, plies, solver, compact, seed):
    import torch
    from caro_ai_b200 import config as cfg
    from caro_ai_b200.engine import SelfPlayEngine
    plies_max = 42 if game.game_kind == 0 else game.action_space
    cap = 4000 if compact else cfg.MCTS_SEARCHES * cfg.MCTS_BATCH_SIZE * plies_max + 8
    eng = SelfPlayEngine(game, G, trees_per_game=1, max_batch=cfg.MCTS_BATCH_SIZE, node_capacity=cap, seed=seed,
                         compact_tree=compact)
    if solver:
        eng.set_solver(3)
    eng.reset(first_player=-1)
    run = lambda n: SelfPlayEngine.play_multi([eng], dn, moves=n, count=cfg.MCTS_SEARCHES, batch=cfg.MCTS_BATCH_SIZE,
                                              tau_plies=cfg.STEPS_BEFORE_TAU_0, auto_restart=True)
    run(4)  # warm-up: graph capture
    torch.cuda.synchronize()
    c0, s0 = eng.counters(), eng.solver_counters()
    t = time.time()
    run(plies)
    torch.cuda.synchronize()
    dt = time.time() - t
    c1, s1 = eng.counters(), eng.solver_counters()
    assert c1["errors"] == 0
    eng.close()
    games = c1["games"] - c0["games"]
    return {"games_per_s": round(games / dt, 1), "plies_per_game": round((c1["plies"] - c0["plies"]) / max(1, games), 3),
            "leaf_evals_per_game": round((c1["leaf_evals"] - c0["leaf_evals"]) / max(1, games), 2),
            "stopped_per_game": round((s1["stopped"] - s0["stopped"]) / max(1, games), 2),
            "proven_per_game": round((s1["proven"] - s0["proven"]) / max(1, games), 2), "games": games, "seconds": round(dt, 3),
            "plies_per_s": round((c1["plies"] - c0["plies"]) / dt, 1),
            "leaf_evals_per_ply": round((c1["leaf_evals"] - c0["leaf_evals"]) / max(1, c1["plies"] - c0["plies"]), 3),
            "stopped_per_ply": round((s1["stopped"] - s0["stopped"]) / max(1, c1["plies"] - c0["plies"]), 3)}


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
        for searches, batch in ((10, 8), (40, 8), (20, 16)):
            r = strength(c4, trained, args.games, searches, batch)
            print(json.dumps({"kind": "strength", "game": "connect4", "net": "connect4_best_026", "searches": searches,
                              "batch": batch, **r, "card": who}), flush=True)
    workloads = [("connect4", "connect4_best_026", c4, trained, args.c4_games, False),
                 ("connect4", "random_init", c4, rand_c4, args.c4_games, False)]
    if args.caro_games:
        caro = Caro()
        torch.manual_seed(0)
        workloads.append(("caro15", "random_init", caro, DeviceNet(Net(caro.obs_shape, caro.action_space).eval(), caro),
                          args.caro_games, True))
    for name, net, game, dn, G, compact in workloads:
        for rnd in range(args.rounds):
            for solver in (False, True):
                r = self_play(game, dn, G, args.plies, solver, compact, seed=100 + rnd)
                print(json.dumps({"kind": "cost", "game": name, "net": net, "solver": solver, "round": rnd, "G": G, **r,
                                  "card": who}), flush=True)


if __name__ == "__main__":
    main()
