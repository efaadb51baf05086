"""Caro against freestyle 15x15/5 self-play at bench.py's Caro workload: does the both-ends-blocked rule cost anything?

Both arms run 2 pipeline parts x 1,024 games, search_batch(200, 8), tree compaction and the reference-shape 5 x 64
random-init network with precision "auto" -- the only difference is the game id (CARO_GAME_CARO vs CARO_GAME_MNK).
The arms alternate A/B/A/B in one process.  Two numbers per arm:
  * leaf evaluations / s over --plies timed plies (CUDA events, after one warm-up ply), the rate bench.py reports;
  * games / s and plies per game when every game is played to its end at search_batch(--game-count, 8) (a Caro game
    can run longer than a freestyle one, which changes games / s but not the per-ply rate).
Prints one JSON line with the card's name and power limit.

    python tools/caro_rule_bench.py [--plies 20] [--rounds 2] [--game-count 25]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--plies", type=int, default=20, help="timed plies per arm and round")
    ap.add_argument("--rounds", type=int, default=2, help="A/B rounds")
    ap.add_argument("--games-per-part", type=int, default=1024)
    ap.add_argument("--game-count", type=int, default=25, help="search_batch count of the to-the-end games/s run (0 = skip)")
    args = ap.parse_args(argv)
    import torch
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import Caro, TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    arms = {"caro": Caro(15, 5), "freestyle": TicTacToe(15, 5)}
    parts, G, count, batch, tau = 2, args.games_per_part, 200, 8, 10

    def make(game, seed):
        torch.manual_seed(0)
        dn = DeviceNet(Net(game.obs_shape, game.action_space).eval(), game, precision="auto")
        engs = [SelfPlayEngine(game, G, max_batch=batch, node_capacity=8192, seed=seed + 7 * h, compact_tree=True)
                for h in range(parts)]
        return dn, engs

    def close(dn, engs):
        for e in engs:
            e.close()
        dn.close()
        torch.cuda.empty_cache()

    def rate(game):
        dn, engs = make(game, 11)
        SelfPlayEngine.play_multi(engs, dn, moves=1, count=count, batch=batch, tau_plies=tau, auto_restart=True)
        torch.cuda.synchronize()
        c0 = [e.counters() for e in engs]
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        SelfPlayEngine.play_multi(engs, dn, moves=args.plies, count=count, batch=batch, tau_plies=tau, auto_restart=True)
        stop.record()
        torch.cuda.synchronize()
        sec = start.elapsed_time(stop) / 1e3
        c1 = [e.counters() for e in engs]
        d = {k: sum(b[k] - a[k] for a, b in zip(c0, c1)) for k in c1[0]}
        out = {"leaf_evals_per_sec": d["leaf_evals"] / sec, "ms_per_ply": 1e3 * sec / args.plies, "errors": d["errors"],
               "precision": dn.precision}
        close(dn, engs)
        return out

    def to_the_end(game):
        dn, engs = make(game, 23)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(0, game.action_space, 8):
            SelfPlayEngine.play_multi(engs, dn, moves=8, count=args.game_count, batch=batch, tau_plies=tau, auto_restart=False)
            if all(int((e.region("status") == 0).sum().item()) == 0 for e in engs):
                break
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        c = [e.counters() for e in engs]
        games, plies = sum(x["games"] for x in c), sum(x["plies"] for x in c)
        draws = sum(x["draws"] for x in c)
        close(dn, engs)
        return {"games": games, "games_per_sec": games / sec, "plies_per_game": plies / max(1, games), "draws": draws}

    runs = {k: [] for k in arms}
    for _ in range(args.rounds):
        for name, game in arms.items():
            runs[name].append(rate(game))
    ends = {name: to_the_end(game) for name, game in arms.items()} if args.game_count > 0 else {}
    summary = {}
    for name in arms:
        r = [x["leaf_evals_per_sec"] for x in runs[name]]
        summary[name] = {"leaf_evals_per_sec": r, "mean": sum(r) / len(r), "spread": max(r) - min(r),
                         "ms_per_ply": [x["ms_per_ply"] for x in runs[name]], "precision": runs[name][0]["precision"],
                         "errors": sum(x["errors"] for x in runs[name])}
        if name in ends:
            summary[name]["to_the_end"] = ends[name]
    print(json.dumps({"workload": "15x15/5 self-play, %d parts x %d games, search_batch(%d,%d), compact tree, 5x64 random-init "
                                  "net; %d timed plies per arm, A/B x %d" % (parts, G, count, batch, args.plies, args.rounds),
                      "gpu": card(), "arms": summary}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
