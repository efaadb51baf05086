"""What does resignation buy in self-play, and what does it cost when it does not fire?

Three arms, alternated in one process (A/B/C per round):
  * off        -- every game to its end (the reference's behaviour);
  * log-only   -- threshold -1.0 (never fires), every game played through and logged: the statistic's cost;
  * calibrated -- the threshold `choose_resign_threshold` picks from the first log-only run, 10 % playthrough.
Per arm: games/s, mean plies per game, leaf evaluations per finished game, resigned share, and the false-positive rate of
the arm's logged playthrough games at the calibrated threshold (the definition of include/caro_b200.h).

Workloads:
  * Connect4 with the shipped trained checkpoint on both sides, train.py's search settings (10 x 8 searches, tau = 1 for
    10 plies): `SelfPlayWorker` steps (every game to its end, no slot restarts: the step lasts as long as its longest
    game) and an auto-restart `play_multi` run (2 parts, freed slots start new games at once);
  * Caro 15x15 with a random-init 5 x 64 net (no trained Caro checkpoint exists), `SelfPlayWorker` steps with tree
    compaction.
Prints one JSON line per arm and round, then one summary line per workload, each with the card's name and power limit.

    python tools/resign_bench.py [--rounds 2] [--c4-games 1024] [--caro-games 256] [--multi-plies 40]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def fp_rate(records, t):
    from caro_ai_b200.utils import _false_positives
    if t is None or len(records) == 0:
        return None
    return _false_positives(records, t) / len(records)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2, help="A/B/C rounds")
    ap.add_argument("--c4-games", type=int, default=1024, help="Connect4 games per worker step and per play_multi part")
    ap.add_argument("--c4-steps", type=int, default=3, help="worker steps per Connect4 arm and round")
    ap.add_argument("--caro-games", type=int, default=256, help="Caro 15x15 games per worker step (0 = skip)")
    ap.add_argument("--multi-plies", type=int, default=40, help="timed play_multi plies per arm and round (0 = skip)")
    args = ap.parse_args(argv)
    import torch
    from caro_ai_b200 import config as cfg
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import Caro, ConnectFour
    from caro_ai_b200.model import DeviceNet, Net, load_checkpoint
    from caro_ai_b200.utils import SelfPlayWorker, choose_resign_threshold, resign_tallies
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    gpu = card()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    search = (cfg.MCTS_SEARCHES, cfg.MCTS_BATCH_SIZE, cfg.STEPS_BEFORE_TAU_0)

    def emit(d):
        d["card"] = gpu
        print(json.dumps(d), flush=True)

    def worker_arm(game, dn, G, steps, resign, playthrough, compact, seed):
        w = SelfPlayWorker(game, G, *search, replay_steps=1, min_replay=100, seed=seed, compact_tree=compact,
                           resign=resign, resign_playthrough=playthrough)
        tot = {"games": 0, "plies": 0, "leaf_evals": 0, "resigned": 0}
        recs, sec = [], 0.0
        for _ in range(steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s = w.play_step(dn)
            torch.cuda.synchronize()
            sec += time.perf_counter() - t0
            for k in ("games", "plies", "leaf_evals"):
                tot[k] += s[k]
            if resign is not None:
                tot["resigned"] += w.resign_stats()["resigned"]
                r, _ = w.engine.resign_log(w.engine.resign_counters()["logged"] - w.resign_stats()["logged"])
                recs.append(r)
        w.close()
        recs = np.concatenate(recs) if recs else np.zeros(0, dtype=SelfPlayEngine.RESIGN_RECORD_DTYPE)
        return tot, sec, recs

    def multi_arm(game, dn, G, resign, playthrough, seed):
        parts = [SelfPlayEngine(game, G, max_batch=search[1], node_capacity=8192, seed=seed + 7 * h, compact_tree=True)
                 for h in range(2)]
        for e in parts:
            if resign is not None:
                e.set_resign(resign, playthrough)
            e.reset(first_player=-1)
        run = lambda n: SelfPlayEngine.play_multi(parts, dn, moves=n, count=search[0], batch=search[1], tau_plies=search[2],
                                                  auto_restart=True)
        run(60)  # past the first wave of game ends: slots restart at staggered plies
        c0 = [e.counters() for e in parts]
        r0 = [e.resign_counters() for e in parts]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run(args.multi_plies)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        tot = {"games": 0, "plies": 0, "leaf_evals": 0, "resigned": 0}
        recs = []
        for e, c, r in zip(parts, c0, r0):
            c1, rc = e.counters(), e.resign_counters()
            assert c1["errors"] == 0, c1
            for k in ("games", "plies", "leaf_evals"):
                tot[k] += c1[k] - c[k]
            tot["resigned"] += rc["resigned"] - r["resigned"]
            recs.append(e.resign_log(r["logged"])[0])
            e.close()
        return tot, sec, np.concatenate(recs)

    def report(workload, path, arm, rnd, tot, sec, recs, t):
        g = max(1, tot["games"])
        emit({"workload": workload, "path": path, "arm": arm, "round": rnd, "threshold": t, "seconds": sec,
              "games": tot["games"], "games_per_sec": tot["games"] / sec,
              # play_multi: plies of all games in the window over the games that ended in it (steady state)
              "plies_per_game": tot["plies"] / g, "leaf_evals_per_game": tot["leaf_evals"] / g,
              "leaf_evals_per_sec": tot["leaf_evals"] / sec, "resigned_share": tot["resigned"] / g,
              "logged": int(len(recs)), "fp_rate": fp_rate(recs, t)})
        return {"games_per_sec": tot["games"] / sec, "plies_per_game": tot["plies"] / g,
                "leaf_evals_per_game": tot["leaf_evals"] / g, "resigned_share": tot["resigned"] / g}

    def workload(name, game, dn, G, steps, compact, multi):
        # calibration: one log-only worker run of the same seeded games the arms play
        _, _, recs = worker_arm(game, dn, G, steps, -1.0, 1.0, compact, seed=101)
        t = choose_resign_threshold(resign_tallies(recs), min_records=min(200, len(recs)))
        emit({"workload": name, "calibration_records": int(len(recs)), "threshold": t,
              "min_stat_quantiles": np.quantile(np.min(recs["min_stat"], axis=1), [0.01, 0.1, 0.5, 0.9]).tolist()})
        arms = {"off": (None, 0.0), "log-only": (-1.0, 1.0)}
        if t is not None:
            arms["calibrated"] = (t, 0.1)
        paths = [("worker", lambda a: worker_arm(game, dn, G, steps, a[0], a[1], compact, seed=101))]
        if multi:
            paths.append(("play_multi", lambda a: multi_arm(game, dn, G, a[0], a[1], seed=202)))
        for path, fn in paths:
            res = {a: [] for a in arms}
            for rnd in range(args.rounds):
                for arm, a in arms.items():
                    tot, sec, r = fn(a)
                    res[arm].append(report(name, path, arm, rnd, tot, sec, r, t if arm != "off" else None))
            summary = {a: {k: float(np.mean([x[k] for x in v])) for k in v[0]} for a, v in res.items()}
            base = summary["off"]["games_per_sec"]
            emit({"workload": name, "path": path, "summary": summary, "threshold": t,
                  "games_per_sec_vs_off": {a: s["games_per_sec"] / base for a, s in summary.items()}})

    c4 = ConnectFour()
    dn = DeviceNet(load_checkpoint(os.path.join(root, "tests", "golden", "checkpoints", "connect4_best_026_12000.dat"), c4).eval(), c4)
    workload("connect4 trained checkpoint connect4_best_026_12000, %d games, search_batch(%d,%d), tau 10 plies"
             % ((args.c4_games,) + search[:2]), c4, dn, args.c4_games, args.c4_steps, False, args.multi_plies > 0)
    dn.close()
    if args.caro_games > 0:
        caro = Caro(15, 5)
        torch.manual_seed(0)
        dn = DeviceNet(Net(caro.obs_shape, caro.action_space).eval(), caro)
        workload("caro 15x15/5 random-init 5x64 net, %d games, search_batch(%d,%d), compact tree"
                 % ((args.caro_games,) + search[:2]), caro, dn, args.caro_games, 1, True, False)
        dn.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
