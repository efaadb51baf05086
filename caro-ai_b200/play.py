#!/usr/bin/env python3
"""Round-robin tournament with the reference's CLI and output format (play.py:15-76); all rounds of a pair are
played as one lock-step batch on the GPU.

    python -m caro_ai_b200.play -g 0 saves/a.dat saves/b.dat ... -r 1000
"""
from __future__ import annotations

import argparse
import sys
import time
from typing import Dict, Tuple

from . import config as cfg
from .game import get_game
from .model import DeviceNet, load_checkpoint
from .utils import play_games_batched, update_counts


def main(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument("models", nargs="+", help="The list of models (at least 2) to play against each other")
    parser.add_argument("-r", "--rounds", type=int, default=2, help="Count of rounds to perform for every pair")
    parser.add_argument("--cuda", default=False, action="store_true", help="accepted for compatibility (always CUDA)")
    parser.add_argument("-g", "--game", required=True, choices=["0", "1", "2"],
                        help="The type of game. 0: Connect4, 1: TicTacToe, 2: Caro 15x15")
    parser.add_argument("--precision", default="auto", choices=["auto", "bf16", "bf16x3"],
                        help="tensor-core precision: auto (default) keeps the one-pass bf16 tower only while it reproduces the fp32 priors to 1e-3 on probe positions")
    parser.add_argument("--solver", default=False, action="store_true",
                        help="extension: both players' searches use the MCTS solver (proven wins, losses and draws)")
    parser.add_argument("--gumbel", default=False, action="store_true",
                        help="extension: both players search their roots by Gumbel sequential halving")
    args = parser.parse_args(argv)
    game = get_game(args.game)
    nets = []
    for fname in args.models:
        net = load_checkpoint(fname, game).eval()
        nets.append((fname, DeviceNet(net, game, precision=args.precision)))
    total_agent: Dict[str, Tuple[int, int, int]] = {}
    total_pairs: Dict[Tuple[str, str], Tuple[int, int, int]] = {}
    for idx1, n1 in enumerate(nets):
        for idx2, n2 in enumerate(nets):
            if idx1 == idx2:
                continue
            ts = time.time()
            s = play_games_batched(game, args.rounds, n1[1], n2[1], steps_before_tau_0=0, mcts_searches=cfg.PLAY_MCTS_SEARCHES,
                                   mcts_batch_size=cfg.PLAY_MCTS_BATCH_SIZE, trees_per_game=2, seed=idx1 * 1000 + idx2,
                                   solver=args.solver or None, gumbel=args.gumbel or None)
            wins, losses, draws = s["wins"], s["losses"], s["draws"]
            speed_games = args.rounds / (time.time() - ts)
            name_1, name_2 = n1[0], n2[0]
            print("%s vs %s -> w=%d, l=%d, d=%d" % (name_1, name_2, wins, losses, draws))
            sys.stderr.write("Speed %.2f games/s\n" % speed_games)
            sys.stdout.flush()
            update_counts(total_agent, name_1, (wins, losses, draws))
            update_counts(total_agent, name_2, (losses, wins, draws))
            update_counts(total_pairs, (name_1, name_2), (wins, losses, draws))
    total_leaders = list(total_agent.items())
    total_leaders.sort(reverse=True, key=lambda p: p[1][0])
    print("Leaderboard:")
    for name, (wins, losses, draws) in total_leaders:
        print("%s: \t w=%d, l=%d, d=%d" % (name, wins, losses, draws))
    return 0


if __name__ == "__main__":
    sys.exit(main())
