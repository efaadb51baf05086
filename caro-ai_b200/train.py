#!/usr/bin/env python3
"""AlphaZero training loop with the reference's CLI and behaviour (train.py:1-217), self-play and arena
evaluation running as lock-step batches on the GPU engine.

    python -m caro_ai_b200.train -g 0 -n run_name [--games 4096] [--max-steps N]
    torchrun --nproc-per-node 8 -m caro_ai_b200.train -g 0 -n run_name        # games shard by rank

Same pieces as the reference: a replay buffer (here the self-play engine's DEVICE ring, sized in steps of --games games,
never smaller than REPLAY_BUFFER), 10 SGD rounds of 256 samples (MSE + soft-target cross-entropy, lr 0.1, momentum 0.9),
an arena of EVALUATION_ROUNDS games every EVALUATE_EVERY_STEP steps with 20 x 16 searches at tau = 0, promotion above
0.60, checkpoints ``saves/<name>/best_%03d_%05d.dat`` written with ``torch.save(net.state_dict())``, TensorBoard tags
speed_steps / speed_nodes / loss_total / loss_value / loss_policy / eval_win_ratio (plus plies_per_game, and with the
resignation extension resign_threshold / resign_fp_rate / resigned_share).
The SGD step itself is plain PyTorch autograd (out of scope for hand kernels).  The batch never visits the host: the
reference's ``random.sample`` draws entry numbers, a CUDA kernel turns the ring rows into the planes / pi / z tensors.
With several ranks every rank contributes BATCH_SIZE / world rows of its own ring to the step's batch (one NCCL
all-gather, so BatchNorm sees the reference's 256-row batch), the gradients are averaged by one flattened NCCL
all-reduce per round, every collective decision (train or skip, promote or not) is taken on reduced values, and the
weights are re-broadcast from rank 0 before an evaluation and after a promotion.
"""
from __future__ import annotations

import argparse
import os
import random
import sys
import time

import torch
import torch.nn.functional as F
import torch.optim as optim

from . import config as cfg
from . import distributed as D
from .game import get_game
from .model import DeviceNet, Net, NetWrapper, save_checkpoint
from .utils import SelfPlayWorker, TBMeanTracker, play_games_batched


class _NullWriter:
    def add_scalar(self, *a, **k):
        pass

    def close(self):
        pass


def make_writer(name: str):
    try:
        from torch.utils.tensorboard import SummaryWriter
        return SummaryWriter(comment="-" + name)
    except Exception:  # noqa: BLE001
        return _NullWriter()


def self_play(worker: SelfPlayWorker, best: DeviceNet, tb, step_idx: int):
    """train.py:25-59 for the worker's games at once; returns (counters, seconds) like the reference's prints."""
    t = time.time()
    stats = worker.play_step(best)
    dt = time.time() - t
    tb.track("speed_steps", stats["plies"] / dt, step_idx)
    tb.track("speed_nodes", stats["leaf_evals"] / dt, step_idx)
    if stats["games"]:
        tb.track("plies_per_game", stats["plies"] / stats["games"], step_idx)
    rs = worker.resign_stats()
    if rs:
        tb.track("resigned_share", rs["resigned_share"], step_idx)
        if rs["threshold"] is not None:
            tb.track("resign_threshold", rs["threshold"], step_idx)
        if rs["fp_rate"] is not None:
            tb.track("resign_fp_rate", rs["fp_rate"], step_idx)
    return stats, dt


def resign_option(text: str):
    """--resign: "off" -> None, "auto" -> "auto", else a threshold in [-1, 1]."""
    if text in ("off", "auto"):
        return None if text == "off" else "auto"
    try:
        t = float(text)
    except ValueError:
        raise argparse.ArgumentTypeError("expected off, auto or a threshold in [-1, 1], got %r" % text)
    if not -1.0 <= t <= 1.0:
        raise argparse.ArgumentTypeError("resign threshold must be in [-1, 1], got %r" % text)
    return t


def share_option(text: str) -> float:
    v = float(text)
    if not 0.0 <= v <= 1.0:
        raise argparse.ArgumentTypeError("share must be in [0, 1], got %r" % text)
    return v


def sgd_losses(net: Net, planes: torch.Tensor, probs: torch.Tensor, values: torch.Tensor):
    """train.py:95-106: (total, value, policy) losses of one batch."""
    out_logits, out_values = net(planes)
    loss_value = F.mse_loss(out_values.squeeze(-1), values)
    loss_policy = (-F.log_softmax(out_logits, dim=1) * probs).sum(dim=1).mean()
    return loss_policy + loss_value, loss_value, loss_policy


def sample_batch(game, source, count: int, device, augment: bool = False):
    """train.py:85-94: ``count`` random replay rows as (planes, probs, values) tensors on ``device``.
    ``source`` is a ``SelfPlayEngine`` (device ring: the rows never visit the host) or a reference-style deque of
    (state, player, probs, z) tuples (host path: states -> device boards -> CUDA plane encoder)."""
    if hasattr(source, "replay_sample"):
        return source.replay_sample(count, random, augment=augment)
    batch = random.sample(source, count)
    states, who, probs, values = zip(*batch)
    d_boards = torch.from_numpy(game.boards_from_states(states).view("int64")).to(device)
    d_who = torch.tensor(list(who), dtype=torch.uint8, device=device)
    return (game.planes_device(d_boards, d_who, len(states)), torch.tensor(probs, dtype=torch.float32, device=device),
            torch.tensor(values, dtype=torch.float32, device=device))


def train_neural_net(game, net: Net, source, optimizer, tb, step_idx: int, device, bucket=None, exchange: str = "gather",
                     augment: bool = False):
    """train.py:62-117.  ``source``: the self-play engine (device replay ring) or a deque of reference tuples.
    ``bucket``: a ``distributed.FlatGradients`` over the net's parameters (one all-reduce per round, no flatten /
    scatter); without it the gradients are flattened per round (``allreduce_gradients``).
    ``exchange`` (several ranks): "gather" = every rank draws BATCH_SIZE / world rows and the step's batch is their
    all-gather (the reference's batch size, BatchNorm statistics over all 256 rows); "local" = every rank trains on
    BATCH_SIZE rows of its own ring and only the gradients are exchanged (data parallel, world x the batch).
    ``augment`` (extension, default off): random board symmetries on the sampled rows (device ring only)."""
    _, ws = D.world()
    sums = torch.zeros(3, dtype=torch.float64, device=device)
    net.train()
    gather = exchange == "gather" and ws > 1 and cfg.BATCH_SIZE % ws == 0
    for _ in range(cfg.TRAIN_ROUNDS):
        if gather:
            planes, probs, values = D.all_gather_rows(sample_batch(game, source, cfg.BATCH_SIZE // ws, device, augment))
        else:
            planes, probs, values = sample_batch(game, source, cfg.BATCH_SIZE, device, augment)
        if bucket is not None:
            bucket.zero()
        else:
            optimizer.zero_grad()
        loss, loss_value, loss_policy = sgd_losses(net, planes, probs, values)
        loss.backward()
        if bucket is not None:
            bucket.allreduce()
        else:
            D.allreduce_gradients(net.parameters())
        optimizer.step()
        sums += torch.stack([loss.detach(), loss_value.detach(), loss_policy.detach()]).double()
    means = (sums / cfg.TRAIN_ROUNDS).tolist()  # the only host read of the step
    for tag, m in zip(("loss_total", "loss_value", "loss_policy"), means):
        tb.track(tag, m, step_idx)
    return means


def evaluate(game, challenger: Net, champion: DeviceNet, rounds: int, seed: int, device) -> float:
    """train.py:120-149: challenger vs champion, 20 x 16 searches, tau = 0; rounds shard over ranks and the W/L/D
    tallies are summed, so every rank returns the same ratio."""
    rank, ws = D.world()
    _, mine = D.shard_games(rounds, rank, ws)
    was_training = challenger.training
    challenger.eval()
    ch = DeviceNet(challenger, game)  # precision "auto": the one-pass tower only while it holds the 1e-3 contract
    w = l = d = 0
    if mine:
        s = play_games_batched(game, mine, ch, champion, 0, 20, 16, trees_per_game=2, seed=seed + rank)
        w, l, d = s["wins"], s["losses"], s["draws"]
    ch.close()
    challenger.train(was_training)
    w, l, d = D.reduce_tallies(w, l, d, device=device)
    return w / max(1, w + l + d)


def parse_args(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("-n", "--name", required=True, help="Name of the run")
    p.add_argument("--cuda", default=False, action="store_true", help="accepted for compatibility (always CUDA)")
    p.add_argument("-g", "--game", required=True, choices=["0", "1", "2"], help="0: Connect4, 1: TicTacToe, 2: Caro 15x15")
    p.add_argument("--games", type=int, default=256, help="self-play games per step and per rank (reference: PLAY_EPISODES=1)")
    p.add_argument("--max-steps", type=int, default=0, help="stop after this many steps (0 = run forever, like the reference)")
    p.add_argument("--replay-steps", type=int, default=4, help="device replay ring = this many steps of --games games (>= REPLAY_BUFFER)")
    p.add_argument("--replay-exchange", default="gather", choices=["gather", "local"],
                   help="several ranks: all-gather BATCH_SIZE/world rows per rank (default) or train on local rows only")
    p.add_argument("--augment", action="store_true", help="extension: random board symmetries on the sampled replay rows")
    p.add_argument("--compact-tree", action="store_true",
                   help="drop unreachable tree nodes after every move (bit-identical play, small arenas; for large boards)")
    p.add_argument("--resign", type=resign_option, default=None, metavar="{off,auto,<threshold>}",
                   help="extension: resign self-play games whose search says they are lost (default off; auto = calibrated "
                        "from played-through games to keep wrong resignations under 5 %%)")
    p.add_argument("--resign-playthrough", type=share_option, default=0.1,
                   help="share of self-play games played through with resignation off to measure wrong resignations")
    p.add_argument("--solver", action="store_true",
                   help="extension: MCTS solver in the self-play searches (proven wins, losses and draws); the arena keeps "
                        "the reference's search")
    p.add_argument("--gumbel", action="store_true",
                   help="extension: Gumbel sequential halving at the self-play roots, trained on the improved policy; the "
                        "arena keeps the reference's search")
    p.add_argument("--gumbel-m", type=int, default=16, choices=range(1, 33), metavar="{1..32}",
                   help="root moves sampled per self-play search with --gumbel")
    p.add_argument("--evaluate-every", type=int, default=cfg.EVALUATE_EVERY_STEP, help="arena evaluation period in steps")
    p.add_argument("--blocks", type=int, default=5, choices=range(1, 21), metavar="{1..20}",
                   help="residual blocks of the network (reference: 5)")
    p.add_argument("--filters", type=int, default=64, choices=[64, 128], help="filters of every convolution (reference: 64)")
    return p.parse_args(argv)


def main(argv=None):
    args = parse_args(argv)
    if "RANK" in os.environ and not torch.distributed.is_initialized():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        torch.distributed.init_process_group("nccl")
    rank, ws = D.world()
    device = torch.device("cuda", torch.cuda.current_device())
    saves_path = os.path.join("saves", args.name)
    if rank == 0:
        os.makedirs(saves_path, exist_ok=True)
    writer = make_writer(args.name) if rank == 0 else _NullWriter()
    game = get_game(args.game)
    net = Net(game.obs_shape, game.action_space, blocks=args.blocks, filters=args.filters).to(device)
    D.broadcast_state_dict(net)
    best_net = NetWrapper(net)
    best_dev = DeviceNet(best_net.target_model, game)  # precision "auto", re-checked on every update()
    if rank == 0:
        print(net)
    optimizer = optim.SGD(net.parameters(), lr=cfg.LEARNING_RATE, momentum=0.9)
    bucket = D.FlatGradients(net.parameters())
    worker = SelfPlayWorker(game, args.games, cfg.MCTS_SEARCHES, cfg.MCTS_BATCH_SIZE, cfg.STEPS_BEFORE_TAU_0,
                            replay_steps=args.replay_steps, min_replay=cfg.REPLAY_BUFFER, seed=1000003 * rank + 17,
                            compact_tree=args.compact_tree, resign=args.resign, resign_playthrough=args.resign_playthrough,
                            solver=args.solver, gumbel=args.gumbel_m if args.gumbel else False)
    step_idx = best_idx = 0
    with TBMeanTracker(writer, batch_size=10) as tb:
        while args.max_steps == 0 or step_idx < args.max_steps:
            stats, dt = self_play(worker, best_dev, tb, step_idx)
            step_idx += 1
            replay_len = worker.replay_len()
            if rank == 0:
                print("Step %d, steps %3d, leaves %4d, steps/s %5.2f, leaves/s %6.2f, best_idx %d, replay %d" % (
                    step_idx, stats["plies"], stats["leaf_evals"], stats["plies"] / dt, stats["leaf_evals"] / dt, best_idx,
                    replay_len), end="")
                if args.resign is not None:
                    t = worker.resign_stats()["threshold"]
                    print(", resign %s" % ("-" if t is None else "%.2f" % t), end="")
                print(end="\r")
                sys.stdout.flush()
            # train.py:199 -- decided on the SMALLEST ring of all ranks, so that every rank enters (or skips) the
            # collectives of the SGD rounds together
            need = max(cfg.MIN_REPLAY_TO_TRAIN, cfg.BATCH_SIZE)
            if D.all_min(replay_len, device=device) < need:
                continue
            train_neural_net(game, net, worker.engine, optimizer, tb, step_idx, device, bucket, exchange=args.replay_exchange,
                             augment=args.augment)
            if step_idx % args.evaluate_every == 0:
                D.broadcast_state_dict(net)  # every rank's arena games are played by the same challenger (BN buffers included)
                win_ratio = evaluate(game, net, best_dev, cfg.EVALUATION_ROUNDS, seed=step_idx, device=device)
                if rank == 0:
                    print("Net evaluated, win ratio = %.2f" % win_ratio)
                writer.add_scalar("eval_win_ratio", win_ratio, step_idx)
                if win_ratio > cfg.BEST_NET_WIN_RATIO:  # the same reduced ratio on every rank
                    if rank == 0:
                        print("Net is better than cur best, sync")
                    best_net.sync()
                    D.broadcast_state_dict(best_net.target_model)
                    best_dev.update(best_net.target_model)
                    best_idx += 1
                    if rank == 0:
                        save_checkpoint(net, os.path.join(saves_path, "best_%03d_%05d.dat" % (best_idx, step_idx)))
    worker.close()
    if ws > 1 and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
