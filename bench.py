#!/usr/bin/env python3
"""Benchmark of the MCTS self-play hot path (BASELINE.json: Connect4 leaf evals/s + games/s).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # the CUDA engine (this repo)
    python bench.py --impl reference [--gpus N] --steps K --warmup W   # the reference's CPU algorithm
    python bench.py ... --dump-outputs DIR     # also write what the last timed step computed as DIR/<name>.npy

One "step" = one ply of lock-step self-play for every game of the batch: MCTS.search_batch(100, 8)
(= 800 descents, lib/mcts.py:162-176) on each of the G games, then the policy / sampling / move of
lib/utils.py:76-99, finished games re-seated immediately.  Workload = BASELINE.json configs[1]:
Connect4 6x7, 800 sims/move, >= 4096 concurrent games per B200 (default 2 x 8192: two half-batches pipelined
against each other), random-init 5x64 residual network,
tau = 1 for 10 plies, c_puct 1.0, Dirichlet(0.3) eps 0.25.  Synthetic: no dataset, seeded weights.

Prints ONE JSON line (see the keys in DESIGN.md section 7).  Multi-GPU: one process per GPU under
torchrun, games sharded by rank, no data-path collective (weak scaling); time = max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TRAINED_C4 = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "checkpoints", "connect4_best_026_12000.dat")
# the tower DeviceNet(precision="auto") selects by measuring against the fp32 tower on the device (model.py): the one-pass fp16
# tower for the benchmark's random-init networks -- tcgen05 kind::f16 like bf16, same tensor rate, 11 instead of 8 mantissa bits
# on both operands (3.7e-5 / 8.1e-5 off fp32 where bf16 is 1.1e-4 / 5.0e-4); the bf16 number of the same workload is
# the line's `bf16_same_workload`
DTYPE_OF = {"fp16": "f16", "bf16": "bf16", "bf16x3": "f16 hi+lo x3", "fp32-simt": "f32"}
TOWER_OF = {"fp16": "fp16 tcgen05, fp32 accumulate", "bf16": "bf16 tcgen05, fp32 accumulate",
            "bf16x3": "split-precision fp16 hi + lo tcgen05, fp32 accumulate", "fp32-simt": "fp32 SIMT"}
FLOP_PER_LEAF_C4 = 15598672  # SURVEY.md section 8(d): conv_in 96,768*... + 5 x 3,096,576*... + heads (2 x MAC)
SIMS_COUNT, SIMS_BATCH, TAU_PLIES = 100, 8, 10
GAMES_PER_GPU = 16384  # two software-pipelined half-batches of 8192 (north_star: >= 4096 concurrent games per GPU; the line at
                       # exactly 4096 games is extra.configs.connect4_4096_games)
NODE_CAPACITY = 24576


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"],
                "source": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples nvidia-smi SM clocks / throttle reasons of one GPU during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:  # noqa: BLE001
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------- CPU baseline
REF_DIR = os.path.join(ROOT, "baseline", "_ref")  # the UNMODIFIED reference (lib/ + config.py), vendored by build() in the
                                                  # build container (git-ignored; travels to the GPU box with the snapshot)


def reference_kind():
    return "reference" if os.path.exists(os.path.join(REF_DIR, "lib", "mcts.py")) else "port"


def cpu_reference_worker(args):
    """One process of the reference arm / cpu_baseline: self-play plies driven exactly like lib/utils.py:76-99 drives
    them (search_batch -> get_policy_value(tau) -> np.random.choice -> game.move, one tree per game as in train.py:185),
    train-mode BatchNorm and autograd left on, as the reference runs its self-play.  Classes: the unmodified reference's
    lib.mcts.MCTS / lib.model.Net / ConnectFour when baseline/_ref holds it (kind "reference"), else the oracle port
    (kind "port").  Returns (leaf_evals, plies, games, seconds)."""
    seed, steps, warmup, threads, kind = args
    import numpy as np
    import torch
    torch.set_num_threads(threads)
    if kind == "reference":
        sys.path.insert(0, REF_DIR)
        from lib.game.connect_four.connect_four import ConnectFour as Game
        from lib.mcts import MCTS as Tree
        from lib.model import Net
    else:
        from oracle.games import ConnectFourOracle as Game
        from oracle.mcts import OracleMCTS as Tree
        from oracle.net import OracleNet as Net
    np.random.seed(seed)
    torch.manual_seed(0)
    game = Game()
    net = Net(game.obs_shape, game.action_space)
    counter = {"rows": 0}
    fwd = net.forward

    def counting_forward(x):
        counter["rows"] += int(x.shape[0])
        return fwd(x)

    net.forward = counting_forward
    state, cur, tree, ply = game.initial_state, int(np.random.choice(2)), Tree(game), 0
    leaf = plies = games = 0
    t0 = None
    for step in range(warmup + steps):
        if step == warmup:
            t0 = time.perf_counter()
            counter["rows"] = 0
            plies = games = 0
        tree.search_batch(SIMS_COUNT, SIMS_BATCH, state, cur, net)
        pi, _ = tree.get_policy_value(state, tau=1 if ply < TAU_PLIES else 0)
        action = int(np.random.choice(game.action_space, p=pi))
        state, won = game.move(state, action, cur)
        cur = 1 - cur
        plies += 1
        ply += 1
        if won or not game.possible_moves(state):
            games += 1
            state, cur, tree, ply = game.initial_state, int(np.random.choice(2)), Tree(game), 0
    dt = time.perf_counter() - t0
    leaf = counter["rows"]
    return leaf, plies, games, dt


def run_cpu_reference(steps, warmup, procs, threads):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    kind = reference_kind()
    jobs = [(1000 + i, steps, warmup, threads, kind) for i in range(procs)]
    if procs == 1:
        res = [cpu_reference_worker(jobs[0])]
    else:
        with ctx.Pool(procs) as pool:
            res = pool.map(cpu_reference_worker, jobs)
    leaf = sum(r[0] for r in res)
    plies = sum(r[1] for r in res)
    games = sum(r[2] for r in res)
    dt = max(r[3] for r in res)
    return {"leaf_evals_per_s": leaf / dt, "plies_per_s": plies / dt, "games_per_s": games / dt, "seconds": dt,
            "leaf_evals": leaf, "plies": plies, "kind": kind,
            "what": "unmodified reference (lib.mcts.MCTS + lib.model.Net from baseline/_ref)" if kind == "reference"
                    else "oracle port of the reference (baseline/_ref absent)"}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    procs = max(1, cores)
    r = run_cpu_reference(args.steps, args.warmup, procs, 1)
    line = {
        "impl": "reference", "metric": "connect4_mcts_leaf_evals_per_sec", "value": r["leaf_evals_per_s"], "unit": "leaf_evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * r["seconds"] / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "connect4 6x7 self-play, search_batch(100,8)=800 descents/move, random-init 5x64 net, CPU",
                   "games": procs, "sims_per_move": SIMS_COUNT * SIMS_BATCH},
        "games_per_sec": r["games_per_s"], "plies_per_sec": r["plies_per_s"],
        "cpu_baseline": {"value": r["leaf_evals_per_s"], "unit": "leaf_evals/s", "cores": procs, "kind": r["kind"],
                         "sample": "%d processes x %d plies of CPU self-play (search_batch(100,8) per ply), 1 torch thread each; %s"
                                   % (procs, args.steps, r["what"])},
        "e2e": {"value": r["leaf_evals_per_s"], "unit": "leaf_evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------- extras (not the headline)
def _cuda_ms(torch, fn, repeat=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(repeat):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / repeat


def extra_train(torch, dist, game, ring_engine, world, rank, rounds=20):
    """The only collectives this design has (SURVEY.md section 8e), at this run's world size: `rounds` SGD rounds of
    train.py:82-111 on batches drawn from the self-play engine's DEVICE replay ring -- every rank gathers BATCH_SIZE / N rows
    (CUDA gather kernel), one NCCL all-gather assembles the 256-row batch, forward / backward in plain PyTorch, one NCCL
    all-reduce of the persistent flat gradient bucket (753 KB), SGD step -- then one weight broadcast (best-net promotion)
    and one 3-integer W/L/D reduction (arena).  Times are CUDA-event milliseconds on this rank, max over ranks."""
    import torch.optim as optim
    from caro_ai_b200 import config as cfg, distributed as D, train as T
    from caro_ai_b200.model import Net
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.manual_seed(0)
    net = Net(game.obs_shape, game.action_space).to(dev)
    D.broadcast_state_dict(net)
    opt = optim.SGD(net.parameters(), lr=cfg.LEARNING_RATE, momentum=0.9)
    bucket = D.FlatGradients(net.parameters())
    net.train()
    per = cfg.BATCH_SIZE // world if cfg.BATCH_SIZE % world == 0 else cfg.BATCH_SIZE
    live = ring_engine.replay_live()
    if live < per:
        return {"skipped": "replay ring holds %d entries" % live}
    acc = {"sample": 0.0, "gather": 0.0, "fwd_bwd": 0.0, "allreduce": 0.0, "step": 0.0}
    losses = []

    def one_round(timed):
        box = {}
        t_s = _cuda_ms(torch, lambda: box.__setitem__("rows", ring_engine.replay_sample(per)))
        t_g = _cuda_ms(torch, lambda: box.__setitem__("batch", D.all_gather_rows(box["rows"]) if per != cfg.BATCH_SIZE else box["rows"]))

        def fb():
            bucket.zero()
            loss, _, _ = T.sgd_losses(net, *box["batch"])
            loss.backward()
            box["loss"] = loss.detach()
        t_f = _cuda_ms(torch, fb)
        t_a = _cuda_ms(torch, bucket.allreduce)
        t_o = _cuda_ms(torch, opt.step)
        if timed:
            for k, v in zip(("sample", "gather", "fwd_bwd", "allreduce", "step"), (t_s, t_g, t_f, t_a, t_o)):
                acc[k] += v
            losses.append(float(box["loss"].item()))

    for _ in range(3):
        one_round(False)
    t0 = time.perf_counter()
    for _ in range(rounds):
        one_round(True)
    wall = time.perf_counter() - t0
    bcast_ms = _cuda_ms(torch, lambda: D.broadcast_state_dict(net), 3)
    tally_ms = _cuda_ms(torch, lambda: D.reduce_tallies(1, 2, 3, device=dev), 3)
    # a bare all-reduce of the bucket, back to back: the collective's own latency without the host gaps around it
    bare_ms = _cuda_ms(torch, bucket.allreduce, 20) if world > 1 else 0.0
    out = {"rounds": rounds, "batch": cfg.BATCH_SIZE, "rows_per_rank": per, "gradient_bytes": int(bucket.flat.numel() * 4),
           "sgd_ms_per_round": 1e3 * wall / rounds, "replay_gather_us": 1e3 * acc["sample"] / rounds,
           "allgather_us": 1e3 * acc["gather"] / rounds if world > 1 else None,
           "fwd_bwd_ms": acc["fwd_bwd"] / rounds, "allreduce_us": 1e3 * acc["allreduce"] / rounds if world > 1 else None,
           "allreduce_bare_us": 1e3 * bare_ms if world > 1 else None, "optimizer_step_us": 1e3 * acc["step"] / rounds,
           "broadcast_us": 1e3 * bcast_ms if world > 1 else None, "reduce_tallies_us": 1e3 * tally_ms if world > 1 else None,
           "loss_first": losses[0], "loss_last": losses[-1],
           "limiter": "NCCL launch + all-reduce latency for 753 KB (NVLS / ring, tens of us); the SGD round itself is "
                      "plain PyTorch autograd at batch 256 (launch-bound)"}
    if world > 1:
        t = torch.tensor([out[k] for k in ("sgd_ms_per_round", "allreduce_us", "allgather_us", "broadcast_us")], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out["sgd_ms_per_round"], out["allreduce_us"], out["allgather_us"], out["broadcast_us"] = [float(x) for x in t]
    return out


def extra_configs(torch, dist, world, rank, seed, small=False, net_sms=0):
    """Short, honestly sized runs of the other BASELINE.json configurations.  EVERY rank runs them on its own GPU (games
    shard by rank, no collective on the data path) and the per-rank rates are summed: at N GPUs the entries are the
    aggregate of N x the stated per-GPU workload (weak scaling).  Every number is measured by CUDA events around the plies
    named in `plies` (max over ranks); nothing is scaled or extrapolated."""
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    out = {}

    def run(tag, game, parts, games_per_part, count, batch, cap, warm, plies, note, blocks=5, checkpoint=None, precision="auto", **flags):
        torch.manual_seed(0)
        if checkpoint is not None:  # a TRAINED network: precision "auto" has to pick the split-precision tower for it
            from caro_ai_b200.model import load_checkpoint
            dn = DeviceNet(load_checkpoint(checkpoint, game).eval(), game, precision=precision)
        else:
            dn = DeviceNet(Net(game.obs_shape, game.action_space, blocks=blocks).eval(), game, precision=precision)
        if net_sms:
            dn.set_grid_limit(net_sms)
        engs = [SelfPlayEngine(game, games_per_part, max_batch=batch, node_capacity=cap, seed=seed + 7 * h + 101 * rank, **flags)
                for h in range(parts)]
        SelfPlayEngine.play_multi(engs, dn, moves=warm, count=count, batch=batch, tau_plies=TAU_PLIES, auto_restart=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        c0 = [e.counters() for e in engs]
        ms = _cuda_ms(torch, lambda: SelfPlayEngine.play_multi(engs, dn, moves=plies, count=count, batch=batch, tau_plies=TAU_PLIES,
                                                                auto_restart=True))
        c1 = [e.counters() for e in engs]
        d = {k: sum(b[k] - a[k] for a, b in zip(c0, c1)) for k in c1[0]}
        tot = torch.tensor([d["leaf_evals"], d["descents"], d["plies"], sum(c["errors"] for c in c1)], dtype=torch.float64, device="cuda")
        tmax = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tot)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        sec = float(tmax[0]) / 1e3
        out[tag] = {"workload": note, "gpus": world, "games_per_gpu": parts * games_per_part, "parts": parts, "plies": plies,
                    "warmup_plies": warm, "ms_per_ply": 1e3 * sec / plies, "leaf_evals_per_sec": float(tot[0]) / sec,
                    "descents_per_sec": float(tot[1]) / sec, "plies_per_sec": float(tot[2]) / sec, "precision": dn.precision,
                    "residual_blocks": blocks, "errors": int(tot[3])}
        for e in engs:
            e.close()
        dn.close()
        torch.cuda.empty_cache()  # the arenas of one configuration must not stay cached next to the next one's

    if small:  # the contract test: the same code on toy sizes
        run("connect4_4096_games", ConnectFour(), 2, 64, 8, SIMS_BATCH, 2048, 1, 2, "toy size (--extra-small)")
        run("connect4_4096_games_virtual_loss", ConnectFour(), 2, 64, 8, SIMS_BATCH, 2048, 1, 2, "toy size (--extra-small)",
            virtual_loss=True, mask_priors=True)
        if os.path.exists(TRAINED_C4):
            run("connect4_trained_checkpoint", ConnectFour(), 2, 64, 8, SIMS_BATCH, 2048, 1, 2, "toy size (--extra-small)",
                checkpoint=TRAINED_C4)
        run("caro_15x15_1600_sims", TicTacToe(15, 5), 2, 16, 6, 8, 512, 1, 2, "toy size (--extra-small)")
        run("caro_15x15_1600_sims_20_plies", TicTacToe(15, 5), 2, 16, 6, 8, 512, 1, 4, "toy size (--extra-small)", compact_tree=True)
        run("caro_15x15_1600_sims_deep10", TicTacToe(15, 5), 2, 16, 6, 8, 512, 1, 2, "toy size (--extra-small)", blocks=10)
        return out
    run("connect4_4096_games", ConnectFour(), 2, 2048, SIMS_COUNT, SIMS_BATCH, 12288, 3, 12,
        "BASELINE configs[1] at exactly 4,096 concurrent games per GPU (2 pipeline parts of 2,048), search_batch(100,8)")
    run("connect4_4096_games_virtual_loss", ConnectFour(), 2, 2048, SIMS_COUNT, SIMS_BATCH, 24576, 2, 8,
        "EXTENSION, not the reference's search (CARO_FLAG_VIRTUAL_LOSS + MASK_PRIORS): 4,096 games per GPU, search_batch(100,8); nearly "
        "every descent reaches the network, so a ply costs ~3x the leaf evaluations of the reference-compatible search",
        virtual_loss=True, mask_priors=True)
    if os.path.exists(TRAINED_C4):
        run("connect4_trained_checkpoint", ConnectFour(), 2, 8192, SIMS_COUNT, SIMS_BATCH, 8192, 2, 6,
            "the headline workload (2 x 8,192 games, search_batch(100,8)) with the reference's TRAINED Connect4 checkpoint "
            "best_026_12000.dat instead of a random-init network: DeviceNet(precision='auto') measures the one-pass bf16 tower at "
            "0.24 off fp32 on it and selects the split-precision tower (fp16 hi + lo, 3 MMAs per product, net_rx.cu)",
            checkpoint=TRAINED_C4)
    run("caro_15x15_1600_sims", TicTacToe(15, 5), 2, 1024, 200, 8, 8192, 1, 3,
        "BASELINE configs[3] shape per GPU: Caro 15,15,5, search_batch(200,8) = 1,600 descents/move, reference-shape 5x64 net, "
        "2,048 concurrent games per GPU (2 pipeline parts of 1,024)")
    run("caro_15x15_1600_sims_20_plies", TicTacToe(15, 5), 2, 1024, 200, 8, 8192, 1, 20,
        "the same 2,048 games over 20 timed plies.  A game's tree is kept across its moves (the reference's semantics): 21 x 1,600 "
        "descents would need 36,864-node arenas of 3.6 KB records (276 GB for 2,048 games), so this run sets CARO_FLAG_COMPACT_TREE: "
        "after every move the nodes that can no longer be reached are dropped and the arena packed -- every statistic, policy and "
        "move stays bit-identical to the keep-everything tree (tests/test_gpu_round2.py), the arenas stay below 1,000 nodes",
        compact_tree=True)
    run("caro_15x15_1600_sims_deep10", TicTacToe(15, 5), 2, 1024, 200, 8, 8192, 1, 2,
        "the same with the 'deep residual net' BASELINE configs[3] names and the reference does not define: here 10 residual blocks "
        "of 64 filters (Net(blocks=10); 166.7 MFLOP per leaf)", blocks=10)
    return out


# ----------------------------------------------------------------------------------------- outputs of the timed path
DUMP_LIMIT_BYTES = 64 << 20


def last_ply_outputs(engs):
    """What the self-play path hands its caller after a ply, as float32 / float64 host arrays (parts in order):
    every game's position (device board words: occupied mask, black stones; exact in float64, Connect4 uses bits < 49),
    side to move and ply count after the move, the search policy of the move each game that goes on just made, and the
    replay tuples of the games that ended in the ply (re-seated: ply 0).  The ring holds those games' blocks in the order
    the device reserved them, which varies from run to run, so the tuples are sorted.  Needs auto-restarted play with at
    least one ply before the last one (bench.py's pre-roll)."""
    import numpy as np
    import torch
    boards, players, plies, move_pi, rows = [], [], [], [], []
    for e in engs:
        ply = e.region("ply").long()
        hist = e.fregion("hist_pi")                                   # [games, max plies, A]
        idx = (ply - 1).clamp(0, hist.shape[1] - 1)
        pi = hist[torch.arange(e.G, device=hist.device), idx] * (ply > 0).unsqueeze(1)
        boards.append(e.region("root_board").cpu().numpy().astype(np.float64))
        players.append(e.region("root_player").cpu().numpy().astype(np.float32))
        plies.append(ply.cpu().numpy().astype(np.float32))
        move_pi.append(pi.cpu().numpy())
        cursor, cap = e.replay_cursor(), e.cfg.replay_capacity
        live = min(cursor, cap)
        slots = torch.arange(cursor - live, cursor, device=hist.device) % cap
        ring = np.concatenate([e.region("replay_board")[slots].cpu().numpy().astype(np.float64),
                               e.region("replay_player")[slots].cpu().numpy().astype(np.float64)[:, None],
                               e.fregion("replay_pi")[slots].cpu().numpy().astype(np.float64),
                               e.fregion("replay_z")[slots].cpu().numpy().astype(np.float64)[:, None]], axis=1)
        ended = int((plies[-1] == 0).sum())
        starts = np.flatnonzero(ring[:, 0] == 0)                       # a game's block opens with the empty board
        assert ended <= len(starts), "the replay ring no longer holds the games that ended in the last ply"
        rows.append(ring[starts[len(starts) - ended]:] if ended else ring[:0])
    rows = np.concatenate(rows)
    rows = rows[np.lexsort(rows.T[::-1])]
    out = {"root_board": np.concatenate(boards), "root_player": np.concatenate(players), "root_ply": np.concatenate(plies),
           "move_pi": np.concatenate(move_pi)}
    budget = DUMP_LIMIT_BYTES - sum(a.nbytes for a in out.values())
    row_bytes = 2 * 8 + 4 + 4 * (rows.shape[1] - 4) + 4
    if len(rows) * row_bytes > budget:  # a fixed, seeded sample of the tuples keeps the dump within its limit
        keep = np.sort(np.random.default_rng(0).choice(len(rows), budget // row_bytes, replace=False))
        rows = rows[keep]
    out.update(replay_board=rows[:, :2], replay_player=rows[:, 2].astype(np.float32),
               replay_pi=rows[:, 3:-1].astype(np.float32), replay_z=rows[:, -1].astype(np.float32))
    return out


def dump_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ----------------------------------------------------------------------------------------- CUDA engine
def engine_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour
    from caro_ai_b200.model import DeviceNet, Net

    game = ConnectFour()
    torch.manual_seed(0)
    net = Net(game.obs_shape, game.action_space).eval()
    dnet = DeviceNet(net, game, precision=args.precision)
    if args.net_sms:
        dnet.set_grid_limit(args.net_sms)
    G = args.games
    # the game batch is split in two halves that are software-pipelined against each other (one half's tree kernels
    # run on a side stream underneath the other half's network pass); --no-pipeline keeps one engine, one stream
    halves = 1 if args.no_pipeline else args.parts
    assert G % halves == 0, "--games must be divisible by --parts"
    engs = [SelfPlayEngine(game, G // halves, trees_per_game=1, max_batch=SIMS_BATCH, node_capacity=args.node_capacity,
                           replay_capacity=1 << 19, seed=1234 + 16 * rank + h) for h in range(halves)]
    stream = torch.cuda.current_stream()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def play(n, count=SIMS_COUNT):
        if halves >= 2:
            SelfPlayEngine.play_multi(engs, dnet, moves=n, count=count, batch=SIMS_BATCH, tau_plies=TAU_PLIES, auto_restart=True)
        else:
            engs[0].play(dnet, dnet, moves=n, count=count, batch=SIMS_BATCH, tau_plies=TAU_PLIES, auto_restart=True)

    def counters():
        tot = {}
        for e in engs:
            for k, v in e.counters().items():
                tot[k] = tot.get(k, 0) + v
        return tot

    # untimed pre-roll with a cheap search so that the games de-synchronise (finished games re-seat at once):
    # the timed window then sees a mix of openings, middle games and endgames instead of 4096 identical plies
    play(args.preroll, count=8)
    play(args.warmup)
    barrier()
    c0 = counters()
    # The K timed plies: the first K - P replay one CUDA graph per ply (the production path), the last P are issued
    # launch by launch with CUDA events around every network kernel (events cannot be replayed from a graph); both
    # kinds are inside the timed region, the roofline's per-launch duration comes from the P evented plies.
    evented = args.steps if (args.profile_level >= 2 or halves < 2) else max(1, min(8, args.steps // 4))
    graphed = args.steps - evented
    for e in engs:
        e.profile(0)
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    if graphed:
        play(graphed)
    for e in engs:
        e.profile(args.profile_level)  # host-side switch, no synchronisation
    play(evented)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    prof = {}
    for e in engs:
        for k, v in e.profile_read().items():
            prof[k] = prof.get(k, 0) + v
        e.profile(0)
    c1 = counters()
    if args.dump_outputs:  # before the legs below play on with the same engines
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, "rank%d" % rank), last_ply_outputs(engs))

    # ---- end-to-end: same plies driven through HOST buffers: pinned H2D of every game's root position + side to move,
    # D2H of the positions after the move AND of the self-play product -- the replay tuples (position, side, pi, z;
    # lib/utils.py:101-106) the finished games wrote during the ply
    Gh = G // halves
    boards_h = [torch.empty((Gh, 2), dtype=torch.int64).pin_memory() for _ in engs]
    players_h = [torch.empty((Gh,), dtype=torch.uint8).pin_memory() for _ in engs]
    rcap = engs[0].cfg.replay_capacity
    replay_h = [{"board": torch.empty((rcap, 2), dtype=torch.int64).pin_memory(), "player": torch.empty((rcap,), dtype=torch.uint8).pin_memory(),
                 "pi": torch.empty((rcap, game.action_space), dtype=torch.float32).pin_memory(),
                 "z": torch.empty((rcap,), dtype=torch.float32).pin_memory()} for _ in engs]
    for e, bh, ph in zip(engs, boards_h, players_h):
        bh.copy_(e.region("root_board"))
        ph.copy_(e.region("root_player"))
    torch.cuda.synchronize()
    e2e_steps = max(1, args.steps // 2)
    barrier()
    ce0 = counters()
    cursors = [e.replay_cursor() for e in engs]
    d2h_bytes = 0
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ee0.record(stream)
    for _ in range(e2e_steps):
        for e, bh, ph in zip(engs, boards_h, players_h):
            e.set_roots_pinned(bh, ph)                      # H2D: this ply's positions + side to move
        play(1)
        for i, (e, bh, ph) in enumerate(zip(engs, boards_h, players_h)):
            bh.copy_(e.region("root_board"), non_blocking=True)   # D2H: positions after the move (re-seated if finished)
            ph.copy_(e.region("root_player"), non_blocking=True)
            cursors[i], nb = e.replay_to_pinned(cursors[i], replay_h[i])  # D2H: the replay tuples of the games that ended
            d2h_bytes += nb + Gh * 17
        stream.synchronize()  # the host owns the buffers between plies
    ee1.record(stream)
    barrier()
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    e2e_ms = ee0.elapsed_time(ee1)
    ce1 = counters()
    workspace_gb = sum(e.workspace_bytes for e in engs) / 1e9
    # the same engines, mid-game states and plies with the one-pass BF16 tower forced -- the dtype BASELINE.json's north_star
    # names -- when the device check selected another tower for the headline
    bf16_same = None
    if dnet.precision != "bf16" and not args.no_extra:
        dn_b = DeviceNet(net, game, precision="bf16")
        if args.net_sms:
            dn_b.set_grid_limit(args.net_sms)
        main_net, dnet = dnet, dn_b
        n_b = max(4, min(16, args.steps // 3))
        play(2)
        barrier()
        cb0 = counters()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record(stream)
        play(n_b)
        b1.record(stream)
        barrier()
        cb1 = counters()
        t = torch.tensor([float(cb1["leaf_evals"] - cb0["leaf_evals"])], dtype=torch.float64, device="cuda")
        tm = torch.tensor([b0.elapsed_time(b1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        bf16_same = {"precision": "bf16", "plies": n_b, "value": float(t[0]) / (float(tm[0]) / 1e3), "unit": "leaf_evals/s",
                     "ms_per_step": float(tm[0]) / n_b}
        dnet = main_net
        dn_b.close()
    extra = {}
    if not args.no_extra:
        extra["train"] = extra_train(torch, dist, game, engs[0], world, rank)
        for e in engs:
            e.close()
        del engs[:]
        torch.cuda.empty_cache()
        extra["configs"] = extra_configs(torch, dist, world, rank, 4321, small=args.extra_small)

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    leaf = allsum(c1["leaf_evals"] - c0["leaf_evals"])
    games = allsum(c1["games"] - c0["games"])
    plies = allsum(c1["plies"] - c0["plies"])
    desc = allsum(c1["descents"] - c0["descents"])
    ms_max = allmax(ms)
    e2e_leaf = allsum(ce1["leaf_evals"] - ce0["leaf_evals"])
    e2e_max = allmax(e2e_ms)
    errors = allsum(c1["errors"])
    if rank == 0:
        peaks = measured_peaks()
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "net_traffic.json")
        if os.path.exists(tpath):  # dram__bytes_read + dram__bytes_write of one `ncu --set full` capture of this kernel
            with open(tpath) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        sec = ms_max / 1000.0
        my_leaf = c1["leaf_evals"] - c0["leaf_evals"]
        net_s = prof["net_ms"] / 1000.0
        n_net_launches = args.steps * SIMS_COUNT * halves
        n_evented = evented * SIMS_COUNT * halves
        avg_launch_s = net_s / max(1, n_evented)
        achieved_tflops = (my_leaf / max(1, n_net_launches)) * FLOP_PER_LEAF_C4 / avg_launch_s / 1e12 if net_s > 0 else 0.0
        graph_launches = graphed * (prof["launches"] / max(1, evented))  # the graph replays exactly the kernels of an evented ply
        line = {
            "metric": "connect4_mcts_leaf_evals_per_sec", "value": leaf / sec, "unit": "leaf_evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPE_OF[dnet.precision], "data": "synthetic",
            "config": {"workload": "connect4 6x7 self-play, search_batch(100,8)=800 descents/move, %d concurrent games per GPU, "
                                   "random-init 5x64 residual net (%s), tau=1 for 10 plies" % (G, TOWER_OF[dnet.precision]),
                       "games_per_gpu": G, "sims_per_move": SIMS_COUNT * SIMS_BATCH, "node_capacity": args.node_capacity,
                       "pipeline": ("%d part-batches of %d games, each part's tree kernels on its own side stream under the other parts' network passes" % (halves, G // halves)) if halves >= 2 else "single stream",
                       "cache": "tree arenas %.1f GB per GPU >> 126 MB L2 (inputs larger than L2, no flush needed)"
                                % workspace_gb},
            "games_per_sec": games / sec, "plies_per_sec": plies / sec, "descents_per_sec": desc / sec,
            "e2e": {"value": e2e_leaf / (e2e_max / 1000.0), "unit": "leaf_evals/s", "steps": e2e_steps,
                    "h2d_bytes_per_step": int(world * G * 17), "d2h_bytes_per_step": int(world * d2h_bytes / e2e_steps),
                    "d2h": "new root positions (17 B/game) + the replay tuples written during the ply (49 B/entry) + ring cursor"},
            "gpu_launches": int(prof["launches"]) + int(graph_launches),
            "roofline": {"kernel": "net_rt_kernel (row-tiled tcgen05 residual tower)", "bound": "tensor", "achieved": achieved_tflops,
                         "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": achieved_tflops / peaks["bf16_tflops_sustained"],
                         "traffic": traffic, "peak_source": peaks["source"] + " (sustained: kernel timed inside a long step; the dense bf16 figure -- fp16 and "
                                        "bf16 operands run the same tcgen05 kind::f16 instruction at the same rate)",
                         "note": "average CUDA-event time per tower launch over the evented plies of the timed region (the other timed "
                                 "plies replay a CUDA graph, where events cannot be recorded); the parts' towers run on their own streams "
                                 "and overlap tail-to-head, so `achieved` is a lower bound (stand-alone: tools/net_bench.py, DESIGN.md "
                                 "section 4)" if halves >= 2 else "",
                         "flop_per_leaf": FLOP_PER_LEAF_C4, "leaves_per_launch": my_leaf / max(1, n_net_launches),
                         "avg_launch_ms": 1e3 * avg_launch_s, "evented_steps": evented, "graph_replayed_steps": graphed},
            "phase_ms_per_step": {k: prof[k] / max(1, evented) for k in ("select_ms", "plan_ms", "net_ms", "expand_backup_ms")
                                  if args.profile_level >= 2 or k == "net_ms"},
            "clocks": sampler.summary(), "engine_errors": int(errors),
            "net_precision": {"selected": dnet.precision, "calibration": dnet.calibration},
            "bf16_same_workload": bf16_same,
        }
        if extra:
            line["extra"] = extra
        if not args.no_cpu_baseline and world == 1:  # the CPU arm is timed beside the single-GPU number only
            cores = os.cpu_count() or 1
            r = run_cpu_reference(args.cpu_plies, 1, cores, 1)  # one process per host core, like the reference arm
            line["cpu_baseline"] = {"value": r["leaf_evals_per_s"], "unit": "leaf_evals/s", "cores": cores, "kind": r["kind"],
                                    "games_per_sec": r["games_per_s"],
                                    "sample": "%d processes x 1 torch thread, %d plies of CPU self-play each "
                                              "(search_batch(100,8) per ply) after 1 warm-up ply; %s" % (cores, args.cpu_plies, r["what"])}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--games", type=int, default=GAMES_PER_GPU)
    ap.add_argument("--node-capacity", type=int, default=NODE_CAPACITY)
    ap.add_argument("--cpu-plies", type=int, default=40)
    ap.add_argument("--preroll", type=int, default=30)
    ap.add_argument("--no-pipeline", action="store_true")
    ap.add_argument("--parts", type=int, default=2, help="software-pipelined parts the game batch is split into")
    ap.add_argument("--net-sms", type=int, default=0, help="SMs the network kernel may occupy (0 = all); the rest serve the tree kernels")
    ap.add_argument("--profile-level", type=int, default=1, help="1: CUDA events around the network kernel only, 2: all phases")
    ap.add_argument("--precision", default="auto", choices=["auto", "fp16", "bf16", "bf16x3"],
                    help="tower of the headline run: auto = the fastest one-pass tower within 1e-3 of fp32 on the device check")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extra-small", action="store_true", help="toy sizes for extra.configs (tests)")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra.train / extra.configs measurements after the headline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (under torchrun: DIR/rank<r>/)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs writes the CUDA engine's outputs (--impl engine)")
    if args.impl == "reference":
        return reference_arm(args)
    return engine_arm(args)


if __name__ == "__main__":
    sys.exit(main())
