"""Measures the 128-filter towers on the GPU and prints JSON lines.

    python tools/wide_bench.py [--seconds S] [--out FILE]

1. Stand-alone tower time (CUDA events, after warm-up): 5x128 Connect4 at 9,472 and 33,152 leaves, 10x128 Caro 15x15 at
   4,096 and 16,384 leaves; the wide tower with fp16 (impl 7), bf16 (impl 0) and bf16 hi + lo (impl 8, split precision)
   operands and, on the same boards, the 64-wide tap-per-MMA tower (impl 3, a 64-filter net of the same depth),
   alternated in rounds; the SIMT tower (impl 1, the fallback of precision "auto") at the smaller size of each board.
   Useful TFLOP/s = leaves x FLOP per leaf / time, with FLOP per leaf from the formula below (the split tower's three
   products per multiply-add are not counted as useful).
2. The phases of one layer (clock64 timeline of CTA 0): MMA phase, weight waits, epilogue, hand-off, against the tensor
   floor, for 10x128 Caro at 16,384 leaves and 5x128 Connect4 at 33,152 leaves, for impls 7, 0 and 8.
3. Self-play leaf evaluations/s: Caro 15,15,5 at search_batch(200, 8), 2 parts x 1,024 games, 10x128 net, compact tree;
   Connect4 at search_batch(100, 8), 2 x 8,192 games, 5x128 net -- both random-init, precision "auto".  Then the
   "trained-like" 10x128 Caro net of tests/wide_split_net.py (policy FC x 100, residual stream x 2^17), which "auto" sends
   to the split tower: at the configuration above, and at a small one (2 x 256 games, search_batch(10, 8)) both on the
   split tower and on the SIMT tower, whose self-play rate the small configuration makes measurable.
The card's name, power limit and SM clock under load are read with a read-only nvidia-smi query in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def flop_per_leaf(h, w, a, blocks, filters):
    """SURVEY.md section 8(d) with width F: 2 FLOP per multiply-add of conv_in (2 -> F, 3x3), the residual convolutions
    (F -> F, 3x3), the 1x1 head convolutions (F -> 1 and F -> 2) and the FC heads (HW -> 20 -> 1, 2 HW -> A)."""
    hw, f = h * w, filters
    conv_in = 2 * hw * f * 2 * 9
    tower = blocks * 2 * hw * f * f * 9
    heads = 2 * hw * f * 3 + 2 * hw * 20 + 2 * 20 + 2 * 2 * hw * a
    return conv_in + tower + heads


assert flop_per_leaf(6, 7, 7, 5, 128) == 62160208
assert flop_per_leaf(15, 15, 225, 10, 128) == 664973140
assert flop_per_leaf(6, 7, 7, 5, 64) == 15598672
assert flop_per_leaf(15, 15, 225, 5, 64) == 83760340


class ClockSampler:
    """nvidia-smi --query-gpu (read-only) every half second while the measurement runs."""
    FIELDS = "name,power.limit,clocks.sm,clocks.max.sm,power.draw"

    def __init__(self, props):
        # nvidia-smi numbers cards its own way (CUDA_VISIBLE_DEVICES does not remap it): address the card by its PCI bus id
        self.index = "%08X:%02X:%02X.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        self.rows, self.stop = [], threading.Event()
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _query(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=10)
        return [x.strip() for x in out.stdout.strip().split(",")] if out.returncode == 0 else None

    def _run(self):
        while not self.stop.is_set():
            r = self._query()
            if r:
                self.rows.append(r)
            self.stop.wait(0.5)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.thread.join()

    def summary(self):
        if not self.rows:
            return {}
        sm = sorted(float(r[2]) for r in self.rows)
        draw = sorted(float(r[4]) for r in self.rows)
        return {"gpu": self.rows[0][0], "power_limit_w": float(self.rows[0][1]), "sm_clock_mhz_median": sm[len(sm) // 2],
                "sm_clock_mhz_min": sm[0], "sm_clock_max_mhz": float(self.rows[0][3]), "power_draw_w_median": draw[len(draw) // 2],
                "samples": len(self.rows)}


def emit(d, out):
    line = json.dumps(d)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def tower_bench(torch, seconds, out):
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet, Net, probe_positions
    cases = [(ConnectFour(), 5, (9472, 33152)), (TicTacToe(15, 5), 10, (4096, 16384))]
    for game, blocks, sizes in cases:
        _, h, w = game.obs_shape
        a = game.action_space
        torch.manual_seed(0)
        wide = DeviceNet(Net(game.obs_shape, a, blocks=blocks, filters=128).eval(), game, precision="fp32-simt")
        torch.manual_seed(0)
        narrow = DeviceNet(Net(game.obs_shape, a, blocks=blocks).eval(), game, precision="fp32-simt")
        base_b, base_w = probe_positions(game, 1024)
        for leaves in sizes:
            towers = [("wide_fp16", wide, 7, 128), ("wide_bf16", wide, 0, 128), ("wide_bf16x3", wide, 8, 128),
                      ("tap_per_mma_64", narrow, 3, 64)]
            if leaves == sizes[0]:  # the SIMT tower at one size per board: a launch takes up to about a second
                towers.append(("simt_128", wide, 1, 128))
            idx = torch.arange(leaves, device="cuda") % base_b.shape[0]
            d_boards, d_who = base_b[idx].contiguous(), base_w[idx].contiguous()
            times = {name: [] for name, *_ in towers}
            iters = {}
            for name, dn, impl, _ in towers:  # warm-up and sizing: each timed window lasts about `seconds`
                for _ in range(2):
                    dn.forward_boards(d_boards, d_who, leaves, impl)
                torch.cuda.synchronize()
                t0 = time.time()
                for _ in range(3):
                    dn.forward_boards(d_boards, d_who, leaves, impl)
                torch.cuda.synchronize()
                iters[name] = max(10 if impl != 1 else 2, int(seconds / max(1e-6, (time.time() - t0) / 3)))
            for _ in range(2):  # rounds, the towers alternate
                for name, dn, impl, _ in towers:
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record()
                    for _ in range(iters[name]):
                        dn.forward_boards(d_boards, d_who, leaves, impl)
                    e.record()
                    e.synchronize()
                    times[name].append(s.elapsed_time(e) / iters[name])
            for name, dn, impl, f in towers:
                ms = min(times[name])
                flop = flop_per_leaf(h, w, a, blocks, f)
                emit({"kind": "tower", "game": type(game).__name__, "board": [h, w], "blocks": blocks, "filters": f, "tower": name,
                      "impl": impl, "leaves": leaves, "launches_per_round": iters[name], "ms_per_launch": ms,
                      "ms_per_launch_rounds": times[name], "flop_per_leaf": flop, "useful_tflops": leaves * flop / (ms * 1e-3) / 1e12},
                     out)
        wide.close()
        narrow.close()


def timeline_bench(torch, out):
    """Splits one layer of the wide tower into its phases with the kernel's clock64 timeline (CTA 0, caro_net_set_trace):
    MMA phase (layer input ready -> every MMA complete; of it, the cycles the MMA warp waited for weight slots), epilogue
    (accumulators complete -> epilogue done) and hand-off (epilogue done -> next layer's input seen by the MMA warp), as
    medians over the residual layers of CTA 0, against the tensor floor of 2 tiles x 72 MMAs x 64 cycles (split
    precision: 3 x 72 MMAs per tile)."""
    import ctypes as C
    from caro_ai_b200 import _cabi
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet, Net, probe_positions
    for game, blocks, leaves in ((TicTacToe(15, 5), 10, 16384), (ConnectFour(), 5, 33152)):
        torch.manual_seed(0)
        dn = DeviceNet(Net(game.obs_shape, game.action_space, blocks=blocks, filters=128).eval(), game, precision="fp32-simt")
        base_b, base_w = probe_positions(game, 1024)
        idx = torch.arange(leaves, device="cuda") % base_b.shape[0]
        d_boards, d_who = base_b[idx].contiguous(), base_w[idx].contiguous()
        trace = torch.zeros(8001, dtype=torch.int64, device="cuda")
        n_layers = blocks + 1
        for name, impl in (("wide_fp16", 7), ("wide_bf16", 0), ("wide_bf16x3", 8)):
            floor = 2 * 72 * 64 * (3 if impl == 8 else 1)
            for _ in range(3):
                dn.forward_boards(d_boards, d_who, leaves, impl)
            trace.zero_()
            _cabi.check(_cabi.lib().caro_net_set_trace(dn.handle, C.c_void_p(trace.data_ptr())))
            dn.forward_boards(d_boards, d_who, leaves, impl)
            torch.cuda.synchronize()
            _cabi.check(_cabi.lib().caro_net_set_trace(dn.handle, None))
            t = trace.cpu().numpy()[:5000].reshape(5, 1000)
            rows = []
            for gl in range(999):
                if gl % n_layers == 0 or (gl + 1) % n_layers == 0 or t[0, gl + 1] == 0 or t[3, gl] == 0:
                    continue  # residual layers followed by a residual layer of the same group
                rows.append((t[2, gl] - t[0, gl], t[4, gl], t[1, gl] - t[0, gl], t[3, gl] - t[2, gl], t[0, gl + 1] - t[3, gl],
                             t[0, gl + 1] - t[0, gl]))
            med = [float(sorted(col)[len(col) // 2]) for col in zip(*rows)]
            emit({"kind": "timeline", "game": type(game).__name__, "blocks": blocks, "leaves": leaves, "tower": name, "impl": impl,
                  "layers_sampled": len(rows), "cycles_per_layer": med[5], "mma_phase_cycles": med[0],
                  "weight_wait_cycles": med[1], "mma_issue_cycles": med[2], "epilogue_cycles": med[3], "handoff_cycles": med[4],
                  "tensor_floor_cycles": floor, "mma_phase_over_floor": med[0] / floor, "epilogue_share": med[3] / med[5]}, out)
        dn.close()


def selfplay_bench(torch, out):
    from caro_ai_b200.engine import SelfPlayEngine
    from caro_ai_b200.game import ConnectFour, TicTacToe
    from caro_ai_b200.model import DeviceNet, Net
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import wide_split_net

    def random_init(game, blocks):
        torch.manual_seed(0)
        return Net(game.obs_shape, game.action_space, blocks=blocks, filters=128).eval().state_dict()

    def trained_like(game, blocks):
        return wide_split_net.trained_like_net(game, blocks)[1]

    caro, c4, compact = TicTacToe(15, 5), ConnectFour(), {"compact_tree": True}
    # (net, game, blocks, precision, parts, games per part, searches, batch, node capacity, warm-up plies, timed plies, flags)
    cases = [("random_init", caro, 10, "auto", 2, 1024, 200, 8, 8192, 1, 3, compact),
             ("random_init", c4, 5, "auto", 2, 8192, 100, 8, 8192, 2, 6, {}),
             ("trained_like", caro, 10, "auto", 2, 1024, 200, 8, 8192, 1, 3, compact),
             ("trained_like", caro, 10, "auto", 2, 256, 10, 8, 2048, 1, 1, compact),
             ("trained_like", caro, 10, "fp32-simt", 2, 256, 10, 8, 2048, 1, 1, compact)]
    for kind, game, blocks, precision, parts, gpp, count, batch, cap, warm, plies, flags in cases:
        sd = random_init(game, blocks) if kind == "random_init" else trained_like(game, blocks)
        dn = DeviceNet(sd, game, precision=precision)
        engs = [SelfPlayEngine(game, gpp, max_batch=batch, node_capacity=cap, seed=11 + 7 * h, **flags) for h in range(parts)]
        SelfPlayEngine.play_multi(engs, dn, moves=warm, count=count, batch=batch, tau_plies=30, auto_restart=True)
        torch.cuda.synchronize()
        c0 = [e.counters() for e in engs]
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        SelfPlayEngine.play_multi(engs, dn, moves=plies, count=count, batch=batch, tau_plies=30, auto_restart=True)
        e.record()
        e.synchronize()
        sec = s.elapsed_time(e) / 1e3
        c1 = [x.counters() for x in engs]
        d = {k: sum(b[k] - a[k] for a, b in zip(c0, c1)) for k in c1[0]}
        emit({"kind": "selfplay", "net": kind, "game": type(game).__name__, "board": list(game.obs_shape[1:]), "blocks": blocks,
              "filters": 128, "games": parts * gpp, "parts": parts, "search_batch": [count, batch],
              "compact_tree": bool(flags.get("compact_tree")), "timed_plies": plies, "ms_per_ply": 1e3 * sec / plies,
              "leaf_evals_per_sec": d["leaf_evals"] / sec, "errors": sum(c["errors"] for c in c1), "precision": dn.precision,
              "impl": dn.impl, "calibration": dn.calibration}, out)
        for x in engs:
            x.close()
        dn.close()
        torch.cuda.empty_cache()


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--seconds", type=float, default=2.0, help="length of one timed window of the tower measurement")
    p.add_argument("--out", default=None, help="also append the JSON lines to this file")
    p.add_argument("--skip-selfplay", action="store_true")
    args = p.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("wide_bench.py needs a CUDA device")
    with ClockSampler(torch.cuda.get_device_properties(torch.cuda.current_device())) as clocks:
        tower_bench(torch, args.seconds, args.out)
        timeline_bench(torch, args.out)
        if not args.skip_selfplay:
            selfplay_bench(torch, args.out)
    emit(dict({"kind": "device"}, **clocks.summary()), args.out)


if __name__ == "__main__":
    main()
