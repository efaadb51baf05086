"""Drop-in for the reference's ``lib/utils.py``: ``play_game`` (one game through the ``MCTS`` facade, same
signature / return value / replay tuples), ``update_counts``, ``TBMeanTracker`` -- plus ``play_games_batched``,
the lock-step GPU version of the same loop for thousands of games (what ``train.py`` / ``play.py`` call here).
"""
from __future__ import annotations

import collections
from typing import Dict, List, Optional, Tuple, Union

import numpy as np
import torch

from . import distributed, mcts, model
from .engine import SelfPlayEngine


def update_counts(counts_dict: Dict, key, counts: Tuple[int, int, int]) -> None:
    """lib/utils.py:9-22."""
    v = counts_dict.get(key, (0, 0, 0))
    counts_dict[key] = (v[0] + counts[0], v[1] + counts[1], v[2] + counts[2])


def play_game(game, mcts_stores, replay_buffer: Optional[collections.deque], net1, net2, steps_before_tau_0: int,
              mcts_searches: int, mcts_batch_size: int, net1_plays_first: Optional[bool] = None, device: str = "cpu"):
    """lib/utils.py:25-108: one game, both sides driven by MCTS; returns (net1_result, step).

    ``mcts_stores``: None (a private tree per side, play.py), one ``MCTS`` (shared, train.py) or a list of two.
    ``device`` is accepted for signature compatibility; the search always runs on the current CUDA device.
    """
    assert isinstance(replay_buffer, (collections.deque, type(None)))
    assert isinstance(mcts_stores, (mcts.MCTS, type(None), list))
    assert isinstance(net1, (model.Net, model.DeviceNet)) and isinstance(net2, (model.Net, model.DeviceNet))
    assert isinstance(steps_before_tau_0, int) and steps_before_tau_0 >= 0
    assert isinstance(mcts_searches, int) and mcts_searches > 0
    assert isinstance(mcts_batch_size, int) and mcts_batch_size > 0
    if mcts_stores is None:
        mcts_stores = [mcts.MCTS(game), mcts.MCTS(game)]
    elif isinstance(mcts_stores, mcts.MCTS):
        mcts_stores = [mcts_stores, mcts_stores]
    state = game.initial_state
    nets = [net1, net2]
    cur_player = int(np.random.choice(2)) if net1_plays_first is None else (0 if net1_plays_first else 1)
    step = 0
    tau = 1 if steps_before_tau_0 > 0 else 0
    history = []
    result = net1_result = None
    while result is None:
        store = mcts_stores[cur_player]
        store.search_batch(mcts_searches, mcts_batch_size, state, cur_player, nets[cur_player], device=device)
        probs, _ = store.get_policy_value(state, tau=tau)
        history.append((state, cur_player, probs))
        action = int(np.random.choice(game.action_space, p=probs))
        if action not in game.possible_moves(state):
            print("Impossible action selected")
        state, won = game.move(state, action, cur_player)
        if won:
            result = 1
            net1_result = 1 if cur_player == 0 else -1
            break
        cur_player = 1 - cur_player
        if len(game.possible_moves(state)) == 0:
            result = 0
            net1_result = 0
            break
        step += 1
        if step >= steps_before_tau_0:
            tau = 0
    if replay_buffer is not None:
        for st, who, probs in reversed(history):
            replay_buffer.append((st, who, probs, result))
            result = -result
    return net1_result, step


def _max_plies(game) -> int:
    return game.action_space if game.game_kind != 0 else 42


def run_to_completion(eng: SelfPlayEngine, dn1, dn2, steps_before_tau_0: int, mcts_searches: int, mcts_batch_size: int,
                      first_player: int) -> None:
    """Plays every game of ``eng`` to its end (no re-seating): chunks of 8 plies, one status read between chunks."""
    max_plies = _max_plies(eng.game)
    plies = 0
    while plies < max_plies:
        chunk = min(8, max_plies - plies)
        eng.play(dn1, dn2, moves=chunk, count=mcts_searches, batch=mcts_batch_size, tau_plies=steps_before_tau_0,
                 auto_restart=False, first_player=first_player)
        plies += chunk
        if int((eng.region("status") == 0).sum().item()) == 0:
            break


def _player_mask(flag) -> int:
    """None / False -> 0, True -> both players, a pair (net1's side, net2's side) -> bits 0 / 1."""
    if flag is None or flag is False:
        return 0
    if flag is True:
        return 3
    return (1 if flag[0] else 0) | (2 if flag[1] else 0)


def play_games_batched(game, n_games: int, net1, net2, steps_before_tau_0: int, mcts_searches: int,
                       mcts_batch_size: int, replay_buffer: Optional[collections.deque] = None,
                       net1_plays_first: Optional[bool] = None, trees_per_game: int = 2, node_capacity: Optional[int] = None,
                       seed: int = 0, solver: Union[None, bool, Tuple[bool, bool]] = None,
                       gumbel: Union[None, bool, Tuple[bool, bool]] = None) -> Dict[str, int]:
    """``n_games`` independent ``play_game`` runs advanced in lock-step on the GPU (fresh trees per game =
    the ``mcts_stores=None`` semantics of play.py when ``trees_per_game=2``).  Returns the W/L/D tallies from
    net1's point of view plus counters; finished games' ``(state, player, probs, z)`` tuples are appended to
    ``replay_buffer`` (lib/utils.py:101-106).

    ``nn.Module`` networks are folded with ``DeviceNet(precision="auto")``: the one-pass bf16 tower only while it
    reproduces the fp32 priors / values within 1e-3 on probe positions, the split-precision tower otherwise.

    Two different networks require lock-step plies, so each half of the games gets a fixed first player when
    ``net1_plays_first`` is None (the reference draws it per game: same distribution, lib/utils.py:66).

    ``solver`` (extension, default off): True runs the MCTS solver for both sides, a pair (net1's, net2's) for each side
    on its own (two trees per game); the counts ``solver_stopped`` / ``solver_proven`` are added to the result.

    ``gumbel`` (extension, default off): True searches both sides' roots by Gumbel sequential halving with the default
    parameters (``SelfPlayEngine.set_gumbel``), a pair (net1's, net2's) each side on its own (two trees per game)."""
    mask, gmask = _player_mask(solver), _player_mask(gumbel)
    dn1 = net1 if isinstance(net1, model.DeviceNet) else model.DeviceNet(net1, game)
    dn2 = dn1 if net2 is net1 else (net2 if isinstance(net2, model.DeviceNet) else model.DeviceNet(net2, game))
    max_plies = _max_plies(game)
    cap = node_capacity or min(1 << 16, mcts_searches * mcts_batch_size * max_plies + 8)
    totals = {"wins": 0, "losses": 0, "draws": 0, "games": 0, "plies": 0, "leaf_evals": 0}
    if mask:
        totals.update(solver_stopped=0, solver_proven=0)
    if dn1 is dn2:
        plans = [(n_games, -1 if net1_plays_first is None else (0 if net1_plays_first else 1))]
    elif net1_plays_first is None:
        plans = [(n_games - n_games // 2, 0), (n_games // 2, 1)]
    else:
        plans = [(n_games, 0 if net1_plays_first else 1)]
    for part, (count, first) in enumerate(plans):
        if count == 0:
            continue
        eng = SelfPlayEngine(game, count, trees_per_game=trees_per_game, max_batch=mcts_batch_size, node_capacity=cap,
                             replay_capacity=count * max_plies if replay_buffer is not None else 0, seed=seed + part)
        if mask:
            eng.set_solver(mask)
        if gmask:
            eng.set_gumbel(gmask)
        eng.reset(first_player=first)
        run_to_completion(eng, dn1, dn2, steps_before_tau_0, mcts_searches, mcts_batch_size, first)
        if mask:
            sc = eng.solver_counters()
            totals["solver_stopped"] += sc["stopped"]
            totals["solver_proven"] += sc["proven"]
        c = eng.counters()
        assert c["errors"] == 0, "engine reported errors: %d" % c["errors"]
        totals["wins"] += c["wins_p0"]
        totals["losses"] += c["wins_p1"]
        totals["draws"] += c["draws"]
        totals["games"] += c["games"]
        totals["plies"] += c["plies"]
        totals["leaf_evals"] += c["leaf_evals"]
        if replay_buffer is not None:
            entries, _ = eng.drain_replay()
            replay_buffer.extend(entries)
        eng.close()
    for dn, src in ((dn1, net1), (dn2, net2)):
        if dn is not src:
            dn.close()
    return totals


# ------------------------------------------------------------------ resignation calibration (extension)
# Thresholds the calibration can choose: -0.99, -0.98, ..., -0.50.
RESIGN_GRID = tuple(round(-0.99 + 0.01 * i, 2) for i in range(50))
RESIGN_WINDOW = 2000  # logged playthrough games per rank the "auto" calibration looks at


def resign_tallies(records) -> np.ndarray:
    """int64 [len(RESIGN_GRID), 2]: for every threshold t of the grid, (false positives, records) over the playthrough
    games ``records`` (``SelfPlayEngine.resign_log``).  A game is a false positive at t when some player whose smallest
    statistic was < t did not lose (won or drew): resigning there would have been wrong.  Tallies of several ranks or
    windows add element-wise."""
    out = np.zeros((len(RESIGN_GRID), 2), dtype=np.int64)
    for i, t in enumerate(RESIGN_GRID):
        out[i] = _false_positives(records, t), len(records)
    return out


def _false_positives(records, t: float) -> int:
    if len(records) == 0:
        return 0
    mins = np.asarray(records["min_stat"], dtype=np.float64).reshape(-1, 2)
    result = np.asarray(records["result"], dtype=np.int64).reshape(-1)
    not_lost = np.stack([result != -1, result != 1], axis=1)  # player 0 lost iff result == -1, player 1 iff +1
    return int(((mins < t) & not_lost).any(axis=1).sum())


def choose_resign_threshold(tallies, target: float = 0.05, min_records: int = 200) -> Optional[float]:
    """The largest threshold of RESIGN_GRID whose false-positive rate is <= ``target``; None while the tallies hold fewer
    than ``min_records`` games, or when no threshold qualifies."""
    tallies = np.asarray(tallies, dtype=np.int64)
    n = int(tallies[0, 1])
    if n < min_records:
        return None
    best = None
    for i, t in enumerate(RESIGN_GRID):
        if tallies[i, 0] <= target * n:
            best = t
    return best


def resign_threshold_over_ranks(records, target: float = 0.05, min_records: int = 200,
                                device=None) -> Tuple[Optional[float], np.ndarray]:
    """``choose_resign_threshold`` on the tallies of ``records`` summed over all ranks (one all-reduce, entered by every
    rank whether or not it holds records): every rank gets the same threshold.  Returns (threshold, summed tallies)."""
    tallies = distributed.sum_counts(resign_tallies(records), device=device)
    return choose_resign_threshold(tallies, target, min_records), tallies


def _fp_rate(records, tallies, threshold: Optional[float]) -> Optional[float]:
    """False-positive rate at ``threshold``: from the (rank-summed) tallies on the grid, from ``records`` off it."""
    if threshold is None or tallies[0, 1] == 0:
        return None
    if threshold in RESIGN_GRID:
        i = RESIGN_GRID.index(threshold)
        return float(tallies[i, 0]) / float(tallies[i, 1])
    return _false_positives(records, threshold) / len(records)


class SelfPlayWorker:
    """The trainer's self-play side (train.py:25-59 for ``games`` games at once): ONE engine that lives as long as the
    training run -- its arenas are re-seated every step, not re-allocated -- and whose device replay ring is the
    replay buffer (``replay_capacity`` entries; SURVEY.md section 8(d)-3: the reference's 5,000 positions are ~200
    single-game steps, so the ring is sized in steps of ``games`` games, not in positions)."""

    def __init__(self, game, games: int, mcts_searches: int, mcts_batch_size: int, steps_before_tau_0: int,
                 replay_steps: int = 4, min_replay: int = 5000, seed: int = 0, node_capacity: Optional[int] = None,
                 compact_tree: bool = False, resign: Union[None, float, str] = None, resign_playthrough: float = 0.1,
                 solver: bool = False, gumbel: Union[bool, int] = False):
        """``compact_tree``: drop unreachable nodes after every move (CARO_FLAG_COMPACT_TREE: bit-identical play, arenas of a
        few moves' searches instead of a whole game's -- what large boards need).
        ``resign`` (extension, default off): None plays every game to its end; a float is a fixed resignation threshold
        with ``resign_playthrough`` of the games played through and logged; "auto" logs every game and never resigns
        until the log (the last RESIGN_WINDOW games of every rank, summed over ranks) yields a threshold whose
        false-positive rate is <= 5 %, then resigns at that threshold with ``resign_playthrough`` played through.  The
        calibration runs after every step on every rank (one all-reduce).
        ``solver`` (extension, default off): the MCTS solver for the self-play searches (``SelfPlayEngine.set_solver``):
        proven subtrees get no more descents, and pi / the replay rows keep no visit mass on proven-losing moves.
        ``gumbel`` (extension, default off): True, or an ``m`` (root moves sampled per search), searches every self-play
        root by Gumbel sequential halving (``SelfPlayEngine.set_gumbel``); the replay rows then hold the improved policy
        softmax(log P + sigma(completed Q)) instead of the visit distribution."""
        self.game, self.games = game, int(games)
        self.searches, self.batch, self.tau_plies = mcts_searches, mcts_batch_size, steps_before_tau_0
        max_plies = _max_plies(game)
        per_move = mcts_searches * mcts_batch_size
        cap = node_capacity or min(1 << 16, (8 * per_move if compact_tree else per_move * max_plies) + 8)
        if compact_tree:
            cap = min(cap, 40000)  # the compaction kernel's index map lives in shared memory
        self.replay_capacity = max(int(min_replay), replay_steps * self.games * max_plies)
        self.engine = SelfPlayEngine(game, self.games, trees_per_game=1, max_batch=mcts_batch_size, node_capacity=cap,
                                     replay_capacity=self.replay_capacity, seed=seed, compact_tree=compact_tree)
        if solver:
            self.engine.set_solver(3)
        if gumbel:
            self.engine.set_gumbel(3, m=16 if gumbel is True else int(gumbel))
        self._last = self.engine.counters()
        if not (resign is None or resign == "auto" or isinstance(resign, (int, float))):
            raise ValueError("resign must be None, a threshold or 'auto'")
        self.resign = resign
        self.resign_playthrough = float(resign_playthrough)
        self.resign_threshold: Optional[float] = None
        self._resign_window = collections.deque(maxlen=RESIGN_WINDOW)
        self._resign_cursor = 0
        self._resign_last = {"resigned": 0, "logged": 0}
        self._resign_stats: Dict[str, Optional[float]] = {}
        if resign == "auto":
            self.engine.set_resign(-1.0, 1.0)  # log only until calibrated
        elif resign is not None:
            self.resign_threshold = float(resign)
            self.engine.set_resign(self.resign_threshold, self.resign_playthrough)

    def play_step(self, net: "model.DeviceNet") -> Dict[str, int]:
        """Every game slot plays one fresh game to its end with ``net`` on both sides; the finished games' positions go
        to the ring.  Returns this step's counters (plies, leaf_evals, games, wins / losses / draws of player 0)."""
        eng = self.engine
        eng.reset(first_player=-1)  # new game ids -> new Philox streams, cleared trees (MCTS.clear, no memset)
        run_to_completion(eng, net, net, self.tau_plies, self.searches, self.batch, -1)
        c = eng.counters()
        if c["errors"]:
            raise RuntimeError("self-play engine reported error bits %d" % c["errors"])
        d = {k: c[k] - self._last[k] for k in c}
        self._last = c
        if self.resign is not None:
            self._resign_update(d)
        return {"wins": d["wins_p0"], "losses": d["wins_p1"], "draws": d["draws"], "games": d["games"], "plies": d["plies"],
                "leaf_evals": d["leaf_evals"]}

    def _resign_update(self, d: Dict[str, int]) -> None:
        eng = self.engine
        records, self._resign_cursor = eng.resign_log(self._resign_cursor)
        self._resign_window.extend(records.tolist())
        rc = eng.resign_counters()
        resigned = rc["resigned"] - self._resign_last["resigned"]
        logged = rc["logged"] - self._resign_last["logged"]
        self._resign_last = rc
        window = np.array(list(self._resign_window), dtype=SelfPlayEngine.RESIGN_RECORD_DTYPE)
        if self.resign == "auto":
            t, tallies = resign_threshold_over_ranks(window, device=eng.device)
            if t != self.resign_threshold:
                self.resign_threshold = t
                if t is None:
                    eng.set_resign(-1.0, 1.0)
                else:
                    eng.set_resign(t, self.resign_playthrough)
        else:
            tallies = resign_tallies(window)
        self._resign_stats = {"threshold": self.resign_threshold, "fp_rate": _fp_rate(window, tallies, self.resign_threshold),
                              "resigned": resigned, "logged": logged, "window": int(tallies[0, 1]),
                              "resigned_share": resigned / d["games"] if d["games"] else 0.0,
                              "plies_per_game": d["plies"] / d["games"] if d["games"] else 0.0}

    def resign_stats(self) -> Dict[str, Optional[float]]:
        """Resignation statistics of the last step (empty while resignation is off): the threshold in force for the next
        step (None = not calibrated yet), its false-positive rate over the logged window (over all ranks in "auto"
        mode), games resigned and playthrough games logged in the step, the window size, the resigned share of the
        step's games and its plies per game."""
        return dict(self._resign_stats)

    def replay_len(self) -> int:
        return self.engine.replay_live()

    def close(self):
        self.engine.close()


class TBMeanTracker:
    """lib/utils.py:111-160: averages ``batch_size`` values per tag before writing them to TensorBoard."""

    def __init__(self, writer, batch_size: int):
        assert isinstance(batch_size, int)
        assert writer is not None
        self.writer = writer
        self.batch_size = batch_size

    def __enter__(self):
        self._batches = collections.defaultdict(list)
        return self

    def __exit__(self, exc_type, exc_val, exc_tb):
        self.writer.close()

    @staticmethod
    def _as_float(value) -> float:
        assert isinstance(value, (float, int, np.ndarray, np.generic)) or torch.is_tensor(value)
        if torch.is_tensor(value):
            return value.float().mean().item()
        if isinstance(value, np.ndarray):
            return float(np.mean(value))
        return float(value)

    def track(self, param_name: str, value, iter_index: int) -> None:
        assert isinstance(param_name, str)
        assert isinstance(iter_index, int)
        data = self._batches[param_name]
        data.append(self._as_float(value))
        if len(data) >= self.batch_size:
            self.writer.add_scalar(param_name, np.mean(data), iter_index)
            data.clear()
