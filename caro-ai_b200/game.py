"""Host-side mirror of the reference's game interface (lib/game/game.py:9-120,
lib/game/connect_four/connect_four.py:8-281, lib/game/tictactoe/tictactoe.py:10-259).

Same class names, members, argument meaning and error behaviour (``AssertionError`` on illegal
input).  The state integers are the reference's; this module only converts them to and from the
packed device boards (pure integer re-encoding, no game logic) -- the rules themselves (move, win,
legal moves, network planes) run in the CUDA board kernels of libcaro_b200.so
(csrc/rules.cuh, csrc/boards.cu) and there is no CPU implementation of them in this package.
"""
from __future__ import annotations

from abc import ABC, abstractmethod
from typing import List, Sequence, Tuple

import numpy as np

from . import _cabi


class BaseGame(ABC):
    """lib/game/game.py:9-120."""

    @property
    @abstractmethod
    def initial_state(self) -> int: ...

    @property
    @abstractmethod
    def obs_shape(self) -> Tuple[int, ...]: ...

    @property
    @abstractmethod
    def action_space(self) -> int: ...

    @abstractmethod
    def possible_moves(self, mcts_state: int) -> List: ...

    @abstractmethod
    def invalid_moves(self, mcts_state: int) -> List: ...

    @abstractmethod
    def states_to_training_batch(self, state_lists: List, who_moves_lists: List[int]) -> np.ndarray: ...

    @abstractmethod
    def move(self, mcts_state: int, move: int, player: int) -> Tuple[int, bool]: ...

    @abstractmethod
    def render(self, mcts_state: int) -> str: ...


class _DeviceGame(BaseGame):
    """Shared CUDA plumbing: boards <-> device, batched rule kernels."""

    game_kind = -1
    board_words = 0  # uint64 words per board
    n = 0
    k = 0
    player_black = 1
    player_white = 0

    # -- encoding hooks (implemented per game) -----------------------------------------------
    def state_to_words(self, state: int) -> List[int]:
        raise NotImplementedError

    def words_to_state(self, words: Sequence[int]) -> int:
        raise NotImplementedError

    def boards_from_states(self, states: Sequence[int]) -> np.ndarray:
        """uint64 [L, board_words] array in the device layout of include/caro_b200.h."""
        out = np.zeros((len(states), self.board_words), dtype=np.uint64)
        for i, s in enumerate(states):
            out[i] = np.array(self.state_to_words(int(s)), dtype=np.uint64)
        return out

    def states_from_boards(self, boards: np.ndarray) -> List[int]:
        return [self.words_to_state([int(w) for w in row]) for row in np.asarray(boards).reshape(-1, self.board_words)]

    # -- batched device calls ------------------------------------------------------------------
    def _torch(self):
        import torch
        _cabi.require_cuda()
        return torch

    def _stream(self, torch):
        return torch.cuda.current_stream().cuda_stream

    def apply_batch(self, states: Sequence[int], actions: Sequence[int], players: Sequence[int]):
        """game.move for many (state, action, player) triples on the GPU.
        Returns (new_states, won uint8[L], draw uint8[L])."""
        torch = self._torch()
        count = len(states)
        d_boards = torch.from_numpy(self.boards_from_states(states).view(np.int64)).cuda()
        d_act = torch.tensor(list(actions), dtype=torch.int32, device="cuda")
        d_pl = torch.tensor(list(players), dtype=torch.uint8, device="cuda")
        d_out = torch.empty_like(d_boards)
        d_won = torch.empty(count, dtype=torch.uint8, device="cuda")
        d_draw = torch.empty(count, dtype=torch.uint8, device="cuda")
        if count:  # an empty torch tensor has a null data pointer, which the C ABI rejects
            _cabi.check(_cabi.lib().caro_boards_apply(self.game_kind, self.n, self.k, d_boards.data_ptr(), d_act.data_ptr(),
                                                      d_pl.data_ptr(), count, d_out.data_ptr(), d_won.data_ptr(),
                                                      d_draw.data_ptr(), self._stream(torch)))
        new_states = self.states_from_boards(d_out.cpu().numpy().view(np.uint64))
        return new_states, d_won.cpu().numpy(), d_draw.cpu().numpy()

    def legal_masks(self, states: Sequence[int]) -> np.ndarray:
        """bool [L, A]: True where the action is legal."""
        torch = self._torch()
        count = len(states)
        words = (self.action_space + 31) // 32
        d_boards = torch.from_numpy(self.boards_from_states(states).view(np.int64)).cuda()
        d_mask = torch.empty((count, words), dtype=torch.int32, device="cuda")
        if count:
            _cabi.check(_cabi.lib().caro_boards_legal_mask(self.game_kind, self.n, self.k, d_boards.data_ptr(), count,
                                                           d_mask.data_ptr(), self._stream(torch)))
        m = d_mask.cpu().numpy().view(np.uint32)
        bits = (m[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1
        return bits.reshape(count, words * 32)[:, :self.action_space].astype(bool)

    def planes_device(self, d_boards, d_who, count: int):
        """float32 CUDA tensor [count, 2, H, W] from device boards (int64 view) + uint8 movers."""
        torch = self._torch()
        out = torch.empty((count,) + tuple(self.obs_shape), dtype=torch.float32, device="cuda")
        if count:
            _cabi.check(_cabi.lib().caro_boards_encode_planes(self.game_kind, self.n, self.k, d_boards.data_ptr(),
                                                              d_who.data_ptr(), count, out.data_ptr(), self._stream(torch)))
        return out

    # -- BaseGame members ------------------------------------------------------------------------
    def possible_moves(self, mcts_state: int) -> List[int]:
        assert isinstance(mcts_state, int)
        return [int(a) for a in np.nonzero(self.legal_masks([mcts_state])[0])[0]]

    def invalid_moves(self, mcts_state: int) -> List[int]:
        return [int(a) for a in np.nonzero(~self.legal_masks([mcts_state])[0])[0]]

    def states_to_training_batch(self, state_ints: Sequence[int], who_moves_lists: Sequence[int]) -> np.ndarray:
        torch = self._torch()
        d_boards = torch.from_numpy(self.boards_from_states(state_ints).view(np.int64)).cuda()
        d_who = torch.tensor(list(who_moves_lists), dtype=torch.uint8, device="cuda")
        return self.planes_device(d_boards, d_who, len(state_ints)).cpu().numpy()


class ConnectFour(_DeviceGame):
    """lib/game/connect_four/connect_four.py:8-281 (6x7, 1 = black 'X', 0 = white 'O')."""

    game_kind = _cabi.GAME_CONNECT4
    board_words = 2

    def __init__(self):
        super().__init__()
        self.game_rows = 6
        self.game_cols = 7
        self.bits_in_len = 3
        self.player_black = 1
        self.player_white = 0
        self.count_to_win = 4

    @property
    def initial_state(self) -> int:
        return 0b110110110110110110110  # seven 3-bit free counters = 6 (connect_four.py:65-72)

    @property
    def obs_shape(self) -> Tuple[int, int, int]:
        return (2, self.game_rows, self.game_cols)

    @property
    def action_space(self) -> int:
        return self.game_cols

    # state int (connect_four.py:16-55): cell (col,row) at bit 62-(6*col+row), free count of
    # column c at bits [18-3c, 21-3c)  <->  device board {mask, black}, bit 7*col+row
    def state_to_words(self, state: int) -> List[int]:
        mask = black = 0
        for c in range(7):
            height = 6 - ((state >> (18 - 3 * c)) & 7)
            for r in range(max(height, 0)):
                bit = 1 << (7 * c + r)
                mask |= bit
                if (state >> (62 - (6 * c + r))) & 1:
                    black |= bit
        return [mask, black]

    def words_to_state(self, words: Sequence[int]) -> int:
        mask, black = int(words[0]), int(words[1])
        state = 0
        for c in range(7):
            height = bin((mask >> (7 * c)) & 0x3F).count("1")
            state |= (6 - height) << (18 - 3 * c)
            for r in range(height):
                if (black >> (7 * c + r)) & 1:
                    state |= 1 << (62 - (6 * c + r))
        return state

    def encode_lists(self, field_lists) -> int:
        """connect_four.py:108-127."""
        assert isinstance(field_lists, list)
        assert len(field_lists) == self.game_cols
        mask = black = 0
        for c, col in enumerate(field_lists):
            for r, tok in enumerate(col):
                mask |= 1 << (7 * c + r)
                if tok:
                    black |= 1 << (7 * c + r)
        return self.words_to_state([mask, black])

    def decode_binary(self, state_int: int):
        """connect_four.py:129-147."""
        assert isinstance(state_int, int)
        mask, black = self.state_to_words(state_int)
        return [[(black >> (7 * c + r)) & 1 for r in range(bin((mask >> (7 * c)) & 0x3F).count("1"))] for c in range(7)]

    def move(self, state_int: int, col: int, player: int) -> Tuple[int, bool]:
        """connect_four.py:241-265 (assertions included)."""
        assert isinstance(state_int, int)
        assert isinstance(col, (int, np.integer))
        assert 0 <= col < self.game_cols
        assert player == self.player_black or player == self.player_white
        assert ((state_int >> (18 - 3 * int(col))) & 7) > 0  # column not full (connect_four.py:255)
        new_states, won, _ = self.apply_batch([state_int], [int(col)], [int(player)])
        return new_states[0], bool(won[0])

    def render(self, state_int: int) -> str:
        """connect_four.py:267-281."""
        cols = self.decode_binary(state_int)
        grid = [[" "] * self.game_cols for _ in range(self.game_rows)]
        for c, col in enumerate(cols):
            for r, tok in enumerate(col):
                grid[self.game_rows - 1 - r][c] = "X" if tok else "O"
        return "0123456\n-------\n" + "\n".join("".join(row) for row in grid) + "\n-------\n0123456"


class TicTacToe(_DeviceGame):
    """lib/game/tictactoe/tictactoe.py:10-259: the m,n,k family with m == n (3,3,3 by default;
    15,15,5 is Caro/Gomoku)."""

    game_kind = _cabi.GAME_MNK
    board_words = 8

    def __init__(self, n: int = 3, k_to_win: int = 3):
        super().__init__()
        assert 2 <= k_to_win <= n <= 15, "device boards hold n <= 15"
        self.board_len = n
        self.k_to_win = k_to_win
        self.n = n
        self.k = k_to_win
        self.player_black = 1
        self.player_white = 0
        self.empty = 2

    @property
    def initial_state(self) -> int:
        return int("2" * self.board_len ** 2)

    @property
    def obs_shape(self) -> Tuple[int, ...]:
        return (2, self.board_len, self.board_len)

    @property
    def action_space(self) -> int:
        return self.board_len ** 2

    def _pad_mcts_state(self, mcts_state_str: str) -> str:
        return mcts_state_str.rjust(self.board_len ** 2, "0")  # tictactoe.py:89-100

    # state int (tictactoe.py:102-135): n*n decimal digits, cell 0 first; 0 white, 1 black, 2 empty
    # <-> device board {w[4], b[4]}, bit = cell index
    def state_to_words(self, state: int) -> List[int]:
        text = self._pad_mcts_state(str(state))
        w = b = 0
        for i, ch in enumerate(text):
            if ch == "0":
                w |= 1 << i
            elif ch == "1":
                b |= 1 << i
        m = (1 << 64) - 1
        return [(w >> (64 * j)) & m for j in range(4)] + [(b >> (64 * j)) & m for j in range(4)]

    def words_to_state(self, words: Sequence[int]) -> int:
        w = sum(int(words[j]) << (64 * j) for j in range(4))
        b = sum(int(words[4 + j]) << (64 * j) for j in range(4))
        digits = ["0" if (w >> i) & 1 else "1" if (b >> i) & 1 else "2" for i in range(self.board_len ** 2)]
        return int("".join(digits))

    def encode_game_state(self, state_list) -> int:
        return int("".join(str(v) for row in state_list for v in row))  # tictactoe.py:102-114

    def convert_mcts_state_to_list_state(self, mcts_state: int):
        text = self._pad_mcts_state(str(mcts_state))
        n = self.board_len
        return [[int(ch) for ch in text[r * n:(r + 1) * n]] for r in range(n)]  # tictactoe.py:116-135

    def move(self, mcts_state: int, move: int, player: int) -> Tuple[int, bool]:
        """tictactoe.py:210-235 (no emptiness check, like the reference)."""
        assert player == self.player_white or player == self.player_black
        assert 0 <= move < self.action_space
        new_states, won, _ = self.apply_batch([mcts_state], [int(move)], [int(player)])
        return new_states[0], bool(won[0])

    def render(self, mcts_state: int) -> str:
        """tictactoe.py:237-259."""
        n = self.board_len
        sym = {self.player_white: "❌", self.player_black: "⭕"}
        rows = []
        for r, row in enumerate(self.convert_mcts_state_to_list_state(mcts_state)):
            rows.append("|" + "|".join(str(r * n + c) if v == self.empty else sym[v] for c, v in enumerate(row)) + "|")
        return "\n".join(rows)


class Caro(TicTacToe):
    """Caro (Vietnamese gomoku) on an n x n board: k in a row wins unless the run is blocked at both ends.

    Everything but the win test is TicTacToe(n, k)'s: state integers, planes, actions, render and the draw rule.  A
    move wins when, in one of the four directions, the maximal run of the mover's stones through it reaches k
    (overlines count) and does not have an opponent stone just past both of its ends; the board edge never blocks.
    A blocked run stays on the board and the game goes on (rule in csrc/rules.cuh, MnkRules::blocked_ends)."""

    game_kind = _cabi.GAME_CARO

    def __init__(self, n: int = 15, k_to_win: int = 5):
        super().__init__(n, k_to_win)


def get_game(game_type: str):
    """lib/game/game_provider.py:15-22: '0' -> ConnectFour, '2' -> Caro(15, 5), anything else -> TicTacToe()."""
    if game_type == "0":
        return ConnectFour()
    if game_type == "2":
        return Caro()
    return TicTacToe()
