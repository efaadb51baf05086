"""Drop-in for the reference's ``lib/play_session.py:Session`` (human vs bot, one move at a time)."""
from __future__ import annotations

import numpy as np

from . import mcts, model

BOT_MCTS_SEARCHES = 40   # config.py:22
BOT_MCTS_BATCH_SIZE = 8  # config.py:23


class Session:
    def __init__(self, game, model_file, player_moves_first, solver: bool = False, gumbel: bool = False):
        """``solver`` (extension, default off): the bot's search proves wins, losses and draws and never plays a move it
        has proven to lose while another is left.
        ``gumbel`` (extension, default off): the bot searches its root by Gumbel sequential halving and plays the best
        survivor."""
        self.game = game
        self.BOT_PLAYER = game.player_black
        self.USER_PLAYER = game.player_white
        self.model_file = model_file
        self.model = model.load_checkpoint(model_file, game)  # any depth and width the file holds
        self.model.eval()
        self.state = game.initial_state
        self.value = None
        self.player_moves_first = player_moves_first
        self.moves = []
        self.mcts_store = mcts.MCTS(game, solver=solver, gumbel=gumbel)  # one tree for the whole session (play_session.py:20)

    def move_player(self, move: int) -> bool:
        self.moves.append(move)
        self.state, won = self.game.move(self.state, move, self.USER_PLAYER)
        return won

    def move_bot(self) -> bool:
        """play_session.py:28-36: 40 x 8 searches, tau = 0."""
        self.mcts_store.search_batch(BOT_MCTS_SEARCHES, BOT_MCTS_BATCH_SIZE, self.state, self.BOT_PLAYER, self.model)
        probs, values = self.mcts_store.get_policy_value(self.state, tau=0)
        action = int(np.random.choice(self.game.action_space, p=probs))
        self.value = values[action]
        self.moves.append(action)
        self.state, won = self.game.move(self.state, action, self.BOT_PLAYER)
        return won

    def is_valid_move(self, move: int) -> bool:
        return move in self.game.possible_moves(self.state)

    def is_draw(self) -> bool:
        return len(self.game.possible_moves(self.state)) == 0

    def render(self) -> str:
        board = self.game.render(self.state)
        extra = ""
        if self.value is not None:
            extra = "Position evaluation: %.2f\n" % float(self.value)
        return extra + "<pre>%s</pre>" % board
