"""TEST-ONLY: tests/fake_engine.FakeEngine with two network slots, each holding a hash evaluator, and per-lane players
(chessrl_b200.engine.Engine.games_set_players), so that the host logic of the match driver (chessrl_b200/arena.py)
runs in the GPU-less CPU suite.  A lane's search uses the oracle agent of the slot that moves at its root, as the
engine's routing does."""
import numpy as np

import chessrl_oracle as O
from chessrl_b200 import boards as B
from chessrl_b200._lib import EVAL_HASH
from fake_engine import FakeEngine


class FakeArenaEngine(FakeEngine):
    def __init__(self, max_games):
        super().__init__(max_games)
        self.slot_agents = [None, None]
        self.players = np.zeros((2, self.max_games), dtype=np.uint8)     # [white, black] slot of every lane
        self.lane_agents = [None] * self.max_games
        self.row_bounds = []

    def set_evaluator(self, kind, seed=0, policy_bits=24, slot=0):
        assert kind == EVAL_HASH, "the fake engine has hash evaluators only"
        self.slot_agents[slot] = O.OAgent(O.hash_evaluator(seed, policy_bits))

    def load_weights(self, tensors, precision="bf16", calibration=None, slot=0):
        raise AssertionError("the fake engine has hash evaluators only")

    def set_row_bound(self, max_running_games=0):
        self.row_bounds.append(int(max_running_games))

    def games_set_players(self, white, black, first=0):
        self._count("games_set_players")
        w, b = np.atleast_1d(np.asarray(white, dtype=np.uint8)), np.atleast_1d(np.asarray(black, dtype=np.uint8))
        self.players[0, first:first + len(w)] = w
        self.players[1, first:first + len(b)] = b

    def mcts_begin_move(self):
        self._count("mcts_begin_move")
        super().mcts_begin_move()
        for g in range(self.max_games):
            if self.trees[g] is not None:
                side = 0 if self.games[g].board.turn else 1
                self.lane_agents[g] = self.slot_agents[self.players[side, g]]
                assert self.lane_agents[g] is not None, "lane %d: its slot has no evaluator" % g

    def mcts_simulate(self, n_sims, inflight=1):
        for g, t in enumerate(self.trees):
            if t is not None:
                for _ in range(n_sims):
                    t.explore_tree(self.lane_agents[g])
                    self.n_sims += 1

    def root_stats(self, want=("visits",)):
        out = super().root_stats(want)
        out["moves"] = np.full((self.max_games, B.MAX_MOVES), B.MOVE_NONE, dtype=np.uint16)
        for g, t in enumerate(self.trees):
            if t is not None:
                ply = len(t.root.state.board.move_stack)
                for k, c in enumerate(t.root.children):
                    out["moves"][g, k] = B.uci_to_move(c.state.board.move_stack[ply].uci())
        return out
