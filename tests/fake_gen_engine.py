"""TEST-ONLY stand-ins that let chessrl_b200/gen_data.py run in the GPU-less CPU suite:
- FakeGenEngine: tests/fake_engine.FakeEngine with games_ab_pick from the g++ build of the pick
  (tests/hostsim/ab_pick.py, the kernels' code): active, unfinished, masked lanes, the ply of each lane's game;
- FakeScalarEngine: Engine.game_replay on the oracle, so that Game / DatasetGame (a device replay per game) work;
- install(): both behind chessrl_b200.engine.Engine and chessrl_b200.runtime.scalar_engine."""
import numpy as np

import chessrl_oracle as O
from chessrl_b200 import boards as B
from fake_engine import FakeEngine
from hostsim import ab_pick as HP


def lane_record(game):
    """The device record of an oracle game: its position with meta_ply = len(move_stack)."""
    return HP.with_ply(B.record_from_fen(game.board.fen()), len(game.board.move_stack))


class FakeGenEngine(FakeEngine):
    def games_ab_pick(self, depth, qdepth, margin, pick_plies, salt, mask=None):
        self._count("games_ab_pick")
        salt = np.asarray(salt, dtype=np.uint64)
        assert salt.shape == (self.max_games,)
        moves = np.full(self.max_games, B.MOVE_NONE, dtype=np.uint16)
        scores = np.zeros(self.max_games, dtype=np.int32)
        nodes = np.zeros(self.max_games, dtype=np.int64)
        for g in range(self.max_games):
            if self._running(g) and (mask is None or mask[g]):
                moves[g], scores[g], nodes[g] = HP.pick(lane_record(self.games[g]), depth, qdepth, margin, pick_plies,
                                                        int(salt[g]))
        return moves, scores, nodes


class FakeScalarEngine:
    def game_replay(self, start_record, moves, records=False):
        g = O.OGame(board=O.chess.Board(B.fen_from_record(np.asarray(start_record, dtype=np.uint64))))
        accepted, recs = [], [np.asarray(start_record, dtype=np.uint64).copy()]
        for m in moves:
            ok = m != B.MOVE_NONE and g.move(B.move_to_uci(int(m)))
            accepted.append(bool(ok))
            if ok:
                recs.append(lane_record(g))
        out = {"legal": np.array([B.uci_to_move(m) for m in g.get_legal_moves()], dtype=np.uint16),
               "result": g.get_result(), "accepted": np.array(accepted, dtype=bool), "record": recs[-1].copy()}
        if records:
            out["records"] = np.stack(recs)
        return out


def install(monkeypatch_setattr):
    """Puts the fakes behind the package: monkeypatch_setattr(obj, name, value) (pytest's monkeypatch.setattr, or
    setattr in a worker process)."""
    from chessrl_b200 import engine, runtime
    scalar = FakeScalarEngine()
    monkeypatch_setattr(engine, "Engine", lambda max_games=1, **kw: FakeGenEngine(max_games))
    monkeypatch_setattr(runtime, "scalar_engine", lambda *a, **kw: scalar)
