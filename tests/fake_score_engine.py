"""TEST-ONLY: tests/fake_gen_engine.FakeGenEngine with Engine.games_ab_root_scores, so that `gen_data --scores` runs in the
GPU-less CPU suite.  The picks still come from the g++ build of the kernels' code; the root scores of every searched lane
come from the oracle's search (oracle/ab_oracle.py search: the root children's values in generation order)."""
import numpy as np

import ab_oracle as A
import fake_gen_engine
from chessrl_b200 import boards as B
from chessrl_b200._lib import CRL_ESTATE, CrlError


class FakeScoreEngine(fake_gen_engine.FakeGenEngine):
    scores = None

    def games_ab_pick(self, depth, qdepth, margin, pick_plies, salt, mask=None):
        out = super().games_ab_pick(depth, qdepth, margin, pick_plies, salt, mask)
        self.scores = np.zeros((self.max_games, B.MAX_MOVES), dtype=np.int32)
        self.counts = np.full(self.max_games, -1, dtype=np.int32)
        for g in range(self.max_games):
            if self._running(g) and (mask is None or mask[g]):
                vals = A.search(self.games[g].board, depth, qdepth)[2]
                self.scores[g, :len(vals)] = vals
                self.counts[g] = len(vals)
        return out

    def games_ab_root_scores(self):
        self._count("games_ab_root_scores")
        if self.scores is None:
            raise CrlError(CRL_ESTATE, "no alpha-beta call has run on this engine")
        return self.scores.copy(), self.counts.copy()


def install(monkeypatch_setattr):
    """fake_gen_engine.install with FakeScoreEngine behind chessrl_b200.engine.Engine."""
    from chessrl_b200 import engine
    fake_gen_engine.install(monkeypatch_setattr)
    monkeypatch_setattr(engine, "Engine", lambda max_games=1, **kw: FakeScoreEngine(max_games))
