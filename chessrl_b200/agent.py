"""Agent: drop-in for the reference's in-process agent (agent.py:12-98): owns a ChessModel, predicts through the
CUDA engine, trains with the PyTorch training step (chessrl_b200/training.py), saves / loads weights."""

from __future__ import annotations

from .agentdistributed import AgentDistributed
from .dataset import DatasetGame
from .model import ChessModel


class Agent(AgentDistributed):

    def __init__(self, color, weights=None):
        super().__init__(color, endpoint=None, num_threads=1, model=ChessModel(compile_model=True, weights=weights))
        self.model = self._model

    def best_move(self, game, real_game=False, max_iters=900, verbose=False, ai_move=False):
        # the reference's Agent builds the abstract Tree here and returns None (agent.py:45-47, SURVEY.md A13);
        # the working search of AgentDistributed is used instead
        return super().best_move(game, real_game=real_game, max_iters=max_iters, ai_move=ai_move, verbose=verbose)

    def train(self, dataset: DatasetGame, epochs=1, logdir=None, batch_size=1, validation_split=0, targets=None):
        """Trains the model on recorded games (agent.py:64-89): one sample per ply, targets = the move played and the
        white-point-of-view result, or with targets=training.SearchTargets(...) the search targets of DESIGN.md 3.8
        for games that carry root scores."""
        if len(dataset) <= 0:
            return
        from . import training
        training.train(self.model, dataset, epochs=epochs, logdir=logdir, batch_size=batch_size,
                       validation_split=validation_split, targets=targets)

    def save(self, path):
        self.model.save_weights(path)

    def load(self, path):
        self.model.load_weights(path)

    def get_copy(self):
        return self
