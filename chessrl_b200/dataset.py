"""DatasetGame: the reference's container of recorded games and its JSON format (dataset.py:6-97)

    [{"moves": [uci, ...], "result": 1 | 0 | -1 | null, "player_color": bool, "date": "dd/mm/YYYY HH:MM:SS"}, ...]

A game may also carry "scores" (gen_data --scores, DESIGN.md 3.8): one list of ints per move, the alpha-beta root scores of
that ply's legal moves in generation order.  It is written only for games that have it, so a file without scores is the
reference's format byte for byte, and the reference's loader, which reads the four keys above, ignores it.

Same surface -- DatasetGame(games=None), augment_game, load, loads, save (appends to what the file holds), append,
str(), +, len, indexing / slicing -- with the games replayed in bulk on the device when a file is read.
"""

from __future__ import annotations

import json

from . import game as _game


def _record(g):
    return g.get_history()


def _check_scores(j, moves, scores):
    """The "scores" field of game j: one list of ints per move, else ValueError naming the game."""
    if not isinstance(scores, list) or len(scores) != len(moves):
        raise ValueError("game %d: \"scores\" must be a list with one entry per move (%d moves, got %s)"
                         % (j, len(moves), len(scores) if isinstance(scores, list) else type(scores).__name__))
    for i, s in enumerate(scores):
        if not isinstance(s, list) or not all(isinstance(v, int) and not isinstance(v, bool) for v in s):
            raise ValueError("game %d, ply %d: the scores must be a list of ints" % (j, i))


class DatasetGame(object):

    def __init__(self, games=None):
        self.games = [] if games is None else games

    # ---- container protocol -------------------------------------------------------------------------------
    def __len__(self):
        return len(self.games)

    def __getitem__(self, key):
        return self.games[key]

    def __str__(self):
        return json.dumps(list(map(_record, self.games)))

    def append(self, other):
        """A Game is added, another DatasetGame is concatenated; anything else is ignored (dataset.py:73-78)."""
        if isinstance(other, DatasetGame):
            self.games += other.games
        elif isinstance(other, _game.Game):
            self.games.append(other)

    def __add__(self, other):
        self.append(other)
        return self

    __iadd__ = __add__

    # ---- (de)serialisation --------------------------------------------------------------------------------
    def loads(self, string):
        """Games with at least one move are rebuilt from their move lists (dataset.py:50-58): one bulk replay on the
        device per game (Game._sync) instead of one Game.move call per ply."""
        for j, entry in enumerate(json.loads(string)):
            if not entry["moves"]:
                continue
            scores = entry.get("scores")
            if scores is not None:
                _check_scores(j, entry["moves"], scores)
            g = _game.Game(player_color=entry["player_color"], date=entry["date"])
            g._sync(extra=entry["moves"])
            if scores is not None:                 # kept for the moves the replay accepted
                accepted = g._accepted if len(entry["moves"]) > 1 else [len(g._moves) == 1]
                g.search_scores = [s for s, ok in zip(scores, accepted) if ok]
            self.games.append(g)

    def load(self, path):
        with open(path, "r") as f:
            self.loads(f.read())

    def save(self, path):
        """Writes the file's previous content followed by this dataset's games (dataset.py:60-71)."""
        before = DatasetGame()
        try:
            before.load(path)
        except FileNotFoundError:
            pass
        with open(path, "w") as f:
            json.dump([_record(g) for g in before.games + self.games], f)

    # ---- training samples ---------------------------------------------------------------------------------
    def augment_game(self, game_base):
        """One sample per ply: {'game': position before the move, 'next_move': the move played, 'result': the game's
        final result} (dataset.py:21-43).  The first sample's Game carries the stored colour and date, the later ones
        are copies (which take Game's defaults, as in the reference)."""
        h = game_base.get_history()
        position = _game.Game(date=h["date"], player_color=h["player_color"])
        samples = []
        for move in h["moves"]:
            samples.append({"game": position, "next_move": move, "result": h["result"]})
            position = position.get_copy()
            position.move(move)
        return samples
