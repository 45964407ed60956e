"""Game: drop-in for the reference's game.Game (game.py:11-112) whose chess rules run in the CUDA engine.

Kept surface: Game(board=None, player_color=True, date=None), NULL_MOVE / WHITE / BLACK, move(uci) -> bool,
get_legal_moves(final_states=False), get_history(), get_fen() (piece placement only), set_fen(), turn,
get_copy(), reset(), free(), get_result() -> 1 / 0 / -1 / None, len(game) = plies, and game.board exposing
.move_stack (items str() to UCI) and .turn, which mctree / netencoder / treeviewer reach into
(mctree.py:186-188, 308; netencoder.py:83).  plot_board (debug drawing) is out of scope.

A game is (start record, list of moves).  Every query replays that list on the device
(crl_game_replay_host) so legality, Game.get_result -- fifty-move claim, fivefold repetition, insufficient
material, mate -- and the history needed by netencoder come from the same kernels the lockstep path uses.
"""

from __future__ import annotations

from datetime import datetime

import numpy as np

from . import boards as B
from . import runtime


class _MoveView(str):
    """An item of board.move_stack: str(m) and m.uci() give the UCI string (chess.Move surface that is used)."""

    def uci(self):
        return str(self)


class BoardView:
    """The slice of chess.Board that the reference's modules touch on game.board."""

    def __init__(self, game):
        self._game = game

    @property
    def move_stack(self):
        return [_MoveView(m) for m in self._game._moves]

    @property
    def turn(self):
        return self._game.turn

    def board_fen(self):
        return B.board_fen_from_record(self._game._record)

    def fen(self):
        return B.fen_from_record(self._game._record, self._game._ep_legal())

    def set_board_fen(self, fen):
        self._game.set_fen(fen)

    def copy(self, stack=True):
        return self._game.get_copy().board

    def reset(self):
        self._game.reset()

    def __len__(self):
        return len(self._game._moves)


def _from_foreign_board(board):
    """Accepts a python-chess-like Board (copy / pop / fen / move_stack) or a FEN string."""
    if isinstance(board, str):
        return B.record_from_fen(board), []
    if isinstance(board, BoardView):
        g = board._game
        return g._start.copy(), list(g._moves)
    b = board.copy()
    moves = [m.uci() for m in b.move_stack]
    for _ in moves:
        b.pop()
    return B.record_from_fen(b.fen()), moves


class Game(object):

    NULL_MOVE = B.NULL_MOVE
    WHITE = True
    BLACK = False
    # the alpha-beta root scores of every ply (DESIGN.md 3.8): one list of ints per move, the scores of that ply's legal
    # moves in generation order; None for a game recorded without them (copies and new games)
    search_scores = None

    def __init__(self, board=None, player_color=True, date=None):
        self.player_color = player_color
        self.date = date if date is not None else datetime.now().strftime("%d/%m/%Y %H:%M:%S")
        if board is None:
            self._start, moves = B.record_from_fen(), []
        else:
            self._start, moves = _from_foreign_board(board)
        self._moves = []
        self._records = [self._start.copy()]       # record after every ply (history planes need the last 9)
        self._sync(extra=moves)
        self.board = BoardView(self)

    # ---- device round trip --------------------------------------------------------------------------------
    def _sync(self, extra=()):
        """Replays moves (+ candidate moves) on the device in ONE round trip; keeps the accepted ones."""
        eng = runtime.scalar_engine()
        extra = list(extra)
        cand = list(self._moves) + extra
        words = [B.uci_to_move(m) for m in cand]
        n_old = len(self._moves)
        if len(extra) > 1:
            # bulk load: the kernel hands back the record after every accepted ply (crl_game_replay_records_host)
            r = eng.game_replay(self._start, words, records=True)
            self._moves = [m for m, ok in zip(cand, r["accepted"]) if ok]
            self._accepted = r["accepted"][n_old:]        # of `extra` (DatasetGame.loads aligns scores with it)
            self._records = [rec.copy() for rec in r["records"]]
            played = len(self._moves) > n_old
        else:
            r = eng.game_replay(self._start, words)
            played = bool(extra) and bool(r["accepted"][n_old])
            if played:
                self._moves.append(extra[0])
                self._records.append(r["record"].copy())
        self._record = r["record"].copy()
        self._legal = [B.move_to_uci(m) for m in r["legal"]]
        self._result = r["result"]
        return played

    def _ep_legal(self):
        ep = B.meta_fields(self._record[8])["ep"]
        if ep < 0:
            return False
        files = "abcdefgh"
        name = files[ep & 7] + str((ep >> 3) + 1)
        return any(m[2:4] == name and m[0] != m[2] and self._is_pawn(m[:2]) for m in self._legal)

    def _is_pawn(self, sq_name):
        sq = "abcdefgh".index(sq_name[0]) + 8 * (int(sq_name[1]) - 1)
        return bool(int(self._record[0]) >> sq & 1)

    # ---- reference surface --------------------------------------------------------------------------------
    def move(self, movement):
        """Plays a move given in UCI notation if it is legal.  Returns whether it was played (game.py:28-41)."""
        if movement not in self._legal:
            return False
        return self._sync(extra=[movement])

    def get_legal_moves(self, final_states=False):
        moves = list(self._legal)
        if final_states:
            states = []
            for m in moves:
                g = self.get_copy()
                g.move(m)
                states.append(g)
            return moves, states
        return moves

    def get_history(self):
        h = {"moves": list(self._moves), "result": self.get_result(), "player_color": self.player_color,
             "date": self.date}
        if self.search_scores is not None:
            h["scores"] = [list(s) for s in self.search_scores]
        return h

    def get_fen(self):
        return B.board_fen_from_record(self._record)

    def set_fen(self, fen):
        """Board.set_board_fen: replaces the piece placement only (game.py:71-72)."""
        bbs = B.board_fen_to_bitboards(fen)
        rec = self._record.copy()
        for k in range(8):
            rec[k] = bbs[k]
        m = B.meta_fields(rec[8])
        rec[8] = B.pack_meta(m["turn"], m["castle"], m["ep"], m["halfmove"], m["fullmove"])
        self._start = rec
        self._moves = []
        self._records = [rec.copy()]
        self._sync()

    @property
    def turn(self):
        return bool(int(self._record[8]) & 1)

    def get_copy(self):
        g = Game.__new__(Game)
        g.player_color = True                      # Game(board=self.board.copy()) takes the defaults (game.py:79-80)
        g.date = datetime.now().strftime("%d/%m/%Y %H:%M:%S")
        g._start = self._start.copy()
        g._moves = list(self._moves)
        g._records = [r.copy() for r in self._records]
        g._record = self._record.copy()
        g._legal = list(self._legal)
        g._result = self._result
        g.board = BoardView(g)
        return g

    def reset(self):
        self._start = B.record_from_fen()
        self._moves = []
        self._records = [self._start.copy()]
        self._sync()

    def free(self):
        pass

    def get_result(self):
        """Result for the white pieces: 1 / -1 / 0, None while the game is running (game.py:92-109)."""
        return self._result

    def __len__(self):
        return len(self._moves)

    # ---- used by netencoder -------------------------------------------------------------------------------
    def history_records(self):
        """Current record followed by up to 8 previous ones (most recent first)."""
        return self._records[::-1][:9]
