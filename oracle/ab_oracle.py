"""ORACLE / TEST INFRASTRUCTURE ONLY -- never imported by the product path (`chessrl_b200/`).

The fixed-depth alpha-beta opponent (DESIGN.md 3.6), restated from its definition on the python-chess restatement in
oracle/pychess_compat/chess.  It is written from the definition, not from chessrl_b200/csrc/ab_search.cuh: the
evaluation walks the pieces one by one with the table below, and the search is a plain alpha-beta over the moves in
generation order (the kernels order captures first), or a plain minimax with no pruning at all.

    s(p)      centipawns for the side to move: the sum over its pieces minus the sum over the opponent's
    T(p, h)   mate -(32000 - h) for the side to move; stalemate, insufficient material, the fifty-move claim 0
              (no repetition inside the search)
    V(p,d,h)  T if terminal; Q(p, q, h) if d = 0; else max over legal m of -V(p.m, d-1, h+1)
    Q(p,k,h)  T if terminal; s(p) if k = 0; in check: max over legal m of -Q(p.m, k-1, h+1);
              else max(s(p), max over the captures (en passant included) and queen promotions m of -Q(p.m, k-1, h+1))
    root      the first legal move in generation order with the largest -V(root.m, D-1, 1); the score is that value
"""

from __future__ import annotations

import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_COMPAT = os.path.join(_HERE, "pychess_compat")
if _COMPAT not in sys.path:
    sys.path.insert(0, _COMPAT)

import chess  # noqa: E402  (the restatement, not the PyPI package)

MATE = 32000
INF = 10 ** 9

# the evaluation table (centipawns); tests change one entry to show that the comparison notices
WEIGHTS = {
    "pawn": 100, "pawn_rank": 5,                  # 100 + 5 (r - 1)
    "knight": 310, "knight_centre": 10,           # 310 + 10 (3 - cd)
    "bishop": 330, "bishop_centre": 5, "bishop_pair": 30,
    "rook": 500, "rook_seventh": 20,              # +20 on r = 6
    "queen": 900, "queen_centre": 2,
    "king_shelter": 10, "king_centre": 5,         # -10 min(r, 2) while the other side has a queen, else 5 (3 - cd)
}


def centre_distance(sq, colour):
    """cd = max(|2f - 7|, |2r - 7|) // 2 with r the rank seen from `colour`."""
    f = chess.square_file(sq)
    r = relative_rank(sq, colour)
    return max(abs(2 * f - 7), abs(2 * r - 7)) // 2


def relative_rank(sq, colour):
    r = chess.square_rank(sq)
    return r if colour == chess.WHITE else 7 - r


def piece_value(board, sq, w=WEIGHTS):
    pt = board.piece_type_at(sq)
    colour = bool(board.occupied_co[chess.WHITE] & (1 << sq))
    r = relative_rank(sq, colour)
    cd = centre_distance(sq, colour)
    if pt == chess.PAWN:
        return w["pawn"] + w["pawn_rank"] * (r - 1)
    if pt == chess.KNIGHT:
        return w["knight"] + w["knight_centre"] * (3 - cd)
    if pt == chess.BISHOP:
        return w["bishop"] + w["bishop_centre"] * (3 - cd)
    if pt == chess.ROOK:
        return w["rook"] + (w["rook_seventh"] if r == 6 else 0)
    if pt == chess.QUEEN:
        return w["queen"] + w["queen_centre"] * (3 - cd)
    if board.pieces_mask(chess.QUEEN, not colour):
        return -w["king_shelter"] * min(r, 2)
    return w["king_centre"] * (3 - cd)


def side_total(board, colour, w=WEIGHTS):
    total = 0
    for sq in chess.SQUARES:
        if board.occupied_co[colour] & (1 << sq):
            total += piece_value(board, sq, w)
    if chess.popcount(board.pieces_mask(chess.BISHOP, colour)) >= 2:
        total += w["bishop_pair"]
    return total


def evaluate(board, w=WEIGHTS):
    """s(p): centipawns from the point of view of the side to move."""
    return side_total(board, board.turn, w) - side_total(board, not board.turn, w)


def terminal(board, legal, h):
    """T(p, h), or None while the game goes on."""
    if board.halfmove_clock >= 100 and legal:
        return 0                                             # the fifty-move claim
    if not legal:
        return -(MATE - h) if board.is_check() else 0       # mate / stalemate
    if board.is_insufficient_material():
        return 0
    return None


def in_quiescence_set(board, m):
    """C(p): a capture (en passant included) or a promotion to a queen."""
    return bool(board.occupied_co[not board.turn] & (1 << m.to_square)) or board.is_en_passant(m) or \
        m.promotion == chess.QUEEN


class Search:
    """V / Q by plain alpha-beta in generation order (prune=True) or by minimax (prune=False).
    `nodes` counts the positions visited (the kernels order moves differently, so their counts differ)."""

    def __init__(self, qdepth, w=WEIGHTS, prune=True):
        self.q = int(qdepth)
        self.w = w
        self.prune = prune
        self.nodes = 0

    def _children(self, board, moves, h, alpha, beta, best, fn):
        for m in moves:
            board.push(m)
            v = -fn(board, h + 1, -beta, -alpha)
            board.pop()
            if v > best:
                best = v
            if self.prune:
                alpha = max(alpha, v)
                if alpha >= beta:
                    break
        return best

    def value(self, board, d, h, alpha=-INF, beta=INF):
        if d == 0:
            return self.qvalue(board, self.q, h, alpha, beta)
        self.nodes += 1
        legal = list(board.generate_legal_moves())
        t = terminal(board, legal, h)
        if t is not None:
            return t
        return self._children(board, legal, h, alpha, beta, -INF,
                              lambda b, hh, a, bt: self.value(b, d - 1, hh, a, bt))

    def qvalue(self, board, k, h, alpha=-INF, beta=INF):
        self.nodes += 1
        legal = list(board.generate_legal_moves())
        t = terminal(board, legal, h)
        if t is not None:
            return t
        s = evaluate(board, self.w)
        if k == 0:
            return s
        fn = lambda b, hh, a, bt: self.qvalue(b, k - 1, hh, a, bt)     # noqa: E731
        if board.is_check():
            return self._children(board, legal, h, alpha, beta, -INF, fn)
        if self.prune:
            if s >= beta:
                return s
            alpha = max(alpha, s)
        return self._children(board, [m for m in legal if in_quiescence_set(board, m)], h, alpha, beta, s, fn)


def search(board, depth, qdepth, w=WEIGHTS, prune=True, ties="first"):
    """(uci of the move or None, score, the root children's values in generation order) at depth D >= 1.
    ties="last" picks the last maximum instead of the first (a deliberately wrong root rule, for tests)."""
    assert depth >= 1 and qdepth >= 0
    b = board.copy()
    legal = list(b.generate_legal_moves())
    t = terminal(b, legal, 0)
    if t is not None:
        return None, t, []
    se = Search(qdepth, w, prune)
    vals = []
    for m in legal:
        b.push(m)
        vals.append(-se.value(b, depth - 1, 1))
        b.pop()
    best = max(vals)
    k = vals.index(best) if ties == "first" else len(vals) - 1 - vals[::-1].index(best)
    return legal[k].uci(), best, vals


def search_fen(fen, depth, qdepth, **kw):
    return search(chess.Board(fen), depth, qdepth, **kw)[:2]
