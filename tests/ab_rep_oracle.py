"""ORACLE / TEST INFRASTRUCTURE ONLY -- never imported by the product path (`chessrl_b200/`).

The alpha-beta opponent with repetitions on (rule R of DESIGN.md 3.6, crl_games_ab_search_host CRL_AB_REPETITIONS), on
top of oracle/ab_oracle.py's definition, which it leaves as it is.  Before anything else in V and Q:

    a position h >= 1 plies below the root for which python-chess's board.is_repetition(2) holds -- the board's
    move_stack being the game's moves followed by the search path -- scores 0 and counts as one visited position

is_repetition walks back until an irreversible move (Board.is_irreversible), so only the positions of the current
reversible run count.  The root itself is never scored by the rule.  The seeded pick (oracle/ab_pick_oracle.py) applies
unchanged to the root children's values.
"""

from __future__ import annotations

import ab_oracle as A
import ab_pick_oracle as AP

chess = A.chess


def repeats_short(board):
    """board.is_repetition(2) with the window one ply short: the position right after the last irreversible move (or
    the first position of the stack) is not compared (a deliberately wrong rule, for tests)."""
    key = board._transposition_key()
    seen, undone = [], []
    try:
        while board.move_stack:
            move = board.pop()
            undone.append(move)
            if board.is_irreversible(move):
                break
            seen.append(board._transposition_key())
    finally:
        while undone:
            board.push(undone.pop())
    return key in seen[:-1]


class Search(A.Search):
    """ab_oracle.Search with the rule R.  rule="short" applies it with repeats_short (a deliberately wrong rule)."""

    def __init__(self, qdepth, w=A.WEIGHTS, prune=True, rule="is_repetition"):
        super().__init__(qdepth, w, prune)
        self.rule = rule

    def _repeated(self, board, h):
        if h < 1:
            return False
        return repeats_short(board) if self.rule == "short" else board.is_repetition(2)

    def value(self, board, d, h, alpha=-A.INF, beta=A.INF):
        if d != 0 and self._repeated(board, h):
            self.nodes += 1
            return 0
        return super().value(board, d, h, alpha, beta)

    def qvalue(self, board, k, h, alpha=-A.INF, beta=A.INF):
        if self._repeated(board, h):
            self.nodes += 1
            return 0
        return super().qvalue(board, k, h, alpha, beta)


def search(board, depth, qdepth, w=A.WEIGHTS, prune=True, repetitions=True):
    """ab_oracle.search with the rule R when `repetitions`, with board.move_stack as the game before the root;
    repetitions=False is ab_oracle.search itself.  Deliberately wrong variants, for tests: "short" (the window one ply
    short), "root" (the rule also scores the root: no move, score 0) and "path" (only the search path is seen, not the
    game before the root)."""
    if not repetitions:
        return A.search(board, depth, qdepth, w=w, prune=prune)
    assert depth >= 1 and qdepth >= 0
    b = board.copy(stack=repetitions != "path")
    legal = list(b.generate_legal_moves())
    t = A.terminal(b, legal, 0)
    if t is not None:
        return None, t, []
    if repetitions == "root" and b.is_repetition(2):
        return None, 0, []
    se = Search(qdepth, w, prune, rule="short" if repetitions == "short" else "is_repetition")
    vals = []
    for m in legal:
        b.push(m)
        vals.append(-se.value(b, depth - 1, 1))
        b.pop()
    best = max(vals)
    return legal[vals.index(best)].uci(), best, vals


def pick(board, depth, qdepth, margin, pick_plies, salt, repetitions=True):
    """ab_pick_oracle.pick on this module's values: (uci of the picked move or None, its score)."""
    assert margin >= 0 and pick_plies >= 0
    move, score, vals = search(board, depth, qdepth, repetitions=repetitions)
    if move is None:
        return None, score
    legal = list(board.generate_legal_moves())
    k = AP.pick_index(vals, len(board.move_stack), margin, pick_plies, salt)
    return legal[k].uci(), vals[k]
