"""ORACLE / TEST INFRASTRUCTURE ONLY -- never imported by the product path (`chessrl_b200/`).

The seeded near-best root pick of the alpha-beta opponent (DESIGN.md 3.7, crl_games_ab_pick_host), restated from its
definition on top of oracle/ab_oracle.py's search (the root children's exact values in generation order):

    best   = max s_k over the root moves m_0..m_{n-1}
    ply    = len(move_stack) of the game, the record's meta_ply
    pick   = the first k with s_k = best      if margin = 0, ply >= pick_plies or |best| >= MATE - MAX_PLY - 1
             C[splitmix64(salt + ply) mod |C|]  otherwise, C = [k : s_k >= best - margin] in generation order
    score  = s_pick
"""

from __future__ import annotations

import ab_oracle as A
from chessrl_oracle import splitmix64

MAX_PLY = 5 + 8                     # AB_MAX_DEPTH + AB_MAX_QDEPTH: plies below the root one search can hold
MATE_BOUND = A.MATE - MAX_PLY - 1   # |best| at or above this is a mate score: the margin does not apply
_M64 = (1 << 64) - 1


def pick_index(vals, ply, margin, pick_plies, salt, member="draw"):
    """Index of the picked root move among the values `vals` (generation order).  member="last" takes the last member
    of C instead of the drawn one (a deliberately wrong rule, for tests)."""
    best = max(vals)
    first = vals.index(best)
    if margin == 0 or ply >= pick_plies or abs(best) >= MATE_BOUND:
        return first
    cands = [k for k, v in enumerate(vals) if v >= best - margin]
    if member == "last":
        return cands[-1]
    return cands[splitmix64((salt + ply) & _M64) % len(cands)]


def pick(board, depth, qdepth, margin, pick_plies, salt, ply=None, **kw):
    """(uci of the picked move or None, its score) at depth D >= 1.  ply: default len(board.move_stack)."""
    assert margin >= 0 and pick_plies >= 0
    move, score, vals = A.search(board, depth, qdepth)
    if move is None:
        return None, score
    legal = list(board.generate_legal_moves())
    k = pick_index(vals, len(board.move_stack) if ply is None else ply, margin, pick_plies, salt, **kw)
    return legal[k].uci(), vals[k]
