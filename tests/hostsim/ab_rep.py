"""TEST-ONLY: builds tests/hostsim/ab_rep_hostsim.cpp (a g++ build of the alpha-beta search with repetitions on,
chessrl_b200/csrc/ab_search.cuh) and loads it with ctypes.  Built like tests/hostsim/ab.py: one shared object per content
of the sources, in a per-user cache directory, so a read-only checkout works and an edit rebuilds."""
import ctypes
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np

from chessrl_b200 import boards as B

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "ab_rep_hostsim.cpp")
_CSRC = os.path.join(_HERE, "..", "..", "chessrl_b200", "csrc")
_DEPS = [_SRC] + [os.path.join(_CSRC, f) for f in ("ab_search.cuh", "chess_core.cuh")]
_lib = None
_lock = threading.Lock()


def load():
    global _lib
    with _lock:
        if _lib is None:
            h = hashlib.sha256()
            for d in _DEPS:
                with open(d, "rb") as f:
                    h.update(f.read())
            out_dir = os.path.join(tempfile.gettempdir(), "chessrl_b200_hostsim_%d" % os.getuid())
            os.makedirs(out_dir, exist_ok=True)
            so = os.path.join(out_dir, "ab_rep_hostsim_%s.so" % h.hexdigest()[:16])
            if not os.path.exists(so):
                tmp = "%s.%d.%d.tmp" % (so, os.getpid(), threading.get_ident())
                subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", _SRC, "-o", tmp])
                os.replace(tmp, so)
            lib = ctypes.CDLL(so)
            u64p = ctypes.POINTER(ctypes.c_uint64)
            lib.hs_ab_rep.argtypes = [u64p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint16),
                                      ctypes.POINTER(ctypes.c_int32), u64p]
            lib.hs_ab_rep.restype = ctypes.c_int
            _lib = lib
        return _lib


def reversible_run(board):
    """Plies since the last irreversible move of a python-chess board's move_stack (Board.is_irreversible), as the
    engine keeps it in meta_revlen."""
    undone, n = [], 0
    try:
        while board.move_stack:
            move = board.pop()
            undone.append(move)
            if board.is_irreversible(move):
                break
            n += 1
    finally:
        while undone:
            board.push(undone.pop())
    return n


def game_records(board, window=None):
    """The records of the last positions of a python-chess board's game, in game order, the board's own position last
    with the engine's ply (len(move_stack)) and revlen in its meta.  window: how many positions before the root to give
    (default the reversible run, what the search reads)."""
    n = reversible_run(board)
    rev = n
    if window is not None:
        n = min(int(window), len(board.move_stack))
    b = board.copy()
    recs = []
    for i in range(n + 1):
        recs.append(np.array(B.record_from_fen(b.fen()), dtype=np.uint64).reshape(9))
        if i < n:
            b.pop()
    recs.reverse()
    m = B.meta_fields(int(recs[-1][8]))
    recs[-1][8] = B.pack_meta(m["turn"], m["castle"], m["ep"], m["halfmove"], m["fullmove"], len(board.move_stack),
                              rev)
    return np.ascontiguousarray(np.stack(recs))


def search(records, depth, qdepth, margin=0, pick_plies=0, salt=None):
    """(move word, score, nodes) of the host build, as crl_games_ab_search_host with CRL_AB_REPETITIONS reports them for
    one lane: the first best move (salt None) or the seeded pick.  records: game_records(board), or any records of the
    window in game order with the root's ply and revlen."""
    r = np.ascontiguousarray(np.asarray(records, dtype=np.uint64).reshape(-1, 9))
    mv, sc, nd = ctypes.c_uint16(0), ctypes.c_int32(0), ctypes.c_uint64(0)
    rc = load().hs_ab_rep(r.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), len(r), int(depth), int(qdepth),
                          int(salt is not None), int(margin), int(pick_plies), int(salt or 0) & (2 ** 64 - 1),
                          ctypes.byref(mv), ctypes.byref(sc), ctypes.byref(nd))
    if rc == -2:
        raise ValueError("%d records, fewer than the root's repetition window" % len(r))
    if rc != 0:
        raise ValueError("depth %d / qdepth %d / margin %d / pick_plies %d out of range"
                         % (depth, qdepth, margin, pick_plies))
    return int(mv.value), int(sc.value), int(nd.value)


def search_uci(records, depth, qdepth, **kw):
    mv, score, _ = search(records, depth, qdepth, **kw)
    return B.move_to_uci(mv), score
