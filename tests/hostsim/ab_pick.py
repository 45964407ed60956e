"""TEST-ONLY: builds tests/hostsim/ab_pick_hostsim.cpp (a g++ build of the alpha-beta search and its seeded near-best
root pick, chessrl_b200/csrc/ab_search.cuh) and loads it with ctypes.  Built like tests/hostsim/ab.py: one shared object
per content of the sources, in a per-user cache directory, so a read-only checkout works and an edit rebuilds."""
import ctypes
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np

from chessrl_b200 import boards as B

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "ab_pick_hostsim.cpp")
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
            so = os.path.join(out_dir, "ab_pick_hostsim_%s.so" % h.hexdigest()[:16])
            if not os.path.exists(so):
                tmp = "%s.%d.%d.tmp" % (so, os.getpid(), threading.get_ident())
                subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", _SRC, "-o", tmp])
                os.replace(tmp, so)
            lib = ctypes.CDLL(so)
            u64p = ctypes.POINTER(ctypes.c_uint64)
            lib.hs_ab_pick.argtypes = [u64p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint64,
                                       ctypes.POINTER(ctypes.c_uint16), ctypes.POINTER(ctypes.c_int32), u64p]
            lib.hs_ab_pick.restype = ctypes.c_int
            _lib = lib
        return _lib


def with_ply(record, ply):
    """The record with its ply field (meta bits 38..51, len(move_stack)) set to `ply`."""
    r = np.array(record, dtype=np.uint64).reshape(9).copy()
    r[8] = (r[8] & ~np.uint64(16383 << 38)) | (np.uint64(ply) << np.uint64(38))
    return r


def pick(record, depth, qdepth, margin, pick_plies, salt):
    """(move word, score, nodes) of the host build, as crl_games_ab_pick_host reports them for one lane."""
    r = np.ascontiguousarray(np.asarray(record, dtype=np.uint64).reshape(9))
    mv, sc, nd = ctypes.c_uint16(0), ctypes.c_int32(0), ctypes.c_uint64(0)
    rc = load().hs_ab_pick(r.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), int(depth), int(qdepth), int(margin),
                           int(pick_plies), int(salt) & (2 ** 64 - 1), ctypes.byref(mv), ctypes.byref(sc),
                           ctypes.byref(nd))
    if rc != 0:
        raise ValueError("depth %d / qdepth %d / margin %d / pick_plies %d out of range"
                         % (depth, qdepth, margin, pick_plies))
    return int(mv.value), int(sc.value), int(nd.value)


def pick_uci(record, depth, qdepth, margin, pick_plies, salt):
    mv, score, _ = pick(record, depth, qdepth, margin, pick_plies, salt)
    return B.move_to_uci(mv), score
