"""TEST-ONLY: builds tests/hostsim/ab_hostsim.cpp (a g++ build of the alpha-beta search, chessrl_b200/csrc/ab_search.cuh)
and loads it with ctypes.  The shared object goes to a per-user cache directory keyed by the sources' contents, so a
read-only checkout works and an edit rebuilds."""
import ctypes
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "ab_hostsim.cpp")
_CSRC = os.path.join(_HERE, "..", "..", "chessrl_b200", "csrc")
_DEPS = [_SRC] + [os.path.join(_CSRC, f) for f in ("ab_search.cuh", "chess_core.cuh")]
_lib = None
_lock = threading.Lock()


def load():
    """Builds (once per content) and loads the host build; safe to call from several threads."""
    with _lock:
        return _load()


def _load():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha256()
    for d in _DEPS:
        with open(d, "rb") as f:
            h.update(f.read())
    out_dir = os.path.join(tempfile.gettempdir(), "chessrl_b200_hostsim_%d" % os.getuid())
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "ab_hostsim_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(so):
        tmp = "%s.%d.%d.tmp" % (so, os.getpid(), threading.get_ident())
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", _SRC, "-o", tmp])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    u64p = ctypes.POINTER(ctypes.c_uint64)
    lib.hs_ab_eval.argtypes = [u64p]
    lib.hs_ab_eval.restype = ctypes.c_int
    lib.hs_ab_root.argtypes = [u64p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_uint16),
                               ctypes.POINTER(ctypes.c_int32), u64p]
    lib.hs_ab_root.restype = ctypes.c_int
    _lib = lib
    return lib


def _rec(record):
    return np.ascontiguousarray(np.asarray(record, dtype=np.uint64).reshape(9))


def evaluate(record):
    r = _rec(record)
    return int(load().hs_ab_eval(r.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))))


def root(record, depth, qdepth):
    """(move word, score, nodes) of the host build, as crl_games_ab_move_host reports them for one lane."""
    r = _rec(record)
    mv, sc, nd = ctypes.c_uint16(0), ctypes.c_int32(0), ctypes.c_uint64(0)
    rc = load().hs_ab_root(r.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), int(depth), int(qdepth),
                           ctypes.byref(mv), ctypes.byref(sc), ctypes.byref(nd))
    if rc != 0:
        raise ValueError("depth %d / qdepth %d out of range" % (depth, qdepth))
    return int(mv.value), int(sc.value), int(nd.value)
