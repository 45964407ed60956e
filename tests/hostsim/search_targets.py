"""TEST-ONLY: builds tests/hostsim/search_targets_hostsim.cpp (a g++ build of the search-target row,
chessrl_b200/csrc/search_targets.cuh) and loads it with ctypes.  Built like tests/hostsim/ab_pick.py: one shared object
per content of the sources, in a per-user cache directory, so a read-only checkout works and an edit rebuilds."""
import ctypes
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np

from chessrl_b200 import boards as B
from chessrl_b200.netencoder import get_uci_labels

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "search_targets_hostsim.cpp")
_ROOT = os.path.join(_HERE, "..", "..")
_DEPS = [_SRC] + [os.path.join(_ROOT, "chessrl_b200", "csrc", f) for f in ("search_targets.cuh", "chess_core.cuh")] + \
    [os.path.join(_ROOT, "include", "chessrl_b200.h")]
_lib = None
_lock = threading.Lock()
N_LABELS = 1968


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
            so = os.path.join(out_dir, "search_targets_hostsim_%s.so" % h.hexdigest()[:16])
            if not os.path.exists(so):
                tmp = "%s.%d.%d.tmp" % (so, os.getpid(), threading.get_ident())
                subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", _SRC, "-o", tmp])
                os.replace(tmp, so)
            lib = ctypes.CDLL(so)
            vp = ctypes.c_void_p
            lib.hs_search_targets.argtypes = [vp, vp, vp, ctypes.c_int, ctypes.c_float, vp, vp, vp, vp]
            lib.hs_search_targets.restype = None
            _lib = lib
        return _lib


def label_table():
    """label_of[promo * 4096 + from * 64 + to] -> netencoder.get_uci_labels index, -1 where there is none."""
    t = np.full(5 * 4096, -1, dtype=np.int16)
    for i, u in enumerate(get_uci_labels()):
        m = B.uci_to_move(u)
        t[(m >> 12 & 7) * 4096 + (m & 63) * 64 + (m >> 6 & 63)] = i
    return t


_TABLE = None


def targets(records, score_lists, temperature):
    """The host build on rows (record [9], list of root scores): (policy float32 [n, 1968], value float32 [n],
    legal count int32 [n])."""
    global _TABLE
    if _TABLE is None:
        _TABLE = label_table()
    recs = np.ascontiguousarray(np.asarray(records, dtype=np.uint64).reshape(-1, 9))
    n = recs.shape[0]
    counts = np.array([len(s) for s in score_lists], dtype=np.int32)
    offsets = np.zeros(n + 1, dtype=np.int32)
    offsets[1:] = np.cumsum(counts)
    flat = np.ascontiguousarray(np.concatenate([np.asarray(s, dtype=np.int32) for s in score_lists])
                                if n else np.zeros(0, np.int32), dtype=np.int32)
    policy = np.zeros((n, N_LABELS), dtype=np.float32)
    value = np.zeros(n, dtype=np.float32)
    legal = np.zeros(n, dtype=np.int32)
    load().hs_search_targets(recs.ctypes.data, flat.ctypes.data, offsets.ctypes.data, n, float(temperature),
                             _TABLE.ctypes.data, policy.ctypes.data, value.ctypes.data, legal.ctypes.data)
    return policy, value, legal
