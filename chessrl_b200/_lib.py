"""ctypes binding of libchessrl_b200.so (include/chessrl_b200.h).  There is no fallback: if the library cannot
be found or built, importing the compute path raises."""

from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libchessrl_b200.so")

c_u64p = ctypes.POINTER(ctypes.c_uint64)
c_u16p = ctypes.POINTER(ctypes.c_uint16)
c_u8p = ctypes.POINTER(ctypes.c_uint8)
c_i8p = ctypes.POINTER(ctypes.c_int8)
c_i16p = ctypes.POINTER(ctypes.c_int16)
c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_f32p = ctypes.POINTER(ctypes.c_float)
c_f64p = ctypes.POINTER(ctypes.c_double)
vp = ctypes.c_void_p

CRL_OK, CRL_EINVAL, CRL_ECUDA, CRL_ENOMEM, CRL_ESTATE = 0, -1, -2, -3, -4
EVAL_NET, EVAL_HASH = 0, 1
NET_BF16, NET_FP8 = 0, 1
N_LABELS = 1968
MAX_MOVES = 256
N_WEIGHT_TENSORS = 140
KERNEL_CLASSES = ("movegen", "encode", "conv", "heads", "tree", "game", "hasheval")


class NodeHost(ctypes.Structure):
    _fields_ = [("parent", ctypes.c_int32), ("slot", ctypes.c_int32), ("visits", ctypes.c_int32),
                ("n_legal", ctypes.c_int32), ("n_children", ctypes.c_int32), ("result", ctypes.c_int32),
                ("move", ctypes.c_uint16), ("reply", ctypes.c_uint16), ("prior", ctypes.c_float),
                ("value", ctypes.c_double), ("board", ctypes.c_uint64 * 9)]


# name -> (restype, argtypes); every symbol include/chessrl_b200.h declares
SIGNATURES = {
    "crl_create": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]),
    "crl_create_ex": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, vp]),
    "crl_destroy": (ctypes.c_int, [vp]),
    "crl_last_error": (ctypes.c_char_p, []),
    "crl_version": (ctypes.c_int, []),
    "crl_movegen": (ctypes.c_int, [vp, vp, ctypes.c_int, vp, vp, vp]),
    "crl_debug_movegen_warp": (ctypes.c_int, [vp, vp, ctypes.c_int, vp, vp, vp]),
    "crl_make_moves": (ctypes.c_int, [vp, vp, ctypes.c_int, vp]),
    "crl_perft": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]),
    "crl_perft_root_host": (ctypes.c_int, [vp, c_u64p, ctypes.c_int, ctypes.c_int, ctypes.c_int64, c_u64p, c_i64p, c_i32p]),
    "crl_perft_root_shard_host": (ctypes.c_int, [vp, c_u64p, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                                 ctypes.c_int64, c_u64p, c_i64p, c_i32p]),
    "crl_expand_frontier": (ctypes.c_int, [vp, vp, ctypes.c_int, vp, vp, ctypes.c_int64, vp]),
    "crl_game_replay_host": (ctypes.c_int, [vp, c_u64p, c_u16p, ctypes.c_int, c_u16p, c_i32p, c_i8p, c_u8p, c_u64p]),
    "crl_game_replay_records_host": (ctypes.c_int, [vp, c_u64p, c_u16p, ctypes.c_int, c_u16p, c_i32p, c_i8p, c_u8p,
                                                    c_u64p, c_i32p]),
    "crl_encode": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, vp]),
    "crl_policy_index": (ctypes.c_int, [vp, vp, vp, ctypes.c_int, vp]),
    "crl_search_targets": (ctypes.c_int, [vp, vp, vp, vp, ctypes.c_int, ctypes.c_float, vp, vp, vp]),
    "crl_label_table_host": (ctypes.c_int, [vp, c_i16p]),
    "crl_net_load_host": (ctypes.c_int, [vp, ctypes.POINTER(c_f32p), c_i64p, ctypes.c_int]),
    "crl_net_forward": (ctypes.c_int, [vp, vp, ctypes.c_int, vp, vp]),
    "crl_debug_conv": (ctypes.c_int, [vp, ctypes.c_int, vp, ctypes.c_int, ctypes.c_int, vp, vp, ctypes.c_int]),
    "crl_debug_tower": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp]),
    "crl_debug_forward_counted": (ctypes.c_int, [vp, vp, ctypes.c_int, vp, vp, vp]),
    "crl_net_calibrate_host": (ctypes.c_int, [vp, vp, ctypes.c_int, c_f32p]),
    "crl_net_load_fp8_host": (ctypes.c_int, [vp, ctypes.POINTER(c_f32p), c_i64p, ctypes.c_int, c_f32p]),
    "crl_net_set_precision": (ctypes.c_int, [vp, ctypes.c_int]),
    "crl_hash_eval": (ctypes.c_int, [vp, vp, ctypes.c_int, ctypes.c_uint64, ctypes.c_int, vp, vp]),
    "crl_set_evaluator": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_uint64, ctypes.c_int]),
    "crl_games_set_host": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, c_u64p, c_u16p, c_i32p, ctypes.c_int]),
    "crl_games_get_host": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, c_u64p, c_i32p, c_i8p]),
    "crl_games_set_active_host": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, c_u8p]),
    "crl_game_moves_host": (ctypes.c_int, [vp, ctypes.c_int, c_u16p, ctypes.c_int, c_i32p]),
    "crl_games_restart_host": (ctypes.c_int, [vp, c_i32p, ctypes.c_int, c_u64p]),
    "crl_games_moves_host": (ctypes.c_int, [vp, c_i32p, ctypes.c_int, c_u16p, ctypes.c_int, c_i32p]),
    "crl_games_play_host": (ctypes.c_int, [vp, c_u16p, c_u8p]),
    "crl_games_legal_host": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, c_u16p, c_i32p]),
    "crl_games_policy_move_host": (ctypes.c_int, [vp, c_u8p, c_u16p]),
    "crl_games_ab_move_host": (ctypes.c_int, [vp, c_u8p, ctypes.c_int, ctypes.c_int, c_u16p, c_i32p, c_i64p]),
    "crl_games_ab_pick_host": (ctypes.c_int, [vp, c_u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_u64p,
                                              c_u16p, c_i32p, c_i64p]),
    "crl_games_ab_search_host": (ctypes.c_int, [vp, c_u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                ctypes.c_int, c_u64p, c_u16p, c_i32p, c_i64p]),
    "crl_games_ab_root_scores_host": (ctypes.c_int, [vp, c_i32p, c_i32p]),
    "crl_net_select_slot": (ctypes.c_int, [vp, ctypes.c_int]),
    "crl_games_set_players_host": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int, c_u8p, c_u8p]),
    "crl_mcts_begin_move": (ctypes.c_int, [vp]),
    "crl_set_reuse": (ctypes.c_int, [vp, ctypes.c_int]),
    "crl_mcts_set_row_bound": (ctypes.c_int, [vp, ctypes.c_int]),
    "crl_reuse_count_host": (ctypes.c_int, [vp, c_i64p]),
    "crl_mcts_simulate": (ctypes.c_int, [vp, ctypes.c_int, ctypes.c_int]),
    "crl_mcts_root_stats_host": (ctypes.c_int, [vp, c_i32p, c_f64p, c_f32p, c_u16p, c_u16p, c_i8p, c_i32p, c_i32p, c_f64p]),
    "crl_mcts_commit_host": (ctypes.c_int, [vp, c_i32p, c_u16p, ctypes.c_int]),
    "crl_mcts_node_dump_host": (ctypes.c_int, [vp, ctypes.c_int, ctypes.POINTER(NodeHost), ctypes.c_int, c_i32p]),
    "crl_counters_host": (ctypes.c_int, [vp, c_i64p]),
    "crl_profile": (ctypes.c_int, [vp, ctypes.c_int]),
    "crl_profile_read_host": (ctypes.c_int, [vp, c_f64p, c_i64p, ctypes.c_int]),
}

_lib = None


class CrlError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("libchessrl_b200 error %d: %s" % (status, message))
        self.status = status


def load():
    """Loads the CUDA library.  It is built with nvcc first only when the .so is missing or CRL_REBUILD is set --
    deliberately NOT on source mtimes: a snapshot copied to a GPU box carries arbitrary mtimes, and several ranks
    importing at once must not start concurrent builds.  After editing csrc/ run `python -m chessrl_b200.build`
    (or __graft_entry__.build()).  Raises if the library cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) or os.environ.get("CRL_REBUILD"):
        from . import build as _build
        _build.build(force=True)
    if not os.path.exists(LIB_PATH):
        raise ImportError("libchessrl_b200.so is missing and could not be built; the CUDA extension is required "
                          "(there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = the library does not match the header
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status):
    if status != CRL_OK:
        raise CrlError(status, load().crl_last_error().decode("utf-8", "replace"))
