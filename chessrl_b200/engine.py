"""Engine: thin Python host object over one crl_engine handle (one per process and GPU).

PyTorch is used for device memory (tensors handed to the C ABI as raw pointers) and the current CUDA
stream; every computation happens inside libchessrl_b200.so.  If CUDA or the library is missing this module
raises -- there is no CPU path.
"""

from __future__ import annotations

import contextlib
import ctypes

import numpy as np
import torch

from . import _lib
from . import boards as B
from ._lib import check, vp


def _ptr(t):
    return vp(t.data_ptr()) if t is not None else None


def _np(a, ctype):
    return a.ctypes.data_as(ctypes.POINTER(ctype))


NET_SLOTS = 2      # CRL_NET_SLOTS: networks one engine holds (include/chessrl_b200.h crl_net_select_slot)
CRL_AB_REPETITIONS = 1   # crl_games_ab_search_host flag: repetitions below the root score 0 (DESIGN.md 3.6)


class Engine:
    """max_games lockstep lanes, max_nodes tree nodes per game (>= simulations per move + 1), max_inflight
    in-flight simulations per game (the reference's `threads`; 1 = the exact threads=1 schedule only)."""

    def __init__(self, max_games=1, max_nodes=1024, avg_moves=64, device=None, max_inflight=1):
        if not torch.cuda.is_available():
            raise RuntimeError("chessrl_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.max_games = int(max_games)
        self.max_nodes = int(max_nodes)
        self.max_inflight = int(max_inflight)
        self.reuse = False               # evaluation reuse across consecutive searches (set_reuse)
        h = vp()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            check(self.lib.crl_create_ex(ctypes.byref(h), self.device_index, self.max_games, self.max_nodes,
                                         int(avg_moves), self.max_inflight, vp(stream)))
        self.h = h
        self.weights_loaded = False
        self.net_precision = "bf16"                     # slot 0's
        self.slot_precision = ["bf16"] * NET_SLOTS      # every network slot's (load_weights / set_net_precision)

    def close(self):
        if getattr(self, "h", None):
            self.lib.crl_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- helpers ----------------------------------------------------------------------------------------
    def boards_to_device(self, records):
        """records: uint64 [n, 9] (AoS, host) -> device tensor int64 [9, n] (SoA)."""
        rec = np.ascontiguousarray(np.asarray(records, dtype=np.uint64).reshape(-1, 9))
        t = torch.from_numpy(rec.view(np.int64).T.copy())
        return t.to(self.device)

    @staticmethod
    def boards_to_host(boards_t):
        return np.ascontiguousarray(boards_t.cpu().numpy().T).view(np.uint64)

    # ---- rules --------------------------------------------------------------------------------------------
    def movegen(self, boards_t):
        n = boards_t.shape[1]
        moves = torch.empty((n, B.MAX_MOVES), dtype=torch.int16, device=self.device)
        counts = torch.empty((n,), dtype=torch.int32, device=self.device)
        flags = torch.empty((n,), dtype=torch.uint8, device=self.device)
        check(self.lib.crl_movegen(self.h, _ptr(boards_t), n, _ptr(moves), _ptr(counts), _ptr(flags)))
        return moves, counts, flags

    def movegen_warp(self, boards_t):
        """Test hook: movegen() through the warp-cooperative generator (crl_debug_movegen_warp)."""
        n = boards_t.shape[1]
        moves = torch.empty((n, B.MAX_MOVES), dtype=torch.int16, device=self.device)
        counts = torch.empty((n,), dtype=torch.int32, device=self.device)
        flags = torch.empty((n,), dtype=torch.uint8, device=self.device)
        check(self.lib.crl_debug_movegen_warp(self.h, _ptr(boards_t), n, _ptr(moves), _ptr(counts), _ptr(flags)))
        return moves, counts, flags

    def make_moves(self, boards_t, moves_t):
        check(self.lib.crl_make_moves(self.h, _ptr(boards_t), boards_t.shape[1], _ptr(moves_t)))
        return boards_t

    def perft(self, boards_t, depth, bulk=True):
        n = boards_t.shape[1]
        nodes = torch.empty((n,), dtype=torch.int64, device=self.device)
        check(self.lib.crl_perft(self.h, _ptr(boards_t), n, int(depth), int(bool(bulk)), _ptr(nodes)))
        return nodes

    def perft_root(self, record, depth, bulk=True, min_frontier=1 << 20, shard=0, n_shards=1, shard_min_frontier=1 << 16):
        """perft(depth) of one position in ONE call: device-side breadth-first plies to >= min_frontier boards, then a
        depth-first walk per lane.  Returns (total, lanes, bfs_plies).  With n_shards > 1 the call computes shard
        `shard`'s part only (the frontier is split once it holds >= shard_min_frontier boards); the shards' totals add up
        to perft(depth)."""
        rec = np.ascontiguousarray(np.asarray(record, dtype=np.uint64).reshape(9))
        total = ctypes.c_uint64(0)
        lanes = ctypes.c_int64(0)
        plies = ctypes.c_int32(0)
        check(self.lib.crl_perft_root_shard_host(self.h, _np(rec, ctypes.c_uint64), int(depth), int(bool(bulk)),
                                                 int(min_frontier), int(shard), int(n_shards), int(shard_min_frontier),
                                                 ctypes.byref(total), ctypes.byref(lanes), ctypes.byref(plies)))
        return int(total.value), int(lanes.value), int(plies.value)

    def expand_frontier(self, boards_t):
        """One breadth-first ply: returns the SoA tensor of all children (python-chess move order per parent)."""
        n = boards_t.shape[1]
        counts = torch.empty((n,), dtype=torch.int32, device=self.device)
        check(self.lib.crl_expand_frontier(self.h, _ptr(boards_t), n, None, None, 0, _ptr(counts)))
        offsets = torch.cumsum(counts.to(torch.int64), 0) - counts.to(torch.int64)
        total = int(counts.sum().item())
        out = torch.empty((9, total), dtype=torch.int64, device=self.device)
        check(self.lib.crl_expand_frontier(self.h, _ptr(boards_t), n, _ptr(offsets), _ptr(out), total, _ptr(counts)))
        return out, counts

    def game_replay(self, start_record, moves, records=False):
        """Game semantics for one game on slot 0: returns dict(legal, result, accepted, record[, records]).
        records=True also returns the record after every accepted move ([n_accepted + 1, 9], records[0] = start)."""
        start = np.ascontiguousarray(np.asarray(start_record, dtype=np.uint64))
        mv = np.ascontiguousarray(np.asarray(moves, dtype=np.uint16))
        legal = np.zeros(B.MAX_MOVES, dtype=np.uint16)
        n_legal = ctypes.c_int32(0)
        result = ctypes.c_int8(0)
        accepted = np.zeros(max(len(mv), 1), dtype=np.uint8)
        out = {}
        if records:
            recs = np.zeros((len(mv) + 1, 9), dtype=np.uint64)
            n_rec = ctypes.c_int32(0)
            check(self.lib.crl_game_replay_records_host(
                self.h, _np(start, ctypes.c_uint64), _np(mv, ctypes.c_uint16), len(mv), _np(legal, ctypes.c_uint16),
                ctypes.byref(n_legal), ctypes.byref(result), _np(accepted, ctypes.c_uint8), _np(recs, ctypes.c_uint64),
                ctypes.byref(n_rec)))
            out["records"] = recs[:n_rec.value].copy()
            final = out["records"][-1].copy()
        else:
            final = np.zeros(9, dtype=np.uint64)
            check(self.lib.crl_game_replay_host(self.h, _np(start, ctypes.c_uint64), _np(mv, ctypes.c_uint16), len(mv),
                                                _np(legal, ctypes.c_uint16), ctypes.byref(n_legal), ctypes.byref(result),
                                                _np(accepted, ctypes.c_uint8), _np(final, ctypes.c_uint64)))
        out.update({"legal": legal[:n_legal.value].copy(),
                    "result": None if result.value == B.RESULT_NONE else int(result.value),
                    "accepted": accepted[:len(mv)].astype(bool), "record": final})
        return out

    # ---- encoding -----------------------------------------------------------------------------------------
    def encode(self, boards_t, hist_t=None, hist_len_t=None):
        n = boards_t.shape[1]
        planes = torch.empty((n, 8, 8, 128), dtype=torch.bfloat16, device=self.device)
        check(self.lib.crl_encode(self.h, _ptr(boards_t), _ptr(hist_t), _ptr(hist_len_t), n, _ptr(planes)))
        return planes

    def policy_index(self, moves_t, counts_t):
        n = moves_t.shape[0]
        idx = torch.empty((n, B.MAX_MOVES), dtype=torch.int16, device=self.device)
        check(self.lib.crl_policy_index(self.h, _ptr(moves_t), _ptr(counts_t), n, _ptr(idx)))
        return idx

    def search_targets(self, boards_t, scores_t, offsets_t, temperature):
        """Policy and score-value targets from root scores (DESIGN.md 3.8, include/chessrl_b200.h crl_search_targets):
        boards_t uint64 SoA [9, n] on the device, scores_t int32 (all rows' scores concatenated), offsets_t int32 [n+1].
        Returns device tensors (policy float32 [n, 1968], score value float32 [n], legal count int32 [n]); a row whose
        legal count differs from its score count is all zeros.  Does not synchronise."""
        n = boards_t.shape[1]
        policy = torch.empty((n, _lib.N_LABELS), dtype=torch.float32, device=self.device)
        value = torch.empty(n, dtype=torch.float32, device=self.device)
        count = torch.empty(n, dtype=torch.int32, device=self.device)
        check(self.lib.crl_search_targets(self.h, _ptr(boards_t), _ptr(scores_t), _ptr(offsets_t), n, float(temperature),
                                          _ptr(policy), _ptr(value), _ptr(count)))
        return policy, value, count

    def label_table(self):
        t = np.zeros(5 * 4096, dtype=np.int16)
        check(self.lib.crl_label_table_host(self.h, _np(t, ctypes.c_int16)))
        return t.reshape(5, 64, 64)

    # ---- network ------------------------------------------------------------------------------------------
    @contextlib.contextmanager
    def _slot(self, slot):
        """The network calls inside act on network slot `slot`; the engine is back on slot 0 afterwards."""
        slot = int(slot)
        if slot == 0:
            yield
            return
        check(self.lib.crl_net_select_slot(self.h, slot))
        try:
            yield
        finally:
            check(self.lib.crl_net_select_slot(self.h, 0))

    def load_weights(self, tensors, precision="bf16", calibration=None, slot=0):
        """tensors: the 140-array weight pack (chessrl_b200.model.ChessModel.weights).
        precision="fp8" also builds the e4m3 tower (include/chessrl_b200.h crl_net_load_fp8_host) and selects it; its
        activation scales come from `calibration`: 21 per-layer amax values (Engine.calibrate), bf16 planes
        [n,8,8,128] to calibrate on, or None for model.calibration_planes(self).
        slot: the network slot (0 or 1) the weights go to; slot 1 is the second player of games_set_players."""
        if slot != 0:
            with self._slot(slot):
                self._load_weights(tensors, precision, calibration, slot)
            return
        self._load_weights(tensors, precision, calibration, 0)

    def _load_weights(self, tensors, precision, calibration, slot):
        if precision not in ("bf16", "fp8"):
            raise ValueError("precision must be 'bf16' or 'fp8', not %r" % (precision,))
        arrs = [np.ascontiguousarray(np.asarray(t, dtype=np.float32).reshape(-1)) for t in tensors]
        n = len(arrs)
        ptrs = (_lib.c_f32p * n)(*[a.ctypes.data_as(_lib.c_f32p) for a in arrs])
        sizes = (ctypes.c_int64 * n)(*[a.size for a in arrs])
        if precision == "bf16" or calibration is None or torch.is_tensor(calibration):
            # the bf16 tower; for fp8 it is also what calibrates (crl_net_load_fp8_host loads it again below)
            self._set_precision_attr(slot, "bf16")
            check(self.lib.crl_net_load_host(self.h, ptrs, sizes, n))
            if slot == 0:
                self.weights_loaded = True
        if precision == "fp8":
            if calibration is None:
                from .model import calibration_planes
                calibration = calibration_planes(self)
            if torch.is_tensor(calibration):
                calibration = self._calibrate(calibration)
            amax = np.ascontiguousarray(np.asarray(calibration, dtype=np.float32).reshape(-1))
            if amax.size != 21:
                raise ValueError("calibration: 21 per-layer amax values expected, got %d" % amax.size)
            self._set_precision_attr(slot, "bf16")           # what a failed fp8 load leaves the slot in
            check(self.lib.crl_net_load_fp8_host(self.h, ptrs, sizes, n, amax.ctypes.data_as(_lib.c_f32p)))
            if slot == 0:
                self.weights_loaded = True
        self._set_precision_attr(slot, precision)

    def _set_precision_attr(self, slot, precision):
        self.slot_precision[slot] = precision
        if slot == 0:
            self.net_precision = precision

    def calibrate(self, planes_t, slot=0):
        """max |output| of each of the 21 tower convolutions over bf16 planes [n,8,8,128], from the bf16 tower
        -> float32 [21] (the `calibration` of load_weights(precision="fp8"))."""
        with self._slot(slot):
            return self._calibrate(planes_t)

    def _calibrate(self, planes_t):
        amax = np.zeros(21, dtype=np.float32)
        part = np.zeros(21, dtype=np.float32)
        step = self.max_games * self.max_inflight          # rows the engine's buffers hold
        for i in range(0, planes_t.shape[0], step):
            x = planes_t[i:i + step]
            check(self.lib.crl_net_calibrate_host(self.h, _ptr(x), x.shape[0], part.ctypes.data_as(_lib.c_f32p)))
            amax = np.maximum(amax, part)
        return amax

    def set_net_precision(self, precision, slot=0):
        """'bf16' or 'fp8' (the latter needs a load_weights(..., precision="fp8") since the last bf16 load)."""
        code = {"bf16": _lib.NET_BF16, "fp8": _lib.NET_FP8}.get(precision)
        if code is None:
            raise ValueError("precision must be 'bf16' or 'fp8', not %r" % (precision,))
        with self._slot(slot):
            check(self.lib.crl_net_set_precision(self.h, code))
        self._set_precision_attr(int(slot), precision)

    def net_forward(self, planes_t, slot=0):
        n = planes_t.shape[0]
        policy = torch.empty((n, _lib.N_LABELS), dtype=torch.float32, device=self.device)
        value = torch.empty((n,), dtype=torch.float32, device=self.device)
        with self._slot(slot):
            check(self.lib.crl_net_forward(self.h, _ptr(planes_t), n, _ptr(policy), _ptr(value)))
        return policy, value

    def debug_conv(self, layer, x_t, residual_t=None, relu=False):
        n, cin = x_t.shape[0], x_t.shape[3]
        out = torch.empty((n, 8, 8, 256), dtype=torch.bfloat16, device=self.device)
        check(self.lib.crl_debug_conv(self.h, int(layer), _ptr(x_t), cin, n, _ptr(residual_t), _ptr(out), int(relu)))
        return out

    def debug_tower(self, planes_t, layer=20, slot=0):
        """The production forward pass with taps: dict(act = output of convolution `layer` [n,8,8,256] bf16,
        logits [n,1968], pf [n,128] bf16, vf [n,64], policy [n,1968], value [n])."""
        n = planes_t.shape[0]
        dev = self.device
        out = {"act": torch.zeros((n, 8, 8, 256), dtype=torch.bfloat16, device=dev),
               "logits": torch.empty((n, _lib.N_LABELS), dtype=torch.float32, device=dev),
               "pf": torch.empty((n, 128), dtype=torch.bfloat16, device=dev),
               "vf": torch.empty((n, 64), dtype=torch.float32, device=dev),
               "policy": torch.empty((n, _lib.N_LABELS), dtype=torch.float32, device=dev),
               "value": torch.empty((n,), dtype=torch.float32, device=dev)}
        with self._slot(slot):
            check(self.lib.crl_debug_tower(self.h, _ptr(planes_t), n, int(layer), _ptr(out["act"]), _ptr(out["logits"]),
                                           _ptr(out["pf"]), _ptr(out["vf"]), _ptr(out["policy"]), _ptr(out["value"])))
        return out

    def debug_forward_counted(self, planes_t, n_bound, count, policy=None, value=None, slot=0):
        """Test hook: net_forward as a search batch runs it -- launched for n_bound rows, with the row count `count` read
        by the kernels from device memory (int, or a device int32 tensor of one element).  Rows at or after the count
        of `policy` [n_bound,1968] / `value` [n_bound] (allocated when None) are left as they were."""
        dev = self.device
        if policy is None:
            policy = torch.empty((n_bound, _lib.N_LABELS), dtype=torch.float32, device=dev)
        if value is None:
            value = torch.empty((n_bound,), dtype=torch.float32, device=dev)
        if not torch.is_tensor(count):
            count = torch.tensor([int(count)], dtype=torch.int32, device=dev)
        assert count.dtype == torch.int32 and count.device == dev
        with self._slot(slot):
            check(self.lib.crl_debug_forward_counted(self.h, _ptr(planes_t), int(n_bound), _ptr(count), _ptr(policy),
                                                     _ptr(value)))
        return policy, value

    def hash_eval(self, boards_t, seed, policy_bits=24):
        n = boards_t.shape[1]
        policy = torch.empty((n, _lib.N_LABELS), dtype=torch.float32, device=self.device)
        value = torch.empty((n,), dtype=torch.float32, device=self.device)
        check(self.lib.crl_hash_eval(self.h, _ptr(boards_t), n, int(seed), int(policy_bits), _ptr(policy), _ptr(value)))
        return policy, value

    # ---- games + search -----------------------------------------------------------------------------------
    def set_evaluator(self, kind, seed=0, policy_bits=24, slot=0):
        with self._slot(slot):
            check(self.lib.crl_set_evaluator(self.h, int(kind), int(seed), int(policy_bits)))

    def games_set_players(self, white, black, first=0):
        """Network slot (0 or 1) that plays white / black in lanes first..first+len(white)-1 (scalars apply to all
        lanes from `first` on).  A search evaluates a lane's rows with the slot of the side to move at its root
        (include/chessrl_b200.h crl_games_set_players_host).  The players persist across games_set / games_restart."""
        n = self.max_games - int(first)
        w = np.asarray(white, dtype=np.uint8)
        b = np.asarray(black, dtype=np.uint8)
        if w.ndim == 0 and b.ndim == 0:
            w, b = np.full(n, w, dtype=np.uint8), np.full(n, b, dtype=np.uint8)
        elif w.ndim == 0:
            w = np.full(b.shape, w, dtype=np.uint8)
        elif b.ndim == 0:
            b = np.full(w.shape, b, dtype=np.uint8)
        w, b = np.ascontiguousarray(w), np.ascontiguousarray(b)
        if w.shape != b.shape or w.ndim != 1:
            raise ValueError("white and black: one slot per lane, of the same length")
        check(self.lib.crl_games_set_players_host(self.h, int(first), int(w.size), _np(w, ctypes.c_uint8),
                                                  _np(b, ctypes.c_uint8)))

    @staticmethod
    def pack_move_lists(move_lists):
        """list of per-game move-word lists -> (uint16 [n, stride], int32 [n]) host arrays for games_set."""
        n = len(move_lists)
        stride = max(1, max((len(m) for m in move_lists), default=1))
        mv = np.full((n, stride), B.MOVE_NONE, dtype=np.uint16)
        cnt = np.zeros(n, dtype=np.int32)
        for i, m in enumerate(move_lists):
            cnt[i] = len(m)
            mv[i, :len(m)] = m
        return mv, cnt

    def games_set(self, start_records, move_lists=None, first=0):
        """Game(board) + Game.move for every listed move.  move_lists: per-game lists, or the packed pair from
        pack_move_lists (host arrays; skips the per-game Python packing)."""
        rec = np.ascontiguousarray(np.asarray(start_records, dtype=np.uint64).reshape(-1, 9))
        n = rec.shape[0]
        if move_lists is None:
            check(self.lib.crl_games_set_host(self.h, first, n, _np(rec, ctypes.c_uint64), None, None, 0))
            return
        if isinstance(move_lists, tuple):
            mv = np.ascontiguousarray(move_lists[0], dtype=np.uint16)
            cnt = np.ascontiguousarray(move_lists[1], dtype=np.int32)
            assert mv.ndim == 2 and mv.shape[0] == n and cnt.shape == (n,)
        else:
            mv, cnt = self.pack_move_lists(move_lists)
        stride = mv.shape[1]
        check(self.lib.crl_games_set_host(self.h, first, n, _np(rec, ctypes.c_uint64), _np(mv, ctypes.c_uint16),
                                          _np(cnt, ctypes.c_int32), stride))

    def games_get(self, first=0, n=None):
        n = self.max_games - first if n is None else n
        rec = np.zeros((n, 9), dtype=np.uint64)
        plies = np.zeros(n, dtype=np.int32)
        res = np.zeros(n, dtype=np.int8)
        check(self.lib.crl_games_get_host(self.h, first, n, _np(rec, ctypes.c_uint64), _np(plies, ctypes.c_int32),
                                          _np(res, ctypes.c_int8)))
        return rec, plies, res

    def games_set_active(self, active, first=0):
        """Parks (0) / resumes (1) lanes first..first+len(active)-1; parked lanes are skipped by the search."""
        a = np.ascontiguousarray(np.asarray(active, dtype=np.uint8))
        check(self.lib.crl_games_set_active_host(self.h, int(first), len(a), _np(a, ctypes.c_uint8)))

    def game_moves(self, game):
        n = ctypes.c_int32(0)
        buf = np.zeros(2048, dtype=np.uint16)
        check(self.lib.crl_game_moves_host(self.h, int(game), _np(buf, ctypes.c_uint16), len(buf), ctypes.byref(n)))
        return buf[:n.value].copy()

    def games_restart(self, lanes, start_record=None):
        """A new game (from `start_record`, default the start position) in every listed lane: one device round trip."""
        ln = np.ascontiguousarray(np.asarray(lanes, dtype=np.int32))
        if ln.size == 0:
            return
        rec = np.ascontiguousarray(B.record_from_fen() if start_record is None else np.asarray(start_record, dtype=np.uint64))
        check(self.lib.crl_games_restart_host(self.h, _np(ln, ctypes.c_int32), int(ln.size), _np(rec, ctypes.c_uint64)))

    def games_moves(self, lanes, cap=2048):
        """Move lists of the listed lanes in one round trip -> list of uint16 arrays."""
        ln = np.ascontiguousarray(np.asarray(lanes, dtype=np.int32))
        if ln.size == 0:
            return []
        buf = np.zeros((ln.size, cap), dtype=np.uint16)
        cnt = np.zeros(ln.size, dtype=np.int32)
        check(self.lib.crl_games_moves_host(self.h, _np(ln, ctypes.c_int32), int(ln.size), _np(buf, ctypes.c_uint16), int(cap),
                                            _np(cnt, ctypes.c_int32)))
        return [buf[i, :min(int(cnt[i]), cap)].copy() for i in range(ln.size)]

    def games_play(self, moves):
        """Game.move of one optional move word per lane (MOVE_NONE = none) -> bool [max_games] accepted."""
        mv = np.ascontiguousarray(np.asarray(moves, dtype=np.uint16))
        assert mv.shape == (self.max_games,)
        acc = np.zeros(self.max_games, dtype=np.uint8)
        check(self.lib.crl_games_play_host(self.h, _np(mv, ctypes.c_uint16), _np(acc, ctypes.c_uint8)))
        torch.cuda.current_stream(self.device).synchronize()
        return acc.astype(bool)

    def games_legal(self, first=0, n=None):
        """Legal moves (python-chess order) of lanes first..first+n-1 -> (uint16 [n, 256], int32 [n])."""
        n = self.max_games - first if n is None else n
        legal = np.zeros((n, B.MAX_MOVES), dtype=np.uint16)
        cnt = np.zeros(n, dtype=np.int32)
        check(self.lib.crl_games_legal_host(self.h, int(first), int(n), _np(legal, ctypes.c_uint16), _np(cnt, ctypes.c_int32)))
        return legal, cnt

    def policy_move(self, mask=None):
        picks = np.zeros(self.max_games, dtype=np.uint16)
        m = None
        if mask is not None:
            mask = np.ascontiguousarray(np.asarray(mask, dtype=np.uint8))
            m = _np(mask, ctypes.c_uint8)
        check(self.lib.crl_games_policy_move_host(self.h, m, _np(picks, ctypes.c_uint16)))
        torch.cuda.current_stream(self.device).synchronize()
        return picks

    def games_ab_move(self, depth, qdepth=4, mask=None, repetitions=False):
        """Fixed-depth alpha-beta (DESIGN.md 3.6, include/chessrl_b200.h crl_games_ab_move_host) on the current position
        of every active, unfinished lane with mask[g] != 0 (None = all lanes).  Plays nothing.
        repetitions: a position below the root that repeats an earlier one of its reversible run (on the search path or
        in the lane's game) scores 0 (crl_games_ab_search_host CRL_AB_REPETITIONS).
        Returns numpy (moves uint16 [max_games], MOVE_NONE for lanes not searched; scores int32, centipawns for the side
        to move, +-(32000 - plies) for a mate; nodes int64, positions visited)."""
        if repetitions:
            return self.games_ab_search(depth, qdepth, CRL_AB_REPETITIONS, 0, 0, None, mask)
        G = self.max_games
        moves = np.zeros(G, dtype=np.uint16)
        scores = np.zeros(G, dtype=np.int32)
        nodes = np.zeros(G, dtype=np.int64)
        m = self._ab_mask(mask)
        check(self.lib.crl_games_ab_move_host(self.h, m, int(depth), int(qdepth), _np(moves, ctypes.c_uint16),
                                              _np(scores, ctypes.c_int32), _np(nodes, ctypes.c_int64)))
        return moves, scores, nodes

    def games_ab_pick(self, depth, qdepth, margin, pick_plies, salt, mask=None, repetitions=False):
        """games_ab_move with the seeded near-best root pick (DESIGN.md 3.7, include/chessrl_b200.h
        crl_games_ab_pick_host): a lane at ply < pick_plies whose best score is not a mate plays one of the root moves
        within `margin` centipawns of the best, chosen by splitmix64(salt[g] + ply); otherwise the first best move.
        salt: one uint64 per lane.  repetitions: as in games_ab_move.  Returns the same triple as games_ab_move; the
        score is the picked move's."""
        G = self.max_games
        s = np.ascontiguousarray(np.asarray(salt, dtype=np.uint64))
        if s.shape != (G,):
            raise ValueError("salt: one entry per lane (%d), got shape %s" % (G, s.shape))
        if repetitions:
            return self.games_ab_search(depth, qdepth, CRL_AB_REPETITIONS, margin, pick_plies, s, mask)
        moves = np.zeros(G, dtype=np.uint16)
        scores = np.zeros(G, dtype=np.int32)
        nodes = np.zeros(G, dtype=np.int64)
        m = self._ab_mask(mask)
        check(self.lib.crl_games_ab_pick_host(self.h, m, int(depth), int(qdepth), int(margin), int(pick_plies),
                                              _np(s, ctypes.c_uint64), _np(moves, ctypes.c_uint16),
                                              _np(scores, ctypes.c_int32), _np(nodes, ctypes.c_int64)))
        return moves, scores, nodes

    def _ab_mask(self, mask):
        if mask is None:
            return None
        mask = np.ascontiguousarray(np.asarray(mask, dtype=np.uint8))
        if mask.shape != (self.max_games,):
            raise ValueError("mask: one entry per lane (%d), got shape %s" % (self.max_games, mask.shape))
        return _np(mask, ctypes.c_uint8)                 # (the pointer keeps the array alive)

    def games_ab_search(self, depth, qdepth, flags=0, margin=0, pick_plies=0, salt=None, mask=None):
        """include/chessrl_b200.h crl_games_ab_search_host: games_ab_move (salt None; margin and pick_plies must be 0)
        or games_ab_pick (a salt per lane) with option bits `flags` (CRL_AB_REPETITIONS).  Returns the same triple."""
        G = self.max_games
        if salt is not None:
            salt = np.ascontiguousarray(np.asarray(salt, dtype=np.uint64))
            if salt.shape != (G,):
                raise ValueError("salt: one entry per lane (%d), got shape %s" % (G, salt.shape))
        moves = np.zeros(G, dtype=np.uint16)
        scores = np.zeros(G, dtype=np.int32)
        nodes = np.zeros(G, dtype=np.int64)
        m = self._ab_mask(mask)
        check(self.lib.crl_games_ab_search_host(self.h, m, int(depth), int(qdepth), int(flags), int(margin),
                                                int(pick_plies), None if salt is None else _np(salt, ctypes.c_uint64),
                                                _np(moves, ctypes.c_uint16), _np(scores, ctypes.c_int32),
                                                _np(nodes, ctypes.c_int64)))
        return moves, scores, nodes

    def games_ab_root_scores(self):
        """The exact value of every root child from the most recent games_ab_* call (include/chessrl_b200.h
        crl_games_ab_root_scores_host): numpy (scores int32 [max_games, MAX_MOVES] in generation order, 0 past a lane's
        count; counts int32 [max_games], -1 for lanes that call did not search)."""
        scores = np.zeros((self.max_games, B.MAX_MOVES), dtype=np.int32)
        counts = np.zeros(self.max_games, dtype=np.int32)
        check(self.lib.crl_games_ab_root_scores_host(self.h, _np(scores, ctypes.c_int32), _np(counts, ctypes.c_int32)))
        return scores, counts

    def mcts_begin_move(self):
        check(self.lib.crl_mcts_begin_move(self.h))

    def set_reuse(self, enable=True):
        """Evaluation reuse across consecutive move searches (include/chessrl_b200.h crl_set_reuse): expansions take the
        reply / value / priors of nodes the previous move's search already evaluated; results are bit-identical."""
        check(self.lib.crl_set_reuse(self.h, int(bool(enable))))
        self.reuse = bool(enable)

    def set_row_bound(self, max_running_games=0):
        """Promise that at most this many games are running (0 = none): launches shrink to that many rows and small batches
        take the tower's single-tile path (include/chessrl_b200.h crl_mcts_set_row_bound).  A broken promise raises."""
        check(self.lib.crl_mcts_set_row_bound(self.h, int(max_running_games)))

    def mcts_simulate(self, n_sims, inflight=1):
        check(self.lib.crl_mcts_simulate(self.h, int(n_sims), int(inflight)))

    def root_stats(self, want=("visits", "values", "priors", "moves", "replies", "results")):
        G, M = self.max_games, B.MAX_MOVES
        out = {
            "visits": np.zeros((G, M), dtype=np.int32) if "visits" in want else None,
            "values": np.zeros((G, M), dtype=np.float64) if "values" in want else None,
            "priors": np.zeros((G, M), dtype=np.float32) if "priors" in want else None,
            "moves": np.zeros((G, M), dtype=np.uint16) if "moves" in want else None,
            "replies": np.zeros((G, M), dtype=np.uint16) if "replies" in want else None,
            "results": np.zeros((G, M), dtype=np.int8) if "results" in want else None,
            "n_children": np.zeros(G, dtype=np.int32),
            "root_visits": np.zeros(G, dtype=np.int32),
            "root_values": np.zeros(G, dtype=np.float64),
        }

        def p(name, ct):
            return _np(out[name], ct) if out[name] is not None else None

        check(self.lib.crl_mcts_root_stats_host(self.h, p("visits", ctypes.c_int32), p("values", ctypes.c_double),
                                                p("priors", ctypes.c_float), p("moves", ctypes.c_uint16),
                                                p("replies", ctypes.c_uint16), p("results", ctypes.c_int8),
                                                p("n_children", ctypes.c_int32), p("root_visits", ctypes.c_int32),
                                                p("root_values", ctypes.c_double)))
        return out

    def commit(self, picks, apply=True):
        pk = np.ascontiguousarray(np.asarray(picks, dtype=np.int32))
        out = np.zeros((self.max_games, 2), dtype=np.uint16)
        check(self.lib.crl_mcts_commit_host(self.h, _np(pk, ctypes.c_int32), _np(out, ctypes.c_uint16), int(bool(apply))))
        torch.cuda.current_stream(self.device).synchronize()
        return out

    def node_dump(self, game=0, cap=None):
        cap = self.max_nodes + 1 if cap is None else cap
        arr = (_lib.NodeHost * cap)()
        n = ctypes.c_int32(0)
        check(self.lib.crl_mcts_node_dump_host(self.h, int(game), arr, cap, ctypes.byref(n)))
        return [arr[i] for i in range(min(n.value, cap))]

    def counters(self):
        c = np.zeros(3, dtype=np.int64)
        check(self.lib.crl_counters_host(self.h, _np(c, ctypes.c_int64)))
        r = np.zeros(1, dtype=np.int64)
        check(self.lib.crl_reuse_count_host(self.h, _np(r, ctypes.c_int64)))
        return {"simulations": int(c[0]), "evaluations": int(c[1]), "launches": int(c[2]), "reused_evaluations": int(r[0])}

    def profile(self, enable):
        check(self.lib.crl_profile(self.h, int(bool(enable))))

    def profile_read(self):
        k = len(_lib.KERNEL_CLASSES)
        ms = np.zeros(k, dtype=np.float64)
        ln = np.zeros(k, dtype=np.int64)
        check(self.lib.crl_profile_read_host(self.h, _np(ms, ctypes.c_double), _np(ln, ctypes.c_int64), k))
        return {name: {"ms": float(ms[i]), "launches": int(ln[i])} for i, name in enumerate(_lib.KERNEL_CLASSES)}
