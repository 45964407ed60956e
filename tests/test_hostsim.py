"""CPU-side check of the DEVICE rule / tree code: chessrl_b200/csrc/{chess_core,tree_core,hash_eval}.cuh are
compiled by g++ into a test-only harness (tests/hostsim) and compared with the oracle and the goldens.  This is
what lets the kernels' arithmetic be validated in the GPU-less build container; the GPU tests repeat the same
comparisons through the C ABI on the real kernels."""
import ctypes
import json
import os

import numpy as np
import pytest

import chessrl_oracle as O
import hostsim
import perft_kats
import position_fuzz
from chessrl_b200 import boards as B

chess = O.chess
u64p = ctypes.POINTER(ctypes.c_uint64)
u16p = ctypes.POINTER(ctypes.c_uint16)
i32p = ctypes.POINTER(ctypes.c_int)


@pytest.fixture(scope="module")
def lib():
    L = hostsim.load()
    L.hs_tree_new.restype = ctypes.c_void_p
    L.hs_tree_new.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int16)]
    L.hs_game_set.argtypes = [ctypes.c_void_p, u64p, u16p, ctypes.c_int]
    L.hs_game_move.argtypes = [ctypes.c_void_p, ctypes.c_uint16]    # undeclared, the handle would pass as a 32-bit int
    L.hs_search.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_int]
    L.hs_search_wave.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint64, ctypes.c_int]
    L.hs_root_stats.argtypes = [ctypes.c_void_p, i32p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float),
                                u16p, u16p, i32p, i32p, ctypes.POINTER(ctypes.c_double)]
    L.hs_grandchild_visits.argtypes = [ctypes.c_void_p, ctypes.c_int, i32p]
    L.hs_edge_score.restype = ctypes.c_double
    L.hs_edge_score.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_float, ctypes.c_int]
    L.hs_history.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, u64p]
    return L


def movegen(lib, rec):
    out = (ctypes.c_uint16 * 256)()
    fl = (ctypes.c_int * 2)()
    n = lib.hs_movegen(rec.ctypes.data_as(u64p), out, fl)
    assert n >= 0
    return [B.move_to_uci(out[i]) for i in range(n)], fl[0], fl[1]


PERFT = [
    (B.STARTING_FEN, [20, 400, 8902, 197281, 4865609]),
    ("r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1", [48, 2039, 97862, 4085603]),
    ("8/2p5/3p4/KP5r/1R3p1k/8/4P1P1/8 w - - 0 1", [14, 191, 2812, 43238, 674624]),
    ("r3k2r/Pppp1ppp/1b3nbN/nP6/BBP1P3/q4N2/Pp1P2PP/R2Q1RK1 w kq - 0 1", [6, 264, 9467, 422333]),
    ("rnbq1k1r/pp1Pbppp/2p5/8/2B5/8/PPP1NnPP/RNBQK2R w KQ - 1 8", [44, 1486, 62379, 2103487]),
    ("r4rk1/1pp1qppp/p1np1n2/2b1p1B1/2B1P1b1/P1NP1N2/1PP1QPPP/R4RK1 w - - 0 10", [46, 2079, 89890, 3894594]),
]


@pytest.mark.parametrize("fen,expected", PERFT)
def test_device_core_perft(lib, fen, expected):
    rec = B.record_from_fen(fen)
    for d, e in enumerate(expected, 1):
        assert lib.hs_perft(rec.ctypes.data_as(u64p), d, 1) == e           # leaf bulk counting (CountSink: set-wise pawns)
        if d <= 4:
            assert lib.hs_perft(rec.ctypes.data_as(u64p), d, 0) == e       # every leaf generated / made (StoreSink)
    assert lib.hs_perft(rec.ctypes.data_as(u64p), 3, 0) == expected[2]      # without leaf bulk counting


@pytest.mark.parametrize("fen,expected", perft_kats.EDGE)
def test_device_core_perft_rule_corners(lib, fen, expected):
    """Full published depth (the host build runs ~50 M nodes/s), with and without leaf bulk counting."""
    rec = B.record_from_fen(fen)
    for d, e in enumerate(expected, 1):
        assert lib.hs_perft(rec.ctypes.data_as(u64p), d, 1) == e, (fen, d)
        if e <= 300_000:
            assert lib.hs_perft(rec.ctypes.data_as(u64p), d, 0) == e, (fen, d)


@pytest.mark.parametrize("fen", perft_kats.MAX_MOVES)
def test_device_core_most_legal_moves(lib, fen):
    """218 legal moves: same list, same ORDER as the python-chess restatement; children are all distinct."""
    rec = B.record_from_fen(fen)
    ml, chk, epl = movegen(lib, rec)
    assert len(ml) == 218 and not chk and not epl
    assert ml == [m.uci() for m in chess.Board(fen).generate_legal_moves()]
    assert lib.hs_perft(rec.ctypes.data_as(u64p), 1, 1) == 218 and lib.hs_perft(rec.ctypes.data_as(u64p), 1, 0) == 218


def test_device_core_on_unreachable_random_positions(lib):
    """1,000 seeded positions that no game from the start reaches (position_fuzz): move list in python-chess ORDER,
    check / legal-ep flags, FEN, and every child position (make-move) against the restatement."""
    import random
    rng = random.Random(11)
    seen = {"ep": 0, "check": 0, "castle": 0, "promo": 0, "moves": 0}
    for _ in range(1000):
        fen, b = position_fuzz.random_fen(rng)
        rec = B.record_from_fen(fen)
        want = [m.uci() for m in b.generate_legal_moves()]
        got, chk, epl = movegen(lib, rec)
        assert got == want, fen
        assert bool(chk) == b.is_check() and bool(epl) == b.has_legal_en_passant(), fen
        assert B.fen_from_record(rec, epl) == b.fen(), fen
        assert lib.hs_perft(rec.ctypes.data_as(u64p), 1, 1) == len(want), fen          # set-wise counting path
        seen["ep"] += bool(epl)
        seen["check"] += bool(chk)
        for m in want:
            child = rec.copy()
            lib.hs_make(child.ctypes.data_as(u64p), B.uci_to_move(m))
            mv = chess.Move.from_uci(m)
            seen["castle"] += b.is_castling(mv)
            seen["promo"] += len(m) == 5
            b.push(mv)
            ml2, _, epl2 = movegen(lib, child)
            assert B.fen_from_record(child, epl2) == b.fen(), (fen, m)
            assert len(ml2) == sum(1 for _ in b.generate_legal_moves()), (fen, m)
            assert lib.hs_perft(child.ctypes.data_as(u64p), 1, 1) == len(ml2), (fen, m)
            b.pop()
        seen["moves"] += len(want)
    assert seen["ep"] > 50 and seen["check"] > 200 and seen["castle"] > 50 and seen["promo"] > 200, seen


def test_device_core_follows_oracle_along_games(lib, golden_dir):
    cases = json.load(open(os.path.join(golden_dir, "rules.json")))["cases"]
    checked = 0
    for c in cases:
        if c["fen"]:
            ml, _, _ = movegen(lib, B.record_from_fen(c["fen"]))
            assert ml == c["legal"], c["name"]
            continue
        rec, ob, keys = B.record_from_fen(), chess.Board(), []
        for i, m in enumerate(c["moves"]):
            lib.hs_make(rec.ctypes.data_as(u64p), B.uci_to_move(m))
            ob.push(chess.Move.from_uci(m))
            ml, chk, epl = movegen(lib, rec)
            assert ml == [x.uci() for x in ob.generate_legal_moves()], (c["name"], i)
            assert bool(chk) == ob.is_check() and bool(epl) == ob.has_legal_en_passant()
            assert B.fen_from_record(rec, epl) == ob.fen()
            k = lib.hs_key(rec.ctypes.data_as(u64p), epl)
            keys.append(k)
            rev = B.meta_fields(rec[8])["rev"]
            reps = sum(1 for j in range(1, rev + 1) if len(keys) - 1 - j >= 0 and keys[len(keys) - 1 - j] == k)
            res = lib.hs_result(rec.ctypes.data_as(u64p), len(ml), chk, reps)
            assert (None if res == 2 else res) == O.OGame(board=ob).get_result(), (c["name"], i)
            checked += 1
    assert checked > 3000


def _label_table():
    tab = np.full((5, 64, 64), -1, dtype=np.int16)
    for i, u in enumerate(O.uci_labels()):
        m = B.uci_to_move(u)
        tab[(m >> 12) & 7, m & 63, (m >> 6) & 63] = i
    return tab


def test_device_tree_core_matches_reference_mcts(lib, golden_dir):
    tab = _label_table()
    t = lib.hs_tree_new(1024, 1024 * 64, tab.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    cases = json.load(open(os.path.join(golden_dir, "mcts_chess.json")))["cases"]
    for c in cases:
        rec = B.record_from_fen(c["fen"] or B.STARTING_FEN)
        mv = np.array([B.uci_to_move(m) for m in c["moves"]], dtype=np.uint16)
        assert lib.hs_game_set(t, rec.ctypes.data_as(u64p), mv.ctypes.data_as(u16p), len(mv)) == len(mv)
        ev = lib.hs_search(t, c["sims"], c["eval_seed"], c["policy_bits"])
        assert ev >> 24 == 0
        V, W, Pr = (ctypes.c_int * 256)(), (ctypes.c_double * 256)(), (ctypes.c_float * 256)()
        M, R, Rs = (ctypes.c_uint16 * 256)(), (ctypes.c_uint16 * 256)(), (ctypes.c_int * 256)()
        rv, rw = ctypes.c_int(), ctypes.c_double()
        n = lib.hs_root_stats(t, V, W, Pr, M, R, Rs, ctypes.byref(rv), ctypes.byref(rw))
        kids = c["children"]
        assert n == len(kids) and rv.value == c["root_visits"] and rw.value == float.fromhex(c["root_value"])
        for k, kid in enumerate(kids):
            line = [B.move_to_uci(M[k])] + ([B.move_to_uci(R[k])] if R[k] != 0xFFFF else [])
            assert line == kid["line"]
            assert V[k] == kid["visits"] and W[k] == float.fromhex(kid["value"])
            assert (None if Rs[k] == 2 else Rs[k]) == kid["result"]
            G = (ctypes.c_int * 256)()
            ng = lib.hs_grandchild_visits(t, k, G)
            assert [G[j] for j in range(ng)] == kid["grandchild_visits"]
            if float.fromhex(kid["prior"]) != 1.0:
                assert Pr[k] == float.fromhex(kid["prior"])
                assert lib.hs_edge_score(V[k], W[k], Pr[k], Rs[k]) == float.fromhex(kid["score"])


def test_device_tree_core_wave_mode_matches_reference(lib, golden_dir):
    """threads=K > 1 (wave schedule, virtual loss): the device tree code against the reference-driven golden."""
    tab = _label_table()
    t = lib.hs_tree_new(1024, 1024 * 64, tab.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    cases = json.load(open(os.path.join(golden_dir, "mcts_wave.json")))["cases"]
    assert len(cases) >= 60
    for c in cases:
        rec = B.record_from_fen(c["fen"] or B.STARTING_FEN)
        mv = np.array([B.uci_to_move(m) for m in c["moves"]], dtype=np.uint16)
        assert lib.hs_game_set(t, rec.ctypes.data_as(u64p), mv.ctypes.data_as(u16p), len(mv)) == len(mv)
        w = lib.hs_search_wave(t, c["sims"], c["threads"], c["eval_seed"], c["policy_bits"])
        assert w >> 24 == 0 and (w & 0xFFFFFF) == c["waves"], (c["name"], c["threads"], w, c["waves"])
        V, W, Pr = (ctypes.c_int * 256)(), (ctypes.c_double * 256)(), (ctypes.c_float * 256)()
        M, R, Rs = (ctypes.c_uint16 * 256)(), (ctypes.c_uint16 * 256)(), (ctypes.c_int * 256)()
        rv, rw = ctypes.c_int(), ctypes.c_double()
        n = lib.hs_root_stats(t, V, W, Pr, M, R, Rs, ctypes.byref(rv), ctypes.byref(rw))
        kids = c["children"]
        assert n == len(kids) and rv.value == c["root_visits"] and rw.value == float.fromhex(c["root_value"])
        for k, kid in enumerate(kids):
            line = [B.move_to_uci(M[k])] + ([B.move_to_uci(R[k])] if R[k] != 0xFFFF else [])
            assert line == kid["line"]
            assert V[k] == kid["visits"] and W[k] == float.fromhex(kid["value"]), (c["name"], c["threads"], k)
            assert (None if Rs[k] == 2 else Rs[k]) == kid["result"]
            G = (ctypes.c_int * 256)()
            ng = lib.hs_grandchild_visits(t, k, G)
            assert [G[j] for j in range(ng)] == kid["grandchild_visits"]
            if float.fromhex(kid["prior"]) != 1.0:
                assert Pr[k] == float.fromhex(kid["prior"])
                assert lib.hs_edge_score(V[k], W[k], Pr[k], Rs[k]) == float.fromhex(kid["score"])


def test_device_core_results_along_playouts_from_unreachable_positions(lib):
    """80 seeded playouts (<= 90 plies, mostly quiet moves) from position_fuzz positions, a third of them started a
    few plies before the fifty-move claim: legal list, FEN, transposition-key repetitions and Game.get_result
    (game.py:92-109: claim, mate, stalemate, insufficient material) ply by ply against the restatement."""
    import random
    rng = random.Random(31)
    plies, ends, fifty = 0, {}, 0
    for gi in range(80):
        fen, ob = position_fuzz.random_fen(rng)
        if gi % 3 == 0:
            parts = fen.split()
            parts[4] = str(rng.randrange(80, 100))
            fen = " ".join(parts)
            ob = chess.Board(fen)
        rec, keys = B.record_from_fen(fen), []
        for i in range(90):
            legal = [m.uci() for m in ob.generate_legal_moves()]
            ml, chk, epl = movegen(lib, rec)
            assert ml == legal, (fen, i)
            assert B.fen_from_record(rec, epl) == ob.fen(), (fen, i)
            k = lib.hs_key(rec.ctypes.data_as(u64p), epl)
            rev = B.meta_fields(rec[8])["rev"]
            reps = sum(1 for j in range(1, rev + 1) if len(keys) - j >= 0 and keys[len(keys) - j] == k)
            keys.append(k)
            res = lib.hs_result(rec.ctypes.data_as(u64p), len(ml), chk, reps)
            want = O.OGame(board=ob).get_result()
            assert (None if res == 2 else res) == want, (fen, i, res, want)
            if want is not None:
                ends[want] = ends.get(want, 0) + 1
                fifty += ob.halfmove_clock >= 100
                break
            quiet = [m for m in legal if not ob.is_zeroing(chess.Move.from_uci(m))]
            m = rng.choice(quiet if quiet and rng.random() < 0.85 else legal)
            lib.hs_make(rec.ctypes.data_as(u64p), B.uci_to_move(m))
            ob.push(chess.Move.from_uci(m))
            plies += 1
    assert plies > 4000 and ends.get(0, 0) >= 10 and ends.get(1, 0) + ends.get(-1, 0) >= 5 and fifty >= 8, (plies, ends, fifty)


def test_device_tree_core_from_unreachable_roots(lib):
    """Searches rooted at position_fuzz positions (terminal children, promotions, ep and castling inside the tree,
    up to 90 legal moves at the root): visit counts, value sums, results and (move, reply) lines against the
    restated SelfPlayTree with the shared evaluator."""
    import random
    tab = _label_table()
    t = lib.hs_tree_new(1024, 1024 * 220, tab.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    rng = random.Random(21)
    searched = terminal_kids = 0
    for _ in range(60):
        fen, _b = position_fuzz.random_fen(rng)
        sims, seed, bits = rng.choice([5, 33, 90]), rng.randrange(1, 1000), rng.choice([3, 11, 24])
        g = O.OGame(board=chess.Board(fen))
        if g.get_result() is not None:
            continue
        rec = B.record_from_fen(fen)
        none = np.zeros(1, dtype=np.uint16)
        assert lib.hs_game_set(t, rec.ctypes.data_as(u64p), none.ctypes.data_as(u16p), 0) == 0
        assert lib.hs_search(t, sims, seed, bits) >> 24 == 0
        ot = O.OSelfPlayTree(g)
        ot.search_move(O.OAgent(O.hash_evaluator(seed, bits)), max_iters=sims, noise=False)
        V, W, Pr = (ctypes.c_int * 256)(), (ctypes.c_double * 256)(), (ctypes.c_float * 256)()
        M, R, Rs = (ctypes.c_uint16 * 256)(), (ctypes.c_uint16 * 256)(), (ctypes.c_int * 256)()
        rv, rw = ctypes.c_int(), ctypes.c_double()
        n = lib.hs_root_stats(t, V, W, Pr, M, R, Rs, ctypes.byref(rv), ctypes.byref(rw))
        kids = ot.root.children
        assert n == len(kids) and rv.value == ot.root.visits and rw.value == float(ot.root.value), fen
        for k, c in enumerate(kids):
            assert V[k] == c.visits and W[k] == float(c.value), (fen, k)
            r = c.state.get_result()
            terminal_kids += r is not None
            assert (None if Rs[k] == 2 else Rs[k]) == r, (fen, k)
            line = [B.move_to_uci(M[k])] + ([B.move_to_uci(R[k])] if R[k] != 0xFFFF else [])
            assert line == [str(x) for x in c.state.board.move_stack], (fen, k)
        searched += 1
    assert searched >= 50 and terminal_kids >= 3


def test_device_tree_core_wave_mode_from_unreachable_roots(lib):
    """threads=K (wave schedule, virtual loss) rooted at position_fuzz positions: visit counts, value sums, results,
    lines and the NUMBER OF WAVES against the restated SelfPlayTree(threads=K)."""
    import random
    tab = _label_table()
    t = lib.hs_tree_new(1024, 1024 * 220, tab.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    rng = random.Random(23)
    searched = cut = 0
    for _ in range(48):
        fen, _b = position_fuzz.random_fen(rng)
        sims, K = rng.choice([7, 40, 96]), rng.choice([2, 3, 6, 16, 64])
        seed, bits = rng.randrange(1, 1000), rng.choice([3, 11, 24])
        g = O.OGame(board=chess.Board(fen))
        if g.get_result() is not None:
            continue
        rec = B.record_from_fen(fen)
        none = np.zeros(1, dtype=np.uint16)
        assert lib.hs_game_set(t, rec.ctypes.data_as(u64p), none.ctypes.data_as(u16p), 0) == 0
        w = lib.hs_search_wave(t, sims, K, seed, bits)
        ot = O.OSelfPlayTree(g, threads=K)
        ot.search_move(O.OAgent(O.hash_evaluator(seed, bits)), max_iters=sims, noise=False)
        assert w >> 24 == 0 and (w & 0xFFFFFF) == ot.n_waves, (fen, K, sims, w, ot.n_waves)
        cut += ot.n_waves > -(-sims // K)
        V, W, Pr = (ctypes.c_int * 256)(), (ctypes.c_double * 256)(), (ctypes.c_float * 256)()
        M, R, Rs = (ctypes.c_uint16 * 256)(), (ctypes.c_uint16 * 256)(), (ctypes.c_int * 256)()
        rv, rw = ctypes.c_int(), ctypes.c_double()
        n = lib.hs_root_stats(t, V, W, Pr, M, R, Rs, ctypes.byref(rv), ctypes.byref(rw))
        kids = ot.root.children
        assert n == len(kids) and rv.value == ot.root.visits and rw.value == float(ot.root.value), (fen, K)
        for k, c in enumerate(kids):
            assert V[k] == c.visits and W[k] == float(c.value), (fen, K, k)
            assert (None if Rs[k] == 2 else Rs[k]) == c.state.get_result(), (fen, K, k)
            line = [B.move_to_uci(M[k])] + ([B.move_to_uci(R[k])] if R[k] != 0xFFFF else [])
            assert line == [str(x) for x in c.state.board.move_stack], (fen, K, k)
        searched += 1
    assert searched >= 40 and cut >= 3


def test_device_history_walk_matches_planes(lib):
    """The parent-chain walk used for history planes inside the tree reproduces the move-stack walk of
    netencoder._get_game_history for a node deep in a search."""
    tab = _label_table()
    t = lib.hs_tree_new(256, 256 * 64, tab.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    moves = ["e2e4", "e7e5", "g1f3", "b8c6", "f1b5"]
    rec = B.record_from_fen()
    mv = np.array([B.uci_to_move(m) for m in moves], dtype=np.uint16)
    lib.hs_game_set(t, rec.ctypes.data_as(u64p), mv.ctypes.data_as(u16p), len(mv))
    lib.hs_search(t, 120, 1, 24)
    # oracle tree on the same game
    g = O.OGame()
    for m in moves:
        g.move(m)
    ot = O.OSelfPlayTree(g)
    ot.search_move(O.OAgent(O.hash_evaluator(1, 24)), max_iters=120, noise=False)
    # deepest oracle node, and the same node in the device tree by following creation order
    node, path = ot.root, []
    while node.children:
        k = int(np.argmax([c.visits for c in node.children]))
        path.append(k)
        node = node.children[k]
    # device node ids are creation-ordered per game; walk via grandchild bookkeeping is not exported, so compare the
    # history of root children instead (they exercise tree + ring) and of the root itself
    out = (ctypes.c_uint64 * 72)()
    for k, child in enumerate(ot.root.children[:5]):
        cnt = lib.hs_history(t, 1 + k, 2, out)       # root children are nodes 1.. in creation order
        planes = O.planes(child.state)
        got = np.zeros((8, 8, 127))
        for s in range(cnt):
            bb = [out[8 * s + j] for j in range(8)]
            for ci, colour in ((0, 7), (7, 6)):
                occ = bb[colour]
                for sq in range(64):
                    r, f = 7 - (sq >> 3), sq & 7
                    if not (occ >> sq) & 1:
                        got[r, f, 14 * s + ci] = 1
                    for pt in range(6):
                        if (bb[pt] & occ) >> sq & 1:
                            got[r, f, 14 * s + ci + 1 + pt] = 1
        got[:, :, 126] = 1.0 if child.state.turn else 0.0
        assert (got == planes).all(), k


def movegen_warp(lib, rec):
    out = (ctypes.c_uint16 * 256)()
    fl = (ctypes.c_int * 2)()
    n = lib.hs_movegen_warp(rec.ctypes.data_as(u64p), out, fl)
    return [int(out[i]) for i in range(n)], fl[0], fl[1], [int(out[i]) for i in range(n, 256)]


def movegen_words(lib, rec):
    out = (ctypes.c_uint16 * 256)()
    fl = (ctypes.c_int * 2)()
    n = lib.hs_movegen(rec.ctypes.data_as(u64p), out, fl)
    return [int(out[i]) for i in range(n)], fl[0], fl[1]


def test_warp_cooperative_generator_equals_scalar_generator(lib):
    """warp_gen.cuh (32 lanes on one board: per-lane squares + packed prefix sum) run lane by lane on the host:
    the same list in the same ORDER as generate_legal, the same flags, nothing written past the end -- over 6,000
    fuzzed positions (promoted material, checks, double checks, pins, castling, en passant), their children, the perft
    suite, the two 218-move positions and a 300-ply game."""
    import random
    rng = random.Random(31)
    recs = [B.record_from_fen(f) for f, _ in PERFT] + [B.record_from_fen(f) for f in perft_kats.MAX_MOVES] + \
           [B.record_from_fen(f) for f, _ in perft_kats.EDGE]
    seen = {"check": 0, "double": 0, "castle": 0, "promo": 0, "ep": 0, "pinned": 0}
    for _ in range(6000):
        fen, b = position_fuzz.random_fen(rng)
        recs.append(B.record_from_fen(fen))
        if bin(b.checkers_mask()).count("1") > 1:
            seen["double"] += 1
    b = chess.Board()
    for _ in range(300):
        ms = list(b.legal_moves)
        if not ms:
            break
        b.push(rng.choice(ms))
        recs.append(B.record_from_fen(b.fen()))
    extra = []
    for rec in recs[:600]:                                   # one ply deeper: positions after every legal move
        words, _, _ = movegen_words(lib, rec)
        for w in words[:6]:
            child = rec.copy()
            lib.hs_make(child.ctypes.data_as(u64p), w)
            extra.append(child)
    for rec in recs + extra:
        want, chk, epl = movegen_words(lib, rec)
        got, chk2, epl2, tail = movegen_warp(lib, rec)
        assert got == want, B.fen_from_record(rec)
        assert (chk, epl) == (chk2, epl2)
        assert all(x == 0xEEEE for x in tail)                 # no stray writes beyond the list
        seen["check"] += chk
        seen["ep"] += epl
        seen["promo"] += any(w >> 12 for w in want)
        seen["castle"] += any((w & 63) in (4, 60) and abs(((w >> 6) & 63) - (w & 63)) == 2 for w in want)
    assert seen["check"] > 1000 and seen["double"] > 20 and seen["castle"] > 300 and seen["promo"] > 500 and seen["ep"] > 200, seen


def _root_stats(lib, t):
    V, W, Pr = (ctypes.c_int * 256)(), (ctypes.c_double * 256)(), (ctypes.c_float * 256)()
    M, R, Rs = (ctypes.c_uint16 * 256)(), (ctypes.c_uint16 * 256)(), (ctypes.c_int * 256)()
    rv, rw = ctypes.c_int(), ctypes.c_double()
    n = lib.hs_root_stats(t, V, W, Pr, M, R, Rs, ctypes.byref(rv), ctypes.byref(rw))
    return (n, rv.value, rw.value, list(V[:n]), list(W[:n]), [float(x) for x in Pr[:n]], list(M[:n]), list(R[:n]),
            list(Rs[:n]))


def test_evaluation_reuse_plays_the_same_games(lib):
    """Evaluation reuse (tree_core.cuh): a search that takes reply / value / priors from the previous move's tree builds
    exactly the tree a search that evaluates everything builds -- root statistics (visits, value sums, priors, lines,
    results) equal move for move along whole playouts, including games that run into mates / draws inside the tree --
    while running far fewer evaluations whenever the game follows a well-visited child."""
    import random
    lib.hs_search_reuse.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_int]
    lib.hs_commit.argtypes = [ctypes.c_void_p, ctypes.c_int]
    lib.hs_game_result.argtypes = [ctypes.c_void_p]
    tab = _label_table()
    ta = lib.hs_tree_new(256, 256 * 220, tab.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    tb = lib.hs_tree_new(256, 256 * 220, tab.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    rng = random.Random(5)
    none = np.zeros(1, dtype=np.uint16)
    moves_played = evals_plain = evals_reuse = finished = 0
    starts = [B.STARTING_FEN] * 3 + [position_fuzz.random_fen(rng)[0] for _ in range(9)]
    for gi, fen in enumerate(starts):
        if O.OGame(board=chess.Board(fen)).get_result() is not None:
            continue
        rec = B.record_from_fen(fen)
        for t in (ta, tb):
            assert lib.hs_game_set(t, rec.ctypes.data_as(u64p), none.ctypes.data_as(u16p), 0) == 0
        sims, seed, bits = rng.choice([24, 60, 120]), rng.randrange(1, 1000), rng.choice([5, 24])
        for mv in range(40):
            if lib.hs_game_result(ta) != 2:
                finished += 1
                break
            ea = lib.hs_search(ta, sims, seed, bits)
            eb = lib.hs_search_reuse(tb, sims, seed, bits)
            assert ea >> 24 == 0 and eb >> 24 == 0
            sa, sb = _root_stats(lib, ta), _root_stats(lib, tb)
            assert sa == sb, (fen, mv)
            evals_plain += ea
            evals_reuse += eb
            assert eb <= ea
            # the most-visited child three times out of four (reuse pays), a random child otherwise (as the reference's
            # unscaled Dirichlet noise often does); sometimes a move from outside the tree, which must unlink the game
            vis = sa[3]
            k = int(np.argmax(vis)) if rng.random() < 0.75 else rng.randrange(sa[0])
            assert lib.hs_commit(ta, k) == lib.hs_commit(tb, k)
            moves_played += 1
            if rng.random() < 0.1 and lib.hs_game_result(ta) == 2:
                out = (ctypes.c_uint16 * 256)()
                fl = (ctypes.c_int * 2)()
                n = lib.hs_movegen((ctypes.c_uint64 * 9)(*[int(x) for x in _cur_record(lib, ta)]), out, fl)
                if n > 0:
                    m = out[rng.randrange(n)]
                    assert lib.hs_game_move(ta, m) == 1 and lib.hs_game_move(tb, m) == 1
    assert moves_played >= 150 and finished >= 1, (moves_played, finished)
    assert evals_reuse < 0.7 * evals_plain, (evals_reuse, evals_plain)


def _cur_record(lib, t):
    lib.hs_cur_record.argtypes = [ctypes.c_void_p, u64p]
    out = (ctypes.c_uint64 * 9)()
    lib.hs_cur_record(t, out)
    return list(out)
