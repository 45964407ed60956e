"""Repetitions in the alpha-beta search on the GPU (crl_games_ab_search_host CRL_AB_REPETITIONS, DESIGN.md 3.6).

- with flags 0 the new entry point equals crl_games_ab_move_host and crl_games_ab_pick_host bit for bit on the 4,096
  positions of test_gpu_alphabeta.py;
- with repetitions on the device equals the g++ build of the same code (tests/hostsim/ab_rep_hostsim.cpp) in move,
  score and node count on lanes with real games (set with move lists, some longer than the 128-slot key ring, some set
  from a FEN, some parked, finished or unmasked), for the first best move and the seeded pick, and equals the oracle
  (tests/ab_rep_oracle.py) on 64 lanes;
- the call changes no engine state a later search could see, and its CRL_EINVAL cases are refused;
- gen_data --repetitions and an arena match with alphabeta:2:2:r against the host build and the oracle."""
import concurrent.futures as cf
import multiprocessing as mp
import os

import numpy as np
import pytest

import ab_rep_oracle as R
import chessrl_oracle as O
from chessrl_b200 import arena, gen_data
from chessrl_b200 import boards as B
from chessrl_b200._lib import CRL_EINVAL, EVAL_HASH, CrlError
from chessrl_b200.engine import CRL_AB_REPETITIONS, Engine
from hostsim import ab_rep as HR
from test_alphabeta_host import fuzz_fens, playout_fens

pytestmark = pytest.mark.gpu
chess = O.chess
G = 4096


def _threads(fn, items):
    with cf.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:      # (ctypes releases the GIL)
        return list(ex.map(fn, items))


# ---- flags 0 -------------------------------------------------------------------------------------------------------
def test_flags_zero_equals_the_existing_calls():
    fens = fuzz_fens(G // 2, 501) + playout_fens(G // 2, 502)
    eng = Engine(max_games=G, max_nodes=2, avg_moves=64)
    try:
        eng.games_set(np.stack([B.record_from_fen(f) for f in fens]))
        salt = np.arange(G, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
        mask = (np.arange(G) % 5 != 0).astype(np.uint8)
        for d, q in ((1, 0), (2, 2), (3, 4)):
            for a, b in zip(eng.games_ab_move(d, q), eng.games_ab_search(d, q)):
                assert np.array_equal(a, b), (d, q)
            for a, b in zip(eng.games_ab_move(d, q, mask=mask), eng.games_ab_search(d, q, mask=mask)):
                assert np.array_equal(a, b), (d, q)
            for margin in (0, 20):
                for a, b in zip(eng.games_ab_pick(d, q, margin, 1000, salt),
                                eng.games_ab_search(d, q, 0, margin, 1000, salt)):
                    assert np.array_equal(a, b), (d, q, margin)
    finally:
        eng.close()


# ---- lanes with games ----------------------------------------------------------------------------------------------
def build_games(eng, seed, long_share=8):
    """Plays seeded games on the device: per ply each lane plays the reverse of its own previous move when that is
    legal (with probability 0.6), else a random legal move, for a per-lane number of plies (0..160; one lane in
    `long_share` 130..230, past the 128-slot key ring).  Every 16th lane starts from a playout FEN (no history before
    it).  Returns the start records."""
    n = eng.max_games
    rng = np.random.default_rng(seed)
    starts = np.tile(B.record_from_fen(), (n, 1))
    fen_lanes = np.arange(0, n, 16)
    for lane, fen in zip(fen_lanes, playout_fens(len(fen_lanes), seed)):
        starts[lane] = B.record_from_fen(fen)
    eng.games_set(starts)
    target = rng.integers(0, 161, n)
    long = rng.random(n) < 1.0 / long_share
    target[long] = rng.integers(130, 231, int(long.sum()))
    prev = np.full((n, 2), B.MOVE_NONE, dtype=np.int64)          # own previous move, the opponent's last move
    for step in range(int(target.max())):
        legal, cnt = eng.games_legal()
        _, _, res = eng.games_get(0, n)
        go = (step < target) & (res == B.RESULT_NONE) & (cnt > 0)
        pick = legal[np.arange(n), (rng.random(n) * np.maximum(cnt, 1)).astype(np.int64)].astype(np.int64)
        own = prev[:, 0]
        back = ((own >> 6) & 63) | ((own & 63) << 6)
        ok = (own != B.MOVE_NONE) & ((legal == back[:, None]) & (np.arange(B.MAX_MOVES)[None, :] < cnt[:, None])).any(1)
        use_back = ok & (rng.random(n) < 0.6)
        mv = np.where(use_back, back, pick)
        mv = np.where(go, mv, B.MOVE_NONE).astype(np.uint16)
        eng.games_play(mv)
        prev[go] = np.stack([prev[go, 1], mv[go].astype(np.int64)], 1)
    return starts


@pytest.fixture(scope="module")
def games():
    """An engine of G lanes with games, the lanes' records in game order (start first), and the searched lanes' mask:
    lanes 3 and 4 parked, every 7th lane unmasked, and lane 9 finished by a mate."""
    eng = Engine(max_games=G, max_nodes=2, avg_moves=64)
    starts = build_games(eng, 11)
    eng.games_set(B.record_from_fen("6k1/5ppp/8/8/8/8/8/R5K1 w - - 0 1")[None, :], [[B.uci_to_move("a1a8")]], first=9)
    starts[9] = B.record_from_fen("6k1/5ppp/8/8/8/8/8/R5K1 w - - 0 1")
    active = np.ones(G, dtype=np.uint8)
    active[[3, 4]] = 0
    eng.games_set_active(active)
    mask = (np.arange(G) % 7 != 6).astype(np.uint8)
    moves = eng.games_moves(np.arange(G))
    replay = Engine(max_games=1, max_nodes=2, avg_moves=64)
    try:
        recs = [replay.game_replay(starts[g], moves[g], records=True)["records"] for g in range(G)]
    finally:
        replay.close()
    _, plies, res = eng.games_get(0, G)
    searched = (mask == 1) & (active == 1) & (res == B.RESULT_NONE)
    assert (plies > 128).sum() >= G // 16 and searched.sum() > G // 2 and not searched[[3, 4, 9]].any()
    yield eng, starts, moves, recs, mask, searched
    eng.close()


def _check(out, want, searched, lanes):
    moves, scores, nodes = out
    for lane, w in zip(lanes, want):
        assert (int(moves[lane]), int(scores[lane]), int(nodes[lane])) == w, lane
    off = ~searched
    assert (moves[off] == B.MOVE_NONE).all() and (scores[off] == 0).all() and (nodes[off] == 0).all()


@pytest.mark.parametrize("depth,qdepth,n", [(1, 0, G), (2, 2, G), (3, 4, G), (4, 4, 512)])
def test_device_equals_host_build(games, depth, qdepth, n):
    eng, _, _, recs, mask, searched = games
    m = mask.copy()
    m[n:] = 0
    s = searched & (m == 1)
    out = eng.games_ab_move(depth, qdepth, mask=m, repetitions=True)
    lanes = np.nonzero(s)[0]
    _check(out, _threads(lambda g: HR.search(recs[g], depth, qdepth), lanes), s, lanes)
    plain = eng.games_ab_move(depth, qdepth, mask=m)
    changed = sum((out[0][g], out[1][g]) != (plain[0][g], plain[1][g]) for g in lanes)
    assert changed > 0                                  # the lanes' games make the rule bite


@pytest.mark.parametrize("margin", [0, 20])
def test_pick_equals_host_build(games, margin):
    eng, _, _, recs, mask, searched = games
    salt = (np.arange(G, dtype=np.uint64) + np.uint64(7)) * np.uint64(0xD1B54A32D192ED03)
    out = eng.games_ab_pick(2, 2, margin, 1000, salt, mask=mask, repetitions=True)
    lanes = np.nonzero(searched)[0]
    want = _threads(lambda g: HR.search(recs[g], 2, 2, margin=margin, pick_plies=1000, salt=int(salt[g])), lanes)
    _check(out, want, searched, lanes)


def _oracle_job(args):
    start_fen, moves, depth, qdepth = args
    b = chess.Board(start_fen)
    for m in moves:
        b.push(chess.Move.from_uci(m))
    return R.search(b, depth, qdepth)[:2]


@pytest.mark.parametrize("depth,qdepth", [(2, 2), (3, 2)])
def test_device_equals_oracle(games, depth, qdepth):
    eng, starts, moves, _, mask, searched = games
    lanes = np.nonzero(searched)[0][::max(1, int(searched.sum()) // 64)][:64]
    m = np.zeros(G, dtype=np.uint8)
    m[lanes] = 1
    out = eng.games_ab_move(depth, qdepth, mask=m, repetitions=True)
    jobs = [(B.fen_from_record(starts[g]), [B.move_to_uci(int(x)) for x in moves[g]], depth, qdepth) for g in lanes]
    with mp.get_context("fork").Pool(min(16, os.cpu_count() or 4)) as pool:
        want = pool.map(_oracle_job, jobs)
    for lane, w in zip(lanes, want):
        assert (B.move_to_uci(int(out[0][lane])), int(out[1][lane])) == w, lane


# ---- engine state and refusals ------------------------------------------------------------------------------------
def _hash_search(with_ab):
    n, sims = 64, 48
    eng = Engine(max_games=n, max_nodes=sims + 1, avg_moves=64)
    try:
        eng.set_evaluator(EVAL_HASH, 5, 24)
        build_games(eng, 3)
        before = eng.games_get(0, n), eng.games_moves(np.arange(n))
        if with_ab:
            eng.games_ab_move(3, 4, repetitions=True)
            eng.games_ab_pick(2, 2, 20, 1000, np.arange(n, dtype=np.uint64), repetitions=True)
        after = eng.games_get(0, n), eng.games_moves(np.arange(n))
        assert all(np.array_equal(x, y) for x, y in zip(before[0], after[0]))
        assert all(np.array_equal(x, y) for x, y in zip(before[1], after[1]))
        eng.mcts_begin_move()
        eng.mcts_simulate(sims)
        return eng.root_stats(), [eng.node_dump(g) for g in (0, 17, 63)]
    finally:
        eng.close()


def test_search_after_a_call_is_bit_identical():
    (a, da), (b, db) = _hash_search(False), _hash_search(True)
    for k in a:
        if a[k] is not None:
            assert np.array_equal(a[k], b[k]), k
    for x, y in zip(da, db):
        assert [bytes(n) for n in x] == [bytes(n) for n in y]


def test_refusals():
    eng = Engine(max_games=4, max_nodes=2, avg_moves=64)
    try:
        eng.games_set(np.tile(B.record_from_fen(), (4, 1)))
        salt = np.arange(4, dtype=np.uint64)
        for kw in (dict(flags=2), dict(flags=-1), dict(depth=0), dict(depth=6), dict(qdepth=9), dict(qdepth=-1),
                   dict(margin=-1, salt=salt), dict(pick_plies=-1, salt=salt), dict(margin=5), dict(pick_plies=3)):
            args = dict(depth=1, qdepth=0, flags=CRL_AB_REPETITIONS)
            args.update(kw)
            with pytest.raises(CrlError) as ei:
                eng.games_ab_search(**args)
            assert ei.value.status == CRL_EINVAL, kw
        assert eng.games_ab_search(1, 0, CRL_AB_REPETITIONS)[0][0] != B.MOVE_NONE
    finally:
        eng.close()


# ---- drivers -------------------------------------------------------------------------------------------------------
KW = dict(depth=2, qdepth=2, margin=20, pick_plies=16, max_plies=160, seed=3, repetitions=True)


def test_gen_data_repetitions():
    a, sa = gen_data.generate_games(64, lanes=16, **KW)
    b, _ = gen_data.generate_games(64, lanes=64, **KW)
    assert a == b
    replay = Engine(max_games=1, max_nodes=2, avg_moves=64)
    try:
        for j, g in enumerate(a):
            mv = [B.uci_to_move(m) for m in g["moves"]]
            recs = replay.game_replay(B.record_from_fen(), mv, records=True)["records"]
            salt = int(gen_data.game_salts(3, j, 1)[0])
            for ply, m in enumerate(mv):
                assert HR.search(recs[:ply + 1], 2, 2, margin=20, pick_plies=16, salt=salt)[0] == m, (j, ply)
            og = O.OGame()
            for m in g["moves"]:
                assert og.move(m)
            assert g["result"] == og.get_result() or (g["result"] is None and len(g["moves"]) >= 160)
    finally:
        replay.close()
    assert sa["games"] == 64


def test_arena_alphabeta_with_repetitions_equals_the_oracle():
    ab = arena.AlphaBetaPlayer.parse("alphabeta:2:2:r")
    out, summary = arena.play_match(arena.HashPlayer(3), ab, games=4, sims=16, lanes=4, opening_plies=4, max_plies=40,
                                    seed=9)
    checked = 0
    for g in out:
        b = chess.Board()
        for ply, m in enumerate(g["moves"]):
            if ply >= 4 and (ply % 2 == 0) != g["a_white"] and ply % 4 < 2:
                assert R.search(b, 2, 2)[0] == m, (ply, m)
                checked += 1
            b.push(chess.Move.from_uci(m))
    assert checked >= 8 and summary["played"] == 4
