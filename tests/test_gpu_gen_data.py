"""Generating training games on the GPU (crl_games_ab_pick_host, Engine.games_ab_pick, chessrl_b200/gen_data.py,
DESIGN.md 3.7).

- margin 0 is games_ab_move: moves, scores and node counts on 4,096 positions;
- margin > 0: the device equals the g++ build of the same code (tests/hostsim/ab_pick_hostsim.cpp) on 4,096 positions at
  (2,2) and (3,4), with random salts and plies on both sides of pick_plies, and the oracle on 64 positions at (2,2);
- masked, parked and finished lanes and every other engine state are untouched, a later search is bit-identical, and
  out-of-range arguments are refused;
- generate_games: the same games on 16 and 64 lanes, every ply the host build's pick, a sample the oracle's, every game
  replays under the oracle with its result; a file written by the CLI trains with supervised.train."""
import concurrent.futures as cf
import json
import multiprocessing as mp
import os
import random

import numpy as np
import pytest

import ab_oracle as A
import ab_pick_oracle as P
import chessrl_oracle as O
from chessrl_b200 import boards as B
from chessrl_b200 import gen_data
from chessrl_b200._lib import CRL_EINVAL, EVAL_HASH, CrlError
from chessrl_b200.engine import Engine
from fake_gen_engine import lane_record
from hostsim import ab_pick as HP
from test_alphabeta_host import fuzz_fens, playout_fens

pytestmark = pytest.mark.gpu
chess = O.chess
G = 4096
PICK_PLIES = 16


@pytest.fixture(scope="module")
def positions():
    """4,096 fuzz and playout positions, each followed by 0..31 seeded random legal plies (so the lane's ply, its move
    count, lies on both sides of PICK_PLIES) that do not end the game; a random salt per lane.
    Returns (FEN after the plies, ply, start records, move lists, salts)."""
    rng = random.Random(7)
    fens, plies, starts, lists = [], [], [], []
    for f in fuzz_fens(G // 2, 601) + playout_fens(G // 2, 602):
        b = chess.Board(f)
        for _ in range(rng.randrange(2 * PICK_PLIES)):
            b.push(rng.choice(list(b.generate_legal_moves())))
            if A.terminal(b, list(b.generate_legal_moves()), 0) is not None:
                b.pop()
                break
        fens.append(b.fen())
        plies.append(len(b.move_stack))
        starts.append(B.record_from_fen(f))
        lists.append([B.uci_to_move(m.uci()) for m in b.move_stack])
    salts = np.array([rng.getrandbits(64) for _ in range(G)], dtype=np.uint64)
    return fens, np.array(plies), np.stack(starts), lists, salts


@pytest.fixture(scope="module")
def engine(positions):
    eng = Engine(max_games=G, max_nodes=2, avg_moves=64)
    eng.games_set(positions[2], positions[3])
    yield eng
    eng.close()


def _ply(recs):
    return ((recs[:, 8] >> np.uint64(38)) & np.uint64(16383)).astype(np.int64)


def test_lanes_hold_their_plies(engine, positions):
    rec, plies, res = engine.games_get()
    assert np.array_equal(_ply(rec), positions[1]) and np.array_equal(plies, positions[1])
    assert (res == B.RESULT_NONE).all()
    assert (positions[1] < PICK_PLIES).sum() > G // 4 and (positions[1] >= PICK_PLIES).sum() > G // 4


@pytest.mark.parametrize("depth,qdepth", [(2, 2), (3, 4)])
def test_margin_zero_is_games_ab_move(engine, positions, depth, qdepth):
    want = engine.games_ab_move(depth, qdepth)
    got = engine.games_ab_pick(depth, qdepth, 0, 1000, positions[4])
    for a, b in zip(got, want):
        assert np.array_equal(a, b)


def _host_all(recs, depth, qdepth, margin, salts):
    with cf.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:      # (ctypes releases the GIL)
        return list(ex.map(lambda a: HP.pick(a[0], depth, qdepth, margin, PICK_PLIES, int(a[1])), zip(recs, salts)))


@pytest.mark.parametrize("depth,qdepth,margin", [(2, 2, 25), (3, 4, 15)])
def test_device_equals_host_build(engine, positions, depth, qdepth, margin):
    fens, salts = positions[0], positions[4]
    recs = engine.games_get()[0]                          # the records as the device holds them
    moves, scores, nodes = engine.games_ab_pick(depth, qdepth, margin, PICK_PLIES, salts)
    best = engine.games_ab_move(depth, qdepth)
    host = _host_all(recs, depth, qdepth, margin, salts)
    for lane, (hm, hs, hn) in enumerate(host):
        assert (int(moves[lane]), int(scores[lane]), int(nodes[lane])) == (hm, hs, hn), (fens[lane], depth, qdepth)
    assert np.array_equal(nodes, best[2])
    differ = moves != best[0]
    ply = _ply(recs)
    assert not differ[ply >= PICK_PLIES].any() and differ[ply < PICK_PLIES].sum() > G // 50


def _oracle_job(args):
    fen, ply, salt = args
    return P.pick(chess.Board(fen), 2, 2, 25, PICK_PLIES, salt, ply=ply)


def test_device_equals_oracle(engine, positions):
    fens, ply, salts = positions[0], positions[1], positions[4]
    lanes = np.concatenate([np.arange(32), G // 2 + np.arange(32)])
    mask = np.zeros(G, dtype=np.uint8)
    mask[lanes] = 1
    moves, scores, _ = engine.games_ab_pick(2, 2, 25, PICK_PLIES, salts, mask=mask)
    with mp.get_context("fork").Pool(min(16, os.cpu_count() or 4)) as pool:
        want = pool.map(_oracle_job, [(fens[l], int(ply[l]), int(salts[l])) for l in lanes])
    for lane, (wm, ws) in zip(lanes, want):
        assert (B.move_to_uci(int(moves[lane])), int(scores[lane])) == (wm, ws), fens[lane]
    off = np.ones(G, dtype=bool)
    off[lanes] = False
    assert (moves[off] == B.MOVE_NONE).all()


def test_unselected_parked_and_finished_lanes_are_untouched():
    n = 64
    eng = Engine(max_games=n, max_nodes=2, avg_moves=64)
    try:
        eng.games_set(np.stack([B.record_from_fen(f) for f in playout_fens(n, 17)]))
        eng.games_set(B.record_from_fen("6k1/5ppp/8/8/8/8/8/R5K1 w - - 0 1")[None, :], [[B.uci_to_move("a1a8")]], first=9)
        active = np.ones(n, dtype=np.uint8)
        active[[3, 4]] = 0
        eng.games_set_active(active)
        before = eng.games_get(0, n), [eng.game_moves(g) for g in range(n)]
        mask = np.ones(n, dtype=np.uint8)
        mask[[7, 8]] = 0
        salts = np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
        moves, scores, nodes = eng.games_ab_pick(2, 2, 30, PICK_PLIES, salts, mask=mask)
        after = eng.games_get(0, n), [eng.game_moves(g) for g in range(n)]
        for x, y in zip(before[0], after[0]):
            assert np.array_equal(x, y)
        assert all(np.array_equal(x, y) for x, y in zip(before[1], after[1]))
        idle = [3, 4, 7, 8, 9]
        assert (moves[idle] == B.MOVE_NONE).all() and (scores[idle] == 0).all() and (nodes[idle] == 0).all()
        busy = [g for g in range(n) if g not in idle]
        assert (moves[busy] != B.MOVE_NONE).all() and (nodes[busy] > 1).all()
    finally:
        eng.close()


def _hash_search(with_pick):
    n, sims = 64, 48
    eng = Engine(max_games=n, max_nodes=sims + 1, avg_moves=64)
    try:
        eng.set_evaluator(EVAL_HASH, 5, 24)
        eng.games_set(np.stack([B.record_from_fen(f) for f in playout_fens(n, 8)]))
        if with_pick:
            eng.games_ab_pick(3, 4, 40, 100, np.arange(n, dtype=np.uint64))
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


def test_out_of_range_arguments():
    eng = Engine(max_games=4, max_nodes=2, avg_moves=64)
    try:
        eng.games_set(np.tile(B.record_from_fen(), (4, 1)))
        salt = np.zeros(4, dtype=np.uint64)
        for d, q, m, p in ((0, 0, 10, 16), (6, 0, 10, 16), (1, -1, 10, 16), (1, 9, 10, 16), (1, 0, -1, 16),
                           (1, 0, 10, -1)):
            with pytest.raises(CrlError) as ei:
                eng.games_ab_pick(d, q, m, p, salt)
            assert ei.value.status == CRL_EINVAL
        with pytest.raises(ValueError):
            eng.games_ab_pick(1, 0, 10, 16, np.zeros(3, dtype=np.uint64))
        mv = eng.games_ab_pick(1, 0, 10, 16, np.arange(4, dtype=np.uint64))[0]
        assert (mv != B.MOVE_NONE).all()
    finally:
        eng.close()


# ---- the driver ---------------------------------------------------------------------------------------------------
KW = dict(depth=2, qdepth=2, margin=20, pick_plies=PICK_PLIES, max_plies=160, seed=11)


@pytest.fixture(scope="module")
def games64():
    a, summary = gen_data.generate_games(64, lanes=64, **KW)
    b, _ = gen_data.generate_games(64, lanes=16, **KW)
    return a, b, summary


def _replay_picks(game, salt):
    """Every ply of the game against the host build's pick for that position; returns (the oracle's result, the
    positions as (fen, ply))."""
    g = O.OGame()
    seen = []
    for m in game["moves"]:
        mv, _, _ = HP.pick(lane_record(g), KW["depth"], KW["qdepth"], KW["margin"], KW["pick_plies"], salt)
        assert B.move_to_uci(mv) == m, (len(g.board.move_stack), m)
        seen.append((g.board.fen(), len(g.board.move_stack)))
        assert g.move(m)
    return g.get_result(), seen


def test_generate_games_lanes_host_build_and_oracle(games64):
    a, b, summary = games64
    assert a == b
    assert summary["games"] == 64 and summary["distinct_fraction"] > 0.9
    salts = gen_data.game_salts(KW["seed"], 0, 64)
    with cf.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        replays = list(ex.map(lambda j: _replay_picks(a[j], int(salts[j])), range(64)))
    sample = []
    for j, (game, (res, seen)) in enumerate(zip(a, replays)):
        assert game["result"] == res or (game["result"] is None and len(game["moves"]) >= KW["max_plies"]), j
        assert game["player_color"] == (j % 2 == 0)
        sample += [(fen, ply, int(salts[j]), game["moves"][ply]) for fen, ply in seen[:: max(1, len(seen) // 2)][:2]]
    assert len(sample) >= 64
    with mp.get_context("fork").Pool(min(16, os.cpu_count() or 4)) as pool:
        want = pool.map(_oracle_sample, sample)
    assert want == [s[3] for s in sample]


def _oracle_sample(s):
    fen, ply, salt, _ = s
    return P.pick(chess.Board(fen), KW["depth"], KW["qdepth"], KW["margin"], KW["pick_plies"], salt, ply=ply)[0]


def test_cli_file_trains_with_supervised(tmp_path):
    from chessrl_b200 import supervised
    out = tmp_path / "games.json"
    summary = gen_data.main([str(out), "--games", "8", "--depth", "1", "--qdepth", "2", "--max-plies", "60",
                             "--seed", "2"])
    saved = json.loads(out.read_text())
    assert len(saved) == 8 and summary["games"] == 8
    assert [g["player_color"] for g in saved] == [j % 2 == 0 for j in range(8)]
    model_dir = tmp_path / "model"
    model_dir.mkdir()
    supervised.train(str(model_dir), str(out), epochs=1, batch_size=8)
    assert any(f.endswith(".h5") for f in os.listdir(model_dir))
