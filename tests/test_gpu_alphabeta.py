"""The fixed-depth alpha-beta opponent on the GPU (crl_games_ab_move_host, Engine.games_ab_move, DESIGN.md 3.6).

- device against the g++ build of the same code (tests/hostsim/ab_hostsim.cpp): move, score and node count, on 4,096
  fuzz and playout positions at (1,0), (2,2), (3,4) and a subset at (4,4);
- device against the oracle (oracle/ab_oracle.py) on 64 positions at (2,2) and (3,2);
- lanes are independent, unselected / parked / finished lanes are untouched, the call changes no engine state a later
  search could see, and out-of-range limits are refused;
- matches (arena.play_match) and the policy benchmark loop (benchmark.play_policy_games) with an AlphaBetaPlayer."""
import concurrent.futures as cf
import multiprocessing as mp
import os

import numpy as np
import pytest

import ab_oracle as A
import chessrl_oracle as O
import netpacks
from chessrl_b200 import arena
from chessrl_b200 import boards as B
from chessrl_b200 import model
from chessrl_b200._lib import CRL_EINVAL, EVAL_HASH, CrlError
from chessrl_b200.engine import Engine
from hostsim import ab as H
from test_alphabeta_host import fuzz_fens, oracle_game, playout_fens

pytestmark = pytest.mark.gpu
chess = O.chess
G = 4096


@pytest.fixture(scope="module")
def positions():
    fens = fuzz_fens(G // 2, 501) + playout_fens(G // 2, 502)
    return fens, np.stack([B.record_from_fen(f) for f in fens])


@pytest.fixture(scope="module")
def engine(positions):
    eng = Engine(max_games=G, max_nodes=2, avg_moves=64)
    eng.games_set(positions[1])
    yield eng
    eng.close()


def _host_all(records, depth, qdepth):
    with cf.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:      # (ctypes releases the GIL)
        return list(ex.map(lambda r: H.root(r, depth, qdepth), records))


@pytest.mark.parametrize("depth,qdepth,n", [(1, 0, G), (2, 2, G), (3, 4, G), (4, 4, 512)])
def test_device_equals_host_build(engine, positions, depth, qdepth, n):
    fens, recs = positions
    mask = np.zeros(G, dtype=np.uint8)
    lanes = np.arange(G) if n == G else np.concatenate([np.arange(n // 2), G // 2 + np.arange(n // 2)])
    mask[lanes] = 1
    moves, scores, nodes = engine.games_ab_move(depth, qdepth, mask=None if n == G else mask)
    host = _host_all(recs[lanes], depth, qdepth)
    for lane, (hm, hs, hn) in zip(lanes, host):
        assert (int(moves[lane]), int(scores[lane]), int(nodes[lane])) == (hm, hs, hn), (fens[lane], depth, qdepth)
    off = np.ones(G, dtype=bool)
    off[lanes] = False
    assert (moves[off] == B.MOVE_NONE).all() and (scores[off] == 0).all() and (nodes[off] == 0).all()


def _oracle_job(args):
    fen, depth, qdepth = args
    return A.search_fen(fen, depth, qdepth)


@pytest.mark.parametrize("depth,qdepth", [(2, 2), (3, 2)])
def test_device_equals_oracle(engine, positions, depth, qdepth):
    fens, _ = positions
    lanes = np.concatenate([np.arange(32), G // 2 + np.arange(32)])
    mask = np.zeros(G, dtype=np.uint8)
    mask[lanes] = 1
    moves, scores, _ = engine.games_ab_move(depth, qdepth, mask=mask)
    with mp.get_context("fork").Pool(min(16, os.cpu_count() or 4)) as pool:
        want = pool.map(_oracle_job, [(fens[l], depth, qdepth) for l in lanes])
    for lane, (wm, ws) in zip(lanes, want):
        assert (B.move_to_uci(int(moves[lane])), int(scores[lane])) == (wm, ws), fens[lane]


def test_lane_independence(positions):
    fens, recs = positions
    eng = Engine(max_games=G, max_nodes=2, avg_moves=64)
    try:
        r = recs.copy()
        same = B.record_from_fen("r1bqkbnr/pppp1ppp/2n5/4p3/4P3/5N2/PPPP1PPP/RNBQKB1R w KQkq - 2 3")
        for lane in (0, 1, G - 1):
            r[lane] = same
        eng.games_set(r)
        out = eng.games_ab_move(3, 4)
        for a in out:
            assert a[0] == a[1] == a[G - 1]
        assert out[0][0] == H.root(same, 3, 4)[0]
    finally:
        eng.close()


def test_unselected_parked_and_finished_lanes_are_untouched():
    n = 64
    eng = Engine(max_games=n, max_nodes=2, avg_moves=64)
    try:
        fens = playout_fens(n, 7)
        eng.games_set(np.stack([B.record_from_fen(f) for f in fens]))
        # lane 9 finishes: mate in one, played
        eng.games_set(B.record_from_fen("6k1/5ppp/8/8/8/8/8/R5K1 w - - 0 1")[None, :], [[B.uci_to_move("a1a8")]], first=9)
        active = np.ones(n, dtype=np.uint8)
        active[[3, 4]] = 0
        eng.games_set_active(active)
        before = eng.games_get(0, n), [eng.game_moves(g) for g in range(n)]
        mask = np.ones(n, dtype=np.uint8)
        mask[[7, 8]] = 0
        moves, scores, nodes = eng.games_ab_move(2, 2, mask=mask)
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


def _hash_search(with_ab):
    n, sims = 64, 48
    eng = Engine(max_games=n, max_nodes=sims + 1, avg_moves=64)
    try:
        eng.set_evaluator(EVAL_HASH, 5, 24)
        eng.games_set(np.stack([B.record_from_fen(f) for f in playout_fens(n, 8)]))
        if with_ab:
            eng.games_ab_move(3, 4)
        eng.mcts_begin_move()
        eng.mcts_simulate(sims)
        st = eng.root_stats()
        return st, [eng.node_dump(g) for g in (0, 17, 63)]
    finally:
        eng.close()


def test_search_after_a_call_is_bit_identical():
    (a, da), (b, db) = _hash_search(False), _hash_search(True)
    for k in a:
        if a[k] is not None:
            assert np.array_equal(a[k], b[k]), k
    for x, y in zip(da, db):
        assert [bytes(n) for n in x] == [bytes(n) for n in y]


def test_out_of_range_limits():
    eng = Engine(max_games=4, max_nodes=2, avg_moves=64)
    try:
        eng.games_set(np.tile(B.record_from_fen(), (4, 1)))
        for d, q in ((0, 0), (6, 0), (1, -1), (1, 9), (-3, 4)):
            with pytest.raises(CrlError) as ei:
                eng.games_ab_move(d, q)
            assert ei.value.status == CRL_EINVAL
        assert eng.games_ab_move(5, 0, mask=np.array([1, 0, 0, 0], dtype=np.uint8))[0][0] != B.MOVE_NONE
    finally:
        eng.close()


# ---- matches and the policy benchmark -------------------------------------------------------------------------------
def test_play_match_hash_against_alphabeta_equals_the_oracle_loop():
    players = (arena.HashPlayer(3), arena.AlphaBetaPlayer(2, 1))
    out, summary = arena.play_match(players[0], players[1], games=6, sims=16, lanes=4, opening_plies=4, max_plies=24,
                                    seed=4)
    for j, g in enumerate(out):
        assert (g["moves"], g["result"]) == oracle_game(g["opening"], g["a_white"], players, 16, 24), j
    assert summary["played"] == 6


def _check_ab_plies(moves, start_ply, ab_to_move, player, samples):
    """The game replays under the oracle; `samples` of the alpha-beta side's plies are the oracle search's move."""
    g = O.OGame()
    checked = 0
    for ply, m in enumerate(moves):
        if ply >= start_ply and ab_to_move(ply) and checked < samples:
            assert A.search(g.board, player.depth, player.qdepth)[0] == m, (ply, m)
            checked += 1
        assert g.move(m), (ply, m)
    return g.get_result(), checked


def test_network_against_alphabeta_replays_under_the_oracle():
    m = model.ChessModel()
    m.weights = netpacks.lively_pack()
    ab = arena.AlphaBetaPlayer(2, 2)
    out, summary = arena.play_match(m, ab, games=8, sims=16, lanes=8, opening_plies=4, max_plies=60, seed=6)
    total = 0
    for g in out:
        res, checked = _check_ab_plies(g["moves"], 4, lambda ply: (ply % 2 == 0) != g["a_white"], ab, 6)
        assert g["result"] == res or (g["result"] is None and len(g["moves"]) >= 60)
        total += checked
    assert total >= 16 and summary["played"] == 8


def test_policy_games_against_alphabeta_replay_under_the_oracle():
    from chessrl_b200 import benchmark
    from chessrl_b200.agent import Agent
    agent = Agent(True)
    ab = arena.AlphaBetaPlayer(2, 2)
    games = benchmark.play_policy_games(agent, opponent=ab, games=6, lanes=3, seed=5, max_plies=60)
    assert len(games) == 6 and all(g is not None for g in games)
    total = 0
    for rec in games:
        res, checked = _check_ab_plies(rec["moves"], 0, lambda ply: (ply % 2 == 0) != rec["color"], ab, 6)
        assert rec["result"] == res or (rec["result"] is None and len(rec["moves"]) >= 60)
        total += checked
    assert total >= 12
    again = benchmark.play_policy_games(agent, opponent="alphabeta:2:2", games=6, lanes=3, seed=5, max_plies=60)
    assert [g["moves"] for g in again] == [g["moves"] for g in games]
