"""Two networks in one engine (crl_net_select_slot, crl_games_set_players_host) and the match driver on the GPU.

A lane's search evaluates every row -- root, predicted replies, leaves -- with the slot of the side to move at its root.
Every comparison is bit-exact: against the oracle with the hash evaluator of that slot, and against single-network
engines that ran the same lanes with that lane's network alone (rows do not depend on the batch they sit in,
tests/test_gpu_evalpath.py)."""
import numpy as np
import pytest
import torch

import chessrl_oracle as O
import netpacks
from chessrl_b200 import arena
from chessrl_b200 import boards as B
from chessrl_b200 import model
from chessrl_b200._lib import CRL_EINVAL, CRL_ESTATE, EVAL_HASH, EVAL_NET, CrlError, check
from chessrl_b200.engine import Engine
from test_arena_host import oracle_game
from test_gpu_evalpath import _openings, _search

pytestmark = pytest.mark.gpu

SEEDS = (3, 11)
STAT_KEYS = ("visits", "values", "priors", "moves", "replies", "results", "n_children", "root_visits", "root_values")


def _players(G):
    """Every combination of players: (0, 0), (0, 1), (1, 0), (1, 1) in turn."""
    k = np.arange(G)
    return ((k // 2) % 2).astype(np.uint8), (k % 2).astype(np.uint8)


def _searching_slot(eng, white, black):
    rec, _, _ = eng.games_get()
    white_to_move = (rec[:, 8] & np.uint64(1)).astype(bool)
    return np.where(white_to_move, white, black)


def _hash_engine(G, K=1, nodes=64):
    eng = Engine(max_games=G, max_nodes=nodes, avg_moves=96, max_inflight=K)
    for slot, seed in enumerate(SEEDS):
        eng.set_evaluator(EVAL_HASH, seed, 24, slot=slot)
    return eng


def _oracle_root(game, seed, sims, K):
    agent = O.OAgent(O.hash_evaluator(seed, 24))
    t = O.OSelfPlayTree(game, threads=K)
    left = sims
    while left > 0:
        if K <= 1:
            t.explore_tree(agent)
            left -= 1
        else:
            left -= t.explore_wave(agent, min(K, left))
    return t


@pytest.mark.parametrize("K", [1, 4])
def test_hash_routing_matches_oracle(K):
    G, sims = 48, 40
    eng = _hash_engine(G, K)
    moves = _openings(eng, seed=5, max_plies=30)
    white, black = _players(G)
    eng.games_set_players(white, black)
    slot = _searching_slot(eng, white, black)
    assert set(slot) == {0, 1} and len({(w, b) for w, b in zip(white, black)}) == 4
    eng.mcts_begin_move()
    eng.mcts_simulate(sims, inflight=K)
    st = eng.root_stats()
    n_priors = 0
    for g in range(G):
        game = O.OGame()
        for m in moves[g]:
            game.move(m)
        if game.get_result() is not None:
            continue
        t = _oracle_root(game, SEEDS[slot[g]], sims, K)
        kids = t.root.children
        ply = len(game.board.move_stack)
        assert st["n_children"][g] == len(kids), g
        assert list(st["visits"][g, :len(kids)]) == [c.visits for c in kids], g
        assert [float(v) for v in st["values"][g, :len(kids)]] == [float(c.value) for c in kids], g
        for k, c in enumerate(kids):                 # (Node.prior stays 1 until its parent is fully expanded)
            if c.prior != 1:
                assert np.float32(st["priors"][g, k]) == np.float32(c.prior), (g, k)
                n_priors += 1
        assert st["root_values"][g] == float(t.root.value) and st["root_visits"][g] == t.root.visits, g
        replies = [B.uci_to_move(c.state.board.move_stack[ply + 1].uci()) if len(c.state.board.move_stack) > ply + 1
                   else B.MOVE_NONE for c in kids]
        assert list(st["replies"][g, :len(kids)]) == replies, g
    assert n_priors > 0


def _net_engine(G, packs, precisions=("bf16", "bf16"), amax=None, nodes=33):
    eng = Engine(max_games=G, max_nodes=nodes, avg_moves=96)
    for slot, (pack, prec) in enumerate(zip(packs, precisions)):
        eng.load_weights(pack, precision=prec, calibration=amax if prec == "fp8" else None, slot=slot)
        eng.set_evaluator(EVAL_NET, slot=slot)
    return eng


@pytest.fixture(scope="module")
def packs():
    return netpacks.lively_pack(), netpacks.lively_pack(seed=netpacks.LIVELY_SEED + 7)


@pytest.fixture(scope="module")
def amax_b(packs):
    eng = Engine(max_games=256, max_nodes=2, avg_moves=96)
    eng.load_weights(packs[1])
    x = torch.from_numpy(netpacks.planes_of(netpacks.midgame_games(256, seed=9))).to(eng.device, torch.bfloat16)
    amax = eng.calibrate(x)
    eng.close()
    return amax


def _same_lanes(a, b, lanes):
    """Root statistics and commit pairs of `lanes` in two recordings -> lanes that differ."""
    bad = set()
    for (sa, _, oa), (sb, _, ob) in zip(a, b):
        for key in STAT_KEYS:
            x, y = sa[key][lanes], sb[key][lanes]
            rows = np.nonzero(~np.all((x == y).reshape(len(lanes), -1), axis=1))[0]
            bad.update(int(lanes[r]) for r in rows)
        rows = np.nonzero(~np.all(oa[lanes] == ob[lanes], axis=1))[0]
        bad.update(int(lanes[r]) for r in rows)
    return bad


@pytest.mark.parametrize("case", ["two_tile", "single_tile", "fp8"])
def test_net_routing_matches_single_network_engines(packs, amax_b, case):
    G, run, sims, bound = {"two_tile": (4096, 4096, 32, 0), "single_tile": (512, 296, 32, 296),
                           "fp8": (1024, 1024, 32, 0)}[case]
    precisions = ("bf16", "fp8") if case == "fp8" else ("bf16", "bf16")
    mixed = _net_engine(G, packs, precisions, amax_b)
    singles = [_net_engine(G, (packs[k],), (precisions[k],), amax_b) for k in (0, 1)]
    active = np.zeros(G, dtype=np.uint8)
    active[:run] = 1
    white, black = _players(G)
    mixed.games_set_players(white, black)
    for eng in [mixed] + singles:
        _openings(eng, seed=23, max_plies=40)
        eng.games_set_active(active)
        eng.set_row_bound(bound)
    slot = _searching_slot(mixed, white, black)
    rec = [_search(eng, 2, sims) for eng in [mixed] + singles]
    live = np.arange(run)
    for k in (0, 1):
        lanes = live[slot[:run] == k]
        assert len(lanes) > run // 4
        assert not _same_lanes(rec[0], rec[1 + k], lanes), (case, k)
        # sensitivity: the other network's engine disagrees on these lanes
        assert len(_same_lanes(rec[0], rec[2 - k], lanes)) > len(lanes) // 2, (case, k)


def test_one_network_is_unchanged_by_a_configured_slot_1(packs):
    G, sims = 1024, 32
    plain = _net_engine(G, packs[:1])
    two = _net_engine(G, packs)
    two.games_set_players(0, 0)
    for eng in (plain, two):
        _openings(eng, seed=31, max_plies=40)
    assert not _same_lanes(_search(plain, 2, sims), _search(two, 2, sims), np.arange(G))
    # net_forward(slot=1) is the other pack's forward pass
    other = _net_engine(64, packs[1:])
    x = torch.from_numpy(netpacks.planes_of(netpacks.midgame_games(64, seed=3))).to(two.device, torch.bfloat16)
    p1, v1 = two.net_forward(x, slot=1)
    q1, w1 = other.net_forward(x)
    assert torch.equal(p1, q1) and torch.equal(v1, w1)
    p0, v0 = two.net_forward(x)
    assert not torch.equal(p0, p1)


def test_configuring_one_slot_leaves_the_other_unchanged(packs, amax_b):
    eng = Engine(max_games=64, max_nodes=2, avg_moves=96)
    x = torch.from_numpy(netpacks.planes_of(netpacks.midgame_games(64, seed=4))).to(eng.device, torch.bfloat16)
    eng.load_weights(packs[0])
    p0, v0 = eng.net_forward(x)
    eng.load_weights(packs[1], precision="fp8", calibration=amax_b, slot=1)
    p1, v1 = eng.net_forward(x, slot=1)
    eng.set_net_precision("bf16", slot=1)
    p1b, v1b = eng.net_forward(x, slot=1)
    for _ in range(2):
        q0, w0 = eng.net_forward(x)
        assert torch.equal(p0, q0) and torch.equal(v0, w0)
        eng.set_net_precision("fp8", slot=1)
    eng.set_net_precision("bf16", slot=1)
    # and slot 1 does not see slot 0's changes
    eng.load_weights(packs[1])
    eng.load_weights(packs[0])
    q1, w1 = eng.net_forward(x, slot=1)
    assert torch.equal(p1b, q1) and torch.equal(v1b, w1)
    eng.set_net_precision("fp8", slot=1)
    q1, w1 = eng.net_forward(x, slot=1)
    assert torch.equal(p1, q1) and torch.equal(v1, w1)
    assert not torch.equal(p1, p1b)


def test_policy_move_routes_by_side_to_move():
    G = 64
    eng = _hash_engine(G, nodes=2)
    moves = _openings(eng, seed=8, max_plies=30)
    white, black = _players(G)
    eng.games_set_players(white, black)
    slot = _searching_slot(eng, white, black)
    picks = eng.policy_move()
    agents = [O.OAgent(O.hash_evaluator(s, 24)) for s in SEEDS]
    n = 0
    for g in range(G):
        game = O.OGame()
        for m in moves[g]:
            game.move(m)
        if game.get_result() is not None:
            continue
        assert B.move_to_uci(picks[g]) == agents[slot[g]].policy_move(game), g
        n += agents[slot[g]].policy_move(game) != agents[1 - slot[g]].policy_move(game)
    assert n > 0


def test_errors(packs):
    eng = Engine(max_games=8, max_nodes=16, avg_moves=96)
    eng.set_evaluator(EVAL_HASH, 1, 24)
    eng.games_set(np.tile(B.record_from_fen(), (8, 1)))
    for slot in (2, -1):
        with pytest.raises(CrlError) as ex:
            check(eng.lib.crl_net_select_slot(eng.h, slot))
        assert ex.value.status == CRL_EINVAL
    with pytest.raises(CrlError):
        eng.games_set_players([2], [0])
    # a lane on slot 1, which has no evaluator
    eng.games_set_players([1], [0], first=3)
    for call in (eng.mcts_begin_move, eng.policy_move):
        with pytest.raises(CrlError) as ex:
            call()
        assert ex.value.status == CRL_ESTATE
    # hash and network kinds in one search
    eng.load_weights(packs[1], slot=1)
    eng.set_evaluator(EVAL_NET, slot=1)
    with pytest.raises(CrlError) as ex:
        eng.mcts_begin_move()
    assert ex.value.status == CRL_ESTATE
    eng.set_evaluator(EVAL_HASH, 2, 24, slot=1)
    eng.mcts_begin_move()
    eng.mcts_simulate(4)
    # changing players ends the search: begin a new one
    eng.games_set_players([0], [0], first=3)
    with pytest.raises(CrlError) as ex:
        eng.mcts_simulate(4)
    assert ex.value.status == CRL_ESTATE
    with pytest.raises(CrlError) as ex:
        eng.set_net_precision("fp8", slot=1)
    assert ex.value.status == CRL_ESTATE


def test_reuse_with_players():
    G, sims = 32, 40
    recs = {}
    for reuse in (False, True):
        eng = _hash_engine(G)
        eng.set_reuse(reuse)
        _openings(eng, seed=12, max_plies=20)
        eng.games_set_players(1, 1)
        recs[reuse] = _search(eng, 3, sims)
        if reuse:
            assert eng.counters()["reused_evaluations"] > 0
            # changing every lane's players unlinks every twin: the next search reuses nothing
            eng.games_set_players(0, 0)
            eng.games_set_players(1, 1)
            before = eng.counters()["reused_evaluations"]
            _search(eng, 1, sims)
            assert eng.counters()["reused_evaluations"] == before
    assert not _same_lanes(recs[False], recs[True], np.arange(G))


def test_play_match_with_hash_players_reproduces_the_oracle_match():
    out, summary = arena.play_match(arena.HashPlayer(3), arena.HashPlayer(11), games=8, sims=30, lanes=4,
                                    opening_plies=4, max_plies=24, seed=1)
    for j, g in enumerate(out):
        moves, res = oracle_game(g["opening"], g["a_white"], 30, 24)
        assert g["moves"] == moves and g["result"] == res, j
    assert summary["played"] == 8


def test_play_match_of_a_network_against_itself_is_exactly_even(packs):
    m = model.ChessModel()
    m.weights = packs[0]
    out, summary = arena.play_match(m, m, games=16, sims=16, lanes=16, opening_plies=4, max_plies=60, seed=2)
    for i in range(0, 16, 2):
        assert out[i]["moves"] == out[i + 1]["moves"] and out[i]["result"] == out[i + 1]["result"]
    assert summary["score"] == 0.5 and summary["elo"] == 0.0
