"""The match driver (chessrl_b200/arena.py) on the CPU: play_match on a two-slot fake engine (tests/fake_arena_engine.py)
plays, move for move, the games of a direct oracle loop in which each side searches with OSelfPlayTree and its own
hash evaluator and plays the first most visited root child; and the Elo interval against hand values."""
import math

import numpy as np
import pytest

import chessrl_oracle as O
from chessrl_b200 import arena
from fake_arena_engine import FakeArenaEngine

SEED_A, SEED_B = 3, 11


def oracle_game(opening, a_white, sims, max_plies, seeds=(SEED_A, SEED_B), bits=24):
    agents = [O.OAgent(O.hash_evaluator(s, bits)) for s in seeds]
    g = O.OGame()
    for m in opening:
        assert g.move(m)
    while g.get_result() is None and len(g.board.move_stack) < max_plies:
        white = g.board.turn
        slot = 0 if white == a_white else 1
        t = O.OSelfPlayTree(g)
        for _ in range(sims):
            t.explore_tree(agents[slot])
        k = int(np.argmax([c.visits for c in t.root.children]))          # the first most visited child
        g.move(t.root.children[k].state.board.move_stack[len(g.board.move_stack)].uci())
    return [m.uci() for m in g.board.move_stack], g.get_result()


def check_against_oracle(out, sims, max_plies):
    for j, game in enumerate(out):
        assert game["a_white"] == (j % 2 == 0)
        moves, res = oracle_game(game["opening"], game["a_white"], sims, max_plies)
        assert game["moves"] == moves, j
        assert game["result"] == res, j


def test_random_openings_refill_park_and_cap():
    # 9 games on 4 lanes: lanes are refilled as games end and parked when none is left; a short cap leaves some
    # games unfinished
    eng = FakeArenaEngine(4)
    out, summary = arena.play_match(arena.HashPlayer(SEED_A), arena.HashPlayer(SEED_B), games=9, sims=30, lanes=4,
                                    opening_plies=4, max_plies=14, seed=5, engine=eng)
    assert len(out) == 9 and all(g is not None for g in out)
    for i in range(0, 8, 2):                        # the colour swap inside each opening pair
        assert out[i]["opening"] == out[i + 1]["opening"]
        assert out[i]["a_white"] and not out[i + 1]["a_white"]
    assert len({tuple(g["opening"]) for g in out}) > 1
    assert all(len(g["opening"]) == 4 and g["moves"][:4] == g["opening"] for g in out)
    check_against_oracle(out, 30, 14)
    assert any(g["result"] is None for g in out) and all(len(g["moves"]) <= 14 for g in out)
    assert summary["unfinished"] == sum(g["result"] is None for g in out)
    assert eng.calls["games_set_active"] >= 1          # lanes parked in the drain
    # the same seed draws the same openings
    again, _ = arena.play_match(arena.HashPlayer(SEED_A), arena.HashPlayer(SEED_B), games=9, sims=30, lanes=4,
                                opening_plies=4, max_plies=14, seed=5, engine=FakeArenaEngine(4))
    assert [g["moves"] for g in again] == [g["moves"] for g in out]


def test_given_openings():
    openings = [["e2e4", "e7e5"], ["d2d4"], ["g1f3", "g8f6", "c2c4"]]
    eng = FakeArenaEngine(3)
    out, summary = arena.play_match(arena.HashPlayer(SEED_A), arena.HashPlayer(SEED_B), games=6, sims=30, lanes=3,
                                    openings=openings, max_plies=40, engine=eng)
    assert [g["opening"] for g in out] == [openings[0], openings[0], openings[1], openings[1], openings[2], openings[2]]
    check_against_oracle(out, 30, 40)
    assert summary["played"] == 6
    assert summary["a_wins"] + summary["b_wins"] + summary["draws"] + summary["unfinished"] == 6


def test_swapped_seeds_change_the_games():
    # sensitivity: the oracle loop with the players' evaluators swapped disagrees with what the driver played
    out, _ = arena.play_match(arena.HashPlayer(SEED_A), arena.HashPlayer(SEED_B), games=2, sims=30, lanes=2,
                              openings=[["e2e4"]], max_plies=20, engine=FakeArenaEngine(2))
    swapped = [oracle_game(g["opening"], g["a_white"], 30, 20, seeds=(SEED_B, SEED_A))[0] for g in out]
    assert swapped != [g["moves"] for g in out]


def test_elo_hand_values():
    assert arena.elo_of_score(0.5) == 0.0
    s, elo, lo, hi = arena.elo_interval(7, 7, 3)
    assert s == 0.5 and elo == 0.0 and lo == -hi and hi > 0
    assert arena.elo_of_score(0.75) == pytest.approx(190.848501887865, abs=1e-9)
    s, elo, lo, hi = arena.elo_interval(30, 10, 0)
    assert s == 0.75 and elo == pytest.approx(190.85, abs=5e-3)
    # trinomial normal approximation: var = (30 * 0.25^2 + 10 * 0.75^2) / 40 = 0.1875, half = 1.96 sqrt(0.1875 / 40)
    half = arena.Z95 * math.sqrt(0.1875 / 40)
    assert lo == pytest.approx(arena.elo_of_score(0.75 - half)) and hi == pytest.approx(arena.elo_of_score(0.75 + half))
    s, elo, lo, hi = arena.elo_interval(10, 0, 0)
    assert s == 1.0 and elo == math.inf and hi == math.inf
    s, elo, lo, hi = arena.elo_interval(0, 4, 0)
    assert elo == -math.inf and lo == -math.inf


def test_summary_counts_unfinished_as_draws():
    games = [{"a_white": True, "result": 1}, {"a_white": False, "result": 1}, {"a_white": True, "result": None},
             {"a_white": False, "result": 0}, {"a_white": False, "result": -1}]
    sm = arena.summarize(games)
    assert (sm["a_wins"], sm["b_wins"], sm["draws"], sm["unfinished"]) == (2, 1, 1, 1)
    assert sm["score"] == pytest.approx((2 + 0.5 * 2) / 5)
