"""The fixed-depth alpha-beta opponent (DESIGN.md 3.6) without a GPU.

- oracle/ab_oracle.py, written from the definition, equals a plain minimax and passes hand-derived vectors;
- the g++ build of chessrl_b200/csrc/ab_search.cuh (tests/hostsim/ab_hostsim.cpp, the kernels' code) equals the oracle
  in s(p), move and score on fuzz and playout positions, and that comparison notices a changed weight or tie rule;
- the match driver (chessrl_b200/arena.py) with an AlphaBetaPlayer, on the oracle-backed fake engine, plays the games of
  a direct oracle loop move for move.

CRL_AB_HOST_POSITIONS scales the number of positions of the host-against-oracle checks (default 1.0)."""
import os
import random

import numpy as np
import pytest

import ab_oracle as A
import chessrl_oracle as O
from chessrl_b200 import arena
from chessrl_b200 import boards as B
from fake_arena_engine import FakeArenaEngine
from hostsim import ab as H
from position_fuzz import random_fen

chess = O.chess
SCALE = float(os.environ.get("CRL_AB_HOST_POSITIONS", "1.0"))


def n_of(k):
    return max(1, int(round(k * SCALE)))


def playout_fens(n, seed, plies=(6, 70)):
    """Seeded random playouts from the start position that have not ended."""
    rng = random.Random(seed)
    out = []
    while len(out) < n:
        b = chess.Board()
        for _ in range(rng.randrange(*plies)):
            legal = list(b.generate_legal_moves())
            if not legal:
                break
            b.push(rng.choice(legal))
        if A.terminal(b, list(b.generate_legal_moves()), 0) is None:
            out.append(b.fen())
    return out


def fuzz_fens(n, seed):
    rng = random.Random(seed)
    out = []
    while len(out) < n:
        fen, b = random_fen(rng)
        if A.terminal(b, list(b.generate_legal_moves()), 0) is None:
            out.append(fen)
    return out


def mirror_fen(fen):
    """The colour-mirrored position: ranks flipped, colours swapped, the other side to move."""
    board, turn, castle, ep, half, full = fen.split()
    board = "/".join(r.swapcase() for r in reversed(board.split("/")))
    castle = "".join(sorted(castle.swapcase(), key="KQkq".index)) if castle != "-" else "-"
    ep = ep if ep == "-" else ep[0] + str(9 - int(ep[1]))
    return " ".join((board, "b" if turn == "w" else "w", castle, ep, half, full))


# ---- the oracle ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("depth,qdepth", [(1, 0), (1, 2), (2, 0), (2, 1)])
def test_oracle_alphabeta_equals_minimax(depth, qdepth):
    for fen in playout_fens(n_of(4), 11 + depth) + fuzz_fens(n_of(4), 17 + qdepth):
        board = chess.Board(fen)
        pruned = A.search(board, depth, qdepth)
        plain = A.search(board, depth, qdepth, prune=False)
        assert pruned == plain, fen


def test_oracle_start_position_is_zero():
    assert A.evaluate(chess.Board()) == 0


def test_oracle_evaluation_hand_values():
    # white: king e1 (no black queen: 5 (3 - 3) = 0), rook d1 500;  black: king e8 0, queen d5 900 + 2 (3 - 0) = 906
    assert A.evaluate(chess.Board("4k3/8/8/3q4/8/8/8/3RK3 w - - 0 1")) == 500 - 906
    # pawn on e7 for white: 100 + 5 (6 - 1) = 125; rook on the 7th: 520; a bishop pair: 2 x (330 + 5 (3 - cd)) + 30
    assert A.evaluate(chess.Board("k7/4P3/8/8/8/8/8/K7 w - - 0 1")) == 125
    assert A.evaluate(chess.Board("k7/3R4/8/8/8/8/8/K7 w - - 0 1")) == 520
    assert A.evaluate(chess.Board("k7/8/8/8/3B4/2B5/8/K7 w - - 0 1")) == (330 + 15) + (330 + 10) + 30
    # king shelter while the other side has a queen: white king on its 3rd rank -10 x 2; black king a8 (no white queen)
    # 5 (3 - 3) = 0, queen on the rim h1 900 + 2 (3 - 3)
    assert A.evaluate(chess.Board("k7/8/8/8/8/K7/8/7q w - - 0 1")) == -20 - 900


def test_oracle_evaluation_is_colour_symmetric():
    for fen in playout_fens(n_of(10), 3) + fuzz_fens(n_of(20), 4):
        assert A.evaluate(chess.Board(fen)) == A.evaluate(chess.Board(mirror_fen(fen))), fen


def test_oracle_back_rank_mate_in_one():
    assert A.search_fen("6k1/5ppp/8/8/8/8/8/R5K1 w - - 0 1", 1, 0) == ("a1a8", 31999)


def test_oracle_mate_in_two():
    fen = "k7/8/2K5/8/8/8/8/7R w - - 0 1"
    move, score = A.search_fen(fen, 3, 2)
    assert score == 31997 and A.search_fen(fen, 1, 0)[1] < 31000      # no mate in one
    b = chess.Board(fen)                                                # every reply allows a mate in one
    b.push(chess.Move.from_uci(move))
    replies = list(b.generate_legal_moves())
    assert replies
    for r in replies:
        b.push(r)
        assert A.search(b, 1, 0)[1] == 31999, r.uci()
        b.pop()


def test_oracle_takes_a_hanging_queen():
    assert A.search_fen("4k3/8/8/3q4/8/8/8/3RK3 w - - 0 1", 1, 0) == ("d1d5", 500)


def test_oracle_avoids_a_stalemating_capture():
    fen = "k7/8/1n6/8/8/8/8/1Q5K w - - 0 1"
    b = chess.Board(fen)
    b.push(chess.Move.from_uci("b1b6"))                                 # winning the knight stalemates black
    assert b.is_stalemate()
    for d, q in ((1, 0), (2, 2)):
        move, score = A.search_fen(fen, d, q)
        assert move != "b1b6" and score > 500


# ---- the host build against the oracle -------------------------------------------------------------------------------
def host_positions(seed, n_fuzz, n_play):
    return fuzz_fens(n_fuzz, seed) + playout_fens(n_play, seed + 1)


def test_host_evaluation_equals_oracle():
    fens = host_positions(21, n_of(150), n_of(100)) + [chess.STARTING_FEN]
    for fen in fens:
        assert H.evaluate(B.record_from_fen(fen)) == A.evaluate(chess.Board(fen)), fen
        assert H.evaluate(B.record_from_fen(mirror_fen(fen))) == H.evaluate(B.record_from_fen(fen)), fen


@pytest.mark.parametrize("depth,qdepth,n_fuzz,n_play", [(1, 0, 40, 40), (2, 2, 12, 12), (3, 2, 3, 5)])
def test_host_search_equals_oracle(depth, qdepth, n_fuzz, n_play):
    for fen in host_positions(100 * depth + qdepth, n_of(n_fuzz), n_of(n_play)):
        mv, score, nodes = H.root(B.record_from_fen(fen), depth, qdepth)
        want_move, want_score = A.search_fen(fen, depth, qdepth)
        assert (B.move_to_uci(mv), score) == (want_move, want_score), fen
        assert nodes >= 2


def test_host_hand_vectors():
    def host(fen, d, q):
        mv, score, _ = H.root(B.record_from_fen(fen), d, q)
        return B.move_to_uci(mv), score
    assert host("6k1/5ppp/8/8/8/8/8/R5K1 w - - 0 1", 1, 0) == ("a1a8", 31999)
    assert host("k7/8/2K5/8/8/8/8/7R w - - 0 1", 3, 2)[1] == 31997
    assert host("4k3/8/8/3q4/8/8/8/3RK3 w - - 0 1", 1, 0) == ("d1d5", 500)
    assert host("k7/8/1n6/8/8/8/8/1Q5K w - - 0 1", 1, 0)[0] != "b1b6"
    assert H.evaluate(B.record_from_fen()) == 0
    with pytest.raises(ValueError):
        H.root(B.record_from_fen(), 0, 0)
    with pytest.raises(ValueError):
        H.root(B.record_from_fen(), 1, 9)


def test_comparison_notices_a_changed_weight():
    # an oracle whose knight is worth 10 centipawns more disagrees in score on most positions that hold a knight
    w = dict(A.WEIGHTS, knight=A.WEIGHTS["knight"] + 10)
    fens = [f for f in host_positions(31, n_of(40), n_of(20))
            if chess.Board(f).knights and chess.popcount(chess.Board(f).knights & chess.Board(f).occupied_co[True]) !=
            chess.popcount(chess.Board(f).knights & chess.Board(f).occupied_co[False])]
    assert len(fens) >= 10
    differ = sum(H.root(B.record_from_fen(f), 1, 0)[1] != A.search(chess.Board(f), 1, 0, w=w)[1] for f in fens)
    assert differ > len(fens) // 2, (differ, len(fens))


def test_comparison_notices_the_last_maximum():
    # breaking root ties by the last maximum picks another move on some positions
    fens = host_positions(41, n_of(30), n_of(30))
    differ = 0
    for f in fens:
        mv, _, _ = H.root(B.record_from_fen(f), 1, 0)
        assert B.move_to_uci(mv) == A.search(chess.Board(f), 1, 0)[0]
        differ += B.move_to_uci(mv) != A.search(chess.Board(f), 1, 0, ties="last")[0]
    assert differ >= 1


# ---- the match driver with an alpha-beta side -------------------------------------------------------------------------
class FakeAlphaBetaEngine(FakeArenaEngine):
    """FakeArenaEngine with games_ab_move from the oracle (Engine.games_ab_move: active, unfinished, masked lanes)."""

    def games_ab_move(self, depth, qdepth=4, mask=None):
        self._count("games_ab_move")
        moves = np.full(self.max_games, B.MOVE_NONE, dtype=np.uint16)
        scores = np.zeros(self.max_games, dtype=np.int32)
        nodes = np.zeros(self.max_games, dtype=np.int64)
        for g in range(self.max_games):
            if self._running(g) and (mask is None or mask[g]):
                mv, scores[g] = A.search(self.games[g].board, depth, qdepth)[:2]
                moves[g] = B.uci_to_move(mv)
        return moves, scores, nodes


SEED = 3


def oracle_game(opening, a_white, players, sims, max_plies):
    """The direct oracle loop: a HashPlayer side searches with OSelfPlayTree and plays the first most visited child, an
    AlphaBetaPlayer side plays ab_oracle.search's move."""
    g = O.OGame()
    for m in opening:
        assert g.move(m)
    while g.get_result() is None and len(g.board.move_stack) < max_plies:
        p = players[0] if g.board.turn == a_white else players[1]
        if isinstance(p, arena.AlphaBetaPlayer):
            mv = A.search(g.board, p.depth, p.qdepth)[0]
        else:
            t = O.OSelfPlayTree(g)
            agent = O.OAgent(O.hash_evaluator(p.seed, p.policy_bits))
            for _ in range(sims):
                t.explore_tree(agent)
            k = int(np.argmax([c.visits for c in t.root.children]))
            mv = t.root.children[k].state.board.move_stack[len(g.board.move_stack)].uci()
        assert g.move(mv)
    return [m.uci() for m in g.board.move_stack], g.get_result()


def check_match(players, games, lanes, sims, max_plies, **kw):
    eng = FakeAlphaBetaEngine(lanes)
    out, summary = arena.play_match(players[0], players[1], games=games, sims=sims, lanes=lanes, max_plies=max_plies,
                                    engine=eng, **kw)
    assert len(out) == games and all(g is not None for g in out)
    for j, game in enumerate(out):
        assert game["a_white"] == (j % 2 == 0)
        assert (game["moves"], game["result"]) == oracle_game(game["opening"], game["a_white"], players, sims,
                                                              max_plies), j
    return eng, out, summary


def test_match_hash_against_alphabeta_refill_park_and_cap():
    # 5 games on 2 lanes: both colours, lanes refilled and parked, a cap that leaves games unfinished
    eng, out, summary = check_match((arena.HashPlayer(SEED), arena.AlphaBetaPlayer(1, 1)), games=5, lanes=2, sims=12,
                                    max_plies=16, opening_plies=4, seed=9)
    assert eng.calls["games_ab_move"] >= 1 and eng.calls["games_set_active"] >= 2
    assert any(g["result"] is None for g in out)
    assert summary["played"] == 5


def test_match_alphabeta_first_and_given_openings():
    # the alpha-beta side as A; the hash side searches alone, in slot 0
    openings = [["e2e4", "e7e5"], ["d2d4", "d7d5"]]
    eng, out, _ = check_match((arena.AlphaBetaPlayer(2, 0), arena.HashPlayer(SEED)), games=4, lanes=4, sims=10,
                              max_plies=14, openings=openings)
    assert [g["opening"] for g in out] == [openings[0], openings[0], openings[1], openings[1]]
    assert eng.slot_agents[1] is None


def test_match_two_alphabeta_players():
    # no search at all: both sides move by games_ab_move, each with its own depth
    eng, out, summary = check_match((arena.AlphaBetaPlayer(2, 1), arena.AlphaBetaPlayer(1, 0)), games=2, lanes=2,
                                    sims=1, max_plies=20, openings=[["g1f3"]])
    assert eng.n_sims == 0 and "mcts_begin_move" not in eng.calls


def test_alphabeta_player_parsing():
    assert str(arena.AlphaBetaPlayer.parse("alphabeta")) == "alphabeta:%d:%d" % (arena.AB_DEPTH, arena.AB_QDEPTH)
    p = arena.AlphaBetaPlayer.parse("alphabeta:2")
    assert (p.depth, p.qdepth) == (2, arena.AB_QDEPTH)
    p = arena.AlphaBetaPlayer.parse("alphabeta:4:0")
    assert (p.depth, p.qdepth) == (4, 0)
    assert arena.AlphaBetaPlayer.parse("models/model-3.h5") is None
    for bad in ("alphabeta:0", "alphabeta:6", "alphabeta:2:9", "alphabeta:x"):
        with pytest.raises(ValueError):
            arena.AlphaBetaPlayer.parse(bad)
    assert arena._label("alphabeta:2", "bf16") == "alphabeta:2:%d" % arena.AB_QDEPTH
