"""Repetitions in the alpha-beta search (rule R of DESIGN.md 3.6, crl_games_ab_search_host CRL_AB_REPETITIONS) without a
GPU.

- tests/ab_rep_oracle.py (R on top of oracle/ab_oracle.py): its alpha-beta equals a plain minimax on positions with
  history, and with R off it is ab_oracle.search;
- hand vectors: a knight shuffle, the same position without its history, a perpetual check that saves a lost position,
  and a repeat of the position right after the last irreversible move;
- the g++ build of the kernels' code (tests/hostsim/ab_rep_hostsim.cpp) equals the oracle in move and score on plies of
  plain alpha-beta self-play games and on seeded playouts followed by there-and-back piece moves; R changes a stated
  share of them, and the comparison notices a window one ply short, the rule at the root and a search blind to the game;
- the drivers: the `alphabeta:D:Q:r` spec, and `gen_data --repetitions` reaching the engine call."""
import random

import numpy as np
import pytest

import ab_oracle as A
import ab_rep_oracle as R
import chessrl_oracle as O
import fake_gen_engine
from chessrl_b200 import arena, gen_data
from chessrl_b200 import boards as B
from hostsim import ab as H
from hostsim import ab_rep as HR

chess = O.chess


def board_after(moves, fen=None):
    b = chess.Board(fen) if fen else chess.Board()
    for m in moves:
        b.push(chess.Move.from_uci(m))
    return b


def _reverse(m):
    return chess.Move(m.to_square, m.from_square)


def _reversible(b, m):
    return not b.is_irreversible(m) and m.promotion is None


def shuffle_boards(n, seed):
    """Seeded random playouts followed by seeded there-and-back piece moves (a reversible move and, later, its reverse,
    for both sides) -- positions whose game holds repetitions, and unfinished."""
    rng = random.Random(seed)
    out = []
    while len(out) < n:
        b = chess.Board()
        for _ in range(rng.randrange(4, 40)):
            legal = list(b.generate_legal_moves())
            if not legal:
                break
            b.push(rng.choice(legal))
        for _ in range(rng.randrange(1, 4)):
            there = [m for m in b.generate_legal_moves() if _reversible(b, m)]
            if not there:
                break
            m1 = rng.choice(there)
            b.push(m1)
            reply = [m for m in b.generate_legal_moves() if _reversible(b, m)]
            if not reply:
                break
            m2 = rng.choice(reply)
            b.push(m2)
            for m in (_reverse(m1), _reverse(m2)):
                if m in list(b.generate_legal_moves()):
                    b.push(m)
        if A.terminal(b, list(b.generate_legal_moves()), 0) is None and not b.is_fivefold_repetition():
            out.append(b)
    return out


def selfplay_boards(n, seed):
    """Plies of plain alpha-beta self-play games at depth 1 (host build, first best move) after a seeded random opening:
    a side with no visible gain repeats, so these games cycle.  A ply whose position repeats an earlier one is taken
    with probability 0.3, any other with 0.05."""
    rng = random.Random(seed)
    out = []
    while len(out) < n:
        b = chess.Board()
        for _ in range(rng.randrange(2, 9)):
            b.push(rng.choice(list(b.generate_legal_moves())))
        for ply in range(200):
            if A.terminal(b, list(b.generate_legal_moves()), 0) is not None or b.is_fivefold_repetition():
                break
            if len(out) < n and rng.random() < (0.3 if b.is_repetition(2) else 0.05):
                out.append(b.copy())
            mv = H.root(B.record_from_fen(b.fen()), 1, 0)[0]
            b.push(chess.Move.from_uci(B.move_to_uci(mv)))
    return out


@pytest.fixture(scope="module")
def history_boards():
    return selfplay_boards(24, 5) + shuffle_boards(24, 6)


# ---- the oracle ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("depth,qdepth", [(1, 0), (1, 2), (2, 1)])
def test_oracle_alphabeta_equals_minimax_with_history(depth, qdepth):
    for b in shuffle_boards(6, 20 + depth) + selfplay_boards(6, 30 + qdepth):
        assert R.search(b, depth, qdepth) == R.search(b, depth, qdepth, prune=False), b.fen()
        assert R.search(b, depth, qdepth, repetitions=False) == A.search(b, depth, qdepth), b.fen()


# ---- hand vectors --------------------------------------------------------------------------------------------------
SHUFFLE = ["g1f3", "g8f6", "f3g1", "f6g8"]


@pytest.mark.parametrize("depth,qdepth", [(1, 0), (3, 2)])
def test_knight_shuffle(depth, qdepth):
    """1.Nf3 Nf6 2.Ng1 Ng8: Nf3 again would repeat the position after 1.Nf3, so with R it scores exactly 0 and the
    search plays the next best move at the same +20."""
    b = board_after(SHUFFLE)
    assert A.search(b, depth, qdepth)[:2] == ("g1f3", 20)
    move, score, vals = R.search(b, depth, qdepth)
    assert (move, score) == ("b1c3", 20)
    legal = [m.uci() for m in b.generate_legal_moves()]
    assert vals[legal.index("g1f3")] == 0
    recs = HR.game_records(b)
    assert B.meta_fields(int(recs[-1][8]))["ply"] == 4 and B.meta_fields(int(recs[-1][8]))["rev"] == 4
    assert HR.search_uci(recs, depth, qdepth) == ("b1c3", 20)


def test_knight_shuffle_from_its_fen_has_no_history():
    b = board_after(SHUFFLE)
    fresh = chess.Board(b.fen())
    assert R.search(fresh, 1, 0) == A.search(fresh, 1, 0)
    assert HR.search_uci(HR.game_records(fresh), 1, 0) == ("g1f3", 20)
    # the record a FEN gives has ply and revlen 0: the engine's root record, not the FEN's, carries the window
    assert B.meta_fields(int(B.record_from_fen(b.fen())[8]))["rev"] == 0


# White is a queen and a rook down; 1.Qc8+ Kh7 2.Qf5+ Kh8 came before, so Qc8+ now repeats the position after 1.Qc8+.
PERPETUAL_FEN = "7k/6p1/7p/5Q2/8/q7/r5PP/7K w - - 0 1"
PERPETUAL = ["f5c8", "h8h7", "c8f5", "h7h8"]


def test_perpetual_check_saves_a_lost_position():
    b = board_after(PERPETUAL, PERPETUAL_FEN)
    for depth, qdepth in ((1, 0), (2, 2)):
        plain = A.search(b, depth, qdepth)
        move, score, _ = R.search(b, depth, qdepth)
        assert plain[1] < -400 and (move, score) == ("f5c8", 0), (depth, qdepth, plain, move, score)
        assert HR.search_uci(HR.game_records(b), depth, qdepth) == ("f5c8", 0)
    # checked by hand: Qc8+ is the position after 1.Qc8+ again; Black's replies are Kh7 (the position after 1...Kh7
    # again) and the blocking ...Qf8, which loses the queen to Qxf8+
    after = board_after(PERPETUAL + ["f5c8"], PERPETUAL_FEN)
    assert [m.uci() for m in after.generate_legal_moves()] == ["h8h7", "a3f8"] and after.is_repetition(2)


def test_far_end_of_the_window_counts():
    """1.e4 e6 2.Nf3 Nf6 3.Ng1: Ng8 repeats the position right after 1...e6, the last irreversible move."""
    b = board_after(["e2e4", "e7e6", "g1f3", "g8f6", "f3g1"])
    legal = [m.uci() for m in b.generate_legal_moves()]
    k = legal.index("f6g8")
    assert R.search(b, 1, 0)[2][k] == 0
    assert A.search(b, 1, 0)[2][k] != 0 and R.search(b, 1, 0, repetitions="short")[2][k] != 0
    recs = HR.game_records(b)
    assert len(recs) == 4                      # the window: after 1...e6, 2.Nf3, 2...Nf6 and the root
    with pytest.raises(ValueError):
        HR.search(recs[1:], 1, 0)              # one record short of the window


# 7...f5 is the last irreversible move; 8.Nb1 Na6 9.Nc3, and ...Nb8 repeats the position right after 7...f5.  Black is
# behind, so with R it plays Nb8 for 0; a window one ply short misses the repeat and plays Nc5 for -220.
FAR_END = ["b1c3", "g8f6", "c3e4", "f6h5", "e4c3", "h5g3", "f2f4", "g3e2", "g1e2", "f7f5", "c3b1", "b8a6", "b1c3"]


def test_far_end_of_the_window_decides_the_move():
    b = board_after(FAR_END)
    assert R.search(b, 1, 0)[:2] == ("a6b8", 0)
    assert R.search(b, 1, 0, repetitions="short")[:2] == ("a6c5", -220)
    assert HR.search_uci(HR.game_records(b), 1, 0) == ("a6b8", 0)


# ---- the host build against the oracle -----------------------------------------------------------------------------
def _compare(boards, depth, qdepth, rule=True):
    """Boards on which the host build's (move, score) differs from the oracle's with `rule`."""
    bad = []
    for b in boards:
        mv, sc, _ = HR.search(HR.game_records(b), depth, qdepth)
        want = R.search(b, depth, qdepth, repetitions=rule)[:2]
        if (None if mv == B.MOVE_NONE else B.move_to_uci(mv), sc) != want:
            bad.append(b.fen())
    return bad


@pytest.mark.parametrize("depth,qdepth,n", [(1, 0, 48), (2, 2, 24), (3, 2, 8)])
def test_host_equals_oracle(history_boards, depth, qdepth, n):
    boards = history_boards[:n // 2] + history_boards[24:24 + n // 2]
    assert _compare(boards, depth, qdepth) == []


def test_rule_changes_a_share_and_the_comparison_bites(history_boards):
    changed = sum(R.search(b, 1, 0)[:2] != A.search(b, 1, 0)[:2] for b in history_boards)
    assert changed >= len(history_boards) // 6, changed            # R changes the move or the score of >= 1/6
    boards = history_boards + [board_after(FAR_END)]
    for wrong in ("short", "root", "path"):
        assert _compare(boards, 1, 0, rule=wrong) or _compare(boards[::3], 2, 2, rule=wrong), wrong


def test_host_limits():
    recs = HR.game_records(board_after(SHUFFLE))
    for kw in ({"margin": -1, "salt": 1}, {"pick_plies": -1, "salt": 1}):
        with pytest.raises(ValueError):
            HR.search(recs, 1, 0, **kw)
    for d, q in ((0, 0), (6, 0), (1, 9)):
        with pytest.raises(ValueError):
            HR.search(recs, d, q)


def test_host_pick_equals_oracle(history_boards):
    for j, b in enumerate(history_boards[::4]):
        for margin in (0, 20):
            mv, sc, _ = HR.search(HR.game_records(b), 1, 0, margin=margin, pick_plies=1000, salt=j + 1)
            assert (B.move_to_uci(mv), sc) == R.pick(b, 1, 0, margin, 1000, j + 1), (b.fen(), margin)


# ---- drivers -------------------------------------------------------------------------------------------------------
def test_alphabeta_spec():
    p = arena.AlphaBetaPlayer.parse("alphabeta:2:2:r")
    assert (p.depth, p.qdepth, p.repetitions, str(p)) == (2, 2, True, "alphabeta:2:2:r")
    assert str(arena.AlphaBetaPlayer.parse("alphabeta:2:2")) == "alphabeta:2:2"
    assert not arena.AlphaBetaPlayer.parse("alphabeta").repetitions
    assert str(arena.AlphaBetaPlayer(1, 0, repetitions=True)) == "alphabeta:1:0:r"
    for bad in ("alphabeta:2:2:x", "alphabeta:2:r", "alphabeta:2:2:r:1"):
        if bad.count(":") > 3:
            assert arena.AlphaBetaPlayer.parse(bad) is None
        else:
            with pytest.raises(ValueError):
                arena.AlphaBetaPlayer.parse(bad)


class _Recorder:
    def __init__(self):
        self.calls = []

    def games_ab_move(self, depth, qdepth, mask=None, **kw):
        self.calls.append(("move", depth, qdepth, kw))
        return np.full(len(mask), B.MOVE_NONE, dtype=np.uint16), None, None


def test_player_passes_the_flag():
    rec = _Recorder()
    mask = np.ones(3, dtype=bool)
    arena.AlphaBetaPlayer(2, 1).moves(rec, mask)
    arena.AlphaBetaPlayer.parse("alphabeta:2:1:r").moves(rec, mask)
    assert rec.calls == [("move", 2, 1, {}), ("move", 2, 1, {"repetitions": True})]


class FakeRepEngine(fake_gen_engine.FakeGenEngine):
    """games_ab_pick with the repetitions flag, from the host build of the repetition search."""

    def games_ab_pick(self, depth, qdepth, margin, pick_plies, salt, mask=None, repetitions=False):
        self._count("games_ab_pick_rep" if repetitions else "games_ab_pick")
        if not repetitions:
            return super().games_ab_pick(depth, qdepth, margin, pick_plies, salt, mask)
        moves = np.full(self.max_games, B.MOVE_NONE, dtype=np.uint16)
        scores = np.zeros(self.max_games, dtype=np.int32)
        nodes = np.zeros(self.max_games, dtype=np.int64)
        for g in range(self.max_games):
            if self._running(g) and (mask is None or mask[g]):
                moves[g], scores[g], nodes[g] = HR.search(HR.game_records(self.games[g].board), depth, qdepth,
                                                          margin=margin, pick_plies=pick_plies, salt=int(salt[g]))
        return moves, scores, nodes


def test_gen_data_repetitions_reach_the_engine(tmp_path, monkeypatch):
    kw = dict(depth=1, qdepth=0, margin=20, pick_plies=4, max_plies=40, seed=2)
    eng = FakeRepEngine(3)
    games, summary = gen_data.generate_games(3, lanes=3, engine=eng, repetitions=True, **kw)
    assert eng.calls.get("games_ab_pick_rep", 0) > 0 and eng.calls.get("games_ab_pick", 0) == 0
    for j, g in enumerate(games):                         # every ply is the oracle's pick given the game so far
        b = chess.Board()
        salt = int(gen_data.game_salts(2, j, 1)[0])
        for m in g["moves"]:
            assert R.pick(b, 1, 0, 20, 4, salt)[0] == m
            b.push(chess.Move.from_uci(m))
    fake_gen_engine.install(monkeypatch.setattr)
    monkeypatch.setattr("chessrl_b200.engine.Engine", lambda max_games=1, **k: FakeRepEngine(max_games))
    out = tmp_path / "g.json"
    s = gen_data.main([str(out), "--games", "3", "--depth", "1", "--qdepth", "0", "--pick-plies", "4",
                       "--max-plies", "40", "--seed", "2", "--repetitions"])
    assert s["repetitions"] is True and s["games"] == 3
