"""Generating training games with the seeded near-best root pick (DESIGN.md 3.7), without a GPU.

- oracle/ab_pick_oracle.py: margin 0 is ab_oracle.search; hand vectors for the candidate set, pick_plies and mates;
- the g++ build of the pick (tests/hostsim/ab_pick_hostsim.cpp, the kernels' code) equals the oracle in move and score,
  and that comparison notices a rule that takes the last candidate or is off by one in the ply;
- the driver (chessrl_b200/gen_data.py) on tests/fake_gen_engine.FakeGenEngine: a direct per-game loop, independence of
  the lane count, seeds, refill / park / cap, the JSON round trip and a two-rank gloo run."""
import json
import os
import random
import socket
import subprocess
import sys
import textwrap

import pytest

import ab_oracle as A
import ab_pick_oracle as P
import chessrl_oracle as O
import fake_gen_engine
from chessrl_b200 import boards as B
from chessrl_b200 import gen_data
from conftest import ROOT
from hostsim import ab_pick as HP
from test_alphabeta_host import fuzz_fens, n_of, playout_fens

chess = O.chess
START_D1 = ["g1f3", "b1c3", "h2h4", "g2g4", "f2f4", "e2e4", "d2d4", "c2c4", "b2b4", "a2a4"]   # within 10 cp of +20


# ---- the oracle ----------------------------------------------------------------------------------------------------
def test_oracle_margin_zero_is_the_search():
    rng = random.Random(1)
    for fen in playout_fens(n_of(6), 51) + fuzz_fens(n_of(6), 52):
        b = chess.Board(fen)
        for d, q in ((1, 0), (2, 1)):
            assert P.pick(b, d, q, 0, 1000, rng.getrandbits(64), ply=rng.randrange(40)) == A.search(b, d, q)[:2], fen


def test_oracle_hand_vectors():
    start = chess.Board()
    # depth 1, no quiescence: the knights to c3 / f3 score 20, the double pushes 10, single pushes 5, Na3 / Nh3 0
    assert P.pick_index([0, 20, 20, 0, 5, 10], 0, 10, 16, 0) in (1, 2, 5)
    picks = {P.pick(start, 1, 0, 10, 16, s)[0] for s in range(40)}
    assert picks <= set(START_D1) and len(picks) >= 5
    for s in range(40):                                   # C[splitmix64(salt + ply) mod |C|]
        mv = START_D1[O.splitmix64(s + 3) % 10]
        assert P.pick(start, 1, 0, 10, 16, s, ply=3) == (mv, 20 if mv in ("g1f3", "b1c3") else 10)
    # at or above pick_plies: the first maximum, whatever the salt
    assert {P.pick(start, 1, 0, 10, 16, s, ply=16) for s in range(20)} == {("g1f3", 20)}
    assert {P.pick(start, 1, 0, 10, 16, s, ply=15)[0] for s in range(20)} != {"g1f3"}
    # a mate score ignores the margin: the back-rank mate is played by every salt
    mate = chess.Board("6k1/5ppp/8/8/8/8/8/R5K1 w - - 0 1")
    assert {P.pick(mate, 1, 0, 10 ** 6, 16, s) for s in range(20)} == {("a1a8", 31999)}
    # a terminal root has no move
    assert P.pick(chess.Board("7k/5Q2/6K1/8/8/8/8/8 b - - 0 1"), 1, 0, 10, 16, 0) == (None, 0)


# ---- the host build against the oracle -------------------------------------------------------------------------------
def _cases(seed, n_fuzz, n_play):
    rng = random.Random(seed)
    return [(fen, rng.randrange(24), rng.getrandbits(64)) for fen in fuzz_fens(n_fuzz, seed) +
            playout_fens(n_play, seed + 1)]


@pytest.mark.parametrize("depth,qdepth,n", [(1, 0, 30), (2, 2, 8)])
@pytest.mark.parametrize("margin", [0, 15, 50])
def test_host_pick_equals_oracle(depth, qdepth, n, margin):
    for fen, ply, salt in _cases(100 * depth + margin, n_of(n), n_of(n)):
        got = HP.pick_uci(HP.with_ply(B.record_from_fen(fen), ply), depth, qdepth, margin, 12, salt)
        assert got == P.pick(chess.Board(fen), depth, qdepth, margin, 12, salt, ply=ply), (fen, ply, salt)


def test_comparison_notices_the_last_member_and_a_ply_off_by_one():
    last = ply_off = 0
    for fen, ply, salt in _cases(7, n_of(40), n_of(40)):
        ply = ply % 12
        got = HP.pick_uci(HP.with_ply(B.record_from_fen(fen), ply), 1, 0, 50, 12, salt)
        assert got == P.pick(chess.Board(fen), 1, 0, 50, 12, salt, ply=ply)
        last += got != P.pick(chess.Board(fen), 1, 0, 50, 12, salt, ply=ply, member="last")
        ply_off += got != P.pick(chess.Board(fen), 1, 0, 50, 12, salt, ply=ply + 1)
    assert last >= 10 and ply_off >= 10, (last, ply_off)


def test_host_pick_limits():
    rec = B.record_from_fen()
    for args in ((0, 0, 10, 16), (1, 9, 10, 16), (1, 0, -1, 16), (1, 0, 10, -1)):
        with pytest.raises(ValueError):
            HP.pick(rec, *args, 0)
    assert HP.pick(rec, 1, 0, 0, 0, 0)[:2] == (B.uci_to_move("g1f3"), 20)


# ---- the driver ---------------------------------------------------------------------------------------------------
KW = dict(depth=1, qdepth=0, margin=15, pick_plies=8, max_plies=20)


def direct_game(j, n, seed, depth, qdepth, margin, pick_plies, max_plies):
    """Game j by hand: the host build's pick at every ply of one oracle game."""
    salt = int(gen_data.game_salts(seed, 0, n)[j])
    g = O.OGame()
    while g.get_result() is None and len(g.board.move_stack) < max_plies:
        mv, _ = HP.pick_uci(fake_gen_engine.lane_record(g), depth, qdepth, margin, pick_plies, salt)
        assert g.move(mv)
    return [m.uci() for m in g.board.move_stack], g.get_result()


def run(n, lanes, seed, **kw):
    eng = fake_gen_engine.FakeGenEngine(lanes)
    games, summary = gen_data.generate_games(n, lanes=lanes, seed=seed, engine=eng, **dict(KW, **kw))
    return eng, games, summary


def test_driver_equals_a_direct_loop_for_any_lane_count():
    n = 8
    _, ref, summary = run(n, n, seed=5)
    for j, g in enumerate(ref):
        assert (g["moves"], g["result"]) == direct_game(j, n, 5, **KW), j
        assert g["player_color"] == (j % 2 == 0)
    for lanes in (1, 7):
        assert run(n, lanes, seed=5)[1] == ref
    assert summary["games"] == n and summary["plies"] == sum(len(g["moves"]) for g in ref)
    assert summary["distinct_fraction"] == 1.0
    assert summary["white_wins"] + summary["black_wins"] + summary["draws"] + summary["unfinished"] == n
    assert sum(summary["ends"].values()) == n and summary["ends"]["unfinished"] == summary["unfinished"]


def test_driver_seeds_and_margin_zero():
    a, b = run(4, 4, seed=1)[1], run(4, 4, seed=2)[1]
    assert all(x["moves"] != y["moves"] for x, y in zip(a, b))
    same = run(3, 3, seed=1, margin=0)[1]                 # no margin: every game is the deterministic game
    assert same[0]["moves"] == same[1]["moves"] == same[2]["moves"]


def test_driver_refills_parks_and_caps():
    eng, games, summary = run(5, 2, seed=9, max_plies=12)
    assert len(games) == 5 and all(g is not None for g in games)
    assert all(g["result"] is None and len(g["moves"]) == 12 and g["end"] == "unfinished" for g in games)
    assert eng.calls["games_restart"] >= 2 and eng.calls["games_set_active"] >= 1
    assert eng.calls["games_ab_pick"] == 3 * 12      # three rounds of games, one call per ply for both lanes
    assert summary["unfinished"] == 5


def test_game_end_classification():
    rec = B.record_from_fen("7k/5Q2/6K1/8/8/8/8/8 b - - 0 1")
    assert gen_data.game_end(rec, None, 0) == "unfinished"
    assert gen_data.game_end(rec, 0, 0) == "stalemate"
    assert gen_data.game_end(B.record_from_fen("6Rk/8/6K1/8/8/8/8/8 b - - 0 1"), 1, 0) == "mate"
    assert gen_data.game_end(B.record_from_fen("4k3/8/8/8/8/8/8/R3K3 w - - 100 80"), 0, 15) == "fifty_moves"
    assert gen_data.game_end(B.record_from_fen("4k3/8/8/8/8/8/8/4K3 w - - 0 80"), 0, 5) == "other_draw"


def test_cli_json_round_trips(tmp_path, monkeypatch):
    fake_gen_engine.install(monkeypatch.setattr)
    out = tmp_path / "games.json"
    argv = [str(out), "--games", "5", "--lanes", "2", "--depth", "1", "--qdepth", "0", "--margin", "15",
            "--pick-plies", "8", "--max-plies", "20", "--seed", "3"]
    summary = gen_data.main(argv)
    games = gen_data.generate_games(5, lanes=5, seed=3, engine=fake_gen_engine.FakeGenEngine(5), **KW)[0]
    saved = json.loads(out.read_text())
    assert [(g["moves"], g["result"], g["player_color"]) for g in saved] == \
        [(g["moves"], g["result"], g["player_color"]) for g in games]
    from chessrl_b200.dataset import DatasetGame
    ds = DatasetGame()
    ds.load(str(out))
    assert [(g.get_history()["moves"], g.get_result()) for g in ds.games] == [(g["moves"], g["result"]) for g in games]
    gen_data.main(argv)                                   # appends
    assert len(json.loads(out.read_text())) == 10
    assert summary["games"] == 5 and summary["seed"] == 3


WORKER = textwrap.dedent("""
    import sys
    sys.path[:0] = [%r, %r, %r]
    import fake_gen_engine
    fake_gen_engine.install(setattr)
    from chessrl_b200 import gen_data
    gen_data.main(sys.argv[1:])
""")


def _free_port():
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_two_ranks_write_the_single_process_file(tmp_path, monkeypatch):
    args = ["--games", "5", "--lanes", "2", "--depth", "1", "--qdepth", "0", "--margin", "15", "--pick-plies", "8",
            "--max-plies", "16", "--seed", "4"]
    script = tmp_path / "worker.py"
    script.write_text(WORKER % (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")))
    port = str(_free_port())
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=port, CUDA_VISIBLE_DEVICES="")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", port, str(script), str(tmp_path / "ranks.json")] + args
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    fake_gen_engine.install(monkeypatch.setattr)
    gen_data.main([str(tmp_path / "one.json")] + args)
    strip = lambda path: [{k: v for k, v in g.items() if k != "date"} for g in json.loads(path.read_text())]  # noqa
    assert strip(tmp_path / "ranks.json") == strip(tmp_path / "one.json")
    assert len(strip(tmp_path / "one.json")) == 5
