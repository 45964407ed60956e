"""Search-score training targets on the GPU (crl_games_ab_root_scores_host, crl_search_targets, gen_data --scores,
supervised --targets search; DESIGN.md 3.8).

- export: on 4,096 positions at (2,2) and (3,4), the counts are the legal counts (-1 for masked, parked and finished
  lanes), the first maximum is games_ab_move's move and score, ab_pick_oracle.pick_index on the scores reproduces
  games_ab_pick at margins 0 and 20, with and without repetitions; the oracle's child values bit for bit on 64
  positions; CRL_ESTATE before any search; engine state untouched and a later search bit-identical;
- kernel: equals the g++ build of the same row code within 1e-6 on 4,096+ rows, bit-identical across batch compositions
  and runs, exact zeros off the legal set, rows summing to 1; a count mismatch names the game and the ply;
- gen_data --scores: 64 games on 16 and 64 lanes, the moves of a run without scores, a sample of plies against the
  oracle; a CLI file trains with supervised.train(targets="search"); 20 steps on one batch reduce the soft policy loss;
- the training step with search targets against the fp64 restatement."""
import json
import multiprocessing as mp
import os
import random

import numpy as np
import pytest
import torch

import ab_oracle as A
import ab_pick_oracle as P
import chessrl_oracle as O
from chessrl_b200 import boards as B
from chessrl_b200 import gen_data, model, runtime, training
from chessrl_b200._lib import CRL_ESTATE, EVAL_HASH, CrlError
from chessrl_b200.engine import Engine
from hostsim import search_targets as HS
from test_gpu_gen_data import G, PICK_PLIES, positions  # noqa: F401  (the module's 4,096-position fixture)
from test_search_targets_host import LABELS, _soft_probs, _soft_ref, random_scores

pytestmark = pytest.mark.gpu
chess = O.chess
MASKED, PARKED, FINISHED = [0, 1, 2, 3], [4, 5, 6], 7
MATE = ("6k1/5ppp/8/8/8/8/8/R5K1 w - - 0 1", "a1a8")


@pytest.fixture(scope="module")
def engine(positions):  # noqa: F811
    eng = Engine(max_games=G, max_nodes=2, avg_moves=64)
    eng.games_set(positions[2], positions[3])
    eng.games_set(B.record_from_fen(MATE[0])[None, :], [[B.uci_to_move(MATE[1])]], first=FINISHED)
    active = np.ones(G, dtype=np.uint8)
    active[PARKED] = 0
    eng.games_set_active(active)
    yield eng
    eng.close()


def _mask():
    m = np.ones(G, dtype=np.uint8)
    m[MASKED] = 0
    return m


def _ply(recs):
    return ((recs[:, 8] >> np.uint64(38)) & np.uint64(16383)).astype(np.int64)


def test_export_before_any_search():
    eng = Engine(max_games=2, max_nodes=2, avg_moves=64)
    try:
        with pytest.raises(CrlError) as ei:
            eng.games_ab_root_scores()
        assert ei.value.status == CRL_ESTATE
    finally:
        eng.close()


@pytest.mark.parametrize("repetitions", [False, True])
@pytest.mark.parametrize("depth,qdepth", [(2, 2), (3, 4)])
def test_export_matches_the_search(engine, positions, depth, qdepth, repetitions):  # noqa: F811
    salts = positions[4]
    rec = engine.games_get()[0]
    legal, n_legal = engine.games_legal()
    idle = np.zeros(G, dtype=bool)
    idle[MASKED + PARKED + [FINISHED]] = True
    for margin in (0, 20):
        picks = engine.games_ab_pick(depth, qdepth, margin, PICK_PLIES, salts, mask=_mask(), repetitions=repetitions)[0]
        scores, counts = engine.games_ab_root_scores()
        assert (counts[idle] == -1).all() and np.array_equal(counts[~idle], n_legal[~idle])
        assert (scores[idle] == 0).all()
        ply = _ply(rec)
        for g in np.nonzero(~idle)[0]:
            s = scores[g, :counts[g]].tolist()
            assert not scores[g, counts[g]:].any()
            k = P.pick_index(s, int(ply[g]), margin, PICK_PLIES, int(salts[g]))
            assert legal[g, k] == picks[g], g
    best_mv, best_sc, _ = engine.games_ab_move(depth, qdepth, mask=_mask(), repetitions=repetitions)
    scores, counts = engine.games_ab_root_scores()
    for g in np.nonzero(~idle)[0]:
        s = scores[g, :counts[g]]
        assert s.max() == best_sc[g] and legal[g, int(np.argmax(s))] == best_mv[g], g


def _oracle_vals(fen):
    return A.search(chess.Board(fen), 2, 2)[2]


def test_export_equals_the_oracles_child_values(engine, positions):  # noqa: F811
    lanes = np.concatenate([8 + np.arange(32), G // 2 + np.arange(32)])
    mask = np.zeros(G, dtype=np.uint8)
    mask[lanes] = 1
    engine.games_ab_move(2, 2, mask=mask)
    scores, counts = engine.games_ab_root_scores()
    with mp.get_context("fork").Pool(min(16, os.cpu_count() or 4)) as pool:
        want = pool.map(_oracle_vals, [positions[0][g] for g in lanes])
    for g, w in zip(lanes, want):
        assert scores[g, :counts[g]].tolist() == w, positions[0][g]
    assert (counts[np.setdiff1d(np.arange(G), lanes)] == -1).all()


def _hash_search(with_export):
    n, sims = 64, 48
    from test_alphabeta_host import playout_fens
    eng = Engine(max_games=n, max_nodes=sims + 1, avg_moves=64)
    try:
        eng.set_evaluator(EVAL_HASH, 5, 24)
        eng.games_set(np.stack([B.record_from_fen(f) for f in playout_fens(n, 8)]))
        before = eng.games_get(), [eng.game_moves(g) for g in range(n)]
        if with_export:
            eng.games_ab_pick(2, 2, 40, 100, np.arange(n, dtype=np.uint64))
            eng.games_ab_root_scores()
            after = eng.games_get(), [eng.game_moves(g) for g in range(n)]
            assert all(np.array_equal(x, y) for x, y in zip(before[0], after[0]))
            assert all(np.array_equal(x, y) for x, y in zip(before[1], after[1]))
        eng.mcts_begin_move()
        eng.mcts_simulate(sims)
        return eng.root_stats(), [eng.node_dump(g) for g in (0, 17, 63)]
    finally:
        eng.close()


def test_export_leaves_the_engine_alone():
    (a, da), (b, db) = _hash_search(False), _hash_search(True)
    for k in a:
        if a[k] is not None:
            assert np.array_equal(a[k], b[k]), k
    for x, y in zip(da, db):
        assert [bytes(n) for n in x] == [bytes(n) for n in y]


# ---- the kernel -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rows(positions):  # noqa: F811
    """4,096 + 1 rows: the fixture's positions (and a one-move position) with random score lists, mates and ties."""
    rng = random.Random(41)
    fens = list(positions[0]) + ["4k3/8/8/8/8/8/r7/K6r w - - 0 1"]
    scores = [random_scores(rng, len(list(chess.Board(f).generate_legal_moves()))) for f in fens]
    return fens, np.stack([B.record_from_fen(f) for f in fens]), scores


def _device(records, scores, temperature, eng=None):
    eng = eng or runtime.scalar_engine()
    cnt = np.array([len(s) for s in scores], dtype=np.int32)
    off = np.zeros(len(cnt) + 1, dtype=np.int32)
    off[1:] = np.cumsum(cnt)
    flat = torch.tensor([v for s in scores for v in s], dtype=torch.int32, device=eng.device)
    p, v, n = eng.search_targets(eng.boards_to_device(records), flat, torch.from_numpy(off).to(eng.device), temperature)
    return p.cpu().numpy(), v.cpu().numpy(), n.cpu().numpy()


@pytest.mark.parametrize("temperature", [1.0, 50.0, 1000.0])
def test_kernel_equals_host_build(rows, temperature):
    fens, recs, scores = rows
    p, v, n = _device(recs, scores, temperature)
    hp, hv, hn = HS.targets(recs, scores, temperature)
    assert len(fens) >= 4096 and np.array_equal(n, hn) and (n == [len(s) for s in scores]).all()
    assert np.abs(p - hp).max() <= 1e-6 and np.abs(v - hv).max() <= 1e-6
    assert np.abs(p.astype(np.float64).sum(1) - 1.0).max() <= 1e-6
    for i in range(0, len(fens), 97):                      # exact zeros off the legal set
        on = np.zeros(1968, dtype=bool)
        on[[LABELS[m.uci()] for m in chess.Board(fens[i]).generate_legal_moves()]] = True
        assert (p[i][~on] == 0).all()


def test_kernel_rows_do_not_depend_on_the_batch(rows):
    _, recs, scores = rows
    full = _device(recs, scores, 50.0)
    again = _device(recs, scores, 50.0)
    assert all(np.array_equal(a, b) for a, b in zip(full, again))
    rng = np.random.default_rng(3)
    for size in (1, 37, 4096):
        pick = np.sort(rng.choice(len(scores), size, replace=False)) if size < len(scores) else np.arange(size)
        part = _device(recs[pick], [scores[i] for i in pick], 50.0)
        for a, b in zip(part, full):
            assert np.array_equal(a, b[pick]), size


def test_count_mismatch_names_the_game_and_ply():
    from chessrl_b200.game import Game
    games = []
    for moves in (["e2e4", "e7e5"], ["d2d4", "d7d5", "c2c4"]):
        g = Game()
        g._sync(extra=moves)
        b = chess.Board()
        g.search_scores = []
        for m in moves:
            g.search_scores.append([0] * len(list(b.generate_legal_moves())))
            b.push(chess.Move.from_uci(m))
        games.append(g)
    training.encode_search_games(games, [False, False], training.SearchTargets())
    n = len(games[1].search_scores[2])
    games[1].search_scores[2] = [0] * (n + 1)
    with pytest.raises(ValueError, match=r"dataset game 6, ply 2: %d root scores for %d legal moves" % (n + 1, n)):
        training.encode_search_games(games, [False, False], training.SearchTargets(), first=5)


# ---- gen_data --scores ----------------------------------------------------------------------------------------------
KW = dict(depth=2, qdepth=2, margin=20, pick_plies=PICK_PLIES, max_plies=160, seed=11)


def _plain(games):
    return [{k: ([s.tolist() for s in v] if k == "scores" else v) for k, v in g.items()} for g in games]


@pytest.fixture(scope="module")
def games64():
    a = _plain(gen_data.generate_games(64, lanes=64, scores=True, **KW)[0])
    b = _plain(gen_data.generate_games(64, lanes=16, scores=True, **KW)[0])
    c = gen_data.generate_games(64, lanes=64, **KW)[0]
    return a, b, c


def _oracle_sample(s):
    moves, ply = s
    b = chess.Board()
    for m in moves[:ply]:
        b.push(chess.Move.from_uci(m))
    return A.search(b, KW["depth"], KW["qdepth"])[2]


def test_gen_data_scores(games64):
    a, b, c = games64
    assert a == b
    assert [{k: v for k, v in g.items() if k != "scores"} for g in a] == c
    assert all(len(g["scores"]) == len(g["moves"]) for g in a)
    sample = [(g["moves"], ply) for g in a[:32] for ply in (0, len(g["moves"]) // 2, len(g["moves"]) - 1)]
    with mp.get_context("fork").Pool(min(16, os.cpu_count() or 4)) as pool:
        want = pool.map(_oracle_sample, sample)
    got = [g["scores"][ply] for g in a[:32] for ply in (0, len(g["moves"]) // 2, len(g["moves"]) - 1)]
    assert got == want


def test_cli_file_trains_with_search_targets(tmp_path):
    from chessrl_b200 import supervised
    from chessrl_b200.dataset import DatasetGame
    out = tmp_path / "games.json"
    summary = gen_data.main([str(out), "--games", "8", "--depth", "1", "--qdepth", "2", "--max-plies", "60",
                             "--seed", "2", "--scores"])
    saved = json.loads(out.read_text())
    assert len(saved) == 8 and summary["scores"] and all(len(g["scores"]) == len(g["moves"]) for g in saved)
    ds = DatasetGame()
    ds.load(str(out))
    assert [g.search_scores for g in ds.games] == [g["scores"] for g in saved]
    model_dir = tmp_path / "model"
    model_dir.mkdir()
    supervised.train(str(model_dir), str(out), epochs=1, batch_size=2, targets="search")
    assert any(f.endswith(".h5") for f in os.listdir(model_dir))
    log = [json.loads(line) for line in open(model_dir / "train_log.jsonl")]
    assert log[0]["search_targets"]["games_without_scores"] == 0 and log[0]["search_targets"]["games"] == 8
    assert any("val_loss" in r and np.isfinite(r["val_policy_loss"]) for r in log)


def test_search_targets_are_learnable(games64):
    from chessrl_b200.dataset import DatasetGame
    ds = DatasetGame()
    ds.loads(json.dumps([dict(g, player_color=True, date="01/01/2020 00:00:00") for g in games64[0][:4]]))
    planes, pol, val, probs = training.encode_search_games(ds.games, [False] * 4, training.SearchTargets())
    assert (probs.sum(1) - 1).abs().max() <= 1e-5 and (probs.max(1).values < 1).any()
    params = [torch.tensor(w, device=planes.device) for w in model.random_pack(2)]
    tr = []
    for i in training.trainable_indices():
        params[i].requires_grad_(True)
        tr.append(params[i])
    opt = training.KerasAdam(tr)
    losses = [training.train_step(params, opt, planes, pol, val, probs)["policy_loss"] for _ in range(20)]
    # the soft cross-entropy is bounded below by the targets' entropy: the excess over it must fall
    floor = float(-(probs * torch.log(probs.clamp_min(1e-30))).sum(1).mean())
    assert losses[-1] - floor < 0.85 * (losses[0] - floor), (losses, floor)


def test_training_step_with_search_targets_matches_fp64_restatement():
    from test_training_step import _batch
    pack = model.random_pack(seed=21, perturb_bn=True)
    x, pol, val = _batch(n_positions=24, seed=6)
    probs = _soft_probs(pol, 4)
    tr = training.trainable_indices()
    params = [torch.tensor(w, device="cuda") for w in pack]
    for i in tr:
        params[i].requires_grad_(True)
    with training.arithmetic("fp32"):
        total, loss_p, _, _, _ = training.loss_terms(params, torch.as_tensor(x, device="cuda"),
                                                     torch.as_tensor(pol, device="cuda"),
                                                     torch.as_tensor(val, device="cuda"), training=True,
                                                     probs=torch.as_tensor(probs, device="cuda"))
        grads = torch.autograd.grad(total, [params[i] for i in tr])
    ref_total, ref_ce, ref_grads = _soft_ref(pack, x, probs, val, tr)
    assert abs(total.item() - ref_total) <= 1e-5 * max(1.0, abs(ref_total))
    assert abs(loss_p.item() - ref_ce) <= 1e-5 * max(1.0, abs(ref_ce))
    dead = {3 + 12 * b + 6 * k for b in range(10) for k in range(2)} | {123, 131}
    for i, g in zip(tr, grads):
        if i in dead:
            continue
        g64, g32 = ref_grads[i], g.detach().cpu().numpy().astype(np.float64)
        scale = np.abs(g64).max()
        assert np.abs(g32 - g64).max() / scale <= 2e-2 and np.linalg.norm(g32 - g64) / np.linalg.norm(g64) <= 4e-3, i
