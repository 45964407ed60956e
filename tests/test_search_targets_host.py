"""Search-score training targets (DESIGN.md 3.8) without a GPU.

- the g++ build of the row code (tests/hostsim/search_targets_hostsim.cpp, the kernel's code) against a float64 numpy
  restatement on oracle legal moves and netencoder labels, at T = 1, 50 and 1000, and hand vectors; the comparison
  notices a score list applied in reversed order and a temperature off by a factor of 2;
- the soft-target loss and its gradients against an fp64 restatement; with one-hot targets it is today's loss;
- DatasetGame: scores round-trip, files without scores are unchanged, malformed score lists are refused;
- gen_data --scores on tests/fake_score_engine.FakeScoreEngine (root scores from the oracle's search): every ply's
  scores, the same games as without scores, any lane count, and two gloo ranks."""
import json
import os
import random
import socket
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

import ab_oracle as A
import ab_pick_oracle as P
import chessrl_oracle as O
import fake_gen_engine
import fake_score_engine
from chessrl_b200 import boards as B
from chessrl_b200 import gen_data, model, training
from chessrl_b200.netencoder import get_uci_labels
from conftest import ROOT
from hostsim import search_targets as HS
from test_alphabeta_host import fuzz_fens, n_of, playout_fens

chess = O.chess
LABELS = {u: i for i, u in enumerate(get_uci_labels())}


# ---- the definition in float64 --------------------------------------------------------------------------------------
def oracle_row(fen, scores, temperature):
    """(policy float64 [1968], v_s) of DESIGN.md 3.8 for the position and its root scores."""
    b = chess.Board(fen)
    legal = [m.uci() for m in b.generate_legal_moves()]
    assert len(legal) == len(scores)
    s = np.asarray(scores, dtype=np.float64)
    best = s.max()
    e = np.exp((s - best) / temperature)
    row = np.zeros(1968)
    for m, p in zip(legal, e / e.sum()):
        row[LABELS[m]] = p
    v = np.tanh(best / 400.0)
    return row, (v if b.turn else -v)


def random_scores(rng, n):
    kind = rng.randrange(4)
    if kind == 0:                                        # ordinary centipawns
        return [rng.randrange(-600, 601) for _ in range(n)]
    if kind == 1:                                        # many ties
        return [rng.choice((-40, 0, 0, 25, 25)) for _ in range(n)]
    s = [rng.randrange(-300, 301) for _ in range(n)]     # mate scores for either side
    for _ in range(rng.randrange(1, 3)):
        h = rng.randrange(1, 14)
        s[rng.randrange(n)] = (32000 - h) if kind == 2 else -(32000 - h)
    return s


@pytest.fixture(scope="module")
def cases():
    rng = random.Random(31)
    fens = fuzz_fens(n_of(1000), 301) + playout_fens(n_of(1000), 302) + [SINGLE]
    return [(f, random_scores(rng, len(list(chess.Board(f).generate_legal_moves())))) for f in fens]


SINGLE = "4k3/8/8/8/8/8/r7/K6r w - - 0 1"          # Kxa2 is the only legal move


def host(cases, temperature, transform=lambda s: s):
    return HS.targets([B.record_from_fen(f) for f, _ in cases], [transform(s) for _, s in cases], temperature)


@pytest.mark.parametrize("temperature", [1.0, 50.0, 1000.0])
def test_host_build_equals_the_definition(cases, temperature):
    policy, value, legal = host(cases, temperature)
    assert len(cases) >= n_of(2000)
    assert any(len(s) == 1 for _, s in cases)
    for i, (fen, scores) in enumerate(cases):
        want, v = oracle_row(fen, scores, temperature)
        assert legal[i] == len(scores)
        assert np.abs(policy[i] - want).max() <= 1e-6, (fen, scores)
        assert (policy[i][want == 0] == 0).all()          # exact zeros off the legal set
        assert abs(float(value[i]) - v) <= 1e-6


def test_comparison_notices_reversed_scores_and_a_doubled_temperature(cases):
    want = [oracle_row(f, s, 50.0)[0] for f, s in cases]
    rev = host(cases, 50.0, transform=lambda s: s[::-1])[0]
    hot = host(cases, 100.0)[0]
    bad_rev = sum(np.abs(rev[i] - want[i]).max() > 1e-6 for i in range(len(cases)))
    bad_hot = sum(np.abs(hot[i] - want[i]).max() > 1e-6 for i in range(len(cases)))
    assert bad_rev >= len(cases) // 2 and bad_hot >= len(cases) // 2, (bad_rev, bad_hot)


def test_hand_vectors():
    start = B.record_from_fen()
    first = [m.uci() for m in chess.Board().generate_legal_moves()]
    # one legal move: all the mass, whatever its score
    p, v, n = HS.targets([B.record_from_fen(SINGLE)], [[-250]], 50.0)
    assert n[0] == 1 and p[0, LABELS["a1a2"]] == 1.0 and p[0].sum() == 1.0
    # two equal best scores, the others far below: one half each
    s = [-5000] * 20
    s[3] = s[11] = 17
    p, v, _ = HS.targets([start], [s], 1.0)
    assert p[0, LABELS[first[3]]] == 0.5 and p[0, LABELS[first[11]]] == 0.5 and np.count_nonzero(p[0]) == 2
    # a mating move against ordinary scores takes essentially all the mass, and v_s is +-tanh(~80) = +-1
    s = [rng_s for rng_s in range(-100, 100, 10)]
    s[7] = 31995
    p, v, _ = HS.targets([start], [s], 50.0)
    assert p[0, LABELS[first[7]]] >= 1 - 1e-6 and v[0] == 1.0
    # v_s is from white's point of view: the same best score with black to move changes sign
    black = B.record_from_fen("rnbqkbnr/pppppppp/8/8/8/5N2/PPPPPPPP/RNBQKB1R b KQkq - 1 1")
    s = [100] + [0] * 19
    pw, vw, _ = HS.targets([start], [s], 50.0)
    pb, vb, _ = HS.targets([black], [s], 50.0)
    assert vw[0] == -vb[0] == np.float32(np.tanh(0.25)) and np.array_equal(np.sort(pw[0]), np.sort(pb[0]))
    # a score count that is not the legal count leaves the row zero and reports the legal count
    p, v, n = HS.targets([start], [[0] * 19], 50.0)
    assert n[0] == 20 and not p.any() and v[0] == 0


def test_value_weight_zero_is_todays_value_target():
    r = torch.tensor([1.0, 0.0, -1.0, 0.0])
    vs = torch.tensor([0.3, -0.999, 0.5, 1.0])
    assert torch.equal(training.blend_value(r, vs, 0.0), r)
    assert torch.allclose(training.blend_value(r, vs, 0.5), 0.5 * r + 0.5 * vs)
    assert torch.equal(training.blend_value(r, vs, 1.0), vs)
    for bad in (training.SearchTargets(0.0), training.SearchTargets(float("inf")), training.SearchTargets(50, 1.5),
                training.SearchTargets(50, -0.1), (50, 0.5)):
        with pytest.raises(ValueError):
            training.check_targets(bad)
    assert training.check_targets(None) is None and training.SearchTargets() == (50.0, 0.5)


# ---- the loss -------------------------------------------------------------------------------------------------------
def _soft_ref(pack, x, probs, val, trainable):
    """fp64 restatement: oracle/train_ref.py's forward pass and Keras loss with the one-hot replaced by `probs`."""
    import train_ref
    p = [torch.tensor(np.asarray(w), dtype=torch.float64) for w in pack]
    for i in trainable:
        p[i].requires_grad_(True)
    policy, value, _ = train_ref.forward_train(p, torch.as_tensor(x, dtype=torch.float64))
    q = torch.clamp(policy / policy.sum(dim=-1, keepdim=True), train_ref.KERAS_EPS, 1.0 - train_ref.KERAS_EPS)
    ce = (-(torch.as_tensor(probs, dtype=torch.float64) * torch.log(q)).sum(dim=-1)).mean()
    mse = ((value - torch.as_tensor(val, dtype=torch.float64)) ** 2).mean()
    reg = train_ref.L2 * sum((p[i] ** 2).sum() for i in train_ref.kernel_indices([tuple(t.shape) for t in p]))
    total = ce + mse + reg
    grads = torch.autograd.grad(total, [p[i] for i in trainable])
    return total.item(), ce.item(), {i: g.numpy() for i, g in zip(trainable, grads)}


def _soft_probs(pol, seed):
    rng = np.random.default_rng(seed)
    probs = np.zeros((len(pol), 1968), dtype=np.float32)
    for r in range(len(pol)):
        cols = np.concatenate([[pol[r]], rng.choice(1968, 20, replace=False)])
        w = rng.random(len(cols)).astype(np.float32)
        probs[r, cols] = w / w.sum()
    return probs


def _step(pack, x, pol, val, probs, tr):
    from test_training_step import _fixed_cpu_summation_order
    params = [torch.tensor(w) for w in pack]
    for i in tr:
        params[i].requires_grad_(True)
    with _fixed_cpu_summation_order():
        out = training.loss_terms(params, torch.as_tensor(x), torch.as_tensor(pol), torch.as_tensor(val), training=True,
                                  probs=None if probs is None else torch.as_tensor(probs))
        grads = torch.autograd.grad(out[0], [params[i] for i in tr])
    return out, grads


def check_soft_step(pack, x, pol, val, probs, tr, step):
    """loss and policy term within 1e-5, gradients 2e-2 of a tensor's largest entry / 4e-3 in L2 (the bounds of
    tests/test_training_step.py for today's step)."""
    (total, loss_p, _, _, _), grads = step
    ref_total, ref_ce, ref_grads = _soft_ref(pack, x, probs, val, tr)
    assert abs(total.item() - ref_total) <= 1e-5 * max(1.0, abs(ref_total))
    assert abs(loss_p.item() - ref_ce) <= 1e-5 * max(1.0, abs(ref_ce))
    dead = {3 + 12 * b + 6 * k for b in range(10) for k in range(2)} | {123, 131}
    for i, g in zip(tr, grads):
        if i in dead:
            continue
        g64, g32 = ref_grads[i], g.detach().cpu().numpy().astype(np.float64)
        scale = np.abs(g64).max()
        assert scale > 1e-9, i
        assert np.abs(g32 - g64).max() / scale <= 2e-2 and np.linalg.norm(g32 - g64) / np.linalg.norm(g64) <= 4e-3, i


def test_soft_loss_and_gradients_match_fp64_restatement():
    from test_training_step import _batch
    pack = model.random_pack(seed=21, perturb_bn=True)
    x, pol, val = _batch()
    probs = _soft_probs(pol, 3)
    tr = training.trainable_indices()
    check_soft_step(pack, x, pol, val, probs, tr, _step(pack, x, pol, val, probs, tr))


def test_one_hot_targets_give_todays_loss():
    from test_training_step import _batch
    pack = model.random_pack(seed=5)
    x, pol, val = _batch(n_positions=12, seed=9)
    tr = training.trainable_indices()
    onehot = np.zeros((len(pol), 1968), dtype=np.float32)
    onehot[np.arange(len(pol)), pol] = 1.0
    (a, _), (b, _) = _step(pack, x, pol, val, None, tr), _step(pack, x, pol, val, onehot, tr)
    for ta, tb in zip(a[:4], b[:4]):
        assert abs(ta.item() - tb.item()) <= 1e-6


# ---- DatasetGame ----------------------------------------------------------------------------------------------------
def _entry(moves, scores=None, result=None):
    e = {"moves": moves, "result": result, "player_color": True, "date": "01/01/2020 00:00:00"}
    if scores is not None:
        e["scores"] = scores
    return e


def test_dataset_round_trip_and_unchanged_files(tmp_path, monkeypatch):
    from chessrl_b200.dataset import DatasetGame
    fake_gen_engine.install(monkeypatch.setattr)
    plain = [_entry(["e2e4", "e7e5", "g1f3"], result=None), _entry(["d2d4"], result=None)]
    scored = _entry(["e2e4", "e7e5"], [[5] * 20, list(range(-10, 10))])
    ds = DatasetGame()
    ds.loads(json.dumps(plain + [scored]))
    assert [g.search_scores for g in ds.games] == [None, None, scored["scores"]]
    out = tmp_path / "a.json"
    ds.save(str(out))
    assert json.loads(out.read_text()) == plain + [scored]
    only_plain = DatasetGame(ds.games[:2])
    out2 = tmp_path / "b.json"
    only_plain.save(str(out2))
    assert out2.read_text() == json.dumps(plain)          # the reference's format, byte for byte
    assert "scores" not in ds.games[0].get_history() and ds.games[2].get_copy().search_scores is None
    # a rejected move drops its score list with it
    ds2 = DatasetGame()
    ds2.loads(json.dumps([_entry(["e2e4", "e2e5", "e7e5"], [[1] * 20, [2], [3] * 20])]))
    assert ds2.games[0].get_history()["moves"] == ["e2e4", "e7e5"]
    assert ds2.games[0].search_scores == [[1] * 20, [3] * 20]


@pytest.mark.parametrize("scores", [[[0] * 20], [[0] * 20, [0] * 20, [0]], [[0] * 20, [0.5] * 20], [[0] * 20, "x"],
                                    [[0] * 20, [True] * 20], {"a": 1}])
def test_dataset_refuses_malformed_scores(scores, monkeypatch):
    from chessrl_b200.dataset import DatasetGame
    fake_gen_engine.install(monkeypatch.setattr)
    with pytest.raises(ValueError, match="game 1"):
        DatasetGame().loads(json.dumps([_entry(["e2e4"]), _entry(["e2e4", "e7e5"], scores)]))


# ---- gen_data --scores ----------------------------------------------------------------------------------------------
KW = dict(depth=1, qdepth=0, margin=15, pick_plies=8, max_plies=20)


def run(n, lanes, seed, scores=True, **kw):
    eng = fake_score_engine.FakeScoreEngine(lanes)
    return gen_data.generate_games(n, lanes=lanes, seed=seed, engine=eng, scores=scores, **dict(KW, **kw))[0]


def _plain(games):
    return [{k: ([s.tolist() for s in v] if k == "scores" else v) for k, v in g.items()} for g in games]


@pytest.mark.parametrize("depth,qdepth,n,max_plies", [(1, 0, 6, 20), (2, 2, 2, 8)])
def test_gen_data_scores_are_the_oracles(depth, qdepth, n, max_plies):
    kw = dict(depth=depth, qdepth=qdepth, max_plies=max_plies)
    games = run(n, n, seed=5, **kw)
    assert _plain(run(n, n, seed=5, scores=False, **kw)) == [{k: v for k, v in g.items() if k != "scores"}
                                                            for g in _plain(games)]
    salts = gen_data.game_salts(5, 0, n)
    for j, g in enumerate(games):
        assert len(g["scores"]) == len(g["moves"])
        b = chess.Board()
        for ply, (m, s) in enumerate(zip(g["moves"], g["scores"])):
            _, _, vals = A.search(b, depth, qdepth)
            assert s.tolist() == vals, (j, ply)
            legal = [x.uci() for x in b.generate_legal_moves()]
            assert legal[P.pick_index(vals, ply, KW["margin"], KW["pick_plies"], int(salts[j]))] == m
            b.push(chess.Move.from_uci(m))


def test_gen_data_scores_do_not_depend_on_lanes():
    ref = _plain(run(8, 8, seed=3))
    for lanes in (1, 7):
        assert _plain(run(8, lanes, seed=3)) == ref


def test_gen_data_cli_writes_scores(tmp_path, monkeypatch):
    fake_score_engine.install(monkeypatch.setattr)
    argv = ["--games", "4", "--lanes", "3", "--depth", "1", "--qdepth", "0", "--margin", "15", "--pick-plies", "8",
            "--max-plies", "12", "--seed", "6"]
    summary = gen_data.main([str(tmp_path / "s.json")] + argv + ["--scores"])
    gen_data.main([str(tmp_path / "p.json")] + argv)
    s, p = json.loads((tmp_path / "s.json").read_text()), json.loads((tmp_path / "p.json").read_text())
    assert summary["scores"] is True
    assert [{k: v for k, v in g.items() if k not in ("scores", "date")} for g in s] == \
        [{k: v for k, v in g.items() if k != "date"} for g in p]
    assert all("scores" not in g for g in p)
    want = _plain(run(4, 4, seed=6, max_plies=12))
    assert [g["scores"] for g in s] == [g["scores"] for g in want]
    from chessrl_b200.dataset import DatasetGame
    ds = DatasetGame()
    ds.load(str(tmp_path / "s.json"))
    assert [g.search_scores for g in ds.games] == [g["scores"] for g in want]


WORKER = textwrap.dedent("""
    import sys
    sys.path[:0] = [%r, %r, %r]
    import fake_score_engine
    fake_score_engine.install(setattr)
    from chessrl_b200 import gen_data
    gen_data.main(sys.argv[1:])
""")


def _free_port():
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_two_ranks_write_the_single_process_file_with_scores(tmp_path, monkeypatch):
    args = ["--games", "5", "--lanes", "2", "--depth", "1", "--qdepth", "0", "--margin", "15", "--pick-plies", "8",
            "--max-plies", "16", "--seed", "4", "--scores"]
    script = tmp_path / "worker.py"
    script.write_text(WORKER % (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")))
    port = str(_free_port())
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=port, CUDA_VISIBLE_DEVICES="")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", port, str(script), str(tmp_path / "ranks.json")] + args
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    fake_score_engine.install(monkeypatch.setattr)
    gen_data.main([str(tmp_path / "one.json")] + args)
    strip = lambda path: [{k: v for k, v in g.items() if k != "date"} for g in json.loads(path.read_text())]  # noqa
    one = strip(tmp_path / "one.json")
    assert strip(tmp_path / "ranks.json") == one
    assert len(one) == 5 and all(len(g["scores"]) == len(g["moves"]) > 0 for g in one)
