"""The evaluation path at full width: the network as a search batch runs it -- row count in device memory, launch bound
on the host, the two-tile tower instantiation -- against the uncounted forward pass, and the 4,096-lane search with the
real network against the oracle.

Every comparison here is bit-exact (torch.equal / array equality): the kernels' rows must not depend on the batch they
sit in, on where they sit in it, on the tower instantiation, or on rows that are not part of the batch.  That is what lets the oracle be served by crl_net_forward in small batches while the engine evaluates the same
positions as rows of 4,096-row batches (net_oracle.py).

Default sizes keep this file to a few minutes; CRL_PARITY_SIMS=200 CRL_PARITY_MOVES=4 runs the searches at BASELINE's
size, CRL_EVALPATH_SAMPLES sets how many lanes the oracle replays.
"""
import os
import random

import numpy as np
import pytest
import torch

import chessrl_oracle as O
import model_torch
import netpacks
from chessrl_b200 import boards as B
from chessrl_b200._lib import CRL_EINVAL, EVAL_NET, N_LABELS
from chessrl_b200.engine import Engine
from chessrl_b200.lockstep import compute_policy
from net_oracle import BatchedNetEvaluator, run_oracle_threads

pytestmark = pytest.mark.gpu

SIMS = int(os.environ.get("CRL_PARITY_SIMS", "64"))
MOVES = int(os.environ.get("CRL_PARITY_MOVES", "2"))
SAMPLES = int(os.environ.get("CRL_EVALPATH_SAMPLES", "16"))
SENTINEL = -7.0
SINGLE_TILE_MAX = 296            # 74 CTA pairs x 4 boards: larger launch bounds take the two-tile instantiation (B200)
STAT_KEYS = ("visits", "values", "priors", "moves", "replies", "results", "n_children", "root_visits", "root_values")


@pytest.fixture(autouse=True)
def _fp32_reference_without_tf32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _batch(seed):
    """4,096 rows of bf16 planes: synthetic 0/1 planes with real midgame positions at the start, around the
    single-tile limit, around the persistent grid's round (592) and at the end."""
    x = netpacks.synthetic_planes(4096, seed=seed)
    real = netpacks.planes_of(netpacks.midgame_games(128, seed=seed))
    x[:32], x[280:312], x[576:608], x[-32:] = real[:32], real[32:64], real[64:96], real[96:]
    return x


@pytest.fixture(scope="module")
def pack():
    return netpacks.lively_pack()


@pytest.fixture(scope="module")
def planes(pack):
    """(live planes, different live planes for the stale rows), both [4096,8,8,128] bf16 on the device."""
    x, y = _batch(101), _batch(202)
    rp, rv = model_torch.forward(pack, x[:32, ..., :127], device="cuda")
    netpacks.assert_lively(rp, rv)
    to = lambda a: torch.from_numpy(a).to("cuda").to(torch.bfloat16)       # noqa: E731
    return to(x), to(y)


@pytest.fixture(scope="module")
def wide(pack):
    e = Engine(max_games=4096, max_nodes=2)
    e.load_weights(pack)
    yield e
    e.close()


# ---- a. counted batches --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bound", [296, 297, 592, 593, 4096])
def test_counted_batch_equals_uncounted_forward(wide, planes, bound):
    """Rows below the device count are bit-identical to crl_net_forward of those rows alone; rows from the count to the
    bound (which hold other live positions, as a search's planes buffer holds the previous batch) are neither evaluated
    into the outputs nor leak into the counted rows."""
    x, y = planes
    counts = sorted({min(c, bound) for c in (0, 1, 3, 4, 5, 8, 9, 295, 296, 297, bound - 1, bound)})
    dev = wide.device
    for count in counts:
        inp = torch.cat([x[:count], y[count:bound]]).contiguous()
        pol = torch.full((bound, N_LABELS), SENTINEL, device=dev)
        val = torch.full((bound,), SENTINEL, device=dev)
        cnt = torch.tensor([count], dtype=torch.int32, device=dev)
        wide.debug_forward_counted(inp, bound, cnt, pol, val)
        torch.cuda.synchronize()
        assert (pol[count:] == SENTINEL).all() and (val[count:] == SENTINEL).all(), (bound, count)
        if count == 0:
            continue
        rp, rv = wide.net_forward(x[:count].contiguous())
        assert torch.equal(pol[:count], rp) and torch.equal(val[:count], rv), (bound, count)
        if count >= 2:                                   # the comparison tells rows apart: one row off would fail
            assert not torch.equal(pol[1:count], rp[:count - 1])
    # a count above the bound is the bound
    inp = x[:bound].contiguous()
    p1, v1 = wide.debug_forward_counted(inp, bound, bound)
    p2, v2 = wide.debug_forward_counted(inp, bound, bound + 7)
    assert torch.equal(p1, p2) and torch.equal(v1, v2)


def test_counted_batch_rejects_bad_arguments(wide, planes):
    x, _ = planes
    lib, h = wide.lib, wide.h
    cnt = torch.ones(1, dtype=torch.int32, device=wide.device)
    pol = torch.empty((8, N_LABELS), device=wide.device)
    val = torch.empty((8,), device=wide.device)
    assert lib.crl_debug_forward_counted(h, x.data_ptr(), 8, None, pol.data_ptr(), val.data_ptr()) == CRL_EINVAL
    assert lib.crl_debug_forward_counted(h, x.data_ptr(), -1, cnt.data_ptr(), pol.data_ptr(), val.data_ptr()) == CRL_EINVAL
    assert lib.crl_debug_forward_counted(h, x.data_ptr(), 8, cnt.data_ptr(), None, val.data_ptr()) == CRL_EINVAL
    # a launch bound beyond the engine's row capacity is refused before anything runs
    assert lib.crl_debug_forward_counted(h, x.data_ptr(), 1 << 20, cnt.data_ptr(), pol.data_ptr(), val.data_ptr()) == CRL_EINVAL
    assert lib.crl_debug_forward_counted(h, None, 0, cnt.data_ptr(), None, None) == 0     # an empty launch bound: nothing to do


# ---- b. the bit-identity checks can fail -----------------------------------------------------------------------------
def _rel_err(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def test_bit_identity_is_not_vacuous_per_layer(wide, pack, planes):
    """Layer 1 of the tower recomputed by k_conv_v2 from the tower's own layer-0 output: the same convolution on the same
    bf16 input, but k_conv_v2 accumulates tap-outer / channel-slice-inner where k_trunk4 accumulates channel-slice-outer /
    tap-inner.  It lands within the emulation's tolerance but differs in at least one bit: the outputs are sensitive to
    summation order, so the torch.equal checks in this file mean something."""
    x, _ = planes
    xs = x[:593].contiguous()
    tap0 = wide.debug_tower(xs, layer=0)["act"]
    tap1 = wide.debug_tower(xs, layer=1)["act"]
    conv = wide.debug_conv(1, tap0, None, relu=True)
    torch.cuda.synchronize()
    xf = xs.float().cpu().numpy()[..., :127]
    f32, emu = {}, {}
    rp, rv = model_torch.forward(pack, xf, device="cuda", taps=f32)
    model_torch.forward(pack, xf, device="cuda", emulate_bf16_activations=True, taps=emu)
    netpacks.assert_lively(rp, rv)
    E = _rel_err(emu["act"][1], f32["act"][1])
    assert _rel_err(conv, tap1) <= 2 * E, (_rel_err(conv, tap1), E)
    assert not torch.equal(conv, tap1)


# ---- c. row independence in the two-tile instantiation ----------------------------------------------------------------
@pytest.mark.parametrize("n", [1000, 4096])
def test_rows_do_not_depend_on_their_place_in_the_batch(wide, planes, n):
    """Permuted, shifted (each shift moves a row to another CTA rank / board-in-tile / tile A-B / pair) and duplicated
    rows give bit-identical outputs to the same position anywhere else in the batch."""
    x = planes[0][:n].contiguous()
    p, v = wide.net_forward(x)
    g = torch.Generator().manual_seed(n)
    perm = torch.randperm(n, generator=g).to(x.device)
    pp, vp_ = wide.net_forward(x[perm].contiguous())
    assert torch.equal(pp, p[perm]) and torch.equal(vp_, v[perm])
    swapped = perm.clone()
    swapped[[0, 1]] = swapped[[1, 0]]
    assert not torch.equal(pp, p[swapped])                # two rows swapped would be caught
    for s in (1, 2, 3, 4, 5, 8):
        ps, vs = wide.net_forward(torch.roll(x, s, 0).contiguous())
        assert torch.equal(ps, torch.roll(p, s, 0)) and torch.equal(vs, torch.roll(v, s, 0)), (n, s)
    # eight real positions copied into other groups (both tiles, both CTAs of a pair, the grid's second round)
    offsets = [0, 13, 301, 594, n - 8] + ([1203, 2051, 3000] if n > 3008 else [])
    xc = x.clone()
    for o in offsets:
        xc[o:o + 8] = x[:8]
    pc, vc = wide.net_forward(xc)
    for o in offsets:
        assert torch.equal(pc[o:o + 8], p[:8]) and torch.equal(vc[o:o + 8], v[:8]), (n, o)


# ---- openings for the searches -----------------------------------------------------------------------------------------
def _line(seed, plies):
    rng = random.Random(seed)
    while True:
        g = O.OGame()
        for _ in range(plies):
            if g.get_result() is not None:
                break
            g.move(rng.choice(g.get_legal_moves()))
        if g.get_result() is None:
            return [m.uci() for m in g.board.move_stack]


def _openings(e, seed, max_plies=60, n_lines=0):
    """Seeded random games of 0..max_plies plies in every lane (history rings fill, castling rights go, en-passant
    squares appear), played through the engine's own move generator; with n_lines, every 8th lane instead holds one of
    n_lines fixed lines, lane 8j the line j % n_lines.  Returns the per-lane uci move lists."""
    G = e.max_games
    rng = np.random.default_rng(seed)
    e.games_set(np.tile(B.record_from_fen(), (G, 1)))
    target = rng.integers(0, max_plies + 1, G)
    for ply in range(max_plies):
        legal, cnt = e.games_legal()
        _, _, res = e.games_get()
        mv = np.full(G, B.MOVE_NONE, dtype=np.uint16)
        go = (target > ply) & (cnt > 0) & (res == B.RESULT_NONE)
        pick = (rng.random(G) * np.maximum(cnt, 1)).astype(np.int64)
        mv[go] = legal[np.arange(G), pick][go]
        e.games_play(mv)
    moves = [[B.move_to_uci(m) for m in ms] for ms in e.games_moves(np.arange(G))]
    if n_lines:
        lines = [_line(seed * 100 + j, 20 + 9 * j) for j in range(n_lines)]
        for lane in range(0, G, 8):
            moves[lane] = lines[(lane // 8) % n_lines]
    e.games_set(np.tile(B.record_from_fen(), (G, 1)), [[B.uci_to_move(m) for m in ms] for ms in moves])
    return moves


def _sampled(G, k, seed):
    rest = random.Random(seed).sample(range(1, G - 1), min(k, G) - 2)
    return sorted({0, G - 1, *rest})


def _assert_value_head_alive(recorded, G):
    mean_q = []
    for st, _, _ in recorded:
        for g in range(G):
            k = int(st["n_children"][g])
            if k:
                mean_q.extend(st["values"][g, :k] / np.maximum(st["visits"][g, :k], 1))
    mean_q = np.asarray(mean_q)
    assert mean_q.max() - mean_q.min() > 0.1 and np.count_nonzero(mean_q) > 0.9 * mean_q.size, (mean_q.min(), mean_q.max())


def _search(eng, n_moves, sims, inflight=1, apply=True):
    """n_moves lockstep searches with argmax-of-compute_policy picks -> [(root stats, picks, returned moves)]."""
    G = eng.max_games
    recorded = []
    for _ in range(n_moves):
        eng.mcts_begin_move()
        eng.mcts_simulate(sims, inflight=inflight)
        st = eng.root_stats()
        _, plies, results = eng.games_get()
        picks = np.full(G, -1, dtype=np.int32)
        for g in range(G):
            k = int(st["n_children"][g])
            if results[g] == B.RESULT_NONE and k:
                picks[g] = int(np.argmax(compute_policy(st["visits"][g, :k], st["root_visits"][g], int(plies[g]), False)))
        out = eng.commit(picks, apply=apply)
        recorded.append((st, picks.copy(), out.copy()))
    return recorded


def _oracle_replay(net, moves, lanes, recorded, sims, threads=1):
    """The sampled lanes' searches in the oracle, fed crl_net_forward rows; -> (failures, lanes whose priors were
    compared).  Per move: children count, visits, value sums, root value, priors (float32 bits, where the oracle's root
    is fully expanded -- before that the reference leaves them at 1), the returned (move, reply)."""
    ev = BatchedNetEvaluator(net, len(lanes))
    priors_checked = []

    def worker(i):
        g = lanes[i]
        og = O.OGame()
        for m in moves[g]:
            og.move(m)
        agent = O.OAgent(ev)
        for st, picks, out in recorded:
            if og.get_result() is not None:
                assert picks[g] == -1 and int(st["n_children"][g]) == 0
                continue
            tree = O.OSelfPlayTree(og, threads=threads)
            ret = tree.search_move(agent, max_iters=sims, noise=False, ai_move=True)
            kids = tree.root.children
            n = len(kids)
            assert int(st["n_children"][g]) == n, (g, n)
            assert [c.visits for c in kids] == list(st["visits"][g, :n]), g
            assert [float(c.value) for c in kids] == [float(x) for x in st["values"][g, :n]], g
            assert float(tree.root.value) == float(st["root_values"][g]), g
            assert int(tree.root.visits) == int(st["root_visits"][g]), g
            if not tree.root.unexpanded_actions:
                want = np.array([c.prior for c in kids], dtype=np.float32).view(np.uint32)
                assert np.array_equal(want, st["priors"][g, :n].view(np.uint32)), g
                priors_checked.append(g)
            assert [B.move_to_uci(out[g, 0]), B.move_to_uci(out[g, 1])] == list(ret), g
            og.move(ret[0])
            og.move(ret[1])

    failures = run_oracle_threads(ev, len(lanes), worker)
    return failures, priors_checked


# ---- d. zero-row batches inside a search ---------------------------------------------------------------------------------
def test_search_with_every_lane_parked_then_resumed(pack):
    """Every lane parked: the evaluation batches have a device count of 0 (launch bound 512 rows, two-tile tower).  The
    search returns empty statistics, and a search afterwards is bit-identical to the same search on a fresh engine."""
    G, sims = 512, 16
    eng = Engine(max_games=G, max_nodes=sims + 1, avg_moves=96)
    eng.load_weights(pack)
    eng.set_evaluator(EVAL_NET)
    moves = _openings(eng, seed=5, max_plies=30)
    eng.games_set_active(np.zeros(G, dtype=np.uint8))
    eng.mcts_begin_move()
    eng.mcts_simulate(sims)
    st = eng.root_stats()
    for k in ("visits", "values", "priors", "n_children", "root_visits", "root_values"):
        assert not np.any(st[k]), k
    assert (st["moves"] == B.MOVE_NONE).all() and (st["replies"] == B.MOVE_NONE).all()
    assert (st["results"] == B.RESULT_NONE).all()
    eng.games_set_active(np.ones(G, dtype=np.uint8))
    got = _search(eng, 1, sims, apply=False)[0]
    fresh = Engine(max_games=G, max_nodes=sims + 1, avg_moves=96)
    fresh.load_weights(pack)
    fresh.set_evaluator(EVAL_NET)
    fresh.games_set(np.tile(B.record_from_fen(), (G, 1)), [[B.uci_to_move(m) for m in ms] for ms in moves])
    want = _search(fresh, 1, sims, apply=False)[0]
    assert (got[0]["root_visits"] > 1).sum() > G // 2
    for k in STAT_KEYS:
        assert np.array_equal(got[0][k], want[0][k]), k
    assert np.array_equal(got[2], want[2])
    eng.close()
    fresh.close()


# ---- e. 4,096-lane search parity with the oracle ---------------------------------------------------------------------------
def test_full_width_search_matches_oracle(pack):
    """4,096 lanes x MOVES lockstep moves x SIMS simulations with the real network (two-tile tower, rows placed by
    atomics): copies of the same line anywhere in the batch get identical statistics, and sampled lanes -- lanes 0 and
    4,095 among them -- match the oracle bit for bit."""
    G = int(os.environ.get("CRL_EVALPATH_LANES", "4096"))
    n_lines = 4
    eng = Engine(max_games=G, max_nodes=SIMS + 1, avg_moves=96)
    eng.load_weights(pack)
    eng.set_evaluator(EVAL_NET)
    moves = _openings(eng, seed=17, n_lines=n_lines)
    recorded = _search(eng, MOVES, SIMS)
    eng.close()
    _assert_value_head_alive(recorded, G)

    # the same line in lanes 8j, 8j + 32, ... (all over the batch): identical statistics and returned moves
    for j in range(n_lines):
        lanes = np.arange(8 * j, G, 8 * n_lines)
        assert len(lanes) >= 2
        for st, picks, out in recorded:
            assert int(st["n_children"][lanes[0]]) > 0
            for k in STAT_KEYS:
                assert (st[k][lanes] == st[k][lanes[0]]).all(), (j, k)
            assert (out[lanes] == out[lanes[0]]).all() and (picks[lanes] == picks[lanes[0]]).all(), j

    net = Engine(max_games=SAMPLES, max_nodes=8)           # serves the oracle's evaluations (single-tile tower)
    net.load_weights(pack)
    lanes = _sampled(G, SAMPLES, seed=29)
    failures, priors_checked = _oracle_replay(net, moves, lanes, recorded, SIMS)
    assert not failures, failures[:3]
    assert len(priors_checked) >= len(lanes) // 2, priors_checked
    # the comparison's own sensitivity: the oracle replaying another lane's opening for a sampled lane must fail
    lane = lanes[1]
    other = next(g for g in range(G) if moves[g] != moves[lane])
    wrong = list(moves)
    wrong[lane] = moves[other]
    failures, _ = _oracle_replay(net, wrong, [lane], recorded, SIMS)
    net.close()
    assert failures, (lane, other)


# ---- f. wave mode with the real network -----------------------------------------------------------------------------------
@pytest.mark.parametrize("G,K", [(512, 8), (48, 6)])
def test_wave_mode_real_network_matches_oracle(pack, G, K):
    """K in-flight simulations per game (row cap G*K: 4,096 rows and the two-tile tower at G = 512, K = 8; the
    reference's default K = 6 on 48 lanes, single-tile) against OSelfPlayTree(threads=K)."""
    eng = Engine(max_games=G, max_nodes=SIMS + 1, avg_moves=96, max_inflight=K)
    eng.load_weights(pack)
    eng.set_evaluator(EVAL_NET)
    moves = _openings(eng, seed=G + K)
    recorded = _search(eng, 1, SIMS, inflight=K, apply=False)
    eng.close()
    _assert_value_head_alive(recorded, G)
    net = Engine(max_games=SAMPLES, max_nodes=8)
    net.load_weights(pack)
    lanes = _sampled(G, SAMPLES, seed=G)
    failures, priors_checked = _oracle_replay(net, moves, lanes, recorded, SIMS, threads=K)
    net.close()
    assert not failures, failures[:3]
    assert len(priors_checked) >= len(lanes) // 2, priors_checked


# ---- g. direct calls between searches -------------------------------------------------------------------------------------
def test_direct_forward_calls_do_not_disturb_a_search(pack, planes):
    """crl_net_forward shares the logits / head-input scratch and the cached planes tensor map with the search: calls
    between mcts_begin_move / mcts_simulate calls on the same tree leave its statistics bit-identical, and the search
    leaves crl_net_forward's results unchanged."""
    G, a, b = 512, 12, 12
    x = planes[0]
    fixed = x[:37].contiguous()

    def run(interleave):
        eng = Engine(max_games=G, max_nodes=a + b + 1, avg_moves=96, max_inflight=8)     # 4,096 rows of capacity
        eng.load_weights(pack)
        eng.set_evaluator(EVAL_NET)
        _openings(eng, seed=41, max_plies=40)
        before = eng.net_forward(fixed)
        eng.mcts_begin_move()
        if interleave:
            eng.net_forward(planes[1][:37].contiguous())
        eng.mcts_simulate(a)
        if interleave:
            eng.net_forward(planes[1][:37].contiguous())
            eng.net_forward(x)
        eng.mcts_simulate(b)
        st = eng.root_stats()
        after = eng.net_forward(fixed)
        assert torch.equal(before[0], after[0]) and torch.equal(before[1], after[1])
        eng.close()
        return st

    sa, sb = run(True), run(False)
    assert (sa["root_visits"] == a + b + 1).sum() > G // 2
    for k in STAT_KEYS:
        assert np.array_equal(sa[k], sb[k]), k
