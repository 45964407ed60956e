"""The opt-in fp8 tower (include/chessrl_b200.h crl_net_load_fp8_host) on the GPU: against its emulation
(tests/fp8_emu.py), bit identity within fp8, the search in fp8 against the oracle, switching, and the error paths."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import fp8_emu
import model_torch
import netpacks
from chessrl_b200 import boards as B
from chessrl_b200._lib import CRL_EINVAL, CRL_ESTATE, EVAL_NET, NET_FP8
from chessrl_b200.engine import Engine
from chessrl_b200.model import calibration_planes
from test_gpu_evalpath import _batch, _openings, _oracle_replay, _sampled, _search, STAT_KEYS

pytestmark = pytest.mark.gpu
SIMS = int(os.environ.get("CRL_PARITY_SIMS", "64"))
STEM_MAX_DIFF_FRACTION = 1e-4     # 5 x the 2.0e-5 measured on a B200 (profiles/r03_fp8_stem_parity.txt)
LAYER_MAX_DIFF_FRACTION = 2e-4    # 5 x the largest per-layer fraction measured on a B200 (3.3e-5), same profile


@pytest.fixture(autouse=True)
def _fp32_reference_without_tf32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.fixture(scope="module")
def pack():
    return netpacks.lively_pack()


@pytest.fixture(scope="module")
def wide(pack):
    e = Engine(max_games=4096, max_nodes=2)
    e.load_weights(pack)
    amax = e.calibrate(calibration_planes(e, n=64))
    e.load_weights(pack, precision="fp8", calibration=amax)
    yield e, amax
    e.close()


@pytest.fixture(scope="module")
def planes():
    return torch.from_numpy(_batch(101)).to("cuda").to(torch.bfloat16)


def _err(a, b):
    d = (a.float() - b.float()).abs()
    return float(d.max()), float(d.mean())


def _steps(a, b, s):
    """Distance between a and b in neighbouring e4m3 codes of scale s (values / s rounded to e4m3, saturating)."""
    ia, ib = ((fp8_emu.e4m3(t.float() / s).to(torch.float8_e4m3fn).view(torch.uint8).to(torch.int32)) for t in (a, b))
    ia = torch.where(ia & 0x80 != 0, -(ia & 0x7F), ia & 0x7F)
    ib = torch.where(ib & 0x80 != 0, -(ib & 0x7F), ib & 0x7F)
    return (ia - ib).abs()


def _layer_alone(pack, L, x, taps, amax, mutate=None):
    """Convolution L of the emulation fed with the kernel's own inputs (its taps are code x s, exact in bf16)."""
    s = [fp8_emu.act_scale(a) for a in amax]
    nchw = lambda t: t.float().permute(0, 3, 1, 2).contiguous()                       # noqa: E731
    if L == 0:
        codes_in, s_in = fp8_emu.e4m3(nchw(x[..., :127])), 1.0
    else:
        codes_in, s_in = nchw(taps[L - 1]) / s[L - 1], s[L - 1]
    res = (nchw(taps[L - 2]) / s[L - 2], s[L - 2]) if fp8_emu.is_second(L) else None
    _, val = fp8_emu.layer(pack, L, codes_in, s_in, res, s[L] if L < 20 else 1.0, device="cuda", mutate=mutate)
    return val.permute(0, 2, 3, 1).contiguous(), (s[L] if L < 20 else None)


def _layer_steps(got, want, s, amax):
    # the last layer is stored in bf16: it is compared on the e4m3 grid of its calibrated scale like the others (in bf16
    # steps, values that cancel to almost zero land several steps apart for a last-bit difference of their terms)
    return _steps(got, want, s if s is not None else fp8_emu.act_scale(amax[20]))


def _kernel_taps(e, x):
    out = {"act": []}
    for L in range(21):
        t = e.debug_tower(x, layer=L)
        out["act"].append(t["act"].float())
    for k in ("pf", "vf", "logits", "policy", "value"):
        out[k] = t[k].float()
    return out


def _emu(pack, x, amax, mutate=None):
    taps = {}
    p, v = fp8_emu.forward(pack, x.float().cpu().numpy(), amax, device="cuda", taps=taps, mutate=mutate)
    taps.update({"policy": p, "value": v})
    return taps


def _fp32(pack, x):
    taps = {}
    p, v = model_torch.forward(pack, x.float().cpu().numpy(), device="cuda", taps=taps)
    taps.update({"policy": p, "value": v})
    return taps


# ---- a. the kernel against the emulation ------------------------------------------------------------------------------------
def test_stem_matches_emulation_to_one_e4m3_step(wide, pack, planes):
    e, amax = wide
    x = planes[:512]
    got = e.debug_tower(x, layer=0)["act"].float()
    want = _emu(pack, x, amax)["act"][0]
    steps = _steps(got, want, fp8_emu.act_scale(amax[0]))
    assert int(steps.max()) <= 1
    frac = float((steps > 0).float().mean())
    print("stem elements one e4m3 step from the emulation: %.3e" % frac)
    assert frac <= STEM_MAX_DIFF_FRACTION


@pytest.mark.parametrize("n", [1, 5, 37, 592, 593, 4096])
def test_layers_and_outputs_within_twice_the_emulation_error(wide, pack, planes, n):
    e, amax = wide
    x = planes[:n]
    got, emu, ref = _kernel_taps(e, x), _emu(pack, x, amax), _fp32(pack, x)
    keys = [("act", L) for L in range(21)] + [(k, None) for k in ("pf", "vf", "logits", "policy", "value")]
    for k, L in keys:
        g = got[k][L] if L is not None else got[k]
        w = emu[k][L] if L is not None else emu[k]
        r = ref[k][L] if L is not None else ref[k]
        e8_max, e8_mean = _err(w, r)
        k_max, k_mean = _err(g.reshape(w.shape), w)
        assert k_max <= 2 * e8_max and k_mean <= 2 * e8_mean, (k, L, k_max, e8_max, k_mean, e8_mean)


@pytest.mark.parametrize("n", [37, 593])
def test_every_layer_matches_its_emulation_to_one_step(wide, pack, planes, n):
    """Each convolution of the kernel against the emulation of that convolution alone, fed the kernel's own input and
    block input: every element equal or one e4m3 step away, and few differ (accumulation order)."""
    e, amax = wide
    x = planes[:n]
    taps = _kernel_taps(e, x)["act"]
    fracs, worst = [], []
    for L in range(21):
        want, s = _layer_alone(pack, L, x, taps, amax)
        steps = _layer_steps(taps[L], want, s, amax)
        worst.append(int(steps.max()))
        fracs.append(float((steps > 0).float().mean()))
    print("n=%d elements one step from the emulation per layer: %s" % (n, " ".join("%.1e" % f for f in fracs)))
    assert max(worst) <= 1, worst
    assert max(fracs) <= LAYER_MAX_DIFF_FRACTION, fracs


def _busiest_channel(tap):
    return int((tap != 0).sum(dim=(0, 1, 2)).argmax())


@pytest.mark.parametrize("mutate,layer", [({"shift_tap": 7}, 7), ({"drop_slice": 0}, 0), ({"drop_slice": 12}, 12),
                                          ({"double_scale": 9}, 9), ({"double_ws": (0, None)}, 0),
                                          ({"double_ws": (14, None)}, 14), ({"double_s_res": 10}, 10)])
def test_bound_rejects_wrong_kernels(wide, pack, planes, mutate, layer):
    """A kernel that computed what the mutated emulation computes fails the per-layer check at least fivefold: it differs
    from the kernel in at least 5 x LAYER_MAX_DIFF_FRACTION of the layer's elements (and by more than one step)."""
    e, amax = wide
    x = planes[:37]
    taps = _kernel_taps(e, x)["act"]
    L = layer
    if "double_ws" in mutate:
        mutate = {"double_ws": (L, _busiest_channel(taps[L]))}
    want, s = _layer_alone(pack, L, x, taps, amax, mutate=mutate)
    steps = _layer_steps(taps[L], want, s, amax)
    frac = float((steps > 1).float().mean())
    print(mutate, "differs by more than one step in %.2e of layer %d: %.0fx the allowed fraction"
          % (frac, L, frac / LAYER_MAX_DIFF_FRACTION))
    assert frac >= 5 * LAYER_MAX_DIFF_FRACTION


# ---- b. bit identity within fp8 -------------------------------------------------------------------------------------------------
def test_single_tile_equals_two_tile(wide, planes):
    """A launch bound of 297 rows takes the two-tile instantiation, crl_net_forward of n <= 296 rows the single-tile one."""
    e, _ = wide
    for n in (1, 37, 64):
        p1, v1 = e.net_forward(planes[:n])
        p2, v2 = e.debug_forward_counted(planes[:297], 297, n)
        assert torch.equal(p1, p2[:n]) and torch.equal(v1, v2[:n]), n


@pytest.mark.parametrize("bound", [296, 297, 592, 593, 4096])
def test_counted_batch_equals_forward(wide, planes, bound):
    e, _ = wide
    for count in sorted({0, 1, bound // 2 + 1, bound}):
        pol = torch.full((bound, 1968), -7.0, device="cuda")
        val = torch.full((bound,), -7.0, device="cuda")
        e.debug_forward_counted(planes[:bound], bound, count, pol, val)
        if count:
            p, v = e.net_forward(planes[:count])
            assert torch.equal(pol[:count], p) and torch.equal(val[:count], v), (bound, count)
        assert (pol[count:] == -7.0).all() and (val[count:] == -7.0).all(), (bound, count)


def test_rows_do_not_depend_on_their_place(wide, planes):
    e, _ = wide
    p, v = e.net_forward(planes)
    perm = torch.randperm(4096, generator=torch.Generator().manual_seed(3)).to("cuda")
    pp, vp = e.net_forward(planes[perm])
    assert torch.equal(pp, p[perm]) and torch.equal(vp, v[perm])
    ps, vs = e.net_forward(planes[5:1005])
    assert torch.equal(ps, p[5:1005]) and torch.equal(vs, v[5:1005])


def test_fp8_differs_from_bf16(wide, planes):
    e, _ = wide
    p8, v8 = e.net_forward(planes[:64])
    e.set_net_precision("bf16")
    p16, v16 = e.net_forward(planes[:64])
    e.set_net_precision("fp8")
    assert not torch.equal(v8, v16)
    assert (v8 - v16).abs().mean() < 0.5


# ---- c. the search in fp8 ---------------------------------------------------------------------------------------------------------
def _fp8_engine(pack, amax, **kw):
    eng = Engine(**kw)
    eng.load_weights(pack, precision="fp8", calibration=amax)
    eng.set_evaluator(EVAL_NET)
    return eng


def test_full_width_fp8_search_matches_oracle(wide, pack):
    _, amax = wide
    G = int(os.environ.get("CRL_EVALPATH_LANES", "4096"))
    eng = _fp8_engine(pack, amax, max_games=G, max_nodes=SIMS + 1, avg_moves=96)
    moves = _openings(eng, seed=17)
    recorded = _search(eng, 2, SIMS)
    eng.close()
    net = _fp8_engine(pack, amax, max_games=16, max_nodes=8)
    lanes = _sampled(G, 16, seed=29)
    failures, checked = _oracle_replay(net, moves, lanes, recorded, SIMS)
    net.close()
    assert not failures, failures[:3]
    assert len(checked) >= len(lanes) // 2


def test_wave_fp8_search_matches_oracle(wide, pack):
    _, amax = wide
    G, K = 512, 8
    eng = _fp8_engine(pack, amax, max_games=G, max_nodes=SIMS + 1, avg_moves=96, max_inflight=K)
    moves = _openings(eng, seed=G + K)
    recorded = _search(eng, 1, SIMS, inflight=K, apply=False)
    eng.close()
    net = _fp8_engine(pack, amax, max_games=16, max_nodes=8)
    failures, _ = _oracle_replay(net, moves, _sampled(G, 16, seed=G), recorded, SIMS, threads=K)
    net.close()
    assert not failures, failures[:3]


def test_reuse_on_and_off_play_the_same_games(wide, pack):
    _, amax = wide
    runs = []
    for reuse in (True, False):
        eng = _fp8_engine(pack, amax, max_games=256, max_nodes=33, avg_moves=96)
        eng.set_reuse(reuse)
        _openings(eng, seed=4, max_plies=20)
        runs.append(_search(eng, 3, 32))
        eng.close()
    for (a, pa, oa), (b, pb, ob) in zip(*runs):
        for k in STAT_KEYS:
            assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(oa, ob)


# ---- d. switching and errors ------------------------------------------------------------------------------------------------------
def test_switching_back_to_bf16_is_bit_identical_to_a_fresh_engine(wide, pack, planes):
    _, amax = wide
    G = 64
    fresh = Engine(max_games=G, max_nodes=17, avg_moves=96)
    fresh.load_weights(pack)
    fresh.set_evaluator(EVAL_NET)
    sw = Engine(max_games=G, max_nodes=17, avg_moves=96)
    sw.load_weights(pack)
    sw.set_evaluator(EVAL_NET)
    want_p, want_v = fresh.net_forward(planes[:G])
    _openings(fresh, seed=9, max_plies=20)
    want = _search(fresh, 1, 16, apply=False)[0]
    moves = _openings(sw, seed=9, max_plies=20)
    sw.load_weights(pack, precision="fp8", calibration=amax)
    sw.net_forward(planes[:G])
    _search(sw, 1, 16, apply=False)                          # captures the fp8 search graph
    sw.set_net_precision("bf16")
    p, v = sw.net_forward(planes[:G])
    assert torch.equal(p, want_p) and torch.equal(v, want_v)
    sw.games_set(np.tile(B.record_from_fen(), (G, 1)), [[B.uci_to_move(m) for m in ms] for ms in moves])
    got = _search(sw, 1, 16, apply=False)[0]
    for k in STAT_KEYS:
        assert np.array_equal(got[0][k], want[0][k]), k
    sw.set_net_precision("fp8")
    p8, _ = sw.net_forward(planes[:G])
    assert not torch.equal(p8, want_p)
    sw.load_weights(pack)                                     # a bf16 load drops the fp8 tower
    assert sw.lib.crl_net_set_precision(sw.h, NET_FP8) == CRL_ESTATE
    fresh.close()
    sw.close()


def test_fp8_load_error_paths_leave_bf16(pack):
    e = Engine(max_games=8, max_nodes=2)
    assert e.lib.crl_net_set_precision(e.h, NET_FP8) == CRL_ESTATE        # no fp8 load
    e.load_weights(pack)
    assert e.lib.crl_net_set_precision(e.h, 7) == CRL_EINVAL
    for bad in (float("nan"), float("inf"), -1.0):
        amax = np.ones(21, np.float32)
        amax[3] = bad
        with pytest.raises(RuntimeError):
            e.load_weights(pack, precision="fp8", calibration=amax)
        assert e.net_precision == "bf16"
    # a failed fp8 load after a good one leaves the engine in bf16, not in the old fp8 state
    x = torch.from_numpy(_batch(7)[:8]).to("cuda").to(torch.bfloat16)
    p16, _ = e.net_forward(x)
    e.load_weights(pack, precision="fp8", calibration=np.ones(21, np.float32))
    bad = np.ones(21, np.float32)
    bad[0] = float("nan")
    with pytest.raises(RuntimeError):
        e.load_weights(pack, precision="fp8", calibration=bad)
    assert e.net_precision == "bf16" and torch.equal(e.net_forward(x)[0], p16)
    e.close()


def test_selfplay_fp8_games_replay_under_the_oracle(tmp_path):
    import chessrl_oracle as O
    env = dict(os.environ)
    r = subprocess.run([sys.executable, "-m", "chessrl_b200.selfplay", str(tmp_path), "--games", "2", "--sims", "8",
                        "--max-moves", "6", "--no-train", "--net-precision", "fp8"], env=env, capture_output=True,
                       text=True, timeout=900, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    with open(tmp_path / "gameplays.json") as f:
        data = json.load(f)
    games = data if isinstance(data, list) else data.get("games", data)
    assert len(games) == 2
    for g in games:
        og = O.OGame()
        for m in g["moves"]:
            assert m in [str(x) for x in og.get_legal_moves()]
            og.move(m)
