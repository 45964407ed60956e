"""GPU numerics, network: the tcgen05 convolution kernel and the full forward pass against a plain PyTorch
fp32 reference of the same graph (oracle/model_torch.py, restating model.py:31-63, 111-122).

Tolerances (bf16 operands, fp32 accumulate, bf16 activations between layers; SURVEY.md KAT-6):
  one conv layer vs fp32 conv on the same bf16-rounded operands: max abs err <= 2e-2 * max|ref| (bf16 output rounding)
  full net, policy probabilities: max abs err <= 2e-3 ; value: <= 2e-2
"""
import numpy as np
import pytest
import torch

import model_torch
from chessrl_b200 import boards as B
from chessrl_b200 import model

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def net_engine():
    from chessrl_b200.engine import Engine
    e = Engine(max_games=64, max_nodes=8)
    import netpacks
    pack = netpacks.lively_pack()
    e.load_weights(pack)
    yield e, pack
    e.close()


def _conv_ref(x_bf16_nhwc, k_hwio, scale, shift, residual, relu):
    x = x_bf16_nhwc.float().permute(0, 3, 1, 2)
    w = torch.as_tensor(k_hwio).to(torch.bfloat16).float().permute(3, 2, 0, 1).to(x.device)
    y = torch.nn.functional.conv2d(x, w, None, padding=1)
    y = y * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1)
    if residual is not None:
        y = y + residual.float().permute(0, 3, 1, 2)
    if relu:
        y = torch.relu(y)
    return y.permute(0, 2, 3, 1)


def _fold(pack, layer, dev):
    if layer == 0:
        return torch.ones(256, device=dev), torch.as_tensor(pack[1], device=dev)
    blk, second = (layer - 1) // 2, (layer - 1) % 2
    o = 2 + 12 * blk + 6 * second
    g, b, m, v = (torch.as_tensor(pack[o + 2 + i], device=dev) for i in range(4))
    s = g / torch.sqrt(v + 1e-3)
    return s, (torch.as_tensor(pack[o + 1], device=dev) - m) * s + b


@pytest.mark.parametrize("n", [1, 2, 7, 64])
def test_conv_layer_matches_fp32(net_engine, n):
    e, pack = net_engine
    dev = e.device
    torch.manual_seed(n)
    x = (torch.randn(n, 8, 8, 256, device=dev) * 0.5).to(torch.bfloat16)
    res = (torch.randn(n, 8, 8, 256, device=dev) * 0.5).to(torch.bfloat16)
    for layer, use_res, relu in ((1, False, True), (2, True, True), (20, True, False)):
        blk, second = (layer - 1) // 2, (layer - 1) % 2
        k = pack[2 + 12 * blk + 6 * second]
        s, sh = _fold(pack, layer, dev)
        got = e.debug_conv(layer, x, res if use_res else None, relu).float()
        ref = _conv_ref(x, k, s, sh, res if use_res else None, relu)
        err = (got - ref).abs().max().item()
        assert err <= 2e-2 * max(1.0, ref.abs().max().item()), (layer, n, err)


def test_stem_conv_with_padded_channel(net_engine):
    e, pack = net_engine
    dev = e.device
    x = torch.zeros(5, 8, 8, 128, device=dev, dtype=torch.bfloat16)
    x[..., :127] = (torch.rand(5, 8, 8, 127, device=dev) > 0.7).to(torch.bfloat16)
    got = e.debug_conv(0, x, None, False).float()
    s, sh = _fold(pack, 0, dev)
    k = np.concatenate([pack[0], np.zeros((3, 3, 1, 256), np.float32)], axis=2)
    ref = _conv_ref(x, k, s, sh, None, False)
    assert (got - ref).abs().max().item() <= 2e-2 * max(1.0, ref.abs().max().item())


def _positions(n, seed=0):
    import chessrl_oracle as O
    import random
    rng = random.Random(seed)
    games = []
    for i in range(n):
        g = O.OGame()
        for _ in range(rng.randrange(0, 40)):
            ms = g.get_legal_moves()
            if not ms or g.get_result() is not None:
                break
            g.move(rng.choice(ms))
        games.append(g)
    return games


def test_full_forward_matches_fp32(net_engine):
    import chessrl_oracle as O
    e, pack = net_engine
    games = _positions(33, seed=1)
    planes = np.stack([O.planes(g) for g in games]).astype(np.float32)
    x = torch.zeros(len(games), 8, 8, 128, dtype=torch.bfloat16, device=e.device)
    x[..., :127] = torch.from_numpy(planes).to(e.device).to(torch.bfloat16)
    p, v = e.net_forward(x)
    rp, rv = model_torch.forward(pack, planes, device=e.device)
    ep, ev = model_torch.forward(pack, planes, device=e.device, emulate_bf16_activations=True)
    import netpacks
    netpacks.assert_lively(rp, rv)
    assert torch.allclose(p.sum(1), torch.ones_like(p.sum(1)), atol=1e-4)
    # bf16 pipeline vs fp32: no worse than 3 x the ideal emulation of the same rounding points (and the absolute
    # KAT-6 bounds 2e-3 / 2e-2 on top)
    assert (p - rp).abs().max().item() <= min(2e-3, 3 * (ep - rp).abs().max().item() + 1e-7)
    assert (v - rv).abs().max().item() <= min(2e-2 * 2, 3 * (ev - rv).abs().max().item() + 1e-6)
    # the same rows in a different batch composition give bit-identical outputs (row independence)
    p2, v2 = e.net_forward(x[5:9].contiguous())
    assert torch.equal(p2, p[5:9]) and torch.equal(v2, v[5:9])


def test_search_with_network_evaluator_runs_and_counts(net_engine):
    """Lockstep search with the real network: visit counts sum to the simulation count and the tree is sane."""
    from chessrl_b200._lib import EVAL_NET
    from chessrl_b200.engine import Engine
    e, pack = net_engine
    e2 = Engine(max_games=32, max_nodes=41)
    e2.load_weights(pack)
    e2.set_evaluator(EVAL_NET)
    e2.games_set(np.tile(B.record_from_fen(), (32, 1)))
    e2.mcts_begin_move()
    e2.mcts_simulate(40)
    st = e2.root_stats()
    assert (st["root_visits"] == 41).all()
    assert (st["visits"].sum(1) == 40).all()
    # all 32 lanes hold the same position and the same weights -> identical trees
    assert (st["visits"] == st["visits"][0]).all()
    e2.close()


# ---------------------------------------------------------------------------------------------------------------
# k_trunk4 itself (the kernel every evaluation runs through), layer by layer, through crl_debug_tower's taps.
#
# Reference = model_torch.forward in fp32 (no TF32) and the same graph with the kernel's rounding points emulated
# (bf16 conv / policy-dense kernels, bf16 activations after every epilogue, fp32 accumulation and BatchNorm folding).
# err(a, b) = max|a - b| / max|b|.  The emulation's own distance from fp32, E = err(emulated, fp32), is the unit:
#   * every tapped convolution output, the head inputs and the policy LOGITS must satisfy
#         err(kernel, emulated) <= 2 E      (=> err(kernel, fp32) <= 3 E),
#     and the same with the mean absolute error;
#   * a reference with ONE filter tap of ONE layer displaced, or one 64-channel slice zeroed, must be REJECTED by that
#     bound by a wide margin (the test's own sensitivity check: a broken tap offset / a dropped channel slice in the
#     kernel cannot pass);
#   * the fp32 outputs are asserted to be non-degenerate (netpacks.assert_lively) before anything is compared.
# ---------------------------------------------------------------------------------------------------------------
import netpacks


@pytest.fixture(autouse=True)
def _fp32_reference_without_tf32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _err(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def _err_mean(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().mean() / b.abs().mean().clamp_min(1e-30)).item()


def _reference_taps(pack, planes_np, emulate):
    taps = {}
    p, v = model_torch.forward(pack, planes_np[..., :127], device="cuda", emulate_bf16_activations=emulate, taps=taps)
    taps["policy"], taps["value"] = p, v
    return taps


@pytest.fixture(scope="module")
def tower_engine():
    from chessrl_b200.engine import Engine
    e = Engine(max_games=4096, max_nodes=2)
    pack = netpacks.lively_pack()
    e.load_weights(pack)
    yield e, pack
    e.close()


def _planes_for(n):
    if n <= 64:
        return netpacks.planes_of(netpacks.midgame_games(n, seed=n))
    x = netpacks.synthetic_planes(n, seed=n)
    real = netpacks.planes_of(netpacks.midgame_games(48, seed=n))
    x[:24] = real[:24]                       # real positions at both ends of the batch (first / last CTA-pair groups)
    x[-24:] = real[24:]
    return x


@pytest.mark.parametrize("n", [1, 5, 37, 592, 593, 4096])
def test_trunk4_logits_and_final_activations_match_emulated_graph(tower_engine, n):
    """Batch sizes around the persistent grid's round (74 CTA pairs x 8 boards = 592) and BASELINE's 4,096."""
    e, pack = tower_engine
    x = _planes_for(n)
    xt = torch.from_numpy(x).to(e.device).to(torch.bfloat16)
    got = e.debug_tower(xt, layer=20)
    f32 = _reference_taps(pack, x, False)
    emu = _reference_taps(pack, x, True)
    netpacks.assert_lively(f32["policy"], f32["value"])
    report = {}
    for name, k, r32, rem in (("act20", got["act"], f32["act"][20], emu["act"][20]),
                              ("pf", got["pf"], f32["pf"], emu["pf"]),
                              ("vf", got["vf"], f32["vf"], emu["vf"]),
                              ("logits", got["logits"], f32["logits"], emu["logits"])):
        E, Em = _err(rem, r32), _err_mean(rem, r32)
        d, dm = _err(k, rem), _err_mean(k, rem)
        report[name] = (E, d, Em, dm)
        assert E > 0 and d <= 2 * E and dm <= 2 * Em, (n, name, report[name])
    # outputs: probabilities and value against fp32, bounded by the emulation's own error as well
    Ep = (emu["policy"] - f32["policy"]).abs().max().item()
    Ev = (emu["value"] - f32["value"]).abs().max().item()
    assert (got["policy"] - f32["policy"]).abs().max().item() <= 3 * Ep + 1e-7, (n, Ep)
    assert (got["value"] - f32["value"]).abs().max().item() <= 3 * Ev + 1e-6, (n, Ev)
    assert torch.allclose(got["policy"].sum(1), torch.ones(n, device=e.device), atol=1e-4)
    # crl_net_forward is the same path: bit-identical outputs
    p, v = e.net_forward(xt)
    assert torch.equal(p, got["policy"]) and torch.equal(v, got["value"])
    print("trunk4 parity n=%d: " % n + ", ".join("%s E=%.2e d=%.2e" % (k, v[0], v[1]) for k, v in report.items()))


def test_trunk4_every_layer_matches_emulated_graph(tower_engine):
    """Each of the 21 convolution outputs of k_trunk4 (stem, conv_a / conv_b of the ten blocks) through the tap."""
    e, pack = tower_engine
    x = netpacks.planes_of(netpacks.midgame_games(19, seed=77))
    xt = torch.from_numpy(x).to(e.device).to(torch.bfloat16)
    f32 = _reference_taps(pack, x, False)
    emu = _reference_taps(pack, x, True)
    for layer in range(21):
        got = e.debug_tower(xt, layer=layer)["act"]
        E = _err(emu["act"][layer], f32["act"][layer])
        if layer == 0:
            # the stem has 0/1 inputs: the only rounding is the bf16 kernel and the output
            assert _err(got, emu["act"][0]) <= 2 ** -8, layer
        else:
            assert _err(got, emu["act"][layer]) <= 2 * E, (layer, E, _err(got, emu["act"][layer]))
        assert _err_mean(got, emu["act"][layer]) <= 2 * _err_mean(emu["act"][layer], f32["act"][layer]) + 1e-4, layer


def _displace_tap(pack, layer):
    """Reference pack whose convolution `layer` has filter taps (0,0) and (0,1) exchanged: what a tap-offset bug does."""
    idx = 0 if layer == 0 else 2 + 12 * ((layer - 1) // 2) + 6 * ((layer - 1) % 2)
    bad = list(pack)
    k = pack[idx].copy()
    k[0, 0], k[0, 1] = pack[idx][0, 1].copy(), pack[idx][0, 0].copy()
    bad[idx] = k
    return bad


def _zero_slice(pack, layer, c0):
    idx = 0 if layer == 0 else 2 + 12 * ((layer - 1) // 2) + 6 * ((layer - 1) % 2)
    bad = list(pack)
    k = pack[idx].copy()
    k[:, :, c0:c0 + 64, :] = 0
    bad[idx] = k
    return bad


@pytest.mark.parametrize("fault", ["tap_layer7", "tap_layer20", "slice_layer0", "slice_layer12"])
def test_parity_bound_rejects_a_displaced_tap_or_a_dropped_channel_slice(tower_engine, fault):
    """Sensitivity of the bound: the kernel's outputs compared with a reference that has exactly the defect a broken
    shared-memory descriptor offset / a skipped k-chunk would produce must violate `err <= 2 E` at least fivefold."""
    e, pack = tower_engine
    x = netpacks.planes_of(netpacks.midgame_games(16, seed=5))
    xt = torch.from_numpy(x).to(e.device).to(torch.bfloat16)
    got = e.debug_tower(xt, layer=20)
    layer = int(fault.split("layer")[1])
    bad_pack = _displace_tap(pack, layer) if fault.startswith("tap") else _zero_slice(pack, layer, 64)
    f32 = _reference_taps(pack, x, False)
    emu = _reference_taps(pack, x, True)
    bad = _reference_taps(bad_pack, x, True)
    for name, k in (("act20", got["act"]), ("logits", got["logits"])):
        r32, rem, rbad = (t["act"][20] if name == "act20" else t["logits"] for t in (f32, emu, bad))
        E = _err(rem, r32)
        assert _err(k, rem) <= 2 * E
        assert _err(k, rbad) > 10 * E, (fault, name, _err(k, rbad), E)


@pytest.mark.parametrize("n", [1, 5, 37, 1000])
def test_tower_matches_fp32_reference(n):
    """crl_net_forward of an engine sized for the batch against the fp32 reference, within 3 x the emulation's own error;
    odd batch sizes exercise the partial tile / zero-filled board rows."""
    from chessrl_b200.engine import Engine
    pack = netpacks.lively_pack()
    x = _planes_for(n)
    planes = torch.from_numpy(x).to("cuda").to(torch.bfloat16)
    e = Engine(max_games=max(n, 2), max_nodes=4)
    e.load_weights(pack)
    p, v = e.net_forward(planes)
    p, v = p.cpu(), v.cpu()
    e.close()
    f32 = _reference_taps(pack, x, False)
    emu = _reference_taps(pack, x, True)
    netpacks.assert_lively(f32["policy"], f32["value"])
    Ep = (emu["policy"] - f32["policy"]).abs().max().item()
    Ev = (emu["value"] - f32["value"]).abs().max().item()
    assert (p - f32["policy"].cpu()).abs().max().item() <= 3 * Ep + 1e-7
    assert (v - f32["value"].cpu()).abs().max().item() <= 3 * Ev + 1e-6
