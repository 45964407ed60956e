"""The fp8 numeric definition (tests/fp8_emu.py, csrc/net.cu net_load_fp8) on the CPU: the e4m3 quantiser, the activation
scale rule and the per-channel weight quantisation."""
import numpy as np
import torch

import fp8_emu
import model_torch
import netpacks


def test_quantiser_is_round_to_nearest_even_and_saturating():
    # e4m3 values around 1: step 1/8; the midpoints go to the even mantissa
    x = torch.tensor([1.0625, 1.1875, 1.3125, -1.0625, 0.0, 448.0, 449.0, 464.0, 1e6, -1e6, 2.0 ** -9, 2.0 ** -10])
    want = torch.tensor([1.0, 1.25, 1.25, -1.0, 0.0, 448.0, 448.0, 448.0, 448.0, -448.0, 2.0 ** -9, 0.0])
    assert torch.equal(fp8_emu.e4m3(x), want)
    assert torch.isnan(fp8_emu.e4m3(torch.tensor([float("nan")]))).all()
    # every e4m3 value is a fixed point
    codes = torch.arange(256, dtype=torch.uint8).view(torch.float8_e4m3fn).to(torch.float32)
    finite = codes[~torch.isnan(codes)]
    assert torch.equal(fp8_emu.e4m3(finite), finite)


def test_activation_scale_rule():
    assert fp8_emu.act_scale(0.0) == 1.0
    assert fp8_emu.act_scale(448.0) == 1.0
    assert fp8_emu.act_scale(448.5) == 2.0
    assert fp8_emu.act_scale(224.0) == 0.5
    assert fp8_emu.act_scale(300.0) == 1.0
    assert fp8_emu.act_scale(1.0) == 2.0 ** -8          # 1/448 -> ceil(log2) = -8
    for a in np.float32([1e-3, 0.37, 5.0, 91.0, 4096.0]):
        s = fp8_emu.act_scale(a)
        assert a / s <= 448.0 < 2 * a / s
    # the floor: scales below the smallest normal power of two would have an infinite reciprocal (NaN codes for a = 0)
    floor = 2.0 ** -126
    edge = np.float32(448.0 * floor)
    for a in (np.float32(1e-37), np.float32(1e-40), np.float32(448.0 * 2.0 ** -128),
              np.nextafter(np.float32(0), np.float32(1)), edge):         # ... the smallest subnormal, the floor's own amax
        s = fp8_emu.act_scale(a)
        assert s == floor, (a, s)
        assert np.isfinite(np.float32(1.0) / np.float32(s))
        assert np.float32(a) * (np.float32(1.0) / np.float32(s)) <= 448.0
    assert fp8_emu.act_scale(np.nextafter(edge, np.float32(1))) == 2.0 ** -125


def test_weight_quantisation_maps_each_column_max_to_448():
    pack = netpacks.lively_pack()
    k = np.array(pack[2], dtype=np.float32)
    k[..., 7] = 0.0                                          # an all-zero column gets scale 1
    q, ws = fp8_emu.quantise_weights(k)
    assert ws[7] == 1.0 and not np.any(q[..., 7])
    m = np.abs(k).reshape(-1, 256).max(axis=0)
    qm = np.abs(q).reshape(-1, 256).max(axis=0)
    live = m > 0
    assert np.all(qm[live] == 448.0)
    assert np.all(qm[live] * ws[live] == np.float32(448.0) * ws[live])
    assert np.allclose(qm[live] * ws[live], m[live], rtol=1e-6)


def test_emulation_tracks_the_fp32_graph():
    pack = netpacks.lively_pack()
    x = netpacks.planes_of(netpacks.midgame_games(8, seed=3))
    taps32 = {}
    p32, v32 = model_torch.forward(pack, x, taps=taps32)
    amax = [float(a.abs().max()) for a in taps32["act"]]
    taps8 = {}
    p8, v8 = fp8_emu.forward(pack, x, amax, taps=taps8)
    assert (p8 - p32).abs().max() < 0.05 and (v8 - v32).abs().max() < 1.0
    # the stem sees exact inputs: only the weight quantisation (<= 2^-4 relative) and the output rounding separate it
    rel = (taps8["act"][0] - taps32["act"][0]).abs().max() / taps32["act"][0].abs().max()
    assert rel < 0.1
    # the mutations change the result
    for mut in ({"shift_tap": 3}, {"drop_slice": 0}, {"double_scale": 5}):
        pm, _ = fp8_emu.forward(pack, x, amax, mutate=mut)
        assert (pm - p8).abs().max() > 0
