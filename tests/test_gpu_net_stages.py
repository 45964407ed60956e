"""The network's stages after the tower, each against an fp64 reference fed the kernel's own input to that stage (so
errors do not pile up across stages), and the fp8 calibration against what it measures.

Every input comes from Engine.debug_tower: the act tap of convolution 20 (bf16: exactly the x the fused heads read, in
both precisions), pf, vf, logits, policy and value.

Bounds, derived from the fp32 roundings each kernel performs (u = 2^-24; c = 2 covers an accumulation that truncates
instead of rounding to nearest, as a tensor-core MMA may):
  * a dot product of length K accumulated in fp32:   c K u sum_i |a_i b_i|,  plus u |result| for each rounding after it;
  * the host-side fp32 BatchNorm fold (net_load):   s = g / sqrt(var + eps) is off by <= 3u |s| (add, sqrt, divide),
    t = (bias - mean) s + beta by <= 5u |(bias - mean) s| + u |t|;  both taken c times.
  1. fused 1x1 heads (k_trunk4 epilogue, bf16 and fp8 branch), K = 256, y = h s + t, then ReLU (1-Lipschitz):
         |dy| <= c K u |s| sum|x w| + u (|h s| + |y|) + c (3u |h s| + 5u |(bias - mean) s| + u |t|)
     vf (fp32) is off by |dy|; pf (bf16, Keras order (h*8+w)*2+c) by |dy| + half a bf16 ulp of |ref| + |dy|.
  2. policy GEMM (k_conv_v2, one tap, 8 N tiles; bf16 operands, bf16(W) is part of the definition), K = 128:
         c K u sum_i |pf_i bf16(W)_ij| + u |logit|          (acc x 1 + bias rounds once)
  3. softmax over the 1,968 labels (k_softmax_value), row max m:  exp(l_j - m) is off relatively by
         r_j = 4u (expf, 2 ulp) + u |l_j - m| (the subtraction);  the sum S by r_S = sum_k p_k r_k + c 67 u (62 terms
     per lane, then 5 shuffle levels); 1 / S and the product round once each:
         |dp_j| <= p_j (r_j + r_S + 2u) + c 2.5 2^-149      (expf's 2 ulp and the product's half ulp at a subnormal)
  4. value MLP (k_softmax_value):  z = vf W1 + b1 (K = 64): dz = c 64 u sum|vf_i W1_ij| + u |z|;  y = relu(z) w2 + b2
     (K = 256): dy = sum_j |w2_j| dz_j + c 256 u sum|h_j w2_j| + u |y|;  value = tanh(y):
         sech^2(max(|y| - dy, 0)) dy + 4u |value|           (tanhf, 2 ulp)
Each bound is checked at every element (err / bound <= 1), and a reference with one planted defect must exceed it at
least tenfold somewhere.

The sharp pack scales the lively pack's policy kernel by 24 and its last value kernel by 4: logits spread over 60-130,
probabilities below 2^-126 (with x 8 the spread is 20-40 and the smallest probabilities ~1e-18, nowhere near the
subnormal range), values near +-1."""
import numpy as np
import pytest
import torch

import fp8_emu
import model_torch
import netpacks
from chessrl_b200.engine import Engine
from chessrl_b200.model import calibration_planes
from test_gpu_evalpath import _batch
from test_gpu_fp8 import LAYER_MAX_DIFF_FRACTION, _kernel_taps, _layer_alone, _layer_steps

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
C = 2
TINY = 2.0 ** -149                 # the smallest fp32 subnormal
NS = [1, 7, 8, 9, 255, 256, 257, 296, 297, 593, 4096]
BN_EPS = 1e-3
DEV = "cuda"


def sharp_pack():
    pack = list(netpacks.lively_pack())
    pack[128] = pack[128] * 24.0
    pack[138] = pack[138] * 4.0
    return pack


PACKS = {"lively": netpacks.lively_pack, "sharp": sharp_pack}


@pytest.fixture(autouse=True)
def _fp32_reference_without_tf32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.fixture(scope="module")
def planes():
    return torch.from_numpy(_batch(101)).to("cuda").to(torch.bfloat16)


@pytest.fixture(scope="module")
def nets():
    """name -> (4,096-row engine holding the pack in bf16 and fp8, pack, calibrated amax)."""
    made = {}

    def get(name):
        if name not in made:
            pack = PACKS[name]()
            e = Engine(max_games=4096, max_nodes=2)
            e.load_weights(pack)
            amax = e.calibrate(calibration_planes(e, n=64))
            e.load_weights(pack, precision="fp8", calibration=amax)
            made[name] = (e, pack, amax)
        return made[name]
    yield get
    for e, _, _ in made.values():
        e.close()


def _d(a):
    return torch.as_tensor(np.asarray(a, dtype=np.float64), device=DEV)


# ---- fp64 references and their bounds ---------------------------------------------------------------------------------------
def _heads(pack, act):
    """act20 [n,8,8,256] -> (pre-ReLU y [n,64,3] (policy c0, c1, value), its bound, h, s, t)."""
    n = act.shape[0]
    x = act.double().reshape(n, 64, 256)
    w = torch.cat([_d(pack[122]).reshape(256, 2), _d(pack[130]).reshape(256, 1)], 1)
    cat = lambda i, j: torch.cat([_d(pack[i]).reshape(-1), _d(pack[j]).reshape(-1)])      # noqa: E731
    bias, g, beta, mean, var = cat(123, 131), cat(124, 132), cat(125, 133), cat(126, 134), cat(127, 135)
    s = g / torch.sqrt(var + BN_EPS)
    t = (bias - mean) * s + beta
    h = x @ w
    hs = h * s
    y = hs + t
    bound = (C * 256 * U * s.abs() * (x.abs() @ w.abs()) + U * (hs.abs() + y.abs())
             + C * (3 * U * hs.abs() + 5 * U * ((bias - mean) * s).abs() + U * t.abs()))
    return y, bound, h, s, t


def _half_ulp_bf16(v):
    _, e = torch.frexp(v)                                    # v in [2^(e-1), 2^e): a bf16 ulp is 2^(e-8)
    return torch.where(v > 0, torch.pow(2.0, (e - 9).double()).clamp_min(2.0 ** -134), torch.zeros_like(v))


def _pf_vf(y, bound):
    n = y.shape[0]
    pf = torch.relu(y[..., :2]).reshape(n, 128)              # Keras Flatten of NHWC: (h*8+w)*2+c
    bpf = bound[..., :2].reshape(n, 128)
    return pf, bpf + _half_ulp_bf16(pf + bpf), torch.relu(y[..., 2]), bound[..., 2]


def _gemm(pack, pf):
    p = pf.double()
    w = torch.as_tensor(np.asarray(pack[128], np.float32)).to(torch.bfloat16).double().to(DEV)    # f2bf: RNE
    b = _d(pack[129])
    acc = p @ w
    return acc, b, C * 128 * U * (p.abs() @ w.abs()) + U * (acc + b).abs()


def _softmax(logits, pad=0):
    """fp64 softmax over the kernel's fp32 logits; pad > 0 also sums that many zero logits (a defect)."""
    l = logits.double()
    m = l.max(1, keepdim=True).values
    z = l - m
    ez = torch.exp(z)
    s = ez.sum(1, keepdim=True)
    p = ez / s
    r = 4 * U + U * z.abs()
    r_s = (p * r).sum(1, keepdim=True) + C * 67 * U
    bound = p * (r + r_s + 2 * U) + C * 2.5 * TINY
    return (ez / (s + pad * torch.exp(-m)) if pad else p), bound


def _value(pack, vf):
    v = vf.double()
    w1, b1, w2, b2 = _d(pack[136]).reshape(64, 256), _d(pack[137]), _d(pack[138]).reshape(256), _d(pack[139])
    z = v @ w1 + b1
    dz = C * 64 * U * (v.abs() @ w1.abs()) + U * z.abs()
    hid = torch.relu(z)
    y = hid @ w2 + b2
    dy = dz @ w2.abs() + C * 256 * U * (hid @ w2.abs()) + U * y.abs()
    val = torch.tanh(y)
    bound = torch.cosh((y.abs() - dy).clamp_min(0)) ** -2 * dy + 4 * U * val.abs()
    return val, bound, hid, w2, b2, y


def _ratio(got, want, bound):
    return float(((got.double().reshape(want.shape) - want).abs() / bound).max())


def _stage_ratios(pack, got):
    y, by, _, _, _ = _heads(pack, got["act"])
    pf, bpf, vf, bvf = _pf_vf(y, by)
    acc, b, bl = _gemm(pack, got["pf"])
    p, bp = _softmax(got["logits"])
    v, bv, _, _, _, _ = _value(pack, got["vf"])
    return {"pf": _ratio(got["pf"], pf, bpf), "vf": _ratio(got["vf"], vf, bvf), "logits": _ratio(got["logits"], acc + b, bl),
            "softmax": _ratio(got["policy"], p, bp), "value": _ratio(got["value"], v, bv)}


def _fmt(r):
    return " ".join("%s %.3f" % kv for kv in r.items())


# ---- 1. every stage within its derived bound --------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["bf16", "fp8"])
@pytest.mark.parametrize("name", ["lively", "sharp"])
@pytest.mark.parametrize("n", NS)
def test_head_stages_within_derived_bounds(nets, planes, name, precision, n):
    """n on either side of k_softmax_value's 8-row blocks, the policy GEMM's 256-row M tiles, the single-tile / two-tile
    switch at 296 and the 592-board round of the tower."""
    e, pack, _ = nets(name)
    e.set_net_precision(precision)
    x = planes[:n]
    got = e.debug_tower(x, layer=20)
    r = _stage_ratios(pack, got)
    print("worst err/bound %s %s n=%d: %s" % (name, precision, n, _fmt(r)))
    assert max(r.values()) <= 1.0, r
    p, v = e.net_forward(x)
    assert torch.equal(p, got["policy"]) and torch.equal(v, got["value"])


def test_packs_are_not_vacuous(nets, planes):
    x = planes[:593]
    e, pack, _ = nets("lively")
    e.set_net_precision("bf16")
    p32, v32 = model_torch.forward(pack, x.float().cpu().numpy(), device="cuda")
    netpacks.assert_lively(p32, v32)
    e, pack, _ = nets("sharp")
    e.set_net_precision("bf16")
    got = e.debug_tower(x, layer=20)
    p, _ = _softmax(got["logits"])
    v = _value(pack, got["vf"])[0]
    print("sharp pack: %d probabilities below 2^-126 in %d of 593 rows, %d values with |v| > 0.9"
          % (int((p < 2.0 ** -126).sum()), int((p < 2.0 ** -126).any(1).sum()), int((v.abs() > 0.9).sum())))
    assert bool((p < 2.0 ** -126).any()) and bool((v.abs() > 0.9).any())


def _moved_by_one(n):
    """Each row's neighbour inside its 8-row block (rows 2k and 2k+1 exchanged; an unpaired last row stays)."""
    perm = torch.arange(n, device=DEV) ^ 1
    return torch.where(perm < n, perm, torch.arange(n, device=DEV))


@pytest.mark.parametrize("precision", ["bf16", "fp8"])
def test_bounds_reject_planted_head_defects(nets, planes, precision):
    """What a kernel with each defect would compute, as a defective reference: it must break the stage's bound at least
    tenfold at its worst element (compare test_parity_bound_rejects_a_displaced_tap_or_a_dropped_channel_slice)."""
    e, pack, _ = nets("lively")
    e.set_net_precision(precision)
    n = 257
    got = e.debug_tower(planes[:n], layer=20)
    y, by, h, s, t = _heads(pack, got["act"])
    pf, bpf, vf, bvf = _pf_vf(y, by)
    acc, b, bl = _gemm(pack, got["pf"])
    p, bp = _softmax(got["logits"])
    v, bv, hid, w2, b2, yv = _value(pack, got["vf"])
    assert max(_stage_ratios(pack, got).values()) <= 1.0
    j = int((hid * w2).abs().max(0).values.argmax())                    # a live hidden unit with a large |h_j w2_j|
    assert float(hid[:, j].max()) > 0
    tail = acc.clone()
    tail[:, 1920:] = 0                                                  # the last, partial N tile's products left out
    perm = _moved_by_one(n)
    defects = {
        "pf: policy channels c swapped": (got["pf"], pf.reshape(n, 64, 2).flip(2).reshape(n, 128), bpf),
        "pf: h,w transposed in the flatten": (got["pf"], pf.reshape(n, 8, 8, 2).transpose(1, 2).reshape(n, 128), bpf),
        "vf: value BN shift left out": (got["vf"], torch.relu(h[..., 2] * s[2]), bvf),
        "logits: bias read from column j+1": (got["logits"], acc + torch.roll(b, -1), bl),
        "logits: columns 1920-1967 without products": (got["logits"], tail + b, bl),
        "softmax: 80 zero-padded logits summed": (got["policy"], _softmax(got["logits"], pad=80)[0], bp),
        "softmax: row moved by one": (got["policy"], p[perm], bp),
        "value: hidden unit %d dropped" % j: (got["value"], torch.tanh(yv - hid[:, j] * w2[j]), bv),
        "value: bv2 left out": (got["value"], torch.tanh(yv - b2), bv),
        "value: row moved by one": (got["value"], v[perm], bv),
    }
    margins = {k: _ratio(g, bad, bound) for k, (g, bad, bound) in defects.items()}
    for k, m in margins.items():
        print("%s planted defect '%s': worst err/bound %.3g" % (precision, k, m))
    assert min(margins.values()) >= 10, margins


def test_slot1_heads_read_their_rows_of_the_shared_logits(planes):
    """Slot 1's logits sit at an offset inside the two-slot buffer: both slots' stages against their own packs."""
    lively, sharp = PACKS["lively"](), PACKS["sharp"]()
    x = planes[:593]
    e = Engine(max_games=600, max_nodes=2)
    e.load_weights(lively)
    e.load_weights(sharp, slot=1)
    amax = e.calibrate(calibration_planes(e, n=64), slot=1)
    for precision in ("bf16", "fp8"):
        if precision == "fp8":
            e.load_weights(sharp, precision="fp8", calibration=amax, slot=1)
        got1 = e.debug_tower(x, layer=20, slot=1)
        got0 = e.debug_tower(x, layer=20, slot=0)
        r1, r0 = _stage_ratios(sharp, got1), _stage_ratios(lively, got0)
        print("worst err/bound slot 1 (sharp, %s) n=593: %s\nworst err/bound slot 0 (lively, bf16) n=593: %s"
              % (precision, _fmt(r1), _fmt(r0)))
        assert max(r1.values()) <= 1.0 and max(r0.values()) <= 1.0, (r1, r0)
        p1, v1 = e.net_forward(x, slot=1)
        assert torch.equal(p1, got1["policy"]) and torch.equal(v1, got1["value"])
    e.close()


# ---- 2. calibration against what it measures --------------------------------------------------------------------------------
def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("n", [1, 37, 297, 4096])
def test_calibration_is_the_max_of_the_taps(nets, planes, n):
    """k_absmax_bf16 over the single-tile and the two-tile tower, its grid-stride loop covering more than one block."""
    e, _, _ = nets("lively")
    e.set_net_precision("bf16")
    x = planes[:n]
    got = e.calibrate(x)
    want = np.array([float(e.debug_tower(x, layer=L)["act"].float().abs().max()) for L in range(21)], np.float32)
    assert got.dtype == np.float32 and np.array_equal(_bits(got), _bits(want)), (got, want)


def test_chunked_calibration_equals_one_pass(nets, planes):
    """An engine of 256 rows calibrates 1,000 in four calls (Engine._calibrate) and must find the same bits."""
    e, pack, _ = nets("lively")
    e.set_net_precision("bf16")
    x = planes[:1000]
    want = e.calibrate(x)
    small = Engine(max_games=256, max_nodes=2)
    small.load_weights(pack)
    got = small.calibrate(x)
    small.close()
    assert np.array_equal(_bits(got), _bits(want)), (got, want)


def test_calibration_tracks_the_fp32_graph(nets):
    """Per layer, the calibrated amax is within twice the bf16 emulation's own error of the fp32 graph's max |output|."""
    e, pack, _ = nets("lively")
    e.set_net_precision("bf16")
    xt = calibration_planes(e, n=256)
    amax = e.calibrate(xt)
    x = xt.float().cpu().numpy()[..., :127]
    f32, emu = {}, {}
    model_torch.forward(pack, x, device="cuda", taps=f32)
    model_torch.forward(pack, x, device="cuda", emulate_bf16_activations=True, taps=emu)
    ratios = []
    for L in range(21):
        m32 = float(f32["act"][L].abs().max())
        E = float((emu["act"][L] - f32["act"][L]).abs().max())
        ratios.append(abs(float(amax[L]) - m32) / (2 * E))
        assert abs(float(amax[L]) - m32) <= 2 * E, (L, float(amax[L]), m32, E)
    print("|amax - fp32 max| / (2 x emulation error) per layer: " + " ".join("%.2f" % r for r in ratios))


def test_calibration_leaves_the_precision_and_the_other_slot(planes):
    lively, other = netpacks.lively_pack(), netpacks.lively_pack(seed=netpacks.LIVELY_SEED + 1)
    x = planes[:64]
    ref = Engine(max_games=64, max_nodes=2)
    ref.load_weights(lively)
    want = ref.calibrate(x)
    ref.load_weights(other)
    want_other = ref.calibrate(x)
    ref.close()
    e = Engine(max_games=64, max_nodes=2)
    e.load_weights(lively, precision="fp8", calibration=want)
    p0, v0 = e.net_forward(x)
    got = e.calibrate(x)                                    # measures the bf16 tower of an engine that runs fp8
    assert np.array_equal(_bits(got), _bits(want))
    assert e.net_precision == "fp8"
    p1, v1 = e.net_forward(x)
    assert torch.equal(p1, p0) and torch.equal(v1, v0)
    e.load_weights(other, slot=1)
    got_other = e.calibrate(x, slot=1)
    assert np.array_equal(_bits(got_other), _bits(want_other))
    p2, v2 = e.net_forward(x)
    assert torch.equal(p2, p0) and torch.equal(v2, v0)
    e.close()


# ---- 3. fp8 scale edges -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def edge():
    pack = netpacks.lively_pack()
    e = Engine(max_games=64, max_nodes=2)
    e.load_weights(pack)
    amax = e.calibrate(calibration_planes(e, n=64))
    yield e, pack, amax
    e.close()


def _layers_within_one_step(e, pack, x, amax):
    """The per-layer check of test_gpu_fp8 with these amax values: every element equal to the emulation of its layer
    alone or one e4m3 step away, and no more than LAYER_MAX_DIFF_FRACTION of them one step away.  -> the kernel's taps."""
    e.load_weights(pack, precision="fp8", calibration=amax)
    taps = _kernel_taps(e, x)["act"]
    worst, fracs = [], []
    for L in range(21):
        want, s = _layer_alone(pack, L, x, taps, amax)
        steps = _layer_steps(taps[L], want, s, amax)
        worst.append(int(steps.max()))
        fracs.append(float((steps > 0).float().mean()))
    print("elements one step from the emulation per layer: %s" % " ".join("%.1e" % f for f in fracs))
    assert max(worst) <= 1, worst
    assert max(fracs) <= LAYER_MAX_DIFF_FRACTION, fracs
    return taps


def _codes(taps, amax, L):
    return taps[L].float() / fp8_emu.act_scale(amax[L])


@pytest.mark.parametrize("regime", ["at_448_2k", "above_448_2k", "saturating", "underflowing", "dead_layers"])
def test_fp8_scale_edges(edge, planes, regime):
    e, pack, cal = edge
    x = planes[:37]
    s_cal = [fp8_emu.act_scale(a) for a in cal]
    amax = cal.copy()
    if regime == "at_448_2k":                                # the largest amax of each scale: 448 s exactly
        amax[:20] = np.float32(448.0) * np.float32(s_cal[:20])
        assert [fp8_emu.act_scale(a) for a in amax[:20]] == s_cal[:20]
    elif regime == "above_448_2k":                           # one float above it: the scale doubles
        amax[:20] = np.nextafter(np.float32(448.0) * np.float32(s_cal[:20]), np.float32(np.inf))
        assert [fp8_emu.act_scale(a) for a in amax[:20]] == [2 * s for s in s_cal[:20]]
    elif regime == "saturating":
        amax[:20] = cal[:20] / 16
    elif regime == "underflowing":
        amax[:20] = cal[:20] * 2.0 ** 12
    else:
        amax[[0, 12]] = 0.0                                  # scale 1
        assert fp8_emu.act_scale(amax[0]) == 1.0
    taps = _layers_within_one_step(e, pack, x, amax)
    if regime == "saturating":
        sat = [float((_codes(taps, amax, L).abs() == 448).float().mean()) for L in range(20)]
        print("codes at +-448 per layer: %s" % " ".join("%.3f" % f for f in sat))
        assert max(sat) >= 0.01 and bool((_codes(taps, amax, 0) == -448).any())      # the stem has no ReLU
    if regime == "underflowing":
        small = [float((_codes(taps, amax, L).abs() < 2.0 ** -6).float().mean()) for L in range(20)]
        c0 = _codes(taps, amax, 0)
        sub0 = float(((c0.abs() < 2.0 ** -6) & (c0 != 0)).float().mean())
        print("codes subnormal or zero per layer: %s; nonzero subnormal in the stem %.3f"
              % (" ".join("%.2f" % f for f in small), sub0))
        assert min(small) >= 0.5 and sub0 >= 0.1


# ---- 4. the activation-scale floor ------------------------------------------------------------------------------------------
def test_tiny_amax_is_floored_to_a_finite_scale(edge, planes):
    """amax 1e-37 would give s = 2^-131 and 1 / s = inf: every zero activation of that layer became e4m3(0 x inf), a NaN
    code, which the next ReLU (fmaxf) turns into 0 -- finite, wrong outputs.  With the floor both amax 1e-37 and
    448 x 2^-128 get s = 2^-126, so both loads compute the same bits, and the emulation (which floors the same way)
    still matches every layer to one e4m3 step."""
    e, pack, cal = edge
    x = planes[:64]
    outs = []
    for tiny in (1e-37, 448.0 * 2.0 ** -128):
        amax = cal.copy()
        amax[[0, 7, 19]] = np.float32(tiny)
        e.load_weights(pack, precision="fp8", calibration=amax)
        acts = _kernel_taps(e, x)["act"]
        assert not [L for L in range(21) if not bool(torch.isfinite(acts[L]).all())], tiny
        p, v = e.net_forward(x)
        assert bool(torch.isfinite(p).all()) and bool(torch.isfinite(v).all()), tiny
        assert torch.allclose(p.sum(1), torch.ones(64, device="cuda"), atol=1e-4)
        outs.append((p, v))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert fp8_emu.act_scale(np.float32(1e-37)) == fp8_emu.act_scale(np.float32(448.0 * 2.0 ** -128)) == 2.0 ** -126
    _layers_within_one_step(e, pack, x, amax)
