"""Emulation of the fp8 tower (include/chessrl_b200.h crl_net_load_fp8_host, DESIGN.md section 3.1) in an fp32 torch graph.

The numeric definition, shared with csrc/net.cu:
  - planes are e4m3 (0 / 1: exact);
  - weights per output channel n of convolution L: ws[n] = max_k |W[k][n]| / 448 (1 for an all-zero column),
    Wq = e4m3_rn_satfinite(W / ws[n]);
  - the outputs of convolutions 0..19 are stored as e4m3(a / s_L) with s_L = max(2^ceil(log2(amax_L / 448)), 2^-126)
    (1 for amax 0; the floor is the smallest normal power of two, so that 1 / s_L is finite);
    convolution 20 feeds only the heads and keeps the bf16 rounding of the bf16 tower;
  - epilogue: a = acc * (ws[n] * s_in * bn_scale[n]) + bn_shift[n], + dequant(residual) * s_res, ReLU.
The heads are the bf16 tower's (oracle/model_torch.forward with emulate_bf16_activations=True).
Mutations (for tests that show a tolerance rejects a wrong kernel): mutate={"shift_tap": L} displaces layer L's input by
one column, {"drop_slice": L} drops input channels 0..127 of layer L, {"double_scale": L} stores layer L's codes with
2 s_L while its consumers read them with s_L, {"double_ws": (L, n)} doubles the weight scale of output channel n of
layer L in its epilogue, {"double_s_res": L} reads layer L's residual with twice its scale."""
import numpy as np
import torch
import torch.nn.functional as F

E4M3_MAX = 448.0
SCALE_FLOOR = 2.0 ** -126       # the smallest normal float32 power of two: the least activation scale
BN_EPS = np.float32(1e-3)


def e4m3(x):
    """Round to the nearest e4m3 value, ties to even, saturating at +-448 (torch's cast alone gives NaN above ~464)."""
    return torch.clamp(x, -E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).to(torch.float32)


def act_scale(amax):
    """max(2^ceil(log2(amax / 448)), 2^-126) in float32 arithmetic, 1 for amax = 0 (the floor keeps 1 / s finite)."""
    a = np.float32(amax)
    if not a > 0:
        return 1.0
    if a <= np.float32(E4M3_MAX * SCALE_FLOOR):
        return SCALE_FLOOR
    r = a / np.float32(E4M3_MAX)
    m, e = np.frexp(r)
    return float(np.ldexp(np.float32(1.0), int(e) - 1 if m == 0.5 else int(e)))


def quantise_weights(k):
    """HWIO kernel [3,3,cin,256] -> (e4m3 values of W / ws, same shape, float32; ws [256] float32)."""
    k = np.asarray(k, dtype=np.float32)
    m = np.abs(k).reshape(-1, k.shape[-1]).max(axis=0)
    ws = np.where(m > 0, m / np.float32(E4M3_MAX), np.float32(1.0)).astype(np.float32)
    return e4m3(torch.from_numpy(k / ws)).numpy(), ws


def is_second(L):
    """Convolution L is the second of a residual block: it adds the block input."""
    return L > 0 and (L - 1) % 2 == 1


def _conv_tensors(L):
    if L == 0:
        return 0, 1, -1
    ik = 2 + 12 * ((L - 1) // 2) + 6 * ((L - 1) % 2)
    return ik, ik + 1, ik + 2


def _fold(pack, ib, ibn):
    b = np.asarray(pack[ib], dtype=np.float32)
    if ibn < 0:
        return np.ones(256, np.float32), b
    g, beta, mean, var = (np.asarray(pack[ibn + i], dtype=np.float32) for i in range(4))
    s = g / np.sqrt(var + BN_EPS)
    return s.astype(np.float32), ((b - mean) * s + beta).astype(np.float32)


def layer(pack, L, codes_in, s_in, res=None, s_out=1.0, device="cpu", mutate=None):
    """Convolution L alone: input codes [B,Cin,8,8] (values / s_in), res = (codes, scale) of the block input for the
    second convolution of a block.  Returns (output codes, value): code x s_out for L < 20, the bf16-rounded value
    (codes None) for L = 20."""
    mutate = mutate or {}
    t = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float32, device=device)     # noqa: E731
    ik, ib, ibn = _conv_tensors(L)
    wq, ws = quantise_weights(pack[ik])
    bn_s, bn_b = _fold(pack, ib, ibn)
    scale = (ws * np.float32(s_in) * bn_s).astype(np.float32)
    if mutate.get("double_ws", (None,))[0] == L:
        scale[mutate["double_ws"][1]] *= 2
    xin = codes_in
    if mutate.get("shift_tap") == L:
        xin = torch.roll(xin, 1, dims=3)
    if mutate.get("drop_slice") == L:
        xin = xin.clone()
        xin[:, :128] = 0
    acc = F.conv2d(xin, t(wq).permute(3, 2, 0, 1).contiguous(), None, padding=1)
    a = acc * t(scale).view(1, -1, 1, 1) + t(bn_b).view(1, -1, 1, 1)
    if res is not None:
        a = a + res[0] * (2 * res[1] if mutate.get("double_s_res") == L else res[1])
    if L > 0:
        a = torch.relu(a)
    if L == 20:
        return None, a.to(torch.bfloat16).to(torch.float32)
    s_store = 2 * s_out if mutate.get("double_scale") == L else s_out
    codes = e4m3(a * (1.0 / s_store))
    return codes, codes * s_out


def forward(pack, planes_nhwc, amax, device="cpu", taps=None, mutate=None):
    """planes [B,8,8,127|128] (0 / 1), amax: the 21 calibration values -> (policy [B,1968], value [B]).
    taps receives 'act' (21 NHWC outputs as the kernel's tap writes them: code x s_L, layer 20 in bf16), 'pf', 'vf',
    'logits'."""
    s_act = [act_scale(a) for a in amax]
    t = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float32, device=device)     # noqa: E731
    x = torch.as_tensor(planes_nhwc, dtype=torch.float32, device=device)[..., :127].permute(0, 3, 1, 2).contiguous()
    codes_in, s_in = e4m3(x), 1.0
    acts = []
    block_in = None                       # (codes, scale) of the current residual block's input
    for L in range(21):
        second = is_second(L)
        codes, val = layer(pack, L, codes_in, s_in, block_in if second else None, s_act[L] if L < 20 else 1.0,
                           device=device, mutate=mutate)
        if taps is not None:
            acts.append(val.permute(0, 2, 3, 1).contiguous())
        codes_in, s_in = codes, s_act[L]
        if L == 0 or second:
            block_in = (codes, s_act[L])
    xh = val
    bf = lambda a: a.to(torch.bfloat16).to(torch.float32)                                  # noqa: E731
    p = F.conv2d(xh, t(pack[122]).permute(3, 2, 0, 1).contiguous(), t(pack[123]))
    ps, pb = _fold_head(pack, 124)
    p = torch.relu(p * t(ps).view(1, -1, 1, 1) + t(pb).view(1, -1, 1, 1))
    p = bf(p.permute(0, 2, 3, 1).reshape(p.shape[0], -1))
    logits = p @ bf(t(pack[128])) + t(pack[129])
    policy = torch.softmax(logits, dim=-1)
    v = F.conv2d(xh, t(pack[130]).permute(3, 2, 0, 1).contiguous(), t(pack[131]))
    vs, vb = _fold_head(pack, 132)
    v = torch.relu(v * t(vs).view(1, -1, 1, 1) + t(vb).view(1, -1, 1, 1))
    vf = v.permute(0, 2, 3, 1).reshape(v.shape[0], -1)
    v = torch.relu(vf @ t(pack[136]) + t(pack[137]))
    v = torch.tanh(v @ t(pack[138]) + t(pack[139])).reshape(-1)
    if taps is not None:
        taps.update({"act": acts, "pf": p, "vf": vf, "logits": logits})
    return policy, v


def _fold_head(pack, i):
    g, beta, mean, var = (np.asarray(pack[i + k], dtype=np.float32) for k in range(4))
    return g / np.sqrt(var + BN_EPS), beta - mean * g / np.sqrt(var + BN_EPS)
