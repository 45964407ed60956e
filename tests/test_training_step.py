"""SURVEY 8(f)-1: the training step (chessrl_b200/training.py: loss_terms, KerasAdam, BatchNorm statistics) against the
independent float64 restatement of the Keras definitions in oracle/train_ref.py (model.py:68-72, 33-60, 111-122).

The step is device-agnostic torch code, so the arithmetic is checked here on the CPU in fp32 against fp64;
tests/test_gpu_training.py repeats the comparison on the GPU the step really runs on.

Tolerances (fp32 autograd vs fp64, 21 conv layers deep): losses 1e-5 relative; per-tensor gradients
max|g32 - g64| <= 2e-2 * max|g64| and ||g32 - g64|| <= 4e-3 * ||g64|| -- about twice the fp32 noise floor (the fp64
restatement itself evaluated in fp32 is off by 0.9e-2 / 1.2e-3 on the worst tensor); moving statistics 1e-5; the Adam
update itself (same gradients fed to both) 1e-6.
"""
import contextlib
import random

import numpy as np
import pytest
import torch

import chessrl_oracle as O
import train_ref
from chessrl_b200 import model, training


def _batch(n_positions=10, seed=4):
    rng = random.Random(seed)
    g = O.OGame()
    planes, pol, val = [], [], []
    labels = {u: i for i, u in enumerate(O.uci_labels())}
    while len(planes) < n_positions:
        legal = g.get_legal_moves()
        m = rng.choice(legal)
        planes.append(O.planes(g).astype(np.float32))
        pol.append(labels[m])
        val.append(float(rng.choice((-1, 0, 1))))
        g.move(m)
    x = np.zeros((n_positions, 8, 8, 128), dtype=np.float32)
    x[..., :127] = np.stack(planes)
    return x, np.array(pol, dtype=np.int64), np.array(val, dtype=np.float32)


@pytest.fixture(scope="module")
def step_data():
    pack = model.random_pack(seed=21, perturb_bn=True)
    x, pol, val = _batch()
    tr = training.trainable_indices()
    ref_losses, ref_grads, ref_stats = train_ref.loss_and_grads(pack, x, pol, val, tr)
    return pack, x, pol, val, tr, ref_losses, ref_grads, ref_stats


@contextlib.contextmanager
def _fixed_cpu_summation_order():
    """One thread and ATen's own convolutions (no oneDNN).  The BatchNorm beta gradients are sums over the batch that
    cancel heavily, so their fp32 error depends on how a sum is split: the CPU kernels split it by thread count, and
    with the defaults the worst relative L2 error moves between 1.2e-3 and 7.3e-3 over 1-16 threads, above the bound
    on a 16-core host.  With the order fixed it is 1.7e-3 whatever the host's core count."""
    threads, onednn = torch.get_num_threads(), torch.backends.mkldnn.enabled
    torch.set_num_threads(1)
    torch.backends.mkldnn.enabled = False
    try:
        yield
    finally:
        torch.set_num_threads(threads)
        torch.backends.mkldnn.enabled = onednn


def _torch_step(pack, x, pol, val, tr, device="cpu"):
    params = [torch.tensor(w, device=device) for w in pack]
    for i in tr:
        params[i].requires_grad_(True)
    with _fixed_cpu_summation_order() if device == "cpu" else contextlib.nullcontext():
        total, lp, lv, reg, _ = training.loss_terms(params, torch.as_tensor(x, device=device), torch.as_tensor(pol, device=device),
                                                    torch.as_tensor(val, device=device), training=True)
        grads = torch.autograd.grad(total, [params[i] for i in tr])
    return params, {"loss": total.item(), "policy_loss": lp.item(), "value_loss": lv.item(), "reg": reg.item()}, grads


def check_against_ref(pack, x, pol, val, tr, ref_losses, ref_grads, ref_stats, device="cpu", grad_max=2e-2, grad_l2=4e-3):
    params, losses, grads = _torch_step(pack, x, pol, val, tr, device)
    for k in ("loss", "policy_loss", "value_loss", "reg"):
        assert abs(losses[k] - ref_losses[k]) <= 1e-5 * max(1.0, abs(ref_losses[k])), (k, losses[k], ref_losses[k])
    # the policy target is one of 1968 classes at random init: CE ~ log(1968); the terms must all be alive
    assert 6.0 < ref_losses["policy_loss"] < 9.5 and ref_losses["value_loss"] > 0.05 and ref_losses["reg"] > 1.0
    worst = 0.0
    dead = {3 + 12 * b + 6 * k for b in range(10) for k in range(2)} | {123, 131}
    for i, g in zip(tr, grads):
        g64 = ref_grads[i]
        scale = np.abs(g64).max()
        g32 = g.detach().cpu().numpy().astype(np.float64)
        if i in dead:
            # a conv bias in front of a training-mode BatchNorm: the batch mean removes it, its gradient is exactly 0
            assert scale <= 1e-12 and np.abs(g32).max() <= 1e-5, (i, scale, np.abs(g32).max())
            continue
        assert scale > 1e-9, "dead gradient for tensor %d" % i
        err = np.abs(g32 - g64).max() / scale
        err_l2 = np.linalg.norm(g32 - g64) / np.linalg.norm(g64)
        worst = max(worst, err)
        assert err <= grad_max and err_l2 <= grad_l2, (i, err, err_l2)
    # BatchNorm moving statistics after the forward pass (momentum 0.99, unbiased batch variance)
    bn_slots = [2 + 12 * b + 6 * s + 4 for b in range(10) for s in range(2)] + [126, 134]
    for slot, (m64, v64) in zip(bn_slots, ref_stats):
        assert np.abs(params[slot].detach().cpu().numpy() - m64).max() <= 1e-5
        assert np.abs(params[slot + 1].detach().cpu().numpy() - v64).max() <= 1e-5 * max(1.0, np.abs(v64).max())
    return worst


def test_loss_gradients_and_bn_statistics_match_fp64_restatement(step_data):
    check_against_ref(*step_data, device="cpu")


def test_split_convolution_step_matches_fp64_restatement(step_data):
    """The tf32x3 setting (training._Conv3xTF32: x*w as x_hi*w_hi + x_hi*w_lo + x_lo*w_hi in all three convolution
    passes) against the same fp64 restatement and the same bounds.  On the CPU the three partial convolutions run in
    fp32, so this checks the decomposition and its hand-written backward; the GPU test runs them on the tensor cores."""
    hi, lo = training._tf32_split(torch.tensor([1.0000001, -3.14159265, 1e-20, 123456.789, 0.0]))
    assert torch.equal(hi + lo, torch.tensor([1.0000001, -3.14159265, 1e-20, 123456.789, 0.0]))
    assert (hi.view(torch.int32) & 0x1FFF).abs().sum() == 0               # 13 low mantissa bits clear: TF32-representable
    assert (lo.abs() <= hi.abs() * 2.0 ** -11 + 1e-45).all()
    with training.arithmetic("tf32x3"):
        check_against_ref(*step_data, device="cpu")


def test_keras_adam_update_matches_definition():
    rng = np.random.default_rng(0)
    ws = [rng.normal(size=s).astype(np.float32) for s in ((3, 3, 4, 5), (7,), (11, 2))]
    params = [torch.tensor(w) for w in ws]
    opt = training.KerasAdam(params, lr=0.002, epsilon=1e-7)
    w64 = [w.astype(np.float64) for w in ws]
    m64 = [np.zeros_like(w) for w in w64]
    v64 = [np.zeros_like(w) for w in w64]
    for t in range(1, 6):
        gs = [rng.normal(size=w.shape).astype(np.float32) * (10.0 ** rng.integers(-9, 1)) for w in ws]   # incl. tiny ones
        opt.step([torch.tensor(g) for g in gs])
        for k in range(len(ws)):
            w64[k], m64[k], v64[k] = train_ref.keras_adam_step(w64[k], gs[k].astype(np.float64), m64[k], v64[k], t)
            assert np.abs(params[k].numpy() - w64[k]).max() <= 1e-6, (t, k)
    # epsilon-hat form: with g = 1e-9 the first update is lr * g / (g + eps / sqrt(1 - b2)) -- NOT ~lr as torch's Adam gives
    p = [torch.zeros(1)]
    training.KerasAdam(p).step([torch.full((1,), 1e-9)])
    want = -0.002 * np.sqrt(1 - 0.999) / (1 - 0.9) * (0.1 * 1e-9) / (np.sqrt(0.001 * 1e-18) + 1e-7)
    assert abs(p[0].item() - want) <= 1e-9 and abs(p[0].item()) < 1e-5


def test_trainable_set_is_everything_but_moving_statistics():
    tr = set(training.trainable_indices())
    shapes = model.pack_shapes()
    frozen = [i for i in range(len(shapes)) if i not in tr]
    assert len(frozen) == 2 * 22 and all(len(shapes[i]) == 1 for i in frozen)
    assert sum(int(np.prod(shapes[i])) for i in tr) == model.N_PARAMS - sum(int(np.prod(shapes[i])) for i in frozen)
