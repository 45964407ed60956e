"""The training step behind Agent.train / selfplay's train_model_job / supervised.py (agent.py:64-89,
model.py:68-72, 86-99, netencoder.py:137-181) in PyTorch, which BASELINE.json's north_star allows for the
training step.  Inputs are built on the GPU: every ply of every game is encoded by the CUDA encode kernel
(crl_encode) from the game's per-ply records.

Keras semantics kept: Adam(lr=0.002, eps=1e-7); loss = categorical cross-entropy(one-hot of the move played)
+ mean squared error(value, white-point-of-view result) + l2(0.01) on every conv / dense kernel; BatchNorm in
training mode with momentum 0.99 / eps 1e-3; a batch = `batch_size` games, one sample per ply; each game's
planes are rotated by 180 degrees with probability 0.1 while the policy target is NOT (agent.py:82-84).
"""

from __future__ import annotations

import contextlib
import itertools
import math
import os
import random
from collections import namedtuple

import numpy as np
import torch
import torch.nn.functional as F

from . import boards as B
from . import runtime
from .netencoder import get_uci_labels

N_LABELS = 1968

L2 = 0.01
BN_EPS = 1e-3
_KERNEL_IDX = None

# Arithmetic of the training step.  "fp32" (default) is the parity setting -- fp32 convolutions and matmuls without TF32,
# what the loss / gradient / Adam tests pin against the fp64 restatement of the Keras definitions.  "tf32" and "bf16" are
# opt-in throughput settings (CRL_TRAIN_PRECISION, `--precision` of the CLIs) that put the convolutions on the tensor
# cores: measured on a B200, 640 positions per step: fp32 103.5 ms, tf32 12.6 ms (8.2 x), bf16 autocast 9.9 ms (10.5 x);
# the loss agrees to 1e-6 / 1e-5 relative, individual gradient tensors of the 21-layer tower deviate from a float64 step by
# up to 13 % / 39 % of their largest entry on a random-init pack (fp32: 1 %; scripts/probe/train_precision_probe.py) --
# NOT parity-grade, hence opt-in.
# "tf32x3" keeps fp32-grade numerics ON the tensor cores: every convolution operand is split into a TF32-representable
# head and its (exact) fp32 remainder, x = x_hi + x_lo, and x * w is evaluated as x_hi*w_hi + x_hi*w_lo + x_lo*w_hi with
# fp32 accumulation -- three TF32 convolutions instead of one fp32 convolution on the CUDA cores, forward and both
# backward passes (the dropped x_lo*w_lo term is below 2^-22 of the product).  See _Conv3xTF32.  Measured on a B200, 640
# positions: 41.1 ms per step (2.5 x fp32); loss equal to fp32's to 7 digits; gradients against a float64 step: worst tensor
# 2.0e-2 of its largest entry / 7.7e-3 in L2, where fp32 itself is at 9.8e-3 / 2.7e-3 (plain tf32: 1.3e-1 / 9.9e-2) -- the
# tensor cores' fp32 accumulation, not the split, sets that floor.  fp32-grade, still opt-in.
PRECISIONS = ("fp32", "tf32x3", "tf32", "bf16")


def resolve_precision(precision=None):
    precision = precision or os.environ.get("CRL_TRAIN_PRECISION", "fp32")
    if precision not in PRECISIONS:
        raise ValueError("training precision %r: expected one of %s" % (precision, ", ".join(PRECISIONS)))
    return precision


@contextlib.contextmanager
def arithmetic(precision):
    """TF32 switches (and bf16 autocast) for the duration of a training / validation pass, restored afterwards."""
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    global _CONV_SPLIT
    saved_split = _CONV_SPLIT
    torch.backends.cudnn.allow_tf32 = precision in ("tf32", "tf32x3")     # tf32x3: convolutions only, on split operands
    torch.backends.cuda.matmul.allow_tf32 = precision == "tf32"
    _CONV_SPLIT = precision == "tf32x3"
    try:
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=precision == "bf16"):
            yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
        _CONV_SPLIT = saved_split


_CONV_SPLIT = False


def _tf32_split(x):
    """x = hi + lo with hi representable in TF32 (10 explicit mantissa bits, round half up in magnitude) and lo the exact
    fp32 remainder."""
    hi = ((x.contiguous().view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)
    return hi, x - hi


class _Conv3xTF32(torch.autograd.Function):
    """conv2d (stride 1, 'same' padding) whose three passes each run as three TF32 tensor-core convolutions on split
    operands (see PRECISIONS): fp32-grade results at roughly a third of the fp32 CUDA-core time."""

    @staticmethod
    def forward(ctx, x, w, b, padding):
        ctx.save_for_backward(x, w)
        ctx.padding = padding
        xh, xl = _tf32_split(x)
        wh, wl = _tf32_split(w)
        y = F.conv2d(xh, wh, None, padding=padding)
        y = y + F.conv2d(xh, wl, None, padding=padding)
        y = y + F.conv2d(xl, wh, None, padding=padding)
        return y + b.view(1, -1, 1, 1)

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        pad = ctx.padding
        gh, gl = _tf32_split(gy)
        xh, xl = _tf32_split(x)
        wh, wl = _tf32_split(w)
        gx = gw = None
        if ctx.needs_input_grad[0]:
            gi = torch.nn.grad.conv2d_input
            gx = gi(x.shape, wh, gh, padding=pad) + gi(x.shape, wl, gh, padding=pad) + gi(x.shape, wh, gl, padding=pad)
        if ctx.needs_input_grad[1]:
            gwf = torch.nn.grad.conv2d_weight
            gw = gwf(xh, w.shape, gh, padding=pad) + gwf(xh, w.shape, gl, padding=pad) + gwf(xl, w.shape, gh, padding=pad)
        gb = gy.sum(dim=(0, 2, 3)) if ctx.needs_input_grad[2] else None
        return gx, gw, gb, None


def _kernel_indices():
    global _KERNEL_IDX
    if _KERNEL_IDX is None:
        from .model import pack_shapes
        _KERNEL_IDX = [i for i, s in enumerate(pack_shapes()) if len(s) >= 2]
    return _KERNEL_IDX


def _bn(x, p, o, training):
    return F.batch_norm(x, p[o + 2], p[o + 3], p[o], p[o + 1], training=training, momentum=0.01, eps=BN_EPS)


def forward_logits(p, planes_nhwc, training):
    """p: list of 140 tensors (pack order).  Returns (policy logits [B,1968], value [B])."""
    x = planes_nhwc[..., :127].permute(0, 3, 1, 2).to(p[0].dtype)    # fp32 (fp64 when a probe passes double parameters)

    def conv(x, i):
        if _CONV_SPLIT:
            return _Conv3xTF32.apply(x, p[i].permute(3, 2, 0, 1), p[i + 1], p[i].shape[0] // 2)
        return F.conv2d(x, p[i].permute(3, 2, 0, 1), p[i + 1], padding=p[i].shape[0] // 2)

    x = conv(x, 0)
    for blk in range(10):
        o = 2 + 12 * blk
        y = torch.relu(_bn(conv(x, o), p, o + 2, training))
        y = _bn(conv(y, o + 6), p, o + 8, training)
        x = torch.relu(x + y)
    ph = torch.relu(_bn(conv(x, 122), p, 124, training))
    ph = ph.permute(0, 2, 3, 1).reshape(ph.shape[0], -1)
    logits = ph @ p[128] + p[129]
    vh = torch.relu(_bn(conv(x, 130), p, 132, training))
    vh = vh.permute(0, 2, 3, 1).reshape(vh.shape[0], -1)
    vh = torch.relu(vh @ p[136] + p[137])
    value = torch.tanh(vh @ p[138] + p[139]).reshape(-1)
    return logits, value


_LABEL_IDS = None


def _label_ids():
    global _LABEL_IDS
    if _LABEL_IDS is None:
        _LABEL_IDS = {u: i for i, u in enumerate(get_uci_labels())}
    return _LABEL_IDS


def draw_flips(n_games, random_flips):
    """One `np.random.rand() < random_flips` per game in batch order, the draw DataGameSequence.__getitem__ makes
    (netencoder.py:168) -- same calls, so numpy's global stream advances as the reference's does."""
    return [bool(np.random.rand() < random_flips) for _ in range(n_games)]


def game_samples(games, flips):
    """Host arrays for every ply of every game, the samples DatasetGame.augment_game lists (dataset.py:21-43):
    boards [N,9], history bitboards [N,8,8] (most recent first, zero where the stack is exhausted), history lengths
    [N], policy target index [N], value target [N] (white-point-of-view result, 0 for an unfinished game), flip [N]."""
    labels = _label_ids()
    boards, hists, hlens, pol, val, flip_rows = [], [], [], [], [], []
    for g, flip in zip(games, flips):
        n = len(g._moves)
        if n == 0:
            continue
        recs = np.stack(g._records[:n + 1]).astype(np.uint64)
        ply = np.arange(n)
        idx = ply[:, None] - 1 - np.arange(8)[None, :]            # position i+1 plies back, i = 0..7
        h = recs[np.clip(idx, 0, None)][:, :, :8].copy()
        h[idx < 0] = 0
        result = g.get_result()
        boards.append(recs[:n])
        hists.append(h)
        hlens.append(np.minimum(ply, 8))
        pol.append(np.array([labels[m] for m in g._moves], dtype=np.int64))
        val.append(np.full(n, 0.0 if result is None else float(result), dtype=np.float32))
        flip_rows.append(np.full(n, bool(flip)))
    if not boards:
        z = np.zeros
        return z((0, 9), np.uint64), z((0, 8, 8), np.uint64), z(0, np.uint8), z(0, np.int64), z(0, np.float32), z(0, bool)
    return (np.concatenate(boards), np.concatenate(hists), np.concatenate(hlens).astype(np.uint8), np.concatenate(pol),
            np.concatenate(val), np.concatenate(flip_rows))


def encode_games(games, flips, device=None):
    """Planes [N,8,8,128] bf16 (crl_encode) for every ply of every game plus the targets (policy index, value), the
    batch DataGameSequence.__getitem__ builds (netencoder.py:159-181): a game's planes are rotated by 180 degrees when
    its flip is set, its policy target is not (reference quirk, kept)."""
    eng = runtime.scalar_engine()
    boards, hists, hlens, pol, val, flip_rows = game_samples(games, flips)
    n = boards.shape[0]
    if n == 0:
        return (torch.zeros((0, 8, 8, 128), dtype=torch.bfloat16, device=eng.device),
                torch.zeros(0, dtype=torch.int64, device=eng.device), torch.zeros(0, device=eng.device))
    bt = eng.boards_to_device(boards)
    ht = torch.from_numpy(np.ascontiguousarray(hists.transpose(1, 2, 0)).view(np.int64)).to(eng.device)
    lt = torch.from_numpy(hlens).to(eng.device)
    planes = eng.encode(bt, ht, lt)
    if flip_rows.any():
        fr = torch.from_numpy(flip_rows).to(eng.device)
        planes = torch.where(fr.view(n, 1, 1, 1), planes.flip(1, 2), planes)      # np.rot90(k=2) over (H, W)
    return planes, torch.from_numpy(pol).to(eng.device), torch.from_numpy(val).to(eng.device)


# Opt-in search targets (DESIGN.md 3.8) for games recorded with their alpha-beta root scores (gen_data --scores): the
# policy target is softmax(scores / temperature) over the legal moves, the value target (1 - value_weight) * result +
# value_weight * tanh(best score / 400) from white's point of view.  The defaults are starting points, not tuned values.
SearchTargets = namedtuple("SearchTargets", ("temperature", "value_weight"), defaults=(50.0, 0.5))


def check_targets(targets):
    """targets None (the move played and the result) or a SearchTargets with 0 < temperature < inf, 0 <= weight <= 1."""
    if targets is None:
        return None
    if not isinstance(targets, SearchTargets):
        raise ValueError("targets: None or training.SearchTargets, got %r" % (targets,))
    if not (math.isfinite(targets.temperature) and targets.temperature > 0):
        raise ValueError("search targets: the temperature must be positive and finite, got %r" % (targets.temperature,))
    if not 0.0 <= targets.value_weight <= 1.0:
        raise ValueError("search targets: the value weight must lie in [0, 1], got %r" % (targets.value_weight,))
    return targets


def encode_search_games(games, flips, targets, first=0):
    """encode_games plus the search targets of the games that carry root scores (Game.search_scores): returns (planes,
    policy index, value target, policy probabilities float32 [N, 1968]).  Rows of games without scores keep the one-hot
    of the move played and the result.  One crl_search_targets launch covers every scored row; the kernel's legal count
    is checked against each row's score count, and a mismatch raises ValueError naming the game and the ply.  The game
    is named by its index in DatasetGame.games, `first` + its index in `games` (a file's games without moves are not
    loaded, so this can be below the game's position in the JSON list).  The ply is its index in the game's moves.
    Flipped games keep their targets, as encode_games does (reference quirk)."""
    eng = runtime.scalar_engine()
    planes, pol, val = encode_games(games, flips)
    probs = F.one_hot(pol, N_LABELS).float()
    rows, recs, counts, flat, where = [], [], [], [], []
    off = 0
    for j, g in enumerate(games):
        n = len(g._moves)
        if n and g.search_scores is not None:
            if len(g.search_scores) != n:
                raise ValueError("dataset game %d: %d score lists for %d moves" % (first + j, len(g.search_scores), n))
            rows.append(np.arange(off, off + n))
            recs.append(np.stack(g._records[:n]).astype(np.uint64))
            counts += [len(x) for x in g.search_scores]
            flat += g.search_scores
            where += [(first + j, i) for i in range(n)]
        off += n
    if not rows:
        return planes, pol, val, probs
    cnt = np.array(counts, dtype=np.int32)
    flat = np.fromiter(itertools.chain.from_iterable(flat), dtype=np.int32, count=int(cnt.sum()))
    offsets = np.zeros(len(cnt) + 1, dtype=np.int32)
    offsets[1:] = np.cumsum(cnt)
    dev = eng.device
    policy, score_value, legal = eng.search_targets(eng.boards_to_device(np.concatenate(recs)),
                                                    torch.from_numpy(flat).to(dev),
                                                    torch.from_numpy(offsets).to(dev), targets.temperature)
    bad = np.nonzero(legal.cpu().numpy() != cnt)[0]          # (the step synchronises on its loss anyway)
    if len(bad):
        k = int(bad[0])
        raise ValueError("dataset game %d, ply %d: %d root scores for %d legal moves"
                         % (where[k][0], where[k][1], cnt[k], int(legal[k])))
    idx = torch.from_numpy(np.concatenate(rows)).to(dev)
    probs[idx] = policy
    val = val.clone()
    val[idx] = blend_value(val[idx], score_value, targets.value_weight)
    return planes, pol, val, probs


def blend_value(result, score_value, w):
    """The search-target value (1 - w) * result + w * score value; with w = 0 exactly the result."""
    w = float(w)
    return (1.0 - w) * result + w * score_value


class KerasAdam:
    """tf.keras.optimizers.Adam(lr=0.002) (model.py:69) step for step: beta_1 0.9, beta_2 0.999, epsilon 1e-7 applied
    as the paper's "epsilon hat":  lr_t = lr * sqrt(1 - b2^t) / (1 - b1^t);  w -= lr_t * m / (sqrt(v) + eps).
    (torch.optim.Adam puts eps next to sqrt(v_hat) instead, which differs where gradients are tiny.)"""

    def __init__(self, params, lr=0.002, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
        self.params = list(params)
        self.lr, self.b1, self.b2, self.eps = lr, beta_1, beta_2, epsilon
        self.m = [torch.zeros_like(p) for p in self.params]
        self.v = [torch.zeros_like(p) for p in self.params]
        self.t = 0

    @torch.no_grad()
    def step(self, grads):
        self.t += 1
        lr_t = self.lr * np.sqrt(1.0 - self.b2 ** self.t) / (1.0 - self.b1 ** self.t)
        torch._foreach_mul_(self.m, self.b1)
        torch._foreach_add_(self.m, grads, alpha=1.0 - self.b1)
        torch._foreach_mul_(self.v, self.b2)
        torch._foreach_addcmul_(self.v, grads, grads, value=1.0 - self.b2)
        denom = torch._foreach_sqrt(self.v)
        torch._foreach_add_(denom, self.eps)
        torch._foreach_addcdiv_(self.params, self.m, denom, value=-lr_t)


def loss_terms(params, planes, pol, val, training=True, probs=None):
    """The compiled Keras loss (model.py:68-72 + kernel_regularizer='l2' on every conv / dense layer):
    mean categorical cross-entropy(one-hot of the move played) + mean squared error(value, result) + 0.01 * sum w^2.
    probs: policy target rows [N, 1968] (search targets) in place of the one-hot of `pol`: the policy term is then
    mean(-sum_k probs_k log_softmax(logits)_k).  Returns (total, policy_loss, value_loss, regulariser, logits)."""
    logits, value = forward_logits(params, planes, training=training)
    if probs is None:
        loss_p = F.cross_entropy(logits, pol)
    else:
        loss_p = -(probs * F.log_softmax(logits, dim=1)).sum(dim=1).mean()
    loss_v = F.mse_loss(value, val)
    reg = sum((params[i] ** 2).sum() for i in _kernel_indices()) * L2
    return loss_p + loss_v + reg, loss_p, loss_v, reg, logits


def trainable_indices():
    """Everything but the BatchNorm moving statistics (those are updated by the forward pass, momentum 0.99)."""
    from .model import pack_shapes
    return [i for i, s in enumerate(pack_shapes()) if not (len(s) == 1 and _is_bn_running(i))]


def train_step(params, opt, planes, pol, val, probs=None):
    """One fit_generator batch: forward in training mode (BatchNorm batch statistics, moving statistics updated in
    place), backward, Adam.  probs: search-target policy rows (loss_terms).  Returns the history record of the batch;
    policy_acc is the argmax against the move played in every target mode."""
    total, loss_p, loss_v, reg, logits = loss_terms(params, planes, pol, val, training=True, probs=probs)
    grads = torch.autograd.grad(total, opt.params)
    opt.step(list(grads))
    acc = (logits.argmax(1) == pol).float().mean().item()
    return {"loss": total.item(), "policy_loss": loss_p.item(), "value_loss": loss_v.item(), "reg": reg.item(),
            "policy_acc": acc}


def validate(params, val_games, batch_size, dev, targets=None, first=0):
    """The validation generator of Agent.train (agent.py:73-75): `batch_size` games per batch, no flips; Keras
    averages the per-batch means over the batches.  targets: the training run's search targets (None: the move played);
    `first` is the dataset index of val_games[0], for error messages."""
    bs = max(1, min(batch_size, len(val_games)))
    sums, n = {"val_loss": 0.0, "val_policy_loss": 0.0, "val_value_loss": 0.0, "val_policy_acc": 0.0}, 0
    with torch.no_grad():
        for b in range(len(val_games) // bs):
            batch = val_games[b * bs:(b + 1) * bs]
            probs = None
            if targets is None:
                planes, pol, val = encode_games(batch, [False] * len(batch), dev)
            else:
                planes, pol, val, probs = encode_search_games(batch, [False] * len(batch), targets, first + b * bs)
            total, loss_p, loss_v, _, logits = loss_terms(params, planes, pol, val, training=False, probs=probs)
            sums["val_loss"] += total.item()
            sums["val_policy_loss"] += loss_p.item()
            sums["val_value_loss"] += loss_v.item()
            sums["val_policy_acc"] += (logits.argmax(1) == pol).float().mean().item()
            n += 1
    return {k: v / max(n, 1) for k, v in sums.items()}


def train(model, dataset, epochs=1, logdir=None, batch_size=1, validation_split=0, verbose=True, precision=None,
          targets=None):
    """targets: None (the move played and the game's result, the reference's targets) or a SearchTargets: search
    targets for the games that carry root scores, today's for the others (their number is reported)."""
    precision = resolve_precision(precision)
    targets = check_targets(targets)
    eng = runtime.scalar_engine()
    dev = eng.device
    games = list(dataset.games)
    val_games = []
    if validation_split > 0:
        split = len(games) - int(validation_split * len(games))
        games, val_games = games[:split], games[split:]
    # default: fp32 like the reference's CPU TensorFlow -- no TF32 convolutions / matmuls inside the training step
    with arithmetic(precision):
        params = [torch.tensor(w, device=dev, requires_grad=False) for w in model.weights]
        trainable = []
        for i in trainable_indices():
            params[i].requires_grad_(True)
            trainable.append(params[i])
        opt = KerasAdam(trainable, lr=0.002, epsilon=1e-7)
        bs = max(1, min(batch_size, len(games))) if games else 1
        history = []
        if targets is not None:
            rec = {"search_targets": {"temperature": targets.temperature, "value_weight": targets.value_weight,
                                      "games": len(games) + len(val_games),
                                      "games_without_scores": sum(g.search_scores is None for g in games + val_games)}}
            history.append(rec)
            if verbose:
                print("search targets (T %g, w %g): %d of %d games have no root scores and keep the played-move "
                      "targets" % (targets.temperature, targets.value_weight, rec["search_targets"]["games_without_scores"],
                                   rec["search_targets"]["games"]))
        for ep in range(epochs):
            order = list(range(len(games) // bs))
            random.shuffle(order)                    # fit_generator shuffles a Sequence's batch order every epoch
            for b in order:
                batch = games[b * bs:(b + 1) * bs]
                flips = draw_flips(len(batch), 0.1)                      # agent.py:82-84: random_flips=.1
                if targets is None:
                    planes, pol, val = encode_games(batch, flips, dev)
                    rec = train_step(params, opt, planes, pol, val)
                else:
                    planes, pol, val, probs = encode_search_games(batch, flips, targets, b * bs)
                    rec = train_step(params, opt, planes, pol, val, probs)
                rec.update({"epoch": ep, "batch": b})
                history.append(rec)
                if verbose:
                    print("epoch %d batch %d loss %.4f (policy %.4f value %.4f) acc %.3f" %
                          (ep, b, rec["loss"], rec["policy_loss"], rec["value_loss"], rec["policy_acc"]))
            if val_games:
                rec = validate(params, val_games, batch_size, dev, targets, len(games))
                rec["epoch"] = ep
                history.append(rec)
                if verbose:
                    print("epoch %d val_loss %.4f (policy %.4f value %.4f) val_acc %.3f" %
                          (ep, rec["val_loss"], rec["val_policy_loss"], rec["val_value_loss"], rec["val_policy_acc"]))
    model.weights = [p.detach().cpu().numpy().astype(np.float32) for p in params]
    if logdir is not None:
        import json
        import os
        os.makedirs(logdir, exist_ok=True)
        with open(os.path.join(logdir, "train_log.jsonl"), "a") as f:
            for h in history:
                f.write(json.dumps(h) + "\n")
    return history


def _is_bn_running(i):
    """True for moving_mean / moving_var tensors of the weight pack."""
    if 2 <= i < 122:
        j = (i - 2) % 6
        return j in (4, 5)
    if 124 <= i < 128:
        return i - 124 in (2, 3)
    if 132 <= i < 136:
        return i - 132 in (2, 3)
    return False
