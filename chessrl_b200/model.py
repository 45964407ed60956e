"""ChessModel: the weight container behind the policy/value ResNet of the reference (model.py:15-122).

The forward pass runs in libchessrl_b200.so (tcgen05 convolutions); this class only owns the fp32 master
weights as the 140-tensor "weight pack" in Keras layouts and (de)serialises them.  Architecture (model.py:31-63):
input 8x8x127 -> conv3x3x256 (bias, no BN, no activation) -> 10 residual blocks [conv3x3+bias, BN, ReLU,
conv3x3+bias, BN, +skip, ReLU] -> policy head [conv1x1x2, BN, ReLU, flatten, Dense 1968 softmax] and value head
[conv1x1x1, BN, ReLU, flatten, Dense 256 ReLU, Dense 1 tanh].

Weight pack order (conv kernels HWIO, dense kernels [in][out], BN = gamma, beta, moving_mean, moving_var):
  0-1      stem conv kernel [3,3,127,256], bias
  2+12b..  block b (0..9): conv_a kernel, bias, BN x4, conv_b kernel, bias, BN x4
  122-129  policy: conv kernel [1,1,256,2], bias, BN x4, dense kernel [128,1968], bias
  130-139  value: conv kernel [1,1,256,1], bias, BN x4, dense kernel [64,256], bias, dense kernel [256,1], bias
"""

from __future__ import annotations

import itertools
import os

import numpy as np

_SERIAL = itertools.count(1)     # process-wide: every weight assignment gets a new serial (never reused, unlike id())
_HDF5_MAGIC = b"\x89HDF\r\n\x1a\n"

N_BLOCKS = 10
N_FILTERS = 256
N_TENSORS = 140
N_PARAMS = 12386496


def pack_shapes():
    s = [(3, 3, 127, 256), (256,)]
    for _ in range(N_BLOCKS):
        for _ in range(2):
            s += [(3, 3, 256, 256), (256,), (256,), (256,), (256,), (256,)]
    s += [(1, 1, 256, 2), (2,), (2,), (2,), (2,), (2,), (128, 1968), (1968,)]
    s += [(1, 1, 256, 1), (1,), (1,), (1,), (1,), (1,), (64, 256), (256,), (256, 1), (1,)]
    assert len(s) == N_TENSORS
    return s


def _glorot(rng, shape):
    if len(shape) == 4:
        rf = shape[0] * shape[1]
        fan_in, fan_out = shape[2] * rf, shape[3] * rf
    else:
        fan_in, fan_out = shape
    lim = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


def random_pack(seed=0, perturb_bn=False):
    """Keras-default initialisation: glorot_uniform kernels, zero biases, BN gamma 1 / beta 0 / mean 0 / var 1.
    perturb_bn=True randomises biases and BatchNorm statistics as a trained net would have (tests)."""
    rng = np.random.default_rng(seed)
    out = []
    shapes = pack_shapes()
    i = 0
    while i < len(shapes):
        sh = shapes[i]
        if len(sh) >= 2:                      # kernel followed by its bias
            out.append(_glorot(rng, sh))
            b = np.zeros(shapes[i + 1], np.float32)
            if perturb_bn:
                b = rng.normal(0, 0.05, shapes[i + 1]).astype(np.float32)
            out.append(b)
            i += 2
        else:                                 # BatchNorm quadruple
            n = sh[0]
            if perturb_bn:
                out += [rng.uniform(0.5, 1.5, n).astype(np.float32), rng.normal(0, 0.1, n).astype(np.float32),
                        rng.normal(0, 0.1, n).astype(np.float32), rng.uniform(0.5, 1.5, n).astype(np.float32)]
            else:
                out += [np.ones(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32), np.ones(n, np.float32)]
            i += 4
    return out


def calibration_planes(engine, n=256, seed=0, max_plies=80):
    """The default fp8 calibration set (Engine.load_weights(precision="fp8")): bf16 planes [n,8,8,128] of `n` positions
    reached by seeded uniformly random legal playouts of 0..max_plies plies from the start position, encoded with their
    history like netencoder.get_game_state.  Depends only on (n, seed, max_plies)."""
    import torch
    from . import boards as B
    rng = np.random.default_rng(seed)
    start = B.record_from_fen()
    cur = np.zeros((9, n), dtype=np.uint64)
    hist = np.zeros((8, 8, n), dtype=np.uint64)
    hist_len = np.zeros(n, dtype=np.uint8)
    for i in range(n):
        target = int(rng.integers(0, max_plies + 1))
        moves = []
        r = engine.game_replay(start, moves, records=True)
        while len(moves) < target and r["result"] is None and len(r["legal"]):
            moves.append(int(r["legal"][int(rng.integers(0, len(r["legal"])))]))
            r = engine.game_replay(start, moves, records=True)
        recs = r["records"][::-1][:9]
        cur[:, i] = recs[0]
        for j, rec in enumerate(recs[1:]):
            hist[j, :, i] = rec[:8]
        hist_len[i] = len(recs) - 1
    dev = engine.device
    return engine.encode(torch.from_numpy(cur.view(np.int64)).to(dev), torch.from_numpy(hist.view(np.int64)).to(dev),
                         torch.from_numpy(hist_len).to(dev))


class ChessModel(object):
    """Same constructor surface as the reference (model.py:17): ChessModel(compile_model=True, weights=None)."""

    def __init__(self, compile_model=True, weights=None, seed=0):
        self.weights = random_pack(seed)
        if weights:
            self.load_weights(weights)

    @property
    def weights(self):
        return self._weights

    @weights.setter
    def weights(self, pack):
        """Assigning a pack (constructor, load_weights, the training step, a broadcast) bumps `serial`, the token the
        engines compare to decide whether their device copy is current (runtime.ensure_weights)."""
        self._weights = pack
        self.serial = next(_SERIAL)

    @property
    def version(self):          # older name of the token
        return self.serial

    @version.setter
    def version(self, _):
        self.serial = next(_SERIAL)

    def n_params(self):
        return int(sum(w.size for w in self.weights))

    def load_weights(self, weights_path):
        if not os.path.exists(weights_path):
            raise OSError("weights file not found: %s" % weights_path)      # supervised.py:57-59 catches OSError
        with open(weights_path, "rb") as f:
            magic = f.read(8)
        if magic == _HDF5_MAGIC:
            # a real Keras checkpoint of the reference (model.py:77-81): needs h5py, which this image does not have;
            # scripts/export_keras_weights.py converts it on the reference side
            from .keras_h5 import load_keras_h5
            w = load_keras_h5(weights_path)
        else:
            with np.load(weights_path) as z:
                w = [z["w%03d" % i].astype(np.float32) for i in range(N_TENSORS)]
        for a, sh in zip(w, pack_shapes()):
            if tuple(a.shape) != tuple(sh):
                raise ValueError("weight shape mismatch %s vs %s" % (a.shape, sh))
        self.weights = w

    def save_weights(self, weights_path):
        with open(weights_path, "wb") as f:       # keep the caller's file name (model-<n>.h5 in the reference)
            np.savez(f, **{"w%03d" % i: w for i, w in enumerate(self.weights)})
