"""NumPy restatement of ``DeepQN.forward`` (K2's checker).

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  Follows
/root/reference/Atari/deepqn.py:39-48 at the batch size the reference uses
(1): the "virtual batch norm" layers are plain ``BatchNorm2d`` in TRAIN mode
(SURVEY.md Appendix C #12), so statistics are per frame over H x W, biased
variance, eps 1e-5, affine gamma/beta.  Pinned against the reference module by
``oracle/make_golden.py``.

``dtype=np.float64`` runs every layer in float64 on the same float32 weights and
the same float32 input the model sees (``u8 / 255`` rounded to float32), with eps
float32(1e-5): a reference whose own rounding is ~1e-16 relative, so a kernel's
error against it is the kernel's alone.  The default ``np.float32`` is the
reference's own arithmetic.
"""
from __future__ import annotations

import numpy as np

from . import layout

BN_EPS = np.float32(1e-5)


def _conv2d(x, w, b, stride):
    """x [C,H,W], w fp32[O,C,kh,kw] -> [O,Ho,Wo] (valid padding) in the dtype of x."""
    dt = x.dtype
    C, H, W = x.shape
    O, _, kh, kw = w.shape
    Ho = (H - kh) // stride + 1
    Wo = (W - kw) // stride + 1
    s0, s1, s2 = x.strides
    cols = np.lib.stride_tricks.as_strided(
        x, shape=(Ho, Wo, C, kh, kw),
        strides=(s1 * stride, s2 * stride, s0, s1, s2), writeable=False)
    cols = cols.reshape(Ho * Wo, C * kh * kw).astype(dt)
    out = cols @ w.reshape(O, -1).T.astype(dt) + b.astype(dt)
    return out.T.reshape(O, Ho, Wo).astype(dt)


def _bn_train(x, g, b):
    """Per-frame train-mode BatchNorm2d: stats over H x W per channel."""
    if x.dtype == np.float32:
        mean = x.mean(axis=(1, 2), keepdims=True, dtype=np.float32)
    else:
        # shifted by the channel's first value, so a constant channel has exactly zero deviation and
        # variance and normalises to exactly beta
        x0 = x[:, :1, :1]
        mean = x0 + (x - x0).mean(axis=(1, 2), keepdims=True)
    xc = x - mean
    var = (xc * xc).mean(axis=(1, 2), keepdims=True, dtype=x.dtype)
    return xc / np.sqrt(var + BN_EPS) * g[:, None, None] + b[:, None, None]


def dqn_layers(row, frame, c_in, n_actions, dtype=np.float32):
    """Every stage of the forward for one frame, in order: conv1 (before BatchNorm), layer 1 (after
    BatchNorm + ReLU), conv2, layer 2, conv3, layer 3, fc1 (after ReLU), logits [A]."""
    dt = np.dtype(dtype)
    p = layout.unpack_dqn(np.asarray(row, dtype=np.float32), c_in, n_actions)
    if dt != np.float32:
        p = {k: v.astype(dt) for k, v in p.items()}
    x = (np.asarray(frame, dtype=np.float32) / np.float32(255)).astype(dt)
    out = []
    for i, stride in ((1, 4), (2, 2), (3, 1)):
        y = _conv2d(x, p[f"conv{i}.weight"], p[f"conv{i}.bias"], stride)
        x = np.maximum(_bn_train(y, p[f"vbn{i}.weight"], p[f"vbn{i}.bias"]), 0)
        out += [y, x]
    x = x.reshape(-1).astype(dt)
    x = np.maximum(p["fc1.weight"] @ x + p["fc1.bias"], 0)
    out += [x, (p["output.weight"] @ x + p["output.bias"]).astype(dt)]
    return out


def dqn_forward(row, frame, c_in, n_actions, dtype=np.float32):
    """Logits [A] in ``dtype`` for one frame (uint8 or float [C,84,84])."""
    return dqn_layers(row, frame, c_in, n_actions, dtype)[-1]


def dqn_forward_batch(rows, frames, c_in, n_actions, dtype=np.float32):
    """rows fp32[P,D], frames [P,B,C,84,84] -> (logits [P,B,A] in ``dtype``, actions int32[P,B])
    with the reference's first-maximum argmax (Atari/deepqn.py:55-60)."""
    P, B = frames.shape[:2]
    logits = np.zeros((P, B, n_actions), dtype=dtype)
    for m in range(P):
        for f in range(B):
            logits[m, f] = dqn_forward(rows[m], frames[m, f], c_in, n_actions, dtype)
    return logits, np.argmax(logits, axis=-1).astype(np.int32)
