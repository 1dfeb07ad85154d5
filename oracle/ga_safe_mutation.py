"""CPU restatement of the Co-GA safe mutations through output gradients (the checker of ``cev_ga_safe_scale_f32``,
``cev_ga_repopulate_safe_f32`` and of the GA engine's safe-mutation path): the sensitivity of every parameter by
explicit backpropagation in fp64, the scale rule, and the children.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  SM-G-SUM follows Lehman, Chen, Clune & Stanley, "Safe Mutations for
Deep and Recurrent Neural Networks through Output Gradients" (GECCO 2018): with y_k(x_t) the logits of the FCNetwork
on the probe observations x_t of the novelty search (``oracle/es_novelty.py``),
    G_kj = sum_t dy_k(x_t) / dW_j,   s_j = sqrt(sum_k G_kj^2),   c_j = 1 if s_j == 0 else fl32(1 / max(s_j, floor)),
and child c >= 1 of elite e is fl(p_j + fl(fl(sigma z_j) c_j)).  The zero rule and the floor are this project's.
"""
from __future__ import annotations

import numpy as np

from . import ga_es, layout

LN_EPS = float(np.float32(1e-5))
N_ACTIONS = 5


def _ln_forward(h):
    mu = h.mean(axis=-1, keepdims=True)
    xc = h - mu
    rstd = 1.0 / np.sqrt((xc * xc).mean(axis=-1, keepdims=True) + LN_EPS)
    return xc * rstd, rstd


def _ln_backward(dxh, xh, rstd):
    """d(input) of a LayerNorm from d(xhat) (biased variance): rstd (dxh - mean(dxh) - xhat mean(dxh xhat))."""
    return rstd * (dxh - dxh.mean(axis=-1, keepdims=True) - xh * (dxh * xh).mean(axis=-1, keepdims=True))


def _ln_backward_abs(dxh, xh, rstd):
    """The same chain with absolute values (no cancellation): a bound on the magnitude of the terms."""
    return rstd * (dxh + dxh.mean(axis=-1, keepdims=True) + np.abs(xh) * (dxh * np.abs(xh)).mean(axis=-1, keepdims=True))


def _chain(row, in_dim, obs, absolute):
    """G fp64 [5, D] of one row (``absolute``: the chain with |.| at every step) and the smallest |ReLU input|."""
    p = {k: v.astype(np.float64) for k, v in layout.unpack_fc(np.asarray(row, np.float32), in_dim).items()}
    ab = np.abs if absolute else (lambda v: v)
    back = _ln_backward_abs if absolute else _ln_backward
    x = np.asarray(obs, np.float32).astype(np.float64)                 # [T, in]
    T = x.shape[0]
    xh1, r1 = _ln_forward(x @ p["fc1.weight"].T + p["fc1.bias"])
    y1 = xh1 * p["ln1.weight"] + p["ln1.bias"]
    m1 = y1 > 0
    a1 = np.where(m1, y1, 0.0)
    xh2, r2 = _ln_forward(a1 @ p["fc2.weight"].T + p["fc2.bias"])
    y2 = xh2 * p["ln2.weight"] + p["ln2.bias"]
    m2 = y2 > 0
    a2 = np.where(m2, y2, 0.0)
    margin = min(np.abs(y1).min(), np.abs(y2).min())
    K = N_ACTIONS
    eye = np.eye(K)
    g_outw = eye[:, :, None] * a2.sum(axis=0)[None, None, :]          # [k, k', i]
    g_outb = eye * T
    dy2 = m2[None] * ab(p["output.weight"])[:, None, :]                 # [k, t, 256]
    dz2 = back(dy2 * ab(p["ln2.weight"]), xh2[None], r2[None])
    g_ln2g = (dy2 * ab(xh2)[None]).sum(axis=1)
    g_ln2b = dy2.sum(axis=1)
    g_b2 = dz2.sum(axis=1)
    g_w2 = np.einsum("kti,tj->kij", dz2, a1)
    da1 = np.einsum("kti,ij->ktj", dz2, ab(p["fc2.weight"]))
    dy1 = m1[None] * da1
    dz1 = back(dy1 * ab(p["ln1.weight"]), xh1[None], r1[None])
    g_ln1g = (dy1 * ab(xh1)[None]).sum(axis=1)
    g_ln1b = dy1.sum(axis=1)
    g_b1 = dz1.sum(axis=1)
    g_w1 = np.einsum("ktj,ti->kji", dz1, ab(x))
    parts = [g_w1, g_b1, g_ln1g, g_ln1b, g_w2, g_b2, g_ln2g, g_ln2b, g_outw, g_outb]
    return np.concatenate([g.reshape(K, -1) for g in parts], axis=1), margin


def gradients(row, in_dim, obs):
    """G fp64 [5, D]: the sum over the probes of the gradient of each logit, by explicit backpropagation in fp64 from
    the fp32 row (ReLU' = [input > 0]; LayerNorm with the biased variance and eps = fl32(1e-5))."""
    return _chain(row, in_dim, obs, False)[0]


def sensitivity(row, in_dim, obs):
    """(s, magnitude, margin): s fp64 [D] = sqrt(sum_k G_kj^2); magnitude fp64 [D], the same chain with absolute
    values (the size of the terms a float32 evaluation rounds, for tolerances); margin, the smallest |ReLU input|
    over both hidden layers and all probes (below it a float32 forward may take the other side of a ReLU)."""
    G, margin = _chain(row, in_dim, obs, False)
    Ga, _ = _chain(row, in_dim, obs, True)
    return np.sqrt((G * G).sum(axis=0)), np.sqrt((Ga * Ga).sum(axis=0)), float(margin)


def scale_from_s(s, floor):
    """c fp32: 1 where s == 0, else fl32(1 / max(fl32(s), fl32(floor)))."""
    s32 = np.asarray(s).astype(np.float32)
    c = np.float32(1.0) / np.maximum(s32, np.float32(floor))
    return np.where(s32 == 0, np.float32(1.0), c).astype(np.float32)


def scale_rows(rows, in_dim, obs, floor, pitch=None):
    """fp32 [E, pitch]: the scale rows of ``rows`` fp32 [E, >= D] (padding 0)."""
    D = layout.fc_dim(in_dim)
    rows = np.asarray(rows, np.float32)
    out = np.zeros((rows.shape[0], pitch or rows.shape[1]), np.float32)
    for e, r in enumerate(rows):
        out[e, :D] = scale_from_s(sensitivity(r[:D], in_dim, obs)[0], floor)
    return out


def children(elites, scale, sigma, z, members, crossover_rate=0.0, seed=0, role_id=0, gen=0):
    """Rows ``members`` (global ids) of the next population, fp32 [n, D]: child 0 = elites[0]; child c >= 1 takes
    parameter j (with crossover, from elite A or B under ``ga_es.ga_repopulate_crossover``'s mask) as
    fl(p_j + fl(fl(sigma z_j) c_j)), p and c from the same elite.  ``z`` fp32 [n, D] (the K3 normals)."""
    elites = np.asarray(elites, np.float32)
    E, D = elites.shape
    scale = np.asarray(scale, np.float32)[:, :D]
    # which elite each parameter comes from: the crossover of rows that hold their own index, unmutated
    ids = np.repeat(np.arange(E, dtype=np.float32)[:, None], D, axis=1)
    src = ga_es.ga_repopulate_crossover(ids, 0.0, np.zeros((len(members), D), np.float32), crossover_rate, seed,
                                        role_id, gen, members).astype(np.int64)
    cols = np.arange(D)[None, :]
    p, c = elites[src, cols], scale[src, cols]
    d = ((np.float32(sigma) * np.asarray(z, np.float32)[:, :D]).astype(np.float32) * c).astype(np.float32)
    out = (p + d).astype(np.float32)
    out[np.asarray(members) == 0] = elites[0]
    return out
