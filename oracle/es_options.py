"""CPU restatement of the opt-in Co-ES update options (the checker of the mirrored K5 / K6, the centered-rank kernel
and the fused apply): mirrored sampling, centered-rank fitness shaping and an Adam / L2 step (Salimans et al. 2017,
"Evolution Strategies as a Scalable Alternative to RL").

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  The reference has none of these: its update is SGD on raw
rewards with independent noise per member (evolutionary_strategy.py:120-148; the normalisation is commented out at
:133-135, the Adam optimizer of MPE/mpe_agent.py:20 is never used).
"""
from __future__ import annotations

import math

import numpy as np

#: Philox kind of the pair noise under mirrored sampling (member word = pair id); CEV_KIND_ES_MIRROR in the header
KIND_ES_MIRROR = 6

ADAM_BETA1, ADAM_BETA2, ADAM_EPS = 0.9, 0.999, 1e-8


def es_perturb_mirrored(theta, sigma, z_pairs, pert_idx, row0, n_rows):
    """Mirrored sampling (extends agent.py:31-70): global member c = theta + s*fl(sigma*z_q) on the perturbable
    entries, pair q = c >> 1, s = +1 for even c, -1 for odd c.  ``z_pairs`` fp32 [n_pairs, D] holds the normals of
    the pairs (row0 >> 1) .. ((row0 + n_rows - 1) >> 1).  Returns (rows, noise) for members row0 .. row0+n_rows-1,
    ``noise = s*fl(sigma*z)`` as in ``ga_es.es_perturb``."""
    theta = np.asarray(theta, dtype=np.float32)
    z = np.asarray(z_pairs, dtype=np.float32)
    c = np.arange(row0, row0 + n_rows)
    d = (np.float32(sigma) * z[(c >> 1) - (row0 >> 1)][:, pert_idx]).astype(np.float32)
    noise = np.where((c & 1)[:, None] == 1, -d, d).astype(np.float32)
    rows = np.repeat(theta[None], n_rows, axis=0)
    rows[:, pert_idx] = theta[pert_idx] + noise
    return rows, noise


def rank_keys(fitness):
    """Order-preserving uint64 keys of fp64 values: -0.0 -> +0.0, every NaN -> 0 (below -inf)."""
    f = np.asarray(fitness, dtype=np.float64)
    b = f.view(np.uint64).copy()
    b[f == 0] = 0
    neg = (b >> np.uint64(63)) == 1
    k = np.where(neg, ~b, b | np.uint64(1 << 63))
    k[np.isnan(f)] = 0
    return k


def centered_ranks(fitness):
    """Centered-rank fitness shaping: u_i = r_i / (P-1) - 0.5 (0 when P = 1) with the average rank
    r_i = #{F_j < F_i} + (#{F_j == F_i} - 1) / 2.  -0.0 == +0.0; all NaNs tie and rank below every number."""
    k = rank_keys(fitness)
    P = len(k)
    if P == 1:
        return np.zeros(1)
    s = np.sort(k)
    lt = np.searchsorted(s, k, side="left")
    eq = np.searchsorted(s, k, side="right") - lt
    r = lt.astype(np.float64) + 0.5 * (eq - 1).astype(np.float64)
    return r / float(P - 1) - 0.5


def es_apply(theta, delta, pert_mask, optimizer, lr, l2_coeff=0.0, t=1, m=None, v=None):
    """The fused ES apply (``cev_es_apply_f32``) in float32, one IEEE rounding per operation:
    g = delta - l2*theta; sgd: theta += lr*g; adam: m = b1 m + (1-b1) g, v = b2 v + ((1-b2) g) g,
    theta += (alpha_t m) / (sqrt(v) + eps), alpha_t = lr sqrt(1-b2^t)/(1-b1^t) in fp64 rounded to fp32.
    Only entries where ``pert_mask`` is set change.  Returns new (theta, m, v) arrays."""
    f32 = np.float32
    theta = np.asarray(theta, dtype=f32).copy()
    delta = np.asarray(delta, dtype=f32)
    p = np.asarray(pert_mask, dtype=bool)
    th = theta[p]
    g = delta[p] - f32(l2_coeff) * th
    if optimizer == "sgd":
        theta[p] = th + f32(lr) * g
        return theta, m, v
    m = np.asarray(m, dtype=f32).copy()
    v = np.asarray(v, dtype=f32).copy()
    b1, b2 = f32(ADAM_BETA1), f32(ADAM_BETA2)
    alpha = f32(lr * math.sqrt(1.0 - math.pow(ADAM_BETA2, t)) / (1.0 - math.pow(ADAM_BETA1, t)))
    mi = b1 * m[p] + (f32(1) - b1) * g
    vi = b2 * v[p] + ((f32(1) - b2) * g) * g
    m[p], v[p] = mi, vi
    theta[p] = th + (alpha * mi) / (np.sqrt(vi) + f32(ADAM_EPS))
    return theta, m, v
