"""CPU restatement of separable natural evolution strategies (SNES; Schaul, Glasmachers & Schmidhuber 2011,
"High Dimensions and Heavy Tails for Natural Evolution Strategies"; Wierstra et al., JMLR 2014): the checker of the
diag K5 / K6 and of the diag apply.  The search distribution of a role is N(mu, diag(sigma^2)).

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  The reference searches with one isotropic Gaussian per role and
moves its scalar sigma only through the ``--adaptive`` heuristic (evolutionary_strategy.py:292-316).

fp32 where the kernels are fp32 (numpy float32 arrays: one IEEE rounding per operation); the exp in fp64.
"""
from __future__ import annotations

import numpy as np


def default_sigma_lr(d):
    """SNES's learning rate of log sigma for d parameters: (3 + ln d) / (5 sqrt d), fp64."""
    return (3.0 + np.log(float(d))) / (5.0 * np.sqrt(float(d)))


def perturb(theta, sigma, z, pert_idx, row0=0, mirrored=False):
    """The rows ``cev_es_perturb_diag_f32`` writes: mu + fl(sigma * s z) on the perturbable entries, copies of mu
    elsewhere.  ``z`` fp32 [n, D] holds the normals of the members [row0, row0 + n) (s = 1), or under ``mirrored`` one
    row per member of its PAIR's normals z_{c >> 1}, s = +1 for even c and -1 for odd c.  Returns (rows, noise) with
    noise = s z on the perturbable entries."""
    theta = np.asarray(theta, dtype=np.float32)
    sigma = np.asarray(sigma, dtype=np.float32)
    z = np.asarray(z, dtype=np.float32)[:, pert_idx]
    if mirrored:
        c = np.arange(row0, row0 + z.shape[0])
        z = np.where((c & 1)[:, None] == 1, -z, z).astype(np.float32)
    rows = np.repeat(theta[None], z.shape[0], axis=0)
    rows[:, pert_idx] = theta[pert_idx] + sigma[pert_idx] * z
    return rows, z


def gradients(noise, fitness, n_total):
    """(g_mu, g_sigma) fp32 over the perturbable entries from the members' s z ``noise`` [n, d] and their fitness:
    fl32(1/n_total) * sum_i F_i z_i and fl32(1/n_total) * sum_i F_i (fl(z_i z_i) - 1), the sums in fp32 (not in the
    kernel's order)."""
    noise = np.asarray(noise, dtype=np.float32)
    f = np.asarray(fitness, dtype=np.float64).astype(np.float32)
    inv_n = np.float32(1.0 / n_total)
    zz = noise * noise - np.float32(1)
    return inv_n * (noise.T @ f), inv_n * (zz.T @ f)


def apply(theta, sigma, g_mu, g_sigma, pert_mask, lr, sigma_lr, sigma_min, sigma_max):
    """The diag apply (``cev_es_apply_diag_f32``) on the perturbable entries, the mu step with the old sigma:
    theta += fl(lr * fl(sigma * g_mu)); sigma = clamp(fl(sigma * fl32(exp(sigma_lr / 2 * g_sigma))), min, max), the
    exp and its argument in fp64, the clamp fmin(fmax(x, min), max).  ``sigma_lr``: a scalar or one value per entry.
    Returns new (theta, sigma)."""
    f32 = np.float32
    theta = np.asarray(theta, dtype=f32).copy()
    sigma = np.asarray(sigma, dtype=f32).copy()
    p = np.asarray(pert_mask, dtype=bool)
    half = 0.5 * np.broadcast_to(np.asarray(sigma_lr, dtype=np.float64), p.shape)[p]
    s = sigma[p]
    theta[p] = theta[p] + f32(lr) * (s * np.asarray(g_mu, dtype=f32)[p])
    factor = np.exp(half * np.asarray(g_sigma, dtype=f32)[p].astype(np.float64)).astype(f32)
    sigma[p] = np.fmin(np.fmax(s * factor, f32(sigma_min)), f32(sigma_max))
    return theta, sigma
