"""Checker backend of the ES engine with separable NES: everything ``tests/es_options_backend.py`` provides, plus the
diag K5 / K6 and the diag apply restated with ``oracle/snes.py`` on torch CPU tensors.

TEST-ONLY, like oracle_backend: it lets the gloo tests exercise the engine's separable path without a GPU.
"""
import numpy as np
import torch

from coevonet_b200 import layout
from oracle import es_options as oes, layout as olayout, philox, snes
from es_options_backend import *  # noqa: F401,F403  (the call signatures of coevonet_b200.ops the engine uses)


def _normals(seed, role, gen, row0, n_rows, D, mirrored):
    """One row of normals per member [row0, row0 + n_rows): its own, or under mirroring its pair's."""
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    c = np.arange(row0, row0 + n_rows)
    if not mirrored:
        return philox.normals(seed, philox.KIND_ES, role_id, gen, c, D)
    if n_rows == 0:
        return np.zeros((0, D), np.float32)
    q0 = row0 >> 1
    z = philox.normals(seed, oes.KIND_ES_MIRROR, role_id, gen, np.arange(q0, ((row0 + n_rows - 1) >> 1) + 1), D)
    return z[(c >> 1) - q0]


def es_perturb_diag(theta, sigma, in_dim, seed, role, gen, row0, n_rows, *, mirrored=False, out=None, noise_out=None):
    D = layout.fc_dim(in_dim)
    z = _normals(seed, role, gen, row0, n_rows, D, mirrored)
    rows, _ = snes.perturb(theta.numpy()[:D], sigma.numpy()[:D], z, olayout.fc_perturbable_index(in_dim), row0,
                           mirrored)
    res = torch.zeros((n_rows, layout.fc_pitch(in_dim)), dtype=torch.float32) if out is None else out
    res[:, :D] = torch.from_numpy(rows)
    res[:, D:] = 0
    return res


def es_update_diag(fitness, in_dim, n_total, seed, role, gen, row0, *, mirrored=False, g_mu=None, g_sigma=None):
    D, pitch = layout.fc_dim(in_dim), layout.fc_pitch(in_dim)
    pidx = olayout.fc_perturbable_index(in_dim)
    n = fitness.shape[0]
    z = _normals(seed, role, gen, row0, n, D, mirrored)
    _, noise = snes.perturb(np.zeros(D, np.float32), np.zeros(D, np.float32), z, pidx, row0, mirrored)
    gm, gs = snes.gradients(noise, fitness.numpy(), n_total)
    outs = []
    for g, dst in ((gm, g_mu), (gs, g_sigma)):
        full = np.zeros(pitch, dtype=np.float32)
        full[pidx] = g
        if dst is None:
            dst = torch.empty(pitch, dtype=torch.float32)
        dst.copy_(torch.from_numpy(full))
        outs.append(dst)
    return tuple(outs)


def es_apply_diag(theta, sigma, g_mu, g_sigma, in_dims, *, lr, sigma_lr, sigma_min, sigma_max):
    mask = np.concatenate([np.isin(np.arange(layout.fc_pitch(d)), olayout.fc_perturbable_index(d)) for d in in_dims])
    eta = np.concatenate([np.full(layout.fc_pitch(d), float(e)) for d, e in zip(in_dims, sigma_lr)])
    th, sg = snes.apply(theta.numpy(), sigma.numpy(), g_mu.numpy(), g_sigma.numpy(), mask, lr, eta, sigma_min,
                        sigma_max)
    theta.copy_(torch.from_numpy(th))
    sigma.copy_(torch.from_numpy(sg))
    return theta, sigma
