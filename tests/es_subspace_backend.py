"""Checker backend of the ES engine with guided search: everything ``tests/es_hof_backend.py`` provides, plus the
subspace K5 and the basis restated with ``oracle/es_subspace.py`` on torch CPU tensors.

TEST-ONLY, like oracle_backend: it lets the gloo tests exercise the engine's guided-search path without a GPU.
"""
import numpy as np
import torch

from coevonet_b200 import layout
from oracle import es_subspace as oss, layout as olayout
from es_hof_backend import *  # noqa: F401,F403  (the call signatures of coevonet_b200.ops the engine uses)
from snes_backend import _normals


def es_perturb_subspace(theta, in_dim, sigma, U, k_eff, alpha, seed, role, gen, row0, n_rows, *, mirrored=False,
                        out=None, noise_out=None, coef_out=None):
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    D, k = layout.fc_dim(in_dim), U.shape[0]
    ke = int(k_eff[0])
    z = _normals(seed, role, gen, row0, n_rows, D, mirrored)
    c = np.zeros((n_rows, k), np.float32)
    if n_rows:
        units = np.arange(row0, row0 + n_rows)
        units = units >> 1 if mirrored else units
        c = oss.coefficients(seed, role_id, gen, units, k)
    rows, _ = oss.perturb(theta.numpy()[:D], float(sigma), U.numpy()[:, :D], ke, float(alpha), z, c,
                          olayout.fc_perturbable_index(in_dim), row0, mirrored)
    res = torch.zeros((n_rows, layout.fc_pitch(in_dim)), dtype=torch.float32) if out is None else out
    res[:, :D] = torch.from_numpy(rows)
    res[:, D:] = 0
    return res


def es_subspace_basis(ring, newest, filled, in_dims, *, out=None, k_eff=None):
    segs, start = [], 0
    for d in in_dims:
        segs.append((start, start + layout.fc_pitch(d), olayout.fc_perturbable_index(d)))
        start += layout.fc_pitch(d)
    U, ke = oss.ring_basis(ring.numpy(), newest, filled, segs)
    out = torch.empty_like(ring) if out is None else out
    k_eff = torch.empty(len(in_dims), dtype=torch.int32) if k_eff is None else k_eff
    out.copy_(torch.from_numpy(U))
    k_eff.copy_(torch.tensor(ke, dtype=torch.int32))
    return out, k_eff
