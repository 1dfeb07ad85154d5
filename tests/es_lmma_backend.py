"""Checker backend of the ES engine with LM-MA-ES: everything ``tests/es_subspace_backend.py`` provides, plus the
projection, the LM-MA K5, the recombination and the apply restated with ``oracle/es_lmma.py`` on torch CPU tensors.

TEST-ONLY, like oracle_backend: it lets the gloo tests exercise the engine's LM-MA-ES path without a GPU.
"""
import numpy as np
import torch

from coevonet_b200 import layout
from oracle import es_lmma as olm, layout as olayout
from es_subspace_backend import *  # noqa: F401,F403  (the call signatures of coevonet_b200.ops the engine uses)
from snes_backend import _normals


def _z(seed, role, gen, row0, n_rows, in_dim):
    """Normals of the members [row0, row0 + n_rows) on the Linear entries, zero elsewhere, fp32 [n_rows, fc_dim]."""
    D = layout.fc_dim(in_dim)
    z = _normals(seed, role, gen, row0, n_rows, D, False)
    mask = np.zeros(D, bool)
    mask[olayout.fc_perturbable_index(in_dim)] = True
    return np.where(mask[None, :], z, np.float32(0)).astype(np.float32)


def es_lmma_project(M, k, G, cd, in_dim, seed, role, gen, row0, n_rows, *, beta=None, s_out=None, status=None):
    D = layout.fc_dim(in_dim)
    z = _z(seed, role, gen, row0, n_rows, in_dim)
    s = olm.project(M.numpy()[:k, :D], z, k)
    _, b = olm.transform_compact(s, G.numpy(), k, list(cd))
    b32 = b.astype(np.float32)
    if status is not None and not (np.all(np.isfinite(s)) and np.all(np.isfinite(b32))):
        status.fill_(status.item() | 1)
    res = torch.from_numpy(b32)
    if beta is not None:
        beta.copy_(res)
        res = beta
    if s_out is not None:
        s_out.copy_(torch.from_numpy(s))
    return res


def es_perturb_lmma(theta, in_dim, sigma, M, k, beta, alpha, seed, role, gen, row0, n_rows, *, out=None):
    D = layout.fc_dim(in_dim)
    z = _normals(seed, role, gen, row0, n_rows, D, False)
    rows = olm.perturb(theta.numpy()[:D], np.float32(float(sigma)), M.numpy()[:k, :D], beta.numpy(), alpha, z,
                       olayout.fc_perturbable_index(in_dim))
    res = torch.zeros((n_rows, layout.fc_pitch(in_dim)), dtype=torch.float32) if out is None else out
    res[:, :D] = torch.from_numpy(rows)
    res[:, D:] = 0
    return res


def es_lmma_reduce(ids, w, beta, in_dim, seed, role, gen, row0, n_rows, *, zbar=None, betabar=None):
    pitch = layout.fc_pitch(in_dim)

    def z_of(i):
        row = np.zeros(pitch, np.float32)
        row[:layout.fc_dim(in_dim)] = _z(seed, role, gen, i, 1, in_dim)[0]
        return row
    zb, bb = olm.reduce(ids.numpy(), w.numpy(), z_of, beta.numpy(), row0, n_rows)
    zbar = torch.empty(pitch, dtype=torch.float32) if zbar is None else zbar
    betabar = torch.empty(beta.shape[1], dtype=torch.float32) if betabar is None else betabar
    zbar.copy_(torch.from_numpy(zb))
    betabar.copy_(torch.from_numpy(bb))
    return zbar, betabar


def es_lmma_apply(theta, M, p, zbar, betabar, in_dims, *, k, alpha, c_sigma, mu_w, c_m, c_c, G, gstate, sigma_min,
                  sigma_max, stats=None, status=None):
    from coevonet_b200 import _lib
    stats = torch.empty((len(in_dims), 2), dtype=torch.float64) if stats is None else stats
    th, Mn, pn = theta.numpy().copy(), M.numpy().copy(), p.numpy().copy()
    bb = betabar.numpy().reshape(len(in_dims), -1)
    start = 0
    for s, d in enumerate(in_dims):
        sl = slice(start, start + layout.fc_pitch(d))
        pidx = olayout.fc_perturbable_index(d)
        const = {"c_sigma": c_sigma[s], "mu_w": mu_w[s], "c_c": list(c_c[s])}
        sigma = float(gstate[_lib.GS_SIGMA + s])
        t, Mr, pr, Gs, v, new = olm.apply(th[sl], Mn[:, sl], pn[sl], zbar.numpy()[sl], bb[s], k, alpha[s], sigma, c_m,
                                          const, len(pidx), pidx, sigma_min, sigma_max)
        th[sl], Mn[:, sl], pn[sl] = t, Mr, pr
        G[s].copy_(torch.from_numpy(Gs))
        if not (np.isfinite(v) and np.all(np.isfinite(Gs))) and status is not None:
            status.fill_(status.item() | 1)
        gstate[_lib.GS_SIGMA + s] = new
        stats[s, 0], stats[s, 1] = v, new
        start = sl.stop
    theta.copy_(torch.from_numpy(th))
    M.copy_(torch.from_numpy(Mn))
    p.copy_(torch.from_numpy(pn))
    return stats
