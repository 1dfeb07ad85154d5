"""Checker backend of the engines WITH the opt-in Co-ES update options: everything ``tests/oracle_backend.py``
provides, plus the mirrored K5 / K6, the centered-rank transform and the fused apply restated with
``oracle/es_options.py`` on torch CPU tensors.

TEST-ONLY, like oracle_backend: it lets the gloo tests exercise the engine's option logic without a GPU.
"""
import numpy as np
import torch

from coevonet_b200 import layout
from oracle import es_options as oes, layout as olayout, philox
from oracle_backend import *  # noqa: F401,F403  (the call signatures of coevonet_b200.ops the engine uses)


def _pairs(row0, n_rows):
    return np.arange(row0 >> 1, ((row0 + n_rows - 1) >> 1) + 1) if n_rows else np.zeros(0, dtype=np.int64)


def es_perturb_mirrored(theta, in_dim, sigma, seed, role, gen, row0, n_rows, *, out=None, noise_out=None):
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    D = layout.fc_dim(in_dim)
    pidx = olayout.fc_perturbable_index(in_dim)
    z = philox.normals(seed, oes.KIND_ES_MIRROR, role_id, gen, _pairs(row0, n_rows), D)
    rows, _ = oes.es_perturb_mirrored(theta.numpy()[:D], float(sigma), z, pidx, row0, n_rows)
    res = torch.zeros((n_rows, layout.fc_pitch(in_dim)), dtype=torch.float32) if out is None else out
    res[:, :D] = torch.from_numpy(rows)
    res[:, D:] = 0
    return res


def es_update_mirrored(fitness, in_dim, sigma, lr, n_total, seed, role, gen, row0, *, out=None):
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    sigma = float(sigma)
    D = layout.fc_dim(in_dim)
    pidx = olayout.fc_perturbable_index(in_dim)
    n = fitness.shape[0]
    z = philox.normals(seed, oes.KIND_ES_MIRROR, role_id, gen, _pairs(row0, n), D)
    _, noise = oes.es_perturb_mirrored(np.zeros(D, np.float32), sigma, z, pidx, row0, n)
    f = fitness.numpy().astype(np.float32)
    coef = np.float32(lr / (n_total * sigma))
    delta = np.zeros(layout.fc_pitch(in_dim), dtype=np.float32)
    delta[pidx] = coef * (noise.T @ f)
    res = torch.from_numpy(delta)
    if out is not None:
        out.copy_(res)
        return out
    return res


def centered_ranks(fitness, row0=0, n_rows=None, *, out=None):
    n_rows = fitness.shape[0] - row0 if n_rows is None else n_rows
    return torch.from_numpy(oes.centered_ranks(fitness.numpy())[row0:row0 + n_rows].copy())


def es_apply(theta, delta, in_dims, *, optimizer="sgd", lr, l2_coeff=0.0, t=1, m=None, v=None):
    mask = np.concatenate([np.isin(np.arange(layout.fc_pitch(d)), olayout.fc_perturbable_index(d)) for d in in_dims])
    th, mm, vv = oes.es_apply(theta.numpy(), delta.numpy(), mask, optimizer, lr, l2_coeff, t,
                              None if m is None else m.numpy(), None if v is None else v.numpy())
    theta.copy_(torch.from_numpy(th))
    if optimizer == "adam":
        m.copy_(torch.from_numpy(mm))
        v.copy_(torch.from_numpy(vv))
    return theta
