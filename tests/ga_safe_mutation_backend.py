"""Checker backend of the GA engine with safe mutations: everything ``tests/ga_novelty_backend.py`` provides (the GA
operations of the oracle backend, the probe observations, the characterisation and the GA novelty search), plus the
scale rows and the K3 with scale rows restated with ``oracle/ga_safe_mutation.py`` on torch CPU tensors.

TEST-ONLY, like oracle_backend: it lets the gloo tests exercise the GA engine's safe-mutation path without a GPU.
"""
import numpy as np
import torch

import ga_novelty_backend as _gn
from coevonet_b200 import layout
from oracle import ga_safe_mutation as gsm, philox
from ga_novelty_backend import *  # noqa: F401,F403  (the call signatures of coevonet_b200.ops the engine uses)


def ga_safe_scale(elites, in_dim, probe_obs, floor, *, out=None, status=None):
    D = layout.fc_dim(in_dim)
    rows = elites.numpy()
    res = torch.from_numpy(gsm.scale_rows(rows, in_dim, probe_obs.numpy(), floor, pitch=rows.shape[1]))
    if status is not None and not np.all(np.isfinite(res.numpy()[:, :D])):
        status.fill_(1)
    if out is not None:
        out.copy_(res)
        return out
    return res


def ga_repopulate(elites, dim, sigma, seed, role, gen, row0, n_rows, *, out=None, noise_out=None,
                  crossover_rate=0.0, scale=None):
    if scale is None:
        return _gn.ga_repopulate(elites, dim, sigma, seed, role, gen, row0, n_rows, out=out, noise_out=noise_out,
                                 crossover_rate=crossover_rate)
    role_id = layout.ROLE_ID[role] if isinstance(role, str) else int(role)
    members = np.arange(row0, row0 + n_rows)
    z = philox.normals(seed, philox.KIND_GA, role_id, gen, members, dim)
    rows = gsm.children(elites.numpy()[:, :dim], scale.numpy(), float(sigma), z, members, crossover_rate, seed,
                        role_id, gen)
    res = torch.zeros((n_rows, elites.shape[1]), dtype=torch.float32) if out is None else out
    res[:, :dim] = torch.from_numpy(rows)
    res[:, dim:] = 0
    return res
