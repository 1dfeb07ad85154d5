"""Checker backend of the ES engine with novelty search: everything ``tests/es_subspace_backend.py`` provides, plus the
probe observations, the behaviour characterisation and the k-NN novelty restated with ``oracle/es_novelty.py`` on
torch CPU tensors.

TEST-ONLY, like oracle_backend: it lets the gloo tests exercise the engine's novelty-search path without a GPU.
"""
import numpy as np
import torch

from coevonet_b200 import layout
from oracle import es_novelty as en
from es_subspace_backend import *  # noqa: F401,F403  (the call signatures of coevonet_b200.ops the engine uses)


def novelty_probe_obs(init, role, *, out=None):
    res = torch.from_numpy(en.probe_obs(init.numpy(), role))
    if out is not None:
        out.copy_(res)
        return out
    return res


def novelty_bc(rows, in_dim, probe_obs, *, out=None, status=None):
    bc = en.bc(rows.numpy()[:, :layout.fc_dim(in_dim)], in_dim, probe_obs.numpy())
    if status is not None and not np.all(np.isfinite(bc)):
        status.fill_(1)
    res = torch.from_numpy(bc)
    if out is not None:
        out.copy_(res)
        return out
    return res


def novelty_knn(bc, ring, filled, k, *, out=None):
    res = torch.from_numpy(en.novelty(bc.numpy(), ring.numpy()[:int(filled)], k))
    if out is not None:
        out.copy_(res)
        return out
    return res
