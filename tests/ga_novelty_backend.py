"""Checker backend of the GA engine with novelty search: everything ``tests/es_novelty_backend.py`` provides (the GA
operations of the oracle backend, the centered ranks, the probe observations and the behaviour characterisation),
plus the population + archive k-NN novelty and the archive draws restated with ``oracle/ga_novelty.py`` on torch CPU
tensors.

TEST-ONLY, like oracle_backend: it lets the gloo tests exercise the GA engine's novelty-search path without a GPU.
"""
import torch

from oracle import ga_novelty as gn
from es_novelty_backend import *  # noqa: F401,F403  (the call signatures of coevonet_b200.ops the engine uses)


def ga_novelty_knn(x, row0, pop, ring, filled, k, *, splits=0, out=None):
    res = torch.from_numpy(gn.novelty(x.numpy(), int(row0), pop.numpy(), ring.numpy()[:int(filled)], k))
    if out is not None:
        out.copy_(res)
        return out
    return res


def ga_novelty_draw(seed, gen, role, m, P, device, *, out=None):
    res = torch.from_numpy(gn.draw_ids(seed, gen, role, m, P))
    if out is not None:
        out.copy_(res)
        return out
    return res
