"""Checker backend of the ES engine with the Hall of Fame: everything ``tests/snes_backend.py`` provides, plus the
opponent-slot draw restated with ``oracle/es_hof.py`` on torch CPU tensors.

TEST-ONLY, like oracle_backend: it lets the gloo tests exercise the engine's Hall-of-Fame path without a GPU.
"""
import torch

from oracle import es_hof
from snes_backend import *  # noqa: F401,F403  (the call signatures of coevonet_b200.ops the engine uses)


def es_hof_opponents(seed, gen, K, filled, newest, device, *, out=None):
    res = torch.from_numpy(es_hof.opponent_slots(seed, gen, K, filled, newest))
    if out is not None:
        out.copy_(res)
        return out
    return res
