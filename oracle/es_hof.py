"""CPU restatement of the Co-ES Hall of Fame (the checker of ``cev_es_hof_opponents_i64`` and of the engine's archive
ring): which archive slots a generation's K opponent sets come from, and what the ring holds after g generations.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  The reference's Co-ES evaluates every member against the other
roles' current base agents only (evolutionary_strategy.py:63-116); its Co-GA keeps a Hall of Fame of champions
(genetic_algorithm.py:270-275), which this extends to Co-ES as an archive of past base agents.
"""
from __future__ import annotations

import numpy as np

from . import philox

#: Philox kind of the opponent draws (member word 0, role 0); CEV_KIND_HOF in the header
KIND_HOF = 7


def opponent_slots(seed, gen, K, filled, newest):
    """int64[K]: set 0 is ``newest``; set k >= 1 is (uint64(w_k) * filled) >> 32 with w_k word (k - 1) & 3 of the
    Philox block (k - 1) >> 2 at (member 0, gen, kind KIND_HOF, role 0)."""
    out = np.empty(int(K), dtype=np.int64)
    out[0] = newest
    if K > 1:
        n4 = (K - 1 + 3) // 4
        w = philox.words(seed, KIND_HOF, 0, gen, [0], n4).reshape(-1)[:K - 1].astype(np.uint64)
        out[1:] = ((w * np.uint64(filled)) >> np.uint64(32)).astype(np.int64)
    return out


class Ring:
    """The archive: H slots of snapshots.  The founders go to slot 0; every later snapshot to slot ``head``, which
    then advances modulo H.  ``filled`` = min(snapshots appended, H); ``slot_gen[s]`` is the generation whose base
    agents slot s holds (-1 while empty).  Slots [0, filled) are the filled ones in every state."""

    def __init__(self, H, founders):
        founders = np.asarray(founders)
        self.H = int(H)
        self.rows = np.zeros((self.H, founders.size), dtype=founders.dtype)
        self.slot_gen = np.full(self.H, -1, dtype=np.int64)
        self.head = self.filled = 0
        self.append(founders, 0)

    def append(self, row, gen):
        self.rows[self.head] = row
        self.slot_gen[self.head] = gen
        self.head = (self.head + 1) % self.H
        self.filled = min(self.filled + 1, self.H)

    @property
    def newest(self):
        return (self.head - 1) % self.H
