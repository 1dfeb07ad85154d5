"""CPU restatement of the Co-ES novelty search (the checker of ``cev_novelty_probe_obs_f32``, ``cev_novelty_bc_f32``,
``cev_novelty_knn_f64`` and of the engine's archive ring): the probe observations, the policy-space behaviour
characterisation, the k-NN novelty, the fitness that combines it with the reward, and the archive.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  NS-ES / NSR-ES follow Conti et al., "Improving Exploration in
Evolution Strategies for Deep Reinforcement Learning via a Population of Novelty-Seeking Agents" (NeurIPS 2018); the
characterisation is the policy's action distributions on fixed probe observations, the "behavioural embedding" of
Parker-Holder et al. (NeurIPS 2020).
"""
from __future__ import annotations

import numpy as np

from . import philox, rollout

PROBES = 32
N_ACTIONS = 5
BC_DIM = PROBES * N_ACTIONS
#: Philox stream of the probe world states (cev_init_states_f64); the training states use role + 4 * gen, the
#: evaluation games 0x40000000 + gen and the Hall-of-Fame matrix 0x50000000
PROBE_TAG = 0x60000000
SEAT_INDEX = {"adversary_0": 0, "agent_0": 1, "agent_1": 2}


def probe_states(seed):
    """fp64 [32, 11]: the probe world states of a run, records 0..31 of the Philox stream PROBE_TAG."""
    return philox.init_states(seed, PROBE_TAG, PROBES)


def probe_obs(states, role):
    """fp32 [n, in_dim]: what ``role`` observes in each world state (zero velocities)."""
    s = np.asarray(states, dtype=np.float64)
    n = s.shape[0]
    pos = s[:, 1:7].reshape(n, 3, 2)
    lm = s[:, 7:11].reshape(n, 2, 2)
    goal = s[:, 0].astype(np.int64)
    return rollout.observations(pos, lm, goal)[SEAT_INDEX[role]]


def softmax(logits):
    """Max-subtracted softmax over the last axis in fp32."""
    lg = np.asarray(logits, dtype=np.float32)
    e = np.exp(lg - lg.max(axis=-1, keepdims=True))
    return (e / e.sum(axis=-1, keepdims=True)).astype(np.float32)


def bc(rows, in_dim, obs):
    """fp32 [P, 160]: the softmax action distributions of each network row on the probe observations ``obs``, probe
    after probe (the fp32 NumPy forward of ``oracle/rollout.py``)."""
    return np.stack([softmax(rollout.fc_forward(r, obs, in_dim)).reshape(-1) for r in np.asarray(rows)]) \
        if len(rows) else np.zeros((0, BC_DIM), np.float32)


def distances(x, archive):
    """fp64 [filled]: Euclidean distances from one characterisation to each archive entry, the squares summed over
    the 160 dimensions in order, one rounding per operation."""
    d = np.asarray(x, np.float32).astype(np.float64)[None, :] - np.asarray(archive, np.float32).astype(np.float64)
    s = np.zeros(d.shape[0])
    for t in range(d.shape[1]):
        s = s + d[:, t] * d[:, t]
    return np.sqrt(s)


def novelty(bcs, archive, k):
    """fp64 [n]: the mean of the min(k, filled) smallest distances from each characterisation to the ``filled``
    archive entries, summed in ascending order of (distance, slot)."""
    archive = np.asarray(archive)
    ke = min(int(k), archive.shape[0])
    out = np.empty(len(bcs))
    for i, x in enumerate(bcs):
        dist = distances(x, archive)
        order = np.lexsort((np.arange(len(dist)), dist))
        acc = 0.0
        for v in dist[order[:ke]]:
            acc += float(v)
        out[i] = acc / ke
    return out


def combine(shaped_reward, shaped_novelty, w):
    """The NSR-ES fitness (1 - w) cr(R) + w cr(N) in fp64 (w = 1: NS-ES)."""
    return (1.0 - float(w)) * np.asarray(shaped_reward, np.float64) + float(w) * np.asarray(shaped_novelty, np.float64)


class Ring:
    """The archive of one role: A slots of characterisations.  The founders' goes to slot 0, the one of every later
    base agent to slot ``head``, which then advances modulo A; ``filled`` = min(appended, A)."""

    def __init__(self, A, first):
        self.A = int(A)
        self.rows = np.zeros((self.A, BC_DIM), dtype=np.float32)
        self.head = self.filled = 0
        self.append(first)

    def append(self, row):
        self.rows[self.head] = row
        self.head = (self.head + 1) % self.A
        self.filled = min(self.filled + 1, self.A)
