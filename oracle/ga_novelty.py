"""CPU restatement of the Co-GA novelty search (the checker of ``cev_ga_novelty_knn_f64``, ``cev_ga_novelty_draw_i64``
and of the GA engine's archive rings): the archive draws, the fp32 distances in their fixed operation order, and the
k-NN novelty of a member against the rest of the population plus an archive.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  Novelty against an archive plus the current population follows
Lehman & Stanley, "Abandoning Objectives: Evolution Through the Search for Novelty Alone" (Evolutionary Computation
2011); Such et al., "Deep Neuroevolution" (2017), ran it with a GA on deep networks.  The characterisation and the
archive ring are those of ``oracle/es_novelty.py`` (:func:`es_novelty.bc`, :class:`es_novelty.Ring`), and so is the
combination of the reward and novelty ranks (:func:`es_novelty.combine`).
"""
from __future__ import annotations

import numpy as np

from . import philox
from .es_novelty import BC_DIM, Ring, combine  # noqa: F401  (re-exported: the GA uses the same ring and fitness)

#: Philox kind of the archive draws (member word 0, role = the role); CEV_KIND_GA_NOVELTY in the header
KIND_GA_NOVELTY = 9
NAN_BITS = np.uint32(0x7FFFFFFF)


def draw_ids(seed, gen, role, m, P):
    """int64[m]: the population ids whose characterisations enter ``role``'s archive after generation ``gen``'s
    selection, in draw order: (uint64(w_j) * P) >> 32 with w_j word (j & 3) of the Philox block (j >> 2, 0, gen,
    role | KIND_GA_NOVELTY << 8)."""
    role_id = philox.ROLE_ID[role] if isinstance(role, str) else int(role)
    n4 = (int(m) + 3) // 4
    w = philox.words(seed, KIND_GA_NOVELTY, role_id, gen, [0], n4).reshape(-1)[:int(m)].astype(np.uint64)
    return ((w * np.uint64(P)) >> np.uint64(32)).astype(np.int64)


def fma32(a, b, c):
    """Correctly rounded float32 fmaf(a, b, c), elementwise: the fp64 product is exact, the fp64 sum carries its
    exact error (TwoSum), and a sum that lands on a float32 midpoint is rounded toward the error."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c64 = c.astype(np.float64)
    s = p + c64
    bb = s - p
    e = (p - (s - bb)) + (c64 - bb)
    r = s.astype(np.float32)
    up, dn = np.nextafter(r, np.float32(np.inf)), np.nextafter(r, np.float32(-np.inf))
    r = np.where((s == (r.astype(np.float64) + up) / 2) & (e > 0), up, r)
    r = np.where((s == (r.astype(np.float64) + dn) / 2) & (e < 0), dn, r)
    return r


def distances(q, X):
    """fp32 [len(q), len(X)]: the Euclidean distances from each row of ``q`` to each row of ``X`` (both fp32
    [., 160]): per pair, e = fl(q_t - x_t) and s = fmaf(e, e, s) from +0 over t = 0 .. 159 in order, then the
    correctly rounded fp32 square root."""
    q = np.asarray(q, np.float32)
    X = np.asarray(X, np.float32)
    s = np.zeros((q.shape[0], X.shape[0]), np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        for t in range(q.shape[1]):
            e = (q[:, t:t + 1] - X[None, :, t]).astype(np.float32)
            s = fma32(e, e, s)
        return np.sqrt(s).astype(np.float32)


def sort_keys(dist, index):
    """uint64 keys ordering (distance, index): the fp32 bit pattern of the non-negative distances, every NaN mapped
    above +inf, then the candidate index."""
    bits = np.asarray(dist, np.float32).view(np.uint32).copy()
    bits[np.isnan(dist)] = NAN_BITS
    return (bits.astype(np.uint64) << np.uint64(32)) | np.asarray(index, np.uint64)


def novelty(x, row0, pop, archive, k, chunk=64):
    """fp64 [n]: the novelty of the members ``x`` fp32 [n, 160], global rows row0 .. row0 + n - 1 of the population
    ``pop`` fp32 [P, 160], against the other population rows (indices [0, P)) and the archive entries ``archive``
    fp32 [filled, 160] (index P + slot): the fp64 sum, in ascending order of (distance, index), of the
    k_eff = min(k, P - 1 + filled) smallest distances, divided by k_eff."""
    x = np.asarray(x, np.float32)
    pop = np.asarray(pop, np.float32)
    archive = np.asarray(archive, np.float32).reshape(-1, BC_DIM)
    P, n = pop.shape[0], x.shape[0]
    cands = np.concatenate([pop, archive])
    ke = min(int(k), P - 1 + archive.shape[0])
    if ke < 1:
        raise ValueError("a member needs at least one other candidate")
    idx = np.arange(cands.shape[0], dtype=np.uint64)
    out = np.empty(n)
    for a in range(0, n, chunk):
        d = distances(x[a:a + chunk], cands)
        for r in range(d.shape[0]):
            keep = idx != np.uint64(row0 + a + r)                      # a member is not its own candidate
            dr, ir = d[r][keep], idx[keep]
            order = np.argsort(sort_keys(dr, ir), kind="stable")[:ke]
            acc = 0.0
            for v in dr[order]:
                acc += float(v)
            out[a + r] = acc / ke
    return out


def append(ring, rows):
    """Append ``rows`` (the characterisations of the drawn ids, in draw order) to an :class:`es_novelty.Ring`."""
    for row in np.asarray(rows, np.float32):
        ring.append(row)
    return ring
