"""CPU restatement of Co-ES guided search in the subspace of past update estimates (the checker of
``cev_es_perturb_subspace_f32`` and ``cev_es_subspace_basis_f32``): the member formula given the normals, the
coefficient stream, and the drop-rule basis of the estimate ring in fp64.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  The reference searches with one isotropic Gaussian per role
(agent.py:31-70); this extends it with Guided ES (Maheswaranathan et al., ICML 2019), whose subspace is spanned by
the ES's own last k update estimates (as in ASEBO, Choromanski et al. 2019, and Self-Guided ES, Liu et al. 2020).
"""
from __future__ import annotations

import math

import numpy as np

from . import philox

#: Philox kind of the subspace coefficients c (member word = member id, or pair id under mirroring);
#: CEV_KIND_ES_SUBSPACE in the header
KIND_ES_SUBSPACE = 8
#: an estimate is dropped when its residual norm is <= DROP_TOL of its own norm
DROP_TOL = 1e-4


def scales(alpha, d, k_eff):
    """(A, B) fp32: A = fp32(sqrt(alpha)), B = fp32(sqrt((1 - alpha) d / k_eff)), both from fp64; B = 0 when
    k_eff = 0."""
    A = np.float32(math.sqrt(alpha))
    B = np.float32(math.sqrt((1.0 - alpha) * d / k_eff)) if k_eff else np.float32(0.0)
    return A, B


def coefficients(seed, role, gen, units, k):
    """fp32 [len(units), k]: normals 0..k-1 of each unit (member id, or pair id) in the stream of kind
    KIND_ES_SUBSPACE, ctr = (m // 4, unit, gen, role | kind << 8)."""
    return philox.normals(seed, KIND_ES_SUBSPACE, role, gen, units, k)


def perturb(theta, sigma, U, k_eff, alpha, z, c, pert_idx, row0, mirrored):
    """Member rows row0 .. row0 + n - 1 and their directions, one IEEE fp32 rounding per operation.  ``z`` fp32
    [n, D] and ``c`` fp32 [n, >= k_eff] hold every member's own normals (under mirroring its pair's, UNSIGNED);
    ``U`` fp32 [>= k_eff, D].  eps = fl(fl(A z) + fl(B s)), s = sum_{m < k_eff} fl(U[m] c_m) in order from +0, or
    eps = z when B = 0; member = theta + fl(sigma eps), the odd member of a mirrored pair theta + (-fl(sigma eps)).
    Returns (rows fp32 [n, D], eps fp32 [n, len(pert_idx)] with the member's sign)."""
    f32 = np.float32
    theta = np.asarray(theta, dtype=f32)
    z = np.asarray(z, dtype=f32)[:, pert_idx]
    n = z.shape[0]
    A, B = scales(alpha, len(pert_idx), k_eff)
    if B == 0:
        eps = z.copy()
    else:
        s = np.zeros_like(z)
        for m in range(k_eff):
            s = (s + (np.asarray(U, dtype=f32)[m, pert_idx][None, :] * np.asarray(c, dtype=f32)[:, m:m + 1])).astype(f32)
        eps = ((A * z).astype(f32) + (B * s).astype(f32)).astype(f32)
    d = (f32(sigma) * eps).astype(f32)
    odd = (np.arange(row0, row0 + n) & 1).astype(bool) if mirrored else np.zeros(n, bool)
    d[odd] = -d[odd]
    rows = np.repeat(theta[None], n, axis=0)
    rows[:, pert_idx] = (theta[pert_idx] + d).astype(f32)
    eps[odd] = -eps[odd]
    return rows, eps


def _cholesky_drop(G):
    """Right-looking Cholesky of G over columns 0, 1, ... that drops column a when its squared residual is
    <= DROP_TOL^2 G[a][a] (a zero or non-finite column is always dropped).  Returns (kept columns, R restricted to
    them: upper triangular with G[kept][:, kept] = R^T R)."""
    k = G.shape[0]
    W = G.copy()
    R = np.zeros_like(G)
    kept = []
    for a in range(k):
        diag = W[a, a]                                  # NaN for a non-finite column: dropped below
        if not diag > DROP_TOL ** 2 * G[a, a]:
            continue
        r = math.sqrt(diag)
        R[a, a] = r
        R[a, a + 1:] = W[a, a + 1:] / r
        with np.errstate(invalid="ignore"):            # a dropped non-finite column's row and column only
            W[a + 1:, a + 1:] -= np.outer(R[a, a + 1:], R[a, a + 1:])
        kept.append(a)
    return kept, R[np.ix_(kept, kept)]


def _pass(D):
    """One CholeskyQR pass with the drop rule: D fp32 [k, d] (rows = columns of the method) -> (Q fp32 [n_kept, d])."""
    D64 = np.asarray(D, dtype=np.float64)
    kept, Rk = _cholesky_drop(D64 @ D64.T)
    if not kept:
        return np.zeros((0, D.shape[1]), np.float32)
    T = np.linalg.inv(Rk)                                           # upper triangular
    return (T.T @ D64[kept]).astype(np.float32)


def basis(D):
    """CholeskyQR2 with the drop rule of the estimates ``D`` fp32 [n, d] given newest first: U fp32 [k_eff, d] with
    orthonormal rows spanning the kept estimates."""
    return _pass(_pass(np.asarray(D, dtype=np.float32)))


class Ring:
    """The estimate ring: k slots, the newest estimate goes to slot ``head``, which then advances modulo k;
    ``filled`` = min(estimates appended, k).  ``newest_first()`` lists the filled slots' rows newest first."""

    def __init__(self, k, n):
        self.k = int(k)
        self.rows = np.zeros((self.k, int(n)), dtype=np.float32)
        self.head = self.filled = 0

    def append(self, row):
        self.rows[self.head] = row
        self.head = (self.head + 1) % self.k
        self.filled = min(self.filled + 1, self.k)

    @property
    def newest(self):
        return (self.head - 1) % self.k

    def newest_first(self):
        return self.rows[[(self.newest - a) % self.k for a in range(self.filled)]]


def ring_basis(ring_rows, newest, filled, segments):
    """``cev_es_subspace_basis_f32`` restated: per segment (start, end, perturbable index relative to start) of the
    concatenated rows, the basis of the ring's estimates newest first over the segment's Linear entries.  Returns
    (U fp32 [k, n], k_eff int list)."""
    k, n = ring_rows.shape
    U = np.zeros((k, n), dtype=np.float32)
    k_eff = []
    order = [(newest - a) % k for a in range(filled)]
    for start, end, pidx in segments:
        cols = start + np.asarray(pidx)
        Us = basis(ring_rows[np.ix_(order, cols)]) if filled else np.zeros((0, len(cols)), np.float32)
        U[np.ix_(np.arange(Us.shape[0]), cols)] = Us
        k_eff.append(Us.shape[0])
    return U, k_eff
