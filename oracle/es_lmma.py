"""CPU restatement of Co-ES limited-memory matrix adaptation (LM-MA-ES, Loshchilov, Glasmachers & Beyer, "Large Scale
Black-Box Optimization by Limited-Memory Matrix Adaptation", IEEE TEC 23(2), 2019), the checker of ``es_lmma.cu``:
the constants and weights, the sequential transform (the spec) and its compact form, the projection in the kernel's
summation order, K5 given beta, the recombination, the apply with the path / vector / Gram / step-size updates, and a
small standalone minimiser built from the same functions.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  The reference searches with one isotropic Gaussian per role
(agent.py:31-70) and has no LM-MA-ES.
"""
from __future__ import annotations

import math

import numpy as np

#: column chunk of the projection, column chunk of the apply's Gram / |p|^2 sums, rank splits of the recombination
#: (LM_CHUNK, LM_ACHUNK, LM_SPLIT in es_lmma.cu)
PROJECT_CHUNK, APPLY_CHUNK, REDUCE_SPLIT = 2048, 4096, 8


def constants(lam, n, m):
    """The constants of Algorithm 1 for population lam, dimension n and m vectors, all fp64: mu = lam // 2, the log
    weights w_i = (ln(mu + 1/2) - ln(i + 1)) / sum_j (...) for i < mu, mu_w = 1 / sum w_i^2, c_sigma = 2 lam / n,
    c_d,j = 1 / (1.5^j n) and c_c,j = lam / (4^j n) for j < m."""
    mu = int(lam) // 2
    raw = np.array([math.log(mu + 0.5) - math.log(i + 1) for i in range(mu)], dtype=np.float64)
    w = raw / raw.sum()
    return {"mu": mu, "w": w, "mu_w": float(1.0 / np.sum(w * w)), "c_sigma": 2.0 * lam / n,
            "c_d": [1.0 / (1.5 ** j * n) for j in range(m)], "c_c": [lam / (4.0 ** j * n) for j in range(m)]}


def transform_sequential(M, z, k, c_d):
    """The paper's transform in fp64: d = z; for j < k: d = (1 - c_d,j) d + c_d,j m_j (m_j . d).  M [>= k, n],
    z [n] or [N, n]."""
    d = np.array(z, dtype=np.float64)
    M = np.asarray(M, dtype=np.float64)
    for j in range(k):
        d = (1.0 - c_d[j]) * d + c_d[j] * np.multiply.outer(d @ M[j], M[j]) if d.ndim == 2 else \
            (1.0 - c_d[j]) * d + c_d[j] * M[j] * (M[j] @ d)
    return d


def transform_compact(s, G, k, c_d):
    """The compact form, fp64, one rounding per operation in the kernel's order: s [N, >= k] = M z, G [>= k, >= k].
    Returns (alpha, beta fp64 [N, k]) with d = alpha z + sum_l beta_l m_l."""
    s = np.asarray(s, dtype=np.float64)
    N = s.shape[0]
    beta = np.zeros((N, k), np.float64)
    alpha = 1.0
    for j in range(k):
        q = alpha * s[:, j]
        for l in range(j):
            q = q + beta[:, l] * G[j][l]
        om = 1.0 - c_d[j]
        beta[:, :j] = beta[:, :j] * om
        beta[:, j] = c_d[j] * q
        alpha = alpha * om
    return alpha, beta


def alpha_of(k, c_d):
    """alpha after k steps of the compact form (data independent)."""
    a = 1.0
    for j in range(k):
        a = a * (1.0 - c_d[j])
    return a


def project(M, z, k):
    """s fp64 [N, k] = M[:k] z in the kernel's order: per column chunk of PROJECT_CHUNK, fp64 adds of the exact fp32 x
    fp32 products in column order from +0, then the chunks in order from +0.  M fp32 [>= k, D], z fp32 [N, D] with
    zeros off the Linear entries (D = the row's fc_dim)."""
    M = np.asarray(M, dtype=np.float32)[:k].astype(np.float64)
    z = np.asarray(z, dtype=np.float32).astype(np.float64)
    N, D = z.shape
    n_ch = -(-D // PROJECT_CHUNK)
    pad = n_ch * PROJECT_CHUNK - D
    Mp = np.pad(M, ((0, 0), (0, pad))).reshape(k, n_ch, PROJECT_CHUNK)
    zp = np.pad(z, ((0, 0), (0, pad))).reshape(N, n_ch, PROJECT_CHUNK)
    acc = np.zeros((n_ch, N, k), np.float64)
    for c in range(PROJECT_CHUNK):
        acc = acc + zp[:, :, c].T[:, :, None] * Mp[:, :, c].T[:, None, :]
    s = np.zeros((N, k), np.float64)
    for ch in range(n_ch):
        s = s + acc[ch]
    return s


def perturb(theta, sigma, M, beta, alpha, z, pert_idx):
    """K5 given beta: rows fp32 [N, D].  eps = fl(fl(fp32(alpha) z) + S), S = sum_{l < k} fl(M[l] beta_l) in order from
    +0 (fp32), member = theta + fl(fp32(sigma) eps) on the Linear entries; with k = 0 eps = z."""
    f32 = np.float32
    theta = np.asarray(theta, dtype=f32)
    z = np.asarray(z, dtype=f32)[:, pert_idx]
    beta = np.asarray(beta, dtype=f32)
    N, k = beta.shape
    if k == 0:
        eps = z
    else:
        S = np.zeros_like(z)
        for l in range(k):
            S = (S + (np.asarray(M, dtype=f32)[l, pert_idx][None, :] * beta[:, l:l + 1]).astype(f32)).astype(f32)
        eps = ((f32(alpha) * z).astype(f32) + S).astype(f32)
    rows = np.repeat(theta[None], N, axis=0)
    rows[:, pert_idx] = (theta[pert_idx] + (f32(sigma) * eps).astype(f32)).astype(f32)
    return rows


def reduce(ids, w, z_of, beta, row0, n_rows):
    """This rank's recombination: zbar fp32 [D] = the REDUCE_SPLIT rank splits of [0, mu) summed in order from +0, each
    the fp64 sum in rank order of w_a z_id (exact fp32 x fp32 products) over the local ids; betabar fp32 [k] = the fp64
    sum in rank order of w_a beta[id - row0].  ``z_of(id)`` -> fp32 [D] normals of member id (zero off the Linear
    entries); w fp32 [mu]; beta fp32 [n_rows, k]."""
    mu = len(ids)
    w = np.asarray(w, dtype=np.float32).astype(np.float64)
    beta = np.asarray(beta, dtype=np.float32)
    per = -(-mu // REDUCE_SPLIT)
    total, bb = None, np.zeros(beta.shape[1], np.float64)
    for sp in range(REDUCE_SPLIT):
        acc = None
        for a in range(sp * per, min(mu, (sp + 1) * per)):
            i = int(ids[a])
            if not row0 <= i < row0 + n_rows:
                continue
            t = w[a] * np.asarray(z_of(i), dtype=np.float32).astype(np.float64)
            acc = t if acc is None else acc + t
        if acc is not None:
            total = acc if total is None else total + acc
    for a in range(mu):
        i = int(ids[a])
        if row0 <= i < row0 + n_rows:
            bb = bb + w[a] * beta[i - row0].astype(np.float64)
    D = len(z_of(int(ids[0]))) if total is None else total.shape[0]
    zbar = np.zeros(D, np.float32) if total is None else total.astype(np.float32)
    return zbar, bb.astype(np.float32)


def gram_chunked(X):
    """Gram fp64 of the rows of X fp32 [r, L] in the apply's order: per column chunk of APPLY_CHUNK, fp64 adds of the
    exact products in column order from +0, the chunks in order from +0."""
    X = np.asarray(X, dtype=np.float32).astype(np.float64)
    r, L = X.shape
    n_ch = -(-L // APPLY_CHUNK)
    Xp = np.pad(X, ((0, 0), (0, n_ch * APPLY_CHUNK - L))).reshape(r, n_ch, APPLY_CHUNK)
    acc = np.zeros((n_ch, r, r), np.float64)
    for c in range(APPLY_CHUNK):
        v = Xp[:, :, c].T
        acc = acc + v[:, :, None] * v[:, None, :]
    G = np.zeros((r, r), np.float64)
    for ch in range(n_ch):
        G = G + acc[ch]
    return G


def apply(theta, M, p, zbar, betabar, k, alpha, sigma, c_m, const, n, pert_idx, sigma_min, sigma_max):
    """One role's apply on the Linear entries ``pert_idx`` of the role's row (fp32 theta / p / zbar [L], M [m, L]),
    every operation one fp64 rounding and every store one fp32 rounding.  Returns (theta, M, p, G fp64 [m, m],
    |p|^2 / n, sigma after); sigma is the fp64 mutation power (the step uses fp32(sigma))."""
    f64 = np.float64
    theta, M, p = (np.array(x, dtype=np.float32) for x in (theta, M, p))
    m = M.shape[0]
    idx = np.asarray(pert_idx)
    zb = np.asarray(zbar, dtype=np.float32)[idx].astype(f64)
    bb = np.asarray(betabar, dtype=np.float32).astype(f64)
    d = alpha * zb
    for l in range(k):
        d = d + bb[l] * M[l, idx].astype(f64)
    step = c_m * f64(np.float32(sigma))
    theta[idx] = (theta[idx].astype(f64) + step * d).astype(np.float32)
    cs, mu_w = const["c_sigma"], const["mu_w"]
    p[idx] = ((1.0 - cs) * p[idx].astype(f64) + math.sqrt(mu_w * cs * (2.0 - cs)) * zb).astype(np.float32)
    for l in range(m):
        cc = const["c_c"][l]
        M[l, idx] = ((1.0 - cc) * M[l, idx].astype(f64) + math.sqrt(mu_w * cc * (2.0 - cc)) * zb).astype(np.float32)
    X = np.zeros((m + 1, len(theta)), np.float32)
    X[:m, idx] = M[:, idx]
    X[m, idx] = p[idx]
    full = gram_chunked(X)
    G = full[:m, :m].copy()
    v = full[m, m] / n
    new = sigma
    if np.isfinite(v) and np.all(np.isfinite(G)):
        new = min(max(sigma * math.exp(cs / 2.0 * (v - 1.0)), sigma_min), sigma_max)
    return theta, M, p, G, v, new


def minimize(f, n, lam, m, sigma0, gens, rng, x0=None, target=None):
    """LM-MA-ES (m = 0: plain CSA-ES) minimising ``f`` over R^n with the same constants, compact transform and
    updates in fp64, c_m = 1.  Returns (x, sigma, history of the best f per generation); stops early once the best f
    reaches ``target``."""
    const = constants(lam, n, max(m, 1))
    mu, w = const["mu"], const["w"]
    cs, mu_w = const["c_sigma"], const["mu_w"]
    x = np.zeros(n) if x0 is None else np.array(x0, dtype=np.float64)
    sigma = float(sigma0)
    p = np.zeros(n)
    M = np.zeros((max(m, 1), n))
    hist = []
    for g in range(gens):
        k = min(g, m)
        Z = rng.standard_normal((lam, n))
        s = Z @ M[:k].T
        alpha, beta = transform_compact(s, M[:k] @ M[:k].T, k, const["c_d"])
        D = alpha * Z + beta @ M[:k]
        F = np.array([f(x + sigma * d) for d in D])
        order = np.argsort(F, kind="stable")[:mu]
        zbar = w @ Z[order]
        dbar = alpha * zbar + (w @ beta[order]) @ M[:k]
        x = x + sigma * dbar
        p = (1.0 - cs) * p + math.sqrt(mu_w * cs * (2.0 - cs)) * zbar
        for j in range(m):
            cc = const["c_c"][j]
            M[j] = (1.0 - cc) * M[j] + math.sqrt(mu_w * cc * (2.0 - cc)) * zbar
        sigma = sigma * math.exp(cs / 2.0 * (p @ p / n - 1.0))
        hist.append(float(F[order[0]]))
        if target is not None and hist[-1] <= target:
            break
    return x, sigma, hist
