"""float64 references of ExactPosterior.condition_on, PosteriorMarginals and grf_phi_row_condition
(grf_b200/posterior.py, csrc/grf_posterior.cu), and the bound that holds a conditioned posterior to a posterior
constructed from scratch on the union of the training rows.

Block update.  With K = G^T G + sigma^2 I over the n old and b new training rows (G = Phi_f[x]^T restricted to S):

    L_21 = (L_11^-1 K_21^T)^T,   L_22 = chol(K_22 + sigma^2 I - L_21 L_21^T),   C_new = (G_new - C_old L_21^T) L_22^-T

which is the Cholesky factor of the whole K and C = G L^-T column block by column block (rows of G_new and C_old are
indexed by the slots of the union; C_old is zero on the slots only the new rows touch).

Error bound.  u = 2^-24.  Write C* for the exact C of the union and s_i for candidate i's row of Phi_f restricted to
S (k_i touched entries, float32 weights w).  Both posteriors store C in float32 and project it in float32:
  - from scratch, every element of C is one rounding of a float64 value: |C^ - C*| <= E_f = u |C*|;
  - conditioned, the first columns are the same, and each call appends C_new = (G_new - C^_old L_21^T) L_22^-T,
    computed in float64 from the STORED C^_old and rounded once, so |C^_new - C*_new| <= E_new = u |C*_new| +
    E_old |M| with M = L_21^T L_22^-T (n x b); chains of calls apply this column block by column block.
The float64 stages (Cholesky, triangular solves, the G and K sums) add relative errors of order kappa(K) 2^-53;
the tests keep kappa(K) <= 2^13, so they stay below 2^-40 relative and F64 = 2^-40 covers them.
The projection p_ic = s_i . C^[:, c] of either side then errs by at most

    delta_ic = sum_e |w_e| E[slot e, c] + (2^-22 max(k_i, 1) + F64) A_ic,      A_ic = sum_e |w_e C*_ec|

(tests/predictive_ref.py: the float32 projection bound holds for any order of the entries, so the slots the
conditioned posterior appends out of ascending order cost nothing extra), and |p^^2 - p^2| <= (2 A + delta) delta.
The variance adds the squares in float64 and rounds: q once to float32 (from scratch; the first pass of
PosteriorMarginals too), d - q once to float32; d is the same float32 on both sides.  So, for the difference of the
two variances,

    |var_c - var_f| <= sum_c [(2 A + delta_c) delta_c + (2 A + delta_f) delta_f] + 2u q + 2u var

and likewise the mean (projection of the float32 a: u + 2^-22 max(k, 1) + F64 per side, of sum_e |w_e a_e|), the
covariance (P P^T with P = S* C^: |P_i| delta_j + delta_i |P_j| + delta_i delta_j per column and side) and the
samples (B = C^ z^ with z^ = fl32(L^-1 V) and a float32 GEMM of n terms: |w| (E |z| + (n + 2) u |C*| |z|) plus the
projection of B, per side).  The bounds below double these sums (the O(u^2) terms, with room to spare)."""

from __future__ import annotations

import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp

U = 2.0 ** -24
PB = 2.0 ** -22
F64 = 2.0 ** -40
KAPPA_MAX = 2.0 ** 13


def block_update(L, C_old, G_new, noise, K21, K22):
    """(L of n + b rows, C_new [m, b], M = L_21^T L_22^-T [n, b]) from the old factor L [n, n], C_old [m, n] (rows of
    the union's slots, zero where only the new rows reach), G_new [m, b] and K_21 [b, n], K_22 [b, b]."""
    n, b = L.shape[0], K22.shape[0]
    l21t = sla.solve_triangular(L, K21.T, lower=True) if n else np.zeros((0, b))
    l22 = np.linalg.cholesky(K22 + noise * np.eye(b) - l21t.T @ l21t)
    Lb = np.zeros((n + b, n + b))
    Lb[:n, :n], Lb[n:, :n], Lb[n:, n:] = L, l21t.T, l22
    c_new = sla.solve_triangular(l22, (G_new - C_old @ l21t).T, lower=True).T
    M = sla.solve_triangular(l22, l21t.T, lower=True).T if n else np.zeros((0, b))
    return Lb, c_new, M


def weights(G, L, y):
    """a = G K^-1 y from the factor L of K (float64 [m])."""
    if G.shape[1] == 0:
        return np.zeros(G.shape[0])
    return G @ sla.cho_solve((L, True), np.asarray(y, np.float64))


def row_condition(ti, col, w, n, slot, B, r, with_mean, q, d):
    """(q, var, mean) after grf_phi_row_condition in float64: q + sum_{c < r} p_c^2, max(d - q, 0) (NaN stays),
    p_r (or None)."""
    B = np.asarray(B, np.float64)
    m = B.shape[0]
    s = np.asarray(slot)[col] if col.size else np.zeros(0, np.int64)
    t = s >= 0
    P = sp.csr_matrix((np.asarray(w, np.float64)[t], (ti[t], s[t])), shape=(n, m))
    p = np.asarray(P @ B[:, :r + with_mean]) if m else np.zeros((n, r + with_mean))
    q = np.asarray(q, np.float64) + np.sum(p[:, :r] ** 2, axis=1)
    diff = np.asarray(d, np.float64) - q
    var = np.where(np.isnan(diff), diff, np.maximum(diff, 0.0))
    return q, var, (p[:, r] if with_mean else None)


def chain(G, n0, batches, noise):
    """The exact factor of the union and the error bounds of both sides' C.  G [m, n_total] over the union's
    slots (columns in training order), n0 rows first, then the batch sizes of the successive condition_on calls.
    Returns (L, C*, E_cond, E_fresh, kappa(K))."""
    m, nt = G.shape
    K = G.T @ G + noise * np.eye(nt)
    L = np.linalg.cholesky(K) if nt else np.zeros((0, 0))
    C = sla.solve_triangular(L, G.T, lower=True).T if nt else np.zeros((m, 0))
    E = np.zeros_like(C)
    E[:, :n0] = U * np.abs(C[:, :n0])
    n = n0
    for b in batches:
        l21, l22 = L[n:n + b, :n], L[n:n + b, n:n + b]
        M = sla.solve_triangular(l22, l21, lower=True).T if n else np.zeros((0, b))
        E[:, n:n + b] = U * np.abs(C[:, n:n + b]) + E[:, :n] @ np.abs(M)
        n += b
    kappa = np.linalg.cond(K) if nt else 1.0
    return L, C, E, U * np.abs(C), kappa


def _proj(ti, col, w, n, slot, X):
    s = np.asarray(slot)[col] if col.size else np.zeros(0, np.int64)
    t = s >= 0
    P = sp.csr_matrix((np.abs(np.asarray(w, np.float64))[t], (ti[t], s[t])), shape=(n, X.shape[0]))
    k = np.bincount(ti[t], minlength=n)
    return np.asarray(P @ X), np.maximum(k, 1)


def proj_delta(ti, col, w, n, slot, C, E):
    """(A, delta) [n, r]: sum_e |w_e C*_ec| and the projection error bound of one side."""
    A, k = _proj(ti, col, w, n, slot, np.abs(C))
    EE, _ = _proj(ti, col, w, n, slot, E)
    return A, EE + (PB * k[:, None] + F64) * A


def var_bound(A, dc, df, q, var):
    """Bound on |var_conditioned - var_fresh| per candidate."""
    return 2.0 * (np.sum((2 * A + dc) * dc + (2 * A + df) * df, axis=1) + 2 * U * (np.abs(q) + np.abs(var)))


def mean_bound(ti, col, w, n, slot, a):
    """Bound on |mean_conditioned - mean_fresh| per candidate (a: float64 [m])."""
    Aa, k = _proj(ti, col, w, n, slot, np.abs(np.asarray(a, np.float64))[:, None])
    return 2.0 * 2 * (U + PB * k + F64) * Aa[:, 0]


def cov_bound(P, dc, df):
    """Bound on |cov_conditioned - cov_fresh| ([q, q]) from P = S* C* and the per-side projection bounds."""
    Pa = np.abs(P)
    one = lambda d: Pa @ d.T + d @ Pa.T + d @ d.T
    return 2.0 * (one(dc) + one(df))


def sample_bound(ti, col, w, n, slot, C, E_c, E_f, z, ntrain):
    """Bound on |samples_conditioned - samples_fresh| ([n, s]) for z = L^-1 V (float64 [ntrain, s])."""
    za = np.abs(z)
    Ba = np.abs(C) @ za
    tot = 0.0
    for E in (E_c, E_f):
        dB = E @ za + (ntrain + 2) * U * Ba
        X, k = _proj(ti, col, w, n, slot, dB)
        A, _ = _proj(ti, col, w, n, slot, Ba + dB)
        tot = tot + X + (PB * k[:, None] + F64) * A
    return 2.0 * tot
