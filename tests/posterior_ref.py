"""float64 references of the exact posterior variance (grf_b200/posterior.py) and of grf_phi_row_quadform.

Error bound of q.  Per column c the kernel forms s_c = sum_e w_e C_ec in float32 (w_e = fl(f_l * val_e), one fused
multiply-add per entry), squares it in float64 and adds the squares in float64; q is rounded to float32 once.  With
u = 2^-24, A_c = sum_e |w_e C_ec| and k touched entries, |s^_c - s_c| <= (k + 1) u A_c (1 + O(u)) whatever the
order of the sum, so |s^_c^2 - s_c^2| <= 2 (k + 1) u A_c^2 (1 + O(u)), and the float64 sums and the final rounding
add at most u sum_c A_c^2.  Hence

    |q^ - q| <= (2k + 3) u sum_c A_c^2 <= 2^-21 max(k, 1) sum_c A_c^2          (8 u k >= (2k + 3) u for k >= 1)

and likewise |d^ - d| <= 2^-21 max(len, 1) sum_e w_e^2.  Both hold for any summation order."""

from __future__ import annotations

import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp

QB = 2.0 ** -21


def exact_cache(phi_f, x, noise):
    """slot (int32 [N]), G (m x n) and C = G L^-T (float64) of the contract, from Phi_f (scipy, one entry per
    (row, col)) and the training ids x."""
    phi_f = sp.csr_matrix(phi_f, dtype=np.float64)
    x = np.asarray(x, np.int64)
    n, N = x.size, phi_f.shape[1]
    rows = phi_f[x] if n else sp.csr_matrix((0, N))
    cols = np.unique(rows.indices)
    slot = np.full(N, -1, np.int32)
    slot[cols] = np.arange(cols.size, dtype=np.int32)
    G = rows[:, cols].T.toarray() if n else np.zeros((cols.size, 0))
    if n == 0:
        return slot, G, np.zeros((cols.size, 0))
    L = np.linalg.cholesky(G.T @ G + noise * np.eye(n))
    C = sla.solve_triangular(L, G.T, lower=True).T
    return slot, G, C


def row_entries(indptr, cols, vals, ids):
    """(test index, column, value) of every entry of the rows ``ids`` of a CSR (entries of one row in order)."""
    ids = np.asarray(ids, np.int64)
    b, e = np.asarray(indptr)[ids].astype(np.int64), np.asarray(indptr)[ids + 1].astype(np.int64)
    lens = e - b
    ti = np.repeat(np.arange(ids.size), lens)
    idx = np.repeat(b - np.r_[0, np.cumsum(lens)[:-1]], lens) + np.arange(lens.sum())
    return ti, np.asarray(cols)[idx], np.asarray(vals)[idx]


def quadform(ti, col, w, n, slot, C):
    """q, d (float64 [n]) and their bounds from the entries (test index ti, column col, weight w) of the test rows,
    a slot map and C (m x r, float64 values)."""
    w = np.asarray(w, np.float64)
    C = np.asarray(C, np.float64)
    m, r = C.shape
    s = np.asarray(slot)[col] if col.size else np.zeros(0, np.int64)
    t = s >= 0
    P = sp.csr_matrix((w[t], (ti[t], s[t])), shape=(n, m))
    Pa = sp.csr_matrix((np.abs(w[t]), (ti[t], s[t])), shape=(n, m))
    S = np.asarray(P @ C) if r else np.zeros((n, 0))
    A = np.asarray(Pa @ np.abs(C)) if r else np.zeros((n, 0))
    q = np.sum(S * S, axis=1)
    k = np.bincount(ti[t], minlength=n)
    d = np.bincount(ti, weights=w * w, minlength=n) if ti.size else np.zeros(n)
    lens = np.bincount(ti, minlength=n)
    return q, d, QB * np.maximum(k, 1) * np.sum(A * A, axis=1), QB * np.maximum(lens, 1) * d


def quadform_f32(ti, col, w32, n, slot, C32):
    """The kernel's arithmetic on the host in entry order: float32 column sums (one fma per entry), float64 squares
    and sum, q rounded to float32."""
    C32 = np.asarray(C32, np.float32)
    q = np.zeros(n, np.float32)
    d = np.zeros(n, np.float32)
    for i in range(n):
        sel = ti == i
        wi, ci = np.asarray(w32, np.float32)[sel], col[sel]
        d[i] = np.float32(np.sum(wi.astype(np.float64) ** 2))
        si = np.asarray(slot)[ci]
        s = np.zeros(C32.shape[1], np.float32)
        for wv, sv in zip(wi[si >= 0], si[si >= 0]):
            s = (s.astype(np.float64) + np.float64(wv) * C32[sv].astype(np.float64)).astype(np.float32)   # fma
        q[i] = np.float32(np.sum(s.astype(np.float64) ** 2))
    return q, d


def dense_variance(phi_f, x, xt, noise):
    """diag(K** - K*x (Kxx + sigma^2 I)^-1 Kx*) and diag(K**) in float64 (sparse products, dense n x n solve)."""
    phi_f = sp.csr_matrix(phi_f, dtype=np.float64)
    x, xt = np.asarray(x, np.int64), np.asarray(xt, np.int64)
    rt = phi_f[xt]
    prior = np.asarray(rt.multiply(rt).sum(axis=1)).ravel()
    if x.size == 0:
        return prior, prior
    rx = phi_f[x]
    kxx = (rx @ rx.T).toarray() + noise * np.eye(x.size)
    kst = (rt @ rx.T).toarray()
    sol = sla.cho_solve(sla.cho_factor(kxx, lower=True), kst.T)
    return prior - np.sum(kst * sol.T, axis=1), prior
