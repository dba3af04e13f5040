"""float64 references of the exact posterior mean, joint covariance and pathwise samples (grf_b200/posterior.py) and
of grf_phi_row_project.  The slot map and C come from the cache of tests/posterior_ref.py; the synthetic shards of
the kernel tests from tests/matvec_abi_ref.py.

Error bound of the projection.  Each output element is o = sum_e w_e B_e over the k touched entries of the row,
with w_e = fl(f_l * val_e).  The kernel adds the products by fused multiply-adds into float32 partial sums (per lane,
per entry group) and then adds the partial sums (a shuffle tree; adding a partial of +0 is exact).  With u = 2^-24 and
A = sum_e |w_e B_e|: the k roundings of w contribute at most u A together, and the fmas and additions round at most
2k - 1 times, each time an intermediate bounded by A (1 + O(u)).  Hence, whatever the order and grouping,

    |o^ - o| <= 2k u A (1 + O(u)) <= 2^-22 max(k, 1) A          (k = 0 gives exactly +0)

with a factor of two to spare."""

from __future__ import annotations

import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp

PB = 2.0 ** -22


def project(ti, col, w, n, slot, B):
    """out (float64 [n, r]) and its bound from the entries (test index ti, column col, weight w) of the test rows,
    a slot map and B (m x r)."""
    w = np.asarray(w, np.float64)
    B = np.asarray(B, np.float64)
    m, r = B.shape
    s = np.asarray(slot)[col] if col.size else np.zeros(0, np.int64)
    t = s >= 0
    P = sp.csr_matrix((w[t], (ti[t], s[t])), shape=(n, m))
    Pa = sp.csr_matrix((np.abs(w[t]), (ti[t], s[t])), shape=(n, m))
    out = np.asarray(P @ B) if r else np.zeros((n, 0))
    A = np.asarray(Pa @ np.abs(B)) if r else np.zeros((n, 0))
    k = np.bincount(ti[t], minlength=n)
    return out, PB * np.maximum(k, 1)[:, None] * A


def project_f32(ti, col, w32, n, slot, B32):
    """The kernel's arithmetic on the host in entry order: a float32 partial sum per column, one fma per entry."""
    B32 = np.asarray(B32, np.float32)
    out = np.zeros((n, B32.shape[1]), np.float32)
    for i in range(n):
        sel = ti == i
        wi, si = np.asarray(w32, np.float32)[sel], np.asarray(slot)[col[sel]]
        s = np.zeros(B32.shape[1], np.float32)
        for wv, sv in zip(wi[si >= 0], si[si >= 0]):
            s = (s.astype(np.float64) + np.float64(wv) * B32[sv].astype(np.float64)).astype(np.float32)   # fma
        out[i] = s
    return out


def train_weights(G, noise, y):
    """a = G (G^T G + sigma^2 I)^-1 y (float64 [m]): the projection operand of the mean."""
    n = G.shape[1]
    if n == 0:
        return np.zeros(G.shape[0])
    return G @ sla.cho_solve(sla.cho_factor(G.T @ G + noise * np.eye(n), lower=True), np.asarray(y, np.float64))


def _dense(phi_f, x, xt, noise):
    phi_f = sp.csr_matrix(phi_f, dtype=np.float64)
    x, xt = np.asarray(x, np.int64), np.asarray(xt, np.int64)
    rt, rx = phi_f[xt], phi_f[x]
    kss = (rt @ rt.T).toarray()
    ksx = (rt @ rx.T).toarray()
    kxx = (rx @ rx.T).toarray() + noise * np.eye(x.size)
    return phi_f, kss, ksx, kxx


def dense_mean(phi_f, x, y, xt, noise):
    """K*x (Kxx + sigma^2 I)^-1 y and sum_j |K*x,j| |alpha_j| (the scale of the mean's cancellations)."""
    _, _, ksx, kxx = _dense(phi_f, x, xt, noise)
    if len(x) == 0:
        return np.zeros(len(xt)), np.zeros(len(xt))
    alpha = sla.cho_solve(sla.cho_factor(kxx, lower=True), np.asarray(y, np.float64))
    return ksx @ alpha, np.abs(ksx) @ np.abs(alpha)


def dense_covariance(phi_f, x, xt, noise):
    """K** - K*x (Kxx + sigma^2 I)^-1 Kx* and K** (float64 [q, q])."""
    _, kss, ksx, kxx = _dense(phi_f, x, xt, noise)
    if len(x) == 0:
        return kss, kss
    return kss - ksx @ sla.cho_solve(sla.cho_factor(kxx, lower=True), ksx.T), kss


def dense_sample(phi_f, x, y, xt, noise, eps, eps_noise):
    """Pathwise samples [s, q]: Phi_f[x*] eps + K*x (Kxx + sigma^2 I)^-1 (y - Phi_f[x] eps - sigma E), with eps
    [s, N] and E [s, n] given (SparseGraphGP.predict with an exact solve)."""
    phi_f, _, ksx, kxx = _dense(phi_f, x, xt, noise)
    eps = np.asarray(eps, np.float64)
    prior_t = (phi_f[np.asarray(xt, np.int64)] @ eps.T).T
    if len(x) == 0:
        return prior_t
    prior_x = (phi_f[np.asarray(x, np.int64)] @ eps.T).T
    v = np.asarray(y, np.float64)[None, :] - prior_x - np.sqrt(noise) * np.asarray(eps_noise, np.float64)
    return prior_t + (ksx @ sla.cho_solve(sla.cho_factor(kxx, lower=True), v.T)).T
