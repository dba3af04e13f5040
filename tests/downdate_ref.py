"""float64 references of ExactPosterior.forget / set_targets, PosteriorMarginals across removals and
grf_phi_row_downdate (grf_b200/posterior.py, csrc/grf_posterior.cu), and the bound that holds a posterior changed by
any chain of appends and removals to a posterior constructed from scratch on the rows it keeps.

Downdate.  With B the removed positions (ascending), j0 = min B, R2 the kept positions after j0 and T = L[R2, j0:]:

    L' = [[L[:j0, :j0], 0], [L[R2, :j0], chol(T T^T)]],   C' = [C[:, :j0] | C[:, j0:] M],   M = T^T L'_22^-T
    Z = L^-1 E_B,  Z^T Z = R_B^T R_B,  W = Z R_B^-1,  U = C W:   C C^T - U U^T = C' C'^T

M and W have orthonormal columns.  Rows of C' of slots no kept row touches are exactly zero.

Error bound.  u = 2^-24.  Every slot is numbered in the union S_all of the columns any row of the history touches
(the posterior's slots are a permutation of a subset of it; the projections do not depend on the order, and a
candidate touches at most as many slots of the posterior as of S_all).  E bounds |C^ - C*| elementwise for the stored
C^ against the exact C* of the current rows:
  - built from scratch: E = u |C*|;
  - append (tests/condition_ref.py): E_new = u |C*_new| + E_old |L_21^T L_22^-T|;
  - removal: E'[:, :j0] = E[:, :j0], E'[:, j0:] = u |C*'[:, j0:]| + (E[:, j0:] + F64 |C*[:, j0:]|) |M|, and E' = 0
    on the rows no kept row touches (C' is set to exactly zero there);
  - U of a removal: u |U*| + (E[:, j0:] + F64 |C*[:, j0:]|) |W[j0:]|.
F64 = 2^-40 covers the float64 stages (Cholesky factors, solves, the products in row chunks) for kappa(K) <= 2^13,
as in tests/condition_ref.py.  The variance, mean, covariance and samples of the changed posterior then obey the
bounds of tests/condition_ref.py with E_c = E.

PosteriorMarginals holds q = fl32(|S* C0|^2) + sum over appended blocks |S* X|^2 - sum over removal blocks |S* U|^2,
which is |S* C*|^2 of the current rows in exact arithmetic.  Each block (exact X, bound E_X) contributes
sum_c (2 A + delta) delta (tests/condition_ref.py, proj_delta); the float32 rounding of the first q and of any
block refreshed through row_quadform adds at most u sum (A + delta)^2 per block, the float64 sums 2^-50 of that, and
the final var one float32 rounding.  ``marginal_bound`` doubles the total (O(u^2) terms, with room to spare)."""

from __future__ import annotations

import numpy as np
import scipy.linalg as sla

import condition_ref as CR

U = CR.U
F64 = CR.F64


def downdate(L, C, positions):
    """(L', C', U, M, W) of removing ``positions`` (any order) from the factor L [n, n] and C [m, n]; U is [m, b],
    M [n - j0, n2], W [n - j0, b] (the rows of Z R_B^-1 from j0 on)."""
    n = L.shape[0]
    pos = np.sort(np.asarray(positions, np.int64))
    b = pos.size
    j0 = int(pos[0])
    kept = np.setdiff1d(np.arange(n), pos)
    r2 = kept[kept > j0]
    nn, n2 = n - b, r2.size
    T = L[r2, j0:]
    Lp = np.zeros((nn, nn))
    Lp[:j0, :j0] = L[:j0, :j0]
    Lp[j0:, :j0] = L[r2, :j0]
    M = np.zeros((n - j0, 0))
    if n2:
        l22 = np.linalg.cholesky(T @ T.T)
        Lp[j0:, j0:] = l22
        M = sla.solve_triangular(l22, T, lower=True).T
    Cp = np.c_[C[:, :j0], C[:, j0:] @ M]
    Eb = np.zeros((n, b))
    Eb[pos, np.arange(b)] = 1.0
    Z = sla.solve_triangular(L, Eb, lower=True)
    rb = np.linalg.cholesky(Z.T @ Z).T                   # upper R_B
    W = sla.solve_triangular(rb, Z.T, lower=False, trans="T").T
    return Lp, Cp, C @ W, M, W[j0:]


def row_downdate(ti, col, w, n, slot, B, r, with_mean, q, d):
    """(q, var, mean) after grf_phi_row_downdate in float64: q - sum_{c < r} p_c^2, max(d - q, 0) (NaN stays),
    p_r (or None)."""
    q2, _, mean = CR.row_condition(ti, col, w, n, slot, B, r, with_mean, np.zeros(n), np.zeros(n))
    q = np.asarray(q, np.float64) - q2
    diff = np.asarray(d, np.float64) - q
    return q, np.where(np.isnan(diff), diff, np.maximum(diff, 0.0)), mean


def exact(G, order, noise):
    """(L, C*) of the training columns ``order`` of G [m_all, rows] from scratch."""
    Gx = G[:, order]
    nt = Gx.shape[1]
    if nt == 0:
        return np.zeros((0, 0)), np.zeros((G.shape[0], 0))
    L = np.linalg.cholesky(Gx.T @ Gx + noise * np.eye(nt))
    return L, sla.solve_triangular(L, Gx.T, lower=True).T


class Track:
    """The exact state of a posterior through a chain of appends and removals, the bound E of its stored C, and
    the blocks every PosteriorMarginals made along the way has to replay.  G: [m_all, rows] over the union slots of
    every row the history touches; rows are named by their column in G."""

    def __init__(self, G, order, noise):
        self.G, self.noise = G, noise
        self.order = np.asarray(order, np.int64)
        self.L, self.C = exact(G, self.order, noise)
        self.E = U * np.abs(self.C)
        self.watch = []
        self.kappa = [self._kappa()]

    def _kappa(self):
        Gx = self.G[:, self.order]
        return np.linalg.cond(Gx.T @ Gx + self.noise * np.eye(len(self.order))) if len(self.order) else 1.0

    def append(self, rows):
        n, b = len(self.order), len(rows)
        self.order = np.r_[self.order, np.asarray(rows, np.int64)]
        self.L, self.C = exact(self.G, self.order, self.noise)
        l21, l22 = self.L[n:, :n], self.L[n:, n:]
        M = sla.solve_triangular(l22, l21, lower=True).T if n else np.zeros((0, b))
        e_new = U * np.abs(self.C[:, n:]) + self.E @ np.abs(M)
        self.E = np.c_[self.E, e_new]
        for blocks in self.watch:
            blocks.append((1, self.C[:, n:].copy(), e_new))
        self.kappa.append(self._kappa())

    def remove(self, positions):
        pos = np.sort(np.asarray(positions, np.int64))
        j0 = int(pos[0])
        Lp, Cp, Uq, M, W = downdate(self.L, self.C, pos)
        kept = np.setdiff1d(np.arange(len(self.order)), pos)
        carry = self.E[:, j0:] + F64 * np.abs(self.C[:, j0:])
        e_u = U * np.abs(Uq) + carry @ np.abs(W)
        for blocks in self.watch:
            blocks.append((-1, Uq, e_u))
        self.order = self.order[kept]
        self.L, self.C = exact(self.G, self.order, self.noise)
        assert np.allclose(Lp, self.L, atol=1e-9 * max(1.0, np.abs(self.L).max(initial=0)))
        assert np.allclose(Cp, self.C, atol=1e-9 * max(1.0, np.abs(self.C).max(initial=0)))
        E = np.c_[self.E[:, :j0], U * np.abs(self.C[:, j0:]) + carry @ np.abs(M)]
        E[~self.live()] = 0.0
        self.E = E
        self.kappa.append(self._kappa())

    def live(self):
        """Slots some current training row touches."""
        return np.any(self.G[:, self.order] != 0, axis=1)

    def marginal(self):
        """Start the block list of a PosteriorMarginals made now."""
        blocks = [(1, self.C.copy(), self.E.copy())]
        self.watch.append(blocks)
        return blocks


def marginal_bound(ti, col, w, n, slot, blocks, var):
    """Bound on |var_marginals - var_exact| per candidate for the replayed blocks."""
    tot = np.zeros(n)
    mag = np.zeros(n)
    for _, X, EX in blocks:
        A, dl = CR.proj_delta(ti, col, w, n, slot, X, EX)
        tot += np.sum((2 * A + dl) * dl, axis=1)
        mag += np.sum((A + dl) ** 2, axis=1)
    return 2.0 * (tot + (U + 2.0 ** -50) * mag + U * np.abs(var))


def side_bound(A, dl, q, var):
    """Bound on |var_side - var_exact| for one posterior whose projections err by dl."""
    return 2.0 * (np.sum((2 * A + dl) * dl, axis=1) + 2 * U * (np.abs(q) + np.abs(var)))
