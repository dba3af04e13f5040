"""CPU self-test of the exact posterior mean, covariance and samples contract (grf_b200/posterior.py,
grf_phi_row_project): the projections of the cached factor restated in numpy against the dense float64 formulas of
tests/predictive_ref.py, and the projection bound the -m gpu tests use."""

import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp

import posterior_ref as P
import predictive_ref as Q


def _phi(seed, n, N, per_row, empty=()):
    rng = np.random.default_rng(seed)
    rows, cols = [], []
    for i in range(n):
        if i in empty:
            continue
        c = rng.choice(N, size=per_row, replace=False)
        rows += [i] * per_row
        cols += list(c)
    vals = rng.standard_normal(len(rows)) * 0.5
    return sp.csr_matrix((vals, (rows, cols)), shape=(n, N))


def _posterior(phi_f, x, y, xt, noise, eps, eps_noise):
    """mean, covariance and samples the way ExactPosterior forms them: projections of the rows x* onto a, C and
    C L^-1 V, plus the prior terms."""
    slot, G, C = P.exact_cache(phi_f, x, noise)
    n = len(x)
    ti, col, w = P.row_entries(phi_f.indptr, phi_f.indices, phi_f.data, xt)
    mean = Q.project(ti, col, w, len(xt), slot, Q.train_weights(G, noise, y)[:, None])[0][:, 0]
    p = Q.project(ti, col, w, len(xt), slot, C)[0]
    rt = phi_f[np.asarray(xt)]
    cov = (rt @ rt.T).toarray() - p @ p.T
    prior = (phi_f @ eps.T).T
    samples = prior[:, xt]
    if n:
        L = np.linalg.cholesky(G.T @ G + noise * np.eye(n))
        v = y[None, :] - prior[:, x] - np.sqrt(noise) * eps_noise
        B = C @ sla.solve_triangular(L, v.T, lower=True)
        samples = samples + Q.project(ti, col, w, len(xt), slot, B)[0].T
    return mean, cov, samples, slot


def _check(phi, x, xt, noise, seed=0, s=5):
    rng = np.random.default_rng(seed)
    y = rng.standard_normal(len(x))
    eps = rng.standard_normal((s, phi.shape[1]))
    eps_noise = rng.standard_normal((s, len(x)))
    mean, cov, samples, slot = _posterior(phi, x, y, xt, noise, eps, eps_noise)
    want_m, _ = Q.dense_mean(phi, x, y, xt, noise)
    want_c, kss = Q.dense_covariance(phi, x, xt, noise)
    want_s = Q.dense_sample(phi, x, y, xt, noise, eps, eps_noise)
    scale = np.sqrt(np.outer(np.diag(kss), np.diag(kss))) + 1e-300
    assert np.allclose(mean, want_m, rtol=1e-9, atol=1e-12 * max(1.0, np.abs(want_m).max(initial=0)))
    assert np.all(np.abs(cov - want_c) <= 1e-10 * scale + 1e-14)
    assert np.allclose(samples, want_s, rtol=1e-9, atol=1e-10)
    # the covariance's diagonal is the variance of tests/posterior_ref.py
    var, _ = P.dense_variance(phi, x, xt, noise)
    assert np.allclose(np.diag(cov), var, rtol=1e-9, atol=1e-12 * kss.max(initial=1.0))
    return mean, cov, slot, kss


def test_mean_covariance_and_samples_from_the_factor():
    phi = _phi(0, 60, 90, 6)
    _check(phi, np.array([3, 7, 11, 20, 21, 40, 55]), np.arange(60), 0.3)


def test_repeats_empty_rows_disjoint_rows_and_no_training_rows():
    phi = _phi(1, 50, 400, 4, empty=(5, 9))
    x = np.array([1, 1, 2, 5, 30, 30, 30])          # repeats and an empty training row
    xt = np.arange(50)
    mean, cov, slot, kss = _check(phi, x, xt, 0.05, seed=1)
    disjoint = [i for i in xt if not np.any(slot[phi[i].indices] >= 0)]
    assert disjoint
    # a test row sharing no column with the training rows: mean exactly 0, its covariance row the prior's
    assert all(mean[i] == 0.0 for i in disjoint)
    assert np.array_equal(cov[disjoint], kss[disjoint])
    assert np.all(cov[[5, 9]] == 0.0)               # empty test rows
    # n = 0: the prior
    mean0, cov0, _, _ = _check(phi, np.zeros(0, np.int64), xt, 0.05, seed=2)
    assert np.all(mean0 == 0.0) and np.array_equal(cov0, kss)


def test_projection_bound_holds_for_float32_and_catches_a_dropped_entry():
    rng = np.random.default_rng(2)
    m, r, N = 300, 5, 400
    lens = [257, 5, 0, 40]
    ti = np.repeat(np.arange(len(lens)), lens)
    col = np.concatenate([rng.choice(N, k, replace=False) for k in lens])
    w32 = (2.0 ** rng.uniform(-2, 2, ti.size)).astype(np.float32)
    col[np.flatnonzero(ti == 0)[-1]] = N - 1         # the 257-entry row's last entry: touched and heavy
    w32[np.flatnonzero(ti == 0)[-1]] = 64.0
    slot = np.full(N, -1, np.int32)
    touched = np.r_[rng.choice(N - 1, m - 1, replace=False), N - 1]
    slot[np.sort(touched)] = np.arange(m)
    B32 = rng.uniform(0.5, 1.0, (m, r)).astype(np.float32)
    want, bound = Q.project(ti, col, w32.astype(np.float64), len(lens), slot, B32)
    got = Q.project_f32(ti, col, w32, len(lens), slot, B32)
    assert np.all(np.abs(got - want) <= bound)
    assert np.all(got[2] == 0.0)
    # the same row without its last entry
    keep = np.arange(ti.size) != np.flatnonzero(ti == 0)[-1]
    bad = Q.project_f32(ti[keep], col[keep], w32[keep], len(lens), slot, B32)
    assert np.all(np.abs(bad[0] - want[0]) > bound[0])
