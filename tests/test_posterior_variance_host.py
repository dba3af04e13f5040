"""CPU self-test of the exact posterior variance contract (grf_b200/posterior.py, grf_phi_row_quadform) and of the
float64 references and bounds in tests/posterior_ref.py that the -m gpu tests use."""

import numpy as np
import scipy.sparse as sp

import posterior_ref as P


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


def _variance(phi_f, x, xt, noise):
    slot, G, C = P.exact_cache(phi_f, x, noise)
    ti, col, w = P.row_entries(phi_f.indptr, phi_f.indices, phi_f.data, xt)
    q, d, _, _ = P.quadform(ti, col, w, len(xt), slot, C)
    return np.maximum(d - q, 0.0), q, slot, G


def test_slots_g_and_c_give_the_dense_posterior_variance():
    phi = _phi(0, 60, 90, 6)
    x = np.array([3, 7, 11, 20, 21, 40, 55])
    xt = np.arange(60)
    got, _, slot, G = _variance(phi, x, xt, 0.3)
    want, prior = P.dense_variance(phi, x, xt, 0.3)
    assert np.allclose(got, want, rtol=1e-10, atol=1e-12 * prior.max())
    # slots: ranks of the touched columns in ascending order; G is Phi_f[x]^T restricted to them
    cols = np.flatnonzero(slot >= 0)
    assert np.array_equal(slot[cols], np.arange(cols.size))
    assert np.array_equal(cols, np.unique(phi[x].indices))
    assert np.array_equal(G, phi[x][:, cols].T.toarray())


def test_repeats_empty_rows_disjoint_rows_and_no_training_rows():
    phi = _phi(1, 50, 400, 4, empty=(5, 9))
    x = np.array([1, 1, 2, 5, 30, 30, 30])          # repeats and an empty training row
    xt = np.arange(50)
    got, q, slot, _ = _variance(phi, x, xt, 0.05)
    want, prior = P.dense_variance(phi, x, xt, 0.05)
    assert np.allclose(got, want, rtol=1e-9, atol=1e-12 * prior.max())
    # a test row sharing no column with the training rows: q is exactly zero, the variance is the prior
    disjoint = [i for i in xt if not np.any(slot[phi[i].indices] >= 0)]
    assert disjoint and all(q[i] == 0.0 for i in disjoint)
    assert got[5] == 0.0 and got[9] == 0.0          # empty test rows
    # n = 0: the prior diagonal; the disjoint rows return exactly that
    got0, q0, slot0, _ = _variance(phi, np.zeros(0, np.int64), xt, 0.05)
    assert np.all(slot0 == -1) and np.all(q0 == 0.0) and np.allclose(got0, prior, rtol=1e-14, atol=0)
    assert np.array_equal(got[disjoint], got0[disjoint])


def test_bound_holds_for_float32_and_catches_a_dropped_entry():
    rng = np.random.default_rng(2)
    m, r, N = 300, 37, 400
    lens = [257, 5, 0, 40]
    ti = np.repeat(np.arange(len(lens)), lens)
    col = np.concatenate([rng.choice(N, k, replace=False) for k in lens])
    w32 = (rng.choice([-1.0, 1.0], ti.size) * 2.0 ** rng.uniform(-6, 2, ti.size)).astype(np.float32)
    slot = np.full(N, -1, np.int32)
    touched = rng.choice(N, m, replace=False)
    slot[np.sort(touched)] = np.arange(m)
    C32 = rng.standard_normal((m, r)).astype(np.float32)
    want, dwant, bq, bd = P.quadform(ti, col, w32.astype(np.float64), len(lens), slot, C32)
    got, dgot = P.quadform_f32(ti, col, w32, len(lens), slot, C32)
    assert np.all(np.abs(got - want) <= bq) and np.all(np.abs(dgot - dwant) <= bd)
    assert got[2] == 0.0 and dgot[2] == 0.0
    # drop the heaviest touched entry of the 257-entry row
    row0 = np.flatnonzero((ti == 0) & (slot[col] >= 0))
    drop = row0[np.argmax(np.abs(w32[row0]))]
    keep = np.arange(ti.size) != drop
    bad, _ = P.quadform_f32(ti[keep], col[keep], w32[keep], len(lens), slot, C32)
    assert abs(bad[0] - want[0]) > bq[0]
