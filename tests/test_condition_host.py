"""CPU self-test of the conditioning contract (ExactPosterior.condition_on, PosteriorMarginals,
grf_phi_row_condition): the block update of tests/condition_ref.py against a dense refactor, the row-condition
formula, the bound that compares a conditioned posterior with one built from scratch (it holds for the float32
storage of C and fails when the last appended column is lost), the byte count and the binding's argument errors."""

import numpy as np
import pytest
import scipy.sparse as sp

import condition_ref as CR
import posterior_ref as P


def _phi(seed, n_rows, N, density=0.02):
    rng = np.random.default_rng(seed)
    phi = sp.random(n_rows, N, density=density, random_state=seed, format="csr", dtype=np.float64)
    phi.data = rng.standard_normal(phi.nnz) * 0.5
    return phi


def _slots(phi, x):
    """The union's slot map in condition_on's order: the first rows' columns ascending, then each batch's new
    columns ascending."""
    N = phi.shape[1]
    slot = np.full(N, -1, np.int64)
    m = 0
    for xs in x:
        cols = np.unique(phi[np.asarray(xs, np.int64)].indices) if len(xs) else np.zeros(0, np.int64)
        fresh = cols[slot[cols] < 0]
        slot[fresh] = np.arange(m, m + fresh.size)
        m += fresh.size
    return slot, m


def _G(phi, x, slot, m):
    rows = phi[np.asarray(x, np.int64)].tocoo()
    G = np.zeros((m, len(x)))
    G[slot[rows.col], rows.row] = rows.data
    return G


def _condition_chain(phi, x0, batches, noise, y):
    """L, C (float64) and a after condition_on calls in the reference algebra, with the union's slot map."""
    slot, m = _slots(phi, [x0] + batches)
    x = np.asarray(x0, np.int64)
    G = _G(phi, x, slot, m)
    n = len(x)
    L = np.linalg.cholesky(G.T @ G + noise * np.eye(n)) if n else np.zeros((0, 0))
    C = np.linalg.solve(L, G.T).T if n else np.zeros((m, 0))
    for xb in batches:
        Gn = _G(phi, xb, slot, m)
        Lb, c_new, _ = CR.block_update(L, C, Gn, noise, Gn.T @ G, Gn.T @ Gn)
        L, C, G = Lb, np.c_[C, c_new], np.c_[G, Gn]
        x = np.r_[x, xb]
    return slot, L, C, CR.weights(G, L, y[:len(x)]), G


@pytest.mark.parametrize("b", [1, 7, 64, 100])
def test_block_update_matches_a_dense_refactor(b):
    phi = _phi(b, 400, 900)
    rng = np.random.default_rng(b)
    x0 = rng.integers(0, 400, 60)
    xb = rng.integers(0, 400, b)
    y = rng.standard_normal(60 + b)
    slot, L, C, a, G = _condition_chain(phi, x0, [xb], 0.1, y)
    Lf = np.linalg.cholesky(G.T @ G + 0.1 * np.eye(G.shape[1]))
    assert np.allclose(L, Lf, rtol=0, atol=1e-12)
    assert np.allclose(C, np.linalg.solve(Lf, G.T).T, rtol=0, atol=1e-12)
    assert np.allclose(a, CR.weights(G, Lf, y), rtol=0, atol=1e-10)
    # the same posterior as the contract's from-scratch cache, up to the slot permutation
    sf, Gf, Cf = P.exact_cache(phi, np.r_[x0, xb], 0.1)
    cols = np.flatnonzero(sf >= 0)
    assert np.array_equal(np.sort(cols), np.flatnonzero(slot >= 0))
    assert np.allclose(C[slot[cols]], Cf[sf[cols]], rtol=0, atol=1e-12)


def test_chains_empty_start_repeats_and_no_new_column():
    phi = _phi(3, 300, 700)
    rng = np.random.default_rng(3)
    x0 = rng.integers(0, 300, 30)
    batches = [rng.integers(0, 300, 5) for _ in range(5)]
    batches[2] = np.r_[x0[:3], x0[:3]]                 # repeated ids, already in x: no new column
    y = rng.standard_normal(30 + 35)
    for start in (x0, np.zeros(0, np.int64)):          # n = 0 start too
        slot, L, C, a, G = _condition_chain(phi, start, batches, 0.05, y)
        Lf = np.linalg.cholesky(G.T @ G + 0.05 * np.eye(G.shape[1]))
        assert np.allclose(L, Lf, atol=1e-12) and np.allclose(C, np.linalg.solve(Lf, G.T).T, atol=1e-12)
        assert np.allclose(a, CR.weights(G, Lf, y[:G.shape[1]]), atol=1e-10)
    s_before, m_before = _slots(phi, [x0] + batches[:2])
    s_after, m_after = _slots(phi, [x0] + batches[:3])
    assert m_after == m_before and np.array_equal(s_before, s_after)


def test_row_condition_formula():
    rng = np.random.default_rng(5)
    phi = _phi(5, 50, 120, 0.1)
    slot = np.where(rng.random(120) < 0.5, np.arange(120), -1)
    B = rng.standard_normal((120, 6))
    ti, col, w = P.row_entries(phi.indptr, phi.indices, phi.data, np.arange(50))
    q0 = rng.random(50)
    d = q0 + 3.0
    d[0] = np.nan
    q, var, mean = CR.row_condition(ti, col, w, 50, slot, B, 5, 1, q0, d)
    S = phi.toarray()[:, slot >= 0] @ B[slot[slot >= 0]]
    assert np.allclose(q, q0 + np.sum(S[:, :5] ** 2, 1)) and np.allclose(mean, S[:, 5])
    assert np.isnan(var[0]) and np.all(var[1:] >= 0)
    assert np.allclose(var[1:], np.maximum(d[1:] - q[1:], 0))
    q2, _, none = CR.row_condition(ti, col, w, 50, slot, B, 5, 0, q, d)
    assert none is None and np.allclose(q2, q + np.sum(S[:, :5] ** 2, 1))      # accumulates, not overwritten


def _f32_posterior(phi, x0, batches, noise, xt):
    """Variance at xt the way both sides form it on the device: the conditioned side with C_old stored in float32
    inside the C_new product, the fresh side from the float64 C rounded once; q and d as float32 projections."""
    slot, m = _slots(phi, [x0] + batches)
    x = np.asarray(x0, np.int64)
    G = _G(phi, x, slot, m)
    n = len(x)
    L = np.linalg.cholesky(G.T @ G + noise * np.eye(n))
    C32 = np.linalg.solve(L, G.T).T.astype(np.float32)
    for xb in batches:
        Gn = _G(phi, xb, slot, m)
        Lb, c_new, _ = CR.block_update(L, C32.astype(np.float64), Gn, noise, Gn.T @ G, Gn.T @ Gn)
        L, C32, G = Lb, np.c_[C32, c_new.astype(np.float32)], np.c_[G, Gn]
    ti, col, w = P.row_entries(phi.indptr, phi.indices, phi.data.astype(np.float32), xt)
    q_c = P.quadform_f32(ti, col, w, len(xt), slot, C32)[0].astype(np.float64)
    return slot, G, C32, ti, col, w, q_c


def test_bound_holds_and_catches_a_lost_column():
    phi = _phi(8, 300, 600, 0.03)
    rng = np.random.default_rng(8)
    x0 = rng.integers(0, 300, 40)
    batches = [rng.integers(0, 300, 7), rng.integers(0, 300, 9)]
    xt = np.r_[np.arange(300), batches[-1]]
    slot, G, C32, ti, col, w, q_c = _f32_posterior(phi, x0, batches, 0.1, xt)
    L, C, E_c, E_f, kappa = CR.chain(G, len(x0), [len(b) for b in batches], 0.1)
    assert kappa <= CR.KAPPA_MAX
    nq = len(xt)
    d = np.bincount(ti, weights=w.astype(np.float64) ** 2, minlength=nq)
    q_f = P.quadform_f32(ti, col, w, nq, slot, C.astype(np.float32))[0].astype(np.float64)
    var_c, var_f = np.maximum(d - q_c, 0), np.maximum(d - q_f, 0)
    A, dc = CR.proj_delta(ti, col, w, nq, slot, C, E_c)
    _, df = CR.proj_delta(ti, col, w, nq, slot, C, E_f)
    bound = CR.var_bound(A, dc, df, q_f, var_f)
    assert np.all(np.abs(var_c - var_f) <= bound)
    # the last appended column dropped: the last new training node itself leaves the bound by far
    S = P.quadform(ti, col, w, nq, slot, C[:, -1:])[0]
    lost = np.maximum(d - (q_c - S), 0)
    assert np.abs(lost - var_f)[-1] > 100 * bound[-1]


def test_condition_bytes():
    from grf_b200.posterior import condition_bytes

    # n = 600, b = 50, m = 40000, 9000 old entries: C 4 m 652, L 8 650^2, G_new^T 8 b m, chunk rows 8 (n + 2b),
    # K_21 products 16 nnz_old b
    chunk = min(40000, (1 << 28) // (8 * 600))
    want = 4 * 40000 * 652 + 8 * 650 ** 2 + 8 * 50 * 40000 + 8 * chunk * 700 + 16 * 9000 * 50
    assert condition_bytes(600, 50, 40000, 9000) == want
    assert condition_bytes(0, 3, 10, 0) == 4 * 10 * 4 + 8 * 9 + 8 * 3 * 10 + 8 * 10 * 6


def _cpu_blocks():
    import torch

    from grf_b200.engine import PhiBlocks

    blk = PhiBlocks.__new__(PhiBlocks)
    blk.blk_ptr = torch.zeros(11, dtype=torch.int32)          # on the CPU: the checks run before any launch
    blk.n_steps, blk.n_cols, blk.n_rows, blk.row_lo = 1, 10, 10, 0
    return blk, torch


def test_row_condition_binding_argument_errors():
    """PhiBlocks.row_condition refuses bad operands before it reaches the library."""
    blk, torch = _cpu_blocks()
    one, slot, x = torch.ones(1), torch.zeros(10, dtype=torch.int32), torch.arange(4)
    B = torch.zeros((3, 5))
    q, d, var, mean = torch.zeros(4, dtype=torch.float64), torch.zeros(4), torch.zeros(4), torch.zeros(4)
    bad = [
        dict(r=0, with_mean=False),                      # k = 0
        dict(r=64, with_mean=True),                      # k = 65
        dict(r=-1, with_mean=True),
        dict(B=torch.zeros((3, 3)), r=3, with_mean=True),   # B narrower than k
        dict(B=torch.zeros((3, 5), dtype=torch.float64)),
        dict(col_slot=torch.zeros(9, dtype=torch.int32)),
        dict(q=torch.zeros(4)),                          # q must be float64
        dict(d=torch.zeros(5)),
        dict(var=torch.zeros(8)[::2]),
        dict(mean=None),                                 # with_mean needs mean
        dict(col_slot=torch.full((10,), 3, dtype=torch.int32)),   # names row 3 of a 3-row B
    ]
    good = dict(f=one, x=x, col_slot=slot, B=B, r=4, with_mean=True, q=q, d=d, var=var, mean=mean)
    for b in bad:
        with pytest.raises(ValueError, match="row_condition"):
            blk.row_condition(**dict(good, **b))
