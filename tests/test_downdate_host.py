"""CPU self-test of the downdate contract (ExactPosterior.forget / set_targets, PosteriorMarginals across removals,
grf_phi_row_downdate): the algebra of tests/downdate_ref.py against a dense refactor of the kept rows (front,
middle, end, random subsets, every row, repeated ids), U against C C^T - C' C'^T, the row-downdate formula, the
error bound E of a float32 C carried through chains of appends and removals (it fails when the rows of retired slots
are not zeroed), the byte count and the positions rules."""

import numpy as np
import pytest
import scipy.sparse as sp

import condition_ref as CR
import downdate_ref as DR


def _phi(seed, n_rows, N, density=0.02):
    rng = np.random.default_rng(seed)
    phi = sp.random(n_rows, N, density=density, random_state=seed, format="csr", dtype=np.float64)
    phi.data = rng.standard_normal(phi.nnz) * 0.5
    return phi


def _G(phi, x):
    """G [m, len(x)] over the ascending union of the columns of the rows x."""
    rows = phi[np.asarray(x, np.int64)]
    cols = np.unique(rows.indices)
    return rows[:, cols].T.toarray()


def _state(phi, x, noise):
    G = _G(phi, x)
    L = np.linalg.cholesky(G.T @ G + noise * np.eye(len(x)))
    return G, L, np.linalg.solve(L, G.T).T


CASES = {
    "front": lambda n, rng: np.arange(0, 7),
    "front1": lambda n, rng: np.array([0]),
    "middle": lambda n, rng: np.arange(n // 2 - 8, n // 2 + 8),
    "end": lambda n, rng: np.arange(n - 16, n),
    "last": lambda n, rng: np.array([n - 1]),
    "random": lambda n, rng: rng.choice(n, 50, replace=False),
    "all": lambda n, rng: rng.permutation(n),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_downdate_matches_a_dense_refactor(case):
    phi = _phi(len(case), 300, 900)
    rng = np.random.default_rng(len(case))
    x = rng.integers(0, 300, 120)
    x[10:14] = x[3]                                   # repeated ids: positions, not ids, are removed
    noise = 0.1
    G, L, C = _state(phi, x, noise)
    pos = CASES[case](len(x), rng)
    Lp, Cp, Uq, M, W = DR.downdate(L, C, pos)
    kept = np.setdiff1d(np.arange(len(x)), pos)
    Gk = G[:, kept]
    K = Gk.T @ Gk + noise * np.eye(kept.size)
    assert np.allclose(Lp @ Lp.T, K, atol=1e-10)
    if kept.size:
        assert np.allclose(Lp, np.linalg.cholesky(K), atol=1e-10)
        assert np.allclose(Cp, np.linalg.solve(Lp, Gk.T).T, atol=1e-10)
    assert np.allclose(Cp @ Cp.T, C @ C.T - Uq @ Uq.T, atol=1e-10)
    assert np.allclose(M.T @ M, np.eye(M.shape[1]), atol=1e-10)
    assert np.allclose(W.T @ W, np.eye(W.shape[1]), atol=1e-10)
    j0 = int(np.min(pos))
    assert np.allclose(Uq, C[:, j0:] @ W, atol=1e-12)          # rows of Z before j0 are zero
    if case in ("end", "last"):                                  # trailing positions: a truncation
        assert np.array_equal(Lp, L[:j0, :j0]) and np.array_equal(Cp, C[:, :j0])


def test_repeated_id_positions_are_distinct_rows():
    """Removing any one copy of a repeated id leaves the same posterior: G_k K_k^-1 G_k^T of the kept rows."""
    phi = _phi(3, 200, 600)
    x = np.array([5, 9, 5, 11, 5, 13])
    G, L, C = _state(phi, x, 0.2)
    for p in (0, 2, 4):
        _, Cp, _, _, _ = DR.downdate(L, C, [p])
        Gk = G[:, np.delete(np.arange(6), p)]
        want = Gk @ np.linalg.solve(Gk.T @ Gk + 0.2 * np.eye(5), Gk.T)
        assert np.allclose(Cp @ Cp.T, want, atol=1e-10)


def test_row_downdate_undoes_row_condition():
    rng = np.random.default_rng(1)
    n, m, N = 40, 30, 80
    ti = np.repeat(np.arange(n), 5)
    col = rng.integers(0, N, ti.size)
    w = rng.standard_normal(ti.size)
    slot = np.full(N, -1)
    slot[rng.choice(N, m, replace=False)] = np.arange(m)
    B = rng.standard_normal((m, 6))
    q0, d = rng.uniform(0, 1, n), rng.uniform(5, 50, n)
    d[3] = np.nan
    q1, _, _ = CR.row_condition(ti, col, w, n, slot, B, 5, 1, q0, d)
    q2, var, mean = DR.row_downdate(ti, col, w, n, slot, B, 5, 1, q1, d)
    assert np.allclose(q2, q0, atol=1e-12)
    assert np.isnan(var[3]) and np.all(var[~np.isnan(var)] >= 0)
    _, _, mean_c = CR.row_condition(ti, col, w, n, slot, B, 5, 1, q0, d)
    assert np.array_equal(mean, mean_c)
    big = DR.row_downdate(ti, col, w, n, slot, B, 5, 0, np.zeros(n), d)[1]
    ok = ~np.isnan(d)                                 # q below zero: var = d - q grows, only negatives clamp
    assert np.all(big[ok] >= d[ok]) and np.isnan(big[3])


def _simulate(G_all, steps, noise, zero_dead=True):
    """float32 C of a posterior driven through ``steps`` (("add", rows) / ("remove", positions)), as the device
    computes it (float64 products of the stored float32 C, rounded once), with the exact Track alongside."""
    tr = DR.Track(G_all, steps[0][1], noise)
    C32 = tr.C.astype(np.float32)
    for kind, arg in steps[1:]:
        n = len(tr.order)
        if kind == "add":
            tr.append(arg)
            l21, l22 = tr.L[n:, :n], tr.L[n:, n:]
            Gn = G_all[:, np.asarray(arg)]
            c_new = np.linalg.solve(l22, (Gn - C32.astype(np.float64) @ l21.T).T).T if n else \
                np.linalg.solve(l22, Gn.T).T
            C32 = np.c_[C32, c_new.astype(np.float32)]
        else:
            pos = np.sort(np.asarray(arg))
            j0 = int(pos[0])
            _, _, _, M, _ = DR.downdate(tr.L, tr.C, pos)
            C32 = np.c_[C32[:, :j0], (C32[:, j0:].astype(np.float64) @ M).astype(np.float32)]
            tr.remove(pos)
            if zero_dead:
                C32[~tr.live()] = 0.0
    return tr, C32


def _chain_setup(seed):
    phi = _phi(seed, 400, 1200, 0.01)
    rng = np.random.default_rng(seed)
    rows = rng.permutation(400)[:260]
    G_all = _G(phi, rows)                             # union slots of every row the history touches
    steps = [("init", np.arange(0, 150)), ("remove", np.arange(0, 16)), ("add", np.arange(150, 200)),
             ("remove", rng.choice(184, 30, replace=False)), ("add", np.arange(200, 207)),
             ("remove", np.arange(150, 161)), ("add", np.arange(207, 260))]
    return G_all, steps


def test_chain_bound_holds_for_float32_storage():
    G_all, steps = _chain_setup(7)
    tr, C32 = _simulate(G_all, steps, 0.1)
    assert max(tr.kappa) <= CR.KAPPA_MAX
    err = np.abs(C32.astype(np.float64) - tr.C)
    assert np.all(err <= tr.E), np.max(err - tr.E)
    assert np.any(~tr.live())                         # the chain retires slots
    assert np.all(C32[~tr.live()] == 0)


def test_chain_bound_fails_when_retired_rows_are_kept():
    G_all, steps = _chain_setup(7)
    tr, C32 = _simulate(G_all, steps, 0.1, zero_dead=False)
    err = np.abs(C32.astype(np.float64) - tr.C)
    assert np.any(err > tr.E)


def test_marginal_blocks_replay_to_the_exact_q():
    G_all, steps = _chain_setup(8)
    tr = DR.Track(G_all, steps[0][1], 0.1)
    early = tr.marginal()
    for i, (kind, arg) in enumerate(steps[1:]):
        tr.append(arg) if kind == "add" else tr.remove(arg)
        if i == 2:
            late = tr.marginal()
    for blocks in (early, late):
        QQ = sum(s * X @ X.T for s, X, _ in blocks)
        assert np.allclose(QQ, tr.C @ tr.C.T, atol=1e-9)


def test_downdate_bytes():
    from grf_b200.posterior import downdate_bytes

    n, b, j0, m, nnz = 600, 16, 0, 5000, 40000
    nn, nt = n - b, n - j0
    n2 = nn - j0
    base = downdate_bytes(n, b, j0, m, nnz, logged=False)
    assert base >= 4 * m * ((nn + 3) // 4 * 4) + 8 * nn * nn + 16 * n2 * nt
    assert downdate_bytes(n, b, j0, m, nnz) - base >= 4 * m * b + 8 * nt * b
    assert downdate_bytes(n, b, n - b, m, nnz, logged=False) < base       # trailing removal: no product


def test_positions_rules():
    import torch
    from grf_b200.posterior import ExactPosterior

    class Fake:
        n = 5
        _positions = ExactPosterior._positions

    f = Fake()
    assert f._positions([3, 0, 4], "forget").tolist() == [3, 0, 4]
    assert f._positions([], "forget").numel() == 0
    assert f._positions(torch.tensor([1, 2], dtype=torch.int32), "forget").dtype == torch.int64
    for bad in ([5], [-1], [0, 7]):
        with pytest.raises(IndexError):
            f._positions(bad, "forget")
    with pytest.raises(ValueError, match="repeat"):
        f._positions([1, 2, 1], "forget")
    with pytest.raises(ValueError, match="integers"):
        f._positions([1.0], "forget")
