"""Host-side contract of the exact marginal likelihood (grf_b200/mll.py) and the per-length training Gram
(PhiBlocks.training_gram, csrc/grf_gram.cu): the float64 references of tests/exact_mll_ref.py, the closed-form
gradient, the memory-guard byte counts and the argument errors that need no device."""

import numpy as np
import pytest
import scipy.sparse as sp

import exact_mll_ref as R


def _mats(rng, N=60, L=3, density=0.08, hub=True):
    mats = []
    for _ in range(L):
        m = sp.random(N, N, density=density, random_state=rng, format="lil", dtype=np.float64)
        if hub:
            m[:, 7] = rng.uniform(0.1, 1.0, size=(N, 1))      # a column every row reaches
        mats.append(sp.csr_matrix(m.astype(np.float32)))
    return mats


@pytest.mark.parametrize("T", [0, 1, 3, 10, 10 ** 9])
def test_gram_split_matches_dense(T):
    rng = np.random.default_rng(1)
    mats = _mats(rng)
    x = np.r_[rng.choice(60, 25, replace=False), [4, 4]]              # repeated ids
    want = R.gram(mats, x)
    got, h, p_light = R.gram_split(mats, x, T)
    assert np.all(np.abs(got - want) <= R.gram_bound(mats, x))
    assert np.array_equal(got, got.T)
    a = R.stacked_rows(mats, x).toarray()
    t = (a != 0).sum(axis=0)
    assert h == int((t > T).sum())
    assert p_light == int((t[(t > 0) & (t <= T)].astype(np.int64) ** 2).sum())
    if T == 0:
        assert p_light == 0 and h == int((t > 0).sum())
    if T >= 10 ** 9:
        assert h == 0 and p_light == int((t.astype(np.int64) ** 2).sum())


def _problem(rng, n=12, L=3, N=40):
    a = rng.standard_normal((L * n, N)) * (rng.random((L * n, N)) < 0.3)
    E = (a @ a.T).reshape(L, n, L, n)
    y = rng.standard_normal(n)
    return E, y


@pytest.mark.parametrize("f", [[1.0, -0.4, 0.2], [0.7, 0.0, 0.3]])     # a zero entry keeps its gradient
def test_closed_form_gradient_matches_finite_differences(f):
    rng = np.random.default_rng(2)
    E, y = _problem(rng)
    f = np.asarray(f)
    noise = 0.3
    gf, gn = R.neg_mll_grad(E, f, noise, y)
    h = 1e-6
    for l in range(3):
        d = np.zeros(3)
        d[l] = h
        fd = (R.neg_mll(E, f + d, noise, y) - R.neg_mll(E, f - d, noise, y)) / (2 * h)
        assert abs(gf[l] - fd) <= 1e-6 * max(1.0, abs(fd)), (l, gf[l], fd)
    fd = (R.neg_mll(E, f, noise + h, y) - R.neg_mll(E, f, noise - h, y)) / (2 * h)
    assert abs(gn - fd) <= 1e-6 * max(1.0, abs(fd))
    assert gf[1] != 0.0 or f[1] != 0.0


def test_memory_guard_byte_counts():
    from grf_b200.engine import training_gram_bytes
    from grf_b200.mll import exact_mll_work_bytes

    assert training_gram_bytes(4096, 5, 0) == 8 * 20480 ** 2 == 3_355_443_200
    assert training_gram_bytes(100, 5, 7) == 8 * 500 ** 2 + 8 * 500 * 7
    assert training_gram_bytes(0, 32, 0) == 0
    assert exact_mll_work_bytes(4096, 5) == 8 * 4096 ** 2 * 9
    assert exact_mll_work_bytes(1, 1) == 40


def test_loss_function_routes_gradients_to_parameter_shapes():
    """The autograd Function hands the closed-form gradients back in the dtype and shape of f and sigma^2 (the
    likelihood's noise is a [1] tensor), scaled by the upstream gradient."""
    import torch

    from grf_b200.mll import _ExactLoss

    class Fixed:
        def _evaluate(self, f, noise):
            return {"loss": torch.tensor(1.5, dtype=torch.float64), "grad_f": torch.tensor([1.0, -2.0, 0.5],
                    dtype=torch.float64), "grad_noise": torch.tensor(0.25, dtype=torch.float64)}

    raw = torch.tensor([0.3, 0.1, -0.2], requires_grad=True)
    f = 2.0 * raw
    noise = torch.tensor([0.4], requires_grad=True)
    loss = _ExactLoss.apply(f, noise, Fixed())
    assert loss.dtype == torch.float64 and loss.item() == 1.5
    (3.0 * loss).backward()
    assert raw.grad.dtype == torch.float32 and torch.equal(raw.grad, torch.tensor([6.0, -12.0, 3.0]))
    assert noise.grad.shape == (1,) and float(noise.grad) == 0.75


def test_gram_entry_point_argument_errors():
    import ctypes

    from grf_b200 import _lib

    lib = _lib.lib()
    dummy = ctypes.c_void_p(16)
    rc = lib.grf_gram_light(None, 10, dummy, dummy, dummy, dummy, 3, dummy, 9, None)     # lde < n_rows
    assert rc == _lib.GRF_ERR_INVALID
    with pytest.raises(ValueError, match="grf_gram_light"):
        _lib.check(rc)
    with pytest.raises(ValueError, match="grf_gram_light: null"):
        _lib.check(lib.grf_gram_light(None, 10, None, dummy, dummy, dummy, 3, dummy, 10, None))
    with pytest.raises(ValueError, match="grf_gram_light"):
        _lib.check(lib.grf_gram_light(None, 10, dummy, dummy, dummy, dummy, -1, dummy, 10, None))
    assert lib.grf_gram_light(None, 0, None, None, None, None, 0, None, 0, None) == _lib.GRF_OK
    with pytest.raises(ValueError, match="grf_gram_mirror"):
        _lib.check(lib.grf_gram_mirror(dummy, 10, 4, None))
    with pytest.raises(ValueError, match="grf_gram_mirror: null"):
        _lib.check(lib.grf_gram_mirror(None, 10, 10, None))
    assert lib.grf_gram_mirror(None, 0, 0, None) == _lib.GRF_OK
