"""CPU restatement of the kernel-matrix contract (csrc/grf_kernel_matrix.cu) checked against scipy.

The reference forms Phi = sum_p f_p M_p by scipy additions and returns Phi @ Phi.T.  ``ref_kernel`` below
restates the rules the device code follows -- the Phi fold and zero-drop, the product's left fold over k,
its zero-drop and its row order (descending by (first k that touched j, j)), the index dtype -- and must
equal scipy in indptr, indices, data (bitwise) and dtypes.  The GPU tests compare the device result with
scipy itself."""

import zlib

import numpy as np
import pytest
import scipy.sparse as sp

from grf_b200.kernel_matrix import kernel_index_dtype, modulator_f64


def ref_kernel(mats, f):
    n = mats[0].shape[0]
    fv = modulator_f64(f, len(mats))
    phi = []
    for r in range(n):
        acc = {}
        for p, fp in enumerate(fv):
            m = mats[p]
            for c, v in zip(m.indices[m.indptr[r]:m.indptr[r + 1]], m.data[m.indptr[r]:m.indptr[r + 1]]):
                acc[int(c)] = acc.get(int(c), 0.0) + float(fp) * float(v)
        phi.append(sorted((c, a) for c, a in acc.items() if a != 0))
    cols = [[] for _ in range(mats[0].shape[1])]
    for j, row in enumerate(phi):
        for c, a in row:
            cols[c].append((j, a))
    indptr, indices, data, touched = [0], [], [], 0
    for i in range(n):
        sums, first = {}, {}
        for p, (k, a) in enumerate(phi[i]):
            for j, b in cols[k]:
                if j not in sums:
                    sums[j], first[j] = 0.0, p
                sums[j] = sums[j] + a * b
        touched += len(sums)
        for _, j in sorted(((first[j], j) for j in sums if sums[j] != 0), reverse=True):
            indices.append(j)
            data.append(sums[j])
        indptr.append(len(indices))
    if touched == 0:
        return sp.csr_matrix((n, n))
    idx = kernel_index_dtype(n, touched, len(indices))
    return sp.csr_matrix((np.asarray(data, dtype=np.float64), np.asarray(indices, dtype=idx),
                          np.asarray(indptr, dtype=idx)), shape=(n, n))


def scipy_kernel(mats, f):
    n = mats[0].shape[0]
    phi = sp.csr_matrix((n, n))
    for step, f_p in enumerate(f):
        if step < len(mats):
            phi += f_p * mats[step]
    return phi @ phi.T


def assert_same(got, want):
    assert type(got) is type(want)
    for name in ("indptr", "indices"):
        a, b = getattr(got, name), getattr(want, name)
        assert a.dtype == b.dtype, name
        assert np.array_equal(a, b), name
    assert got.data.dtype == want.data.dtype
    assert np.array_equal(got.data.view(np.int64), want.data.view(np.int64))


def random_steps(rng, n, L, density, ints=False, zeros=False, index_dtype=np.int32):
    mats = []
    for _ in range(L):
        m = sp.random(n, n, density=density, format="csr", random_state=rng,
                      data_rvs=(lambda k: rng.integers(-2, 3, k).astype(float)) if ints else None)
        m.sort_indices()
        if zeros and m.nnz:
            m.data[rng.random(m.nnz) < 0.2] = 0.0      # explicit stored zeros
        m.indices = m.indices.astype(index_dtype)
        m.indptr = m.indptr.astype(index_dtype)
        mats.append(m)
    return mats


MODULATORS = {
    "float64": [1.0, -0.5, 0.25, 0.125],
    "float32": list(np.array([0.7, -1.3, 0.1, 2.2], dtype=np.float32)),
    "int": [1, -1, 2, 0],
    "python_float_short": [0.3, 1.7],
    "long": [1.0, 1.0, -1.0, 0.5, 3.0, 9.0],
    "empty": [],
    "cancel": [1.0, -1.0, 1.0, -1.0],
}


@pytest.mark.parametrize("mod", sorted(MODULATORS))
@pytest.mark.parametrize("case", ["ints_zeros", "floats", "sparse_rows", "wide_index"])
def test_restatement_equals_scipy(mod, case):
    rng = np.random.default_rng(zlib.crc32(f"{mod}/{case}".encode()))
    L = 4
    if case == "ints_zeros":
        mats = random_steps(rng, 30, L, 0.15, ints=True, zeros=True)
    elif case == "floats":
        mats = random_steps(rng, 40, L, 0.1)
    elif case == "sparse_rows":
        mats = random_steps(rng, 50, L, 0.01, ints=True)      # many empty rows
    else:
        mats = random_steps(rng, 25, L, 0.2, ints=True, index_dtype=np.int64)
    f = MODULATORS[mod]
    assert_same(ref_kernel(mats, f), scipy_kernel(mats, f))


def test_exact_cancellation_and_identity_steps():
    # M_1 = -M_0 with f = (1, 1): Phi is empty, nothing is touched -> csr_matrix((N, N))
    rng = np.random.default_rng(3)
    m0 = random_steps(rng, 20, 1, 0.2, ints=True)[0]
    mats = [m0, (-m0).tocsr()]
    want = scipy_kernel(mats, [1.0, 1.0])
    assert want.nnz == 0 and want.indices.dtype == np.int32
    assert_same(ref_kernel(mats, [1.0, 1.0]), want)
    # products that cancel inside K: rows (1, 1) and (1, -1) are orthogonal
    a = sp.csr_matrix(np.array([[1.0, 1.0, 0], [1.0, -1.0, 0], [0, 0, 0]]))
    mats = [a]
    want = scipy_kernel(mats, [1.0])
    assert want[0, 1] == 0 and want.nnz == 2
    assert_same(ref_kernel(mats, [1.0]), want)


def test_nan_is_kept():
    a = sp.csr_matrix(np.array([[np.nan, 1.0], [0.0, 2.0]]))
    assert_same(ref_kernel([a], [1.0]), scipy_kernel([a], [1.0]))


def test_modulator_widening():
    f = modulator_f64([np.float32(0.1), 2, 0.3, True, np.float16(0.5)], 10)
    assert f.dtype == np.float64
    assert f[0] == float(np.float32(0.1)) and f[1] == 2.0 and f[3] == 1.0 and f[4] == 0.5
    assert modulator_f64([1.0, 2.0, 3.0], 2).tolist() == [1.0, 2.0]
    assert modulator_f64(iter([1.0, 2.0]), 5).tolist() == [1.0, 2.0]
    with pytest.raises(TypeError):
        modulator_f64([1 + 2j], 3)
    with pytest.raises(TypeError):
        modulator_f64([np.longdouble(1.0)], 3)


def test_index_dtype_rule_matches_scipy():
    """scipy builds the product with check_contents=True: int64 only when N or the stored count needs it.
    Checked against scipy's own selection on arrays holding the boundary values (no 2^31-entry matrix)."""
    big = 2**31
    m = sp.csr_matrix((2, 2))
    for n, stored in [(10, 5), (10, big - 1), (10, big), (big, 5), (big - 1, big - 1)]:
        indptr = np.array([0, stored], dtype=np.int64)
        indices = np.array([0, n - 1], dtype=np.int64)
        want = m._get_index_dtype((indices, indptr), maxval=n, check_contents=True)
        assert kernel_index_dtype(n, touched=max(stored, 1), stored=stored) == want, (n, stored)
    assert kernel_index_dtype(10, 0, 0) == np.int32
    # int64 inputs with small contents come back as int32, as the rule says
    rng = np.random.default_rng(0)
    mats = random_steps(rng, 20, 2, 0.2, index_dtype=np.int64)
    assert scipy_kernel(mats, [1.0, 0.5]).indices.dtype == np.int32
    assert not scipy_kernel(mats, [1.0, 0.5]).has_sorted_indices
