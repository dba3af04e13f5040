"""CPU checks of the host-side Phi builder and references that tests/test_gpu_matvec_abi.py compares the kernels
with: the host Phi^T is scipy's transpose, the profiles have the shapes the GPU table relies on, and the
per-element bound holds for a float32 evaluation while a dropped entry breaks it."""

import numpy as np
import pytest
import scipy.sparse as sp

import matvec_abi_ref as R


@pytest.fixture(scope="module")
def pl():
    return R.profile("pl")


@pytest.fixture(scope="module")
def l32():
    return R.profile("l32")


def _unpack(words):
    w = np.asarray(words).view(np.uint32)
    return (w >> np.uint32(R.SHIFT)).astype(np.int64), (w & np.uint32(R.COL_MASK)).astype(np.int64)


@pytest.mark.parametrize("name,rows", [("pl", None), ("l32", None), ("pl", (3001, 9000)), ("l32", (1000, 2500))])
def test_host_transpose_is_scipys(name, rows, request):
    hp = request.getfixturevalue(name)
    r0, r1 = rows or (0, hp.n_rows)
    tptr, tent = hp.transpose(r0, r1)
    length, row = _unpack(tent[:, 0])
    val = tent[:, 1].view(np.float32)
    L = hp.L
    for l in range(L):
        mt = sp.csr_matrix(hp.mat(l)[r0:r1].astype(np.float32).T)
        mt.sort_indices()
        for c in range(0, hp.n_cols, 7):
            b, e = tptr[c * L + l], tptr[c * L + l + 1]
            assert np.all(length[b:e] == l)
            assert np.array_equal(row[b:e], mt.indices[mt.indptr[c]:mt.indptr[c + 1]])
            assert np.array_equal(val[b:e].view(np.int32), mt.data[mt.indptr[c]:mt.indptr[c + 1]].view(np.int32))
        seg = np.diff(tptr)[l::L]
        assert np.array_equal(seg, np.diff(mt.indptr))


def test_phi_blocks_pack_the_matrices(l32):
    ent = l32.entries
    length, col = _unpack(ent[:, 0])
    assert (ent[:, 0] < 0).any(), "length 31 sets bit 31 of the packed column"
    ptr = l32.blk_ptr
    for r in (0, 7, 8, 2999):
        for l in range(32):
            b, e = ptr[r * 32 + l], ptr[r * 32 + l + 1]
            m = l32.mat(l)
            assert np.array_equal(col[b:e], m.indices[m.indptr[r]:m.indptr[r + 1]])
            assert np.all(length[b:e] == l)


def test_profiles_have_the_rows_the_table_needs(pl):
    lens, cols = pl.row_len, pl.col_len
    assert list(lens[R.SPECIAL_ROWS]) == [255, 256, 257, 512, 513, 769, 1100, 2000]
    assert (lens == 0).any() and (lens == 1).any() and (cols == 0).any() and cols.max() > 10 ** 4
    assert pl.nnz / pl.n_rows < 64 < R.profile("dense").nnz / 1500
    z = (pl.length == 0) & (pl.col == 0) & (pl.val.view(np.int32) == np.int32(-2 ** 31))
    assert z.sum() == 1, "one entry {length 0, column 0, -0.0}"
    mags = np.abs(pl.val[pl.val != 0])
    assert mags.min() < 2.0 ** -19 and mags.max() > 2.0 ** 3 and (pl.val < 0).any()


def test_band_profile_reaches_tiles_and_fallbacks():
    hp = R.profile("band")
    win, mw = R.windows(hp.blk_ptr, hp.entries, hp.n_rows, hp.L)
    tptr, tent = hp.transpose()
    twin, tmw = R.windows(tptr, tent, hp.n_cols, hp.L)
    for t in (4, 16):
        assert all(R.tiled_plan(win, mw, hp.n_rows, t)) and all(R.tiled_plan(twin, tmw, hp.n_cols, t))
    fwd = R.tiled_plan(win, mw, hp.n_rows, 64)
    assert 0 < sum(fwd) < len(fwd)
    assert R.tiled_plan(twin, tmw, hp.n_cols, 128) is None


def _float32_matvec(hp, f, x1, x2, v, row_lo, drop=None):
    """The product in float32 (scipy sums in the matrix dtype), optionally without entry `drop`."""
    keep = np.ones(hp.nnz, bool)
    if drop is not None:
        keep[drop] = False
    a = (hp.val * f[hp.length]).astype(np.float32)[keep]
    p = sp.csr_matrix((a, (hp.row[keep], hp.col[keep])), shape=(hp.n_rows, hp.n_cols), dtype=np.float32)
    s1 = R.selection(x1, row_lo, hp.n_rows).astype(np.float32)
    s2 = R.selection(x2, row_lo, hp.n_rows).astype(np.float32)
    u = ((s2 @ p).T @ v).astype(np.float32)
    return (s1 @ (p @ u)).astype(np.float32)


def test_bound_holds_for_float32_and_catches_a_dropped_entry(pl):
    rng = np.random.default_rng(3)
    f = np.array([0.75, 0.0, -1.5], np.float32)
    row_lo = 1000
    x1 = np.r_[R.SPECIAL_ROWS, rng.integers(0, pl.n_rows + 2000, 500)].astype(np.int32) + row_lo - 500
    x1[:len(R.SPECIAL_ROWS)] = R.SPECIAL_ROWS + row_lo
    x2 = rng.integers(0, pl.n_rows + 2000, 3000).astype(np.int32) + row_lo - 500
    v = rng.standard_normal((len(x2), 5)).astype(np.float32)
    want, bound = R.ref_matvec(pl, f, x1, x2, v, row_lo)
    got = _float32_matvec(pl, f, x1, x2, v, row_lo)
    assert np.all(np.abs(got - want) <= bound)
    # the classic bound is looser: 2^-22 (len + max_c len(Phi^T_c)) A
    # a 257-entry row that loses its last entry (a chunk bound off by one) leaves the bound
    ptr = pl.blk_ptr
    r = R.SPECIAL_ROWS[2]
    last = ptr[(r + 1) * pl.L] - 1
    for k in range(5):
        if f[pl.length[last - k]] != 0:
            last -= k
            break
    bad = _float32_matvec(pl, f, x1, x2, v, row_lo, drop=last)
    i = np.flatnonzero(x1 == r + row_lo)[0]
    assert np.any(np.abs(bad[i] - want[i]) > bound[i])


def test_fgrad_and_row_dots_references_agree_with_dense(l32):
    rng = np.random.default_rng(5)
    x = rng.integers(0, l32.n_rows, 40).astype(np.int32)
    left = rng.standard_normal((40, 3))
    p = rng.standard_normal((l32.n_cols, 3))
    want, bound = R.ref_fgrad(l32, x, left, p)
    for l in (0, 31):
        dense = l32.mat(l).toarray()[x]
        assert abs(want[l] - np.sum(left * (dense @ p))) <= 1e-9 * (1 + abs(want[l]))
    f = rng.standard_normal(32).astype(np.float32)
    x2 = rng.permutation(x).astype(np.int32)
    dots, dbound, both = R.ref_row_dots(l32, f, x, x2, 40)
    pf = R.HostPhi.phi_f(l32, f)[0].toarray()
    for i in (0, 17):
        for l in (0, 31):
            row = l32.mat(l).toarray()[x[i]]
            assert abs(dots[i, l] - np.sum(row * pf[x2[i]])) <= 1e-9 * (1 + abs(dots[i, l]))
