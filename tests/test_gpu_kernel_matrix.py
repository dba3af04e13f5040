"""-m gpu: the sparse kernel matrix K = Phi_f Phi_f^T formed on the device (csrc/grf_kernel_matrix.cu) equals
scipy's ``Phi @ Phi.T`` on the same step matrices in indptr, indices, data (bitwise) and dtypes."""

import ctypes
import gc

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_golden
from gpu_util import grid_graph, powerlaw_graph, random_graph, ring_graph
from test_kernel_matrix_host import assert_same, scipy_kernel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import torch

    assert torch.cuda.is_available(), "these tests need a B200"
    from grf_b200 import _lib, engine, kernel_matrix
    from oracle import grf_oracle

    return dict(torch=torch, lib=_lib, eng=engine, km=kernel_matrix, o=grf_oracle)


def _steps(env, adj, W, p, L, seed=42, load_mode=0, scale_mode=0, coupling="iid"):
    eng = env["eng"]
    g = eng.DeviceGraph.laplacian_of(adj)
    cfg = eng.WalkConfig(W, p, L, seed=seed, load_mode=load_mode, coupling=coupling)
    return eng.build_step_matrices(g, cfg, scale_mode=scale_mode)


def _check(steps, f):
    got = steps.kernel_matrix(f).to_scipy()
    want = scipy_kernel(steps.to_scipy(), f)
    assert_same(got, want)
    return got


def _kernels(env, fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        env["torch"].cuda.synchronize()
    return {e.key.replace(" ", "") for e in prof.key_averages()}


def test_replayed_golden_kernels(env):
    """The drop-in on the three kernels.npz cases: equal to the old host path and to the golden K."""
    from efficient_graph_gp_sparse.graph_kernels_sparse.fast_grf_kernel_general import fast_general_grf_kernel
    from efficient_graph_gp_sparse.random_walk_samplers_sparse import SparseRandomWalk

    z = load_golden("kernels.npz")
    nproc = int(z["n_processes"])
    for name in ("cycle4", "grid6x4", "gnm40w"):
        adj, f = sp.csr_matrix(z[name + "_adj"]), z[name + "_f"]
        lap = env["o"].normalized_laplacian_sparse(adj)
        _, trace = env["o"].sparse_step_matrices(lap, 10, 0.2, 3, seed=None, n_processes=nproc, record=True)
        got = fast_general_grf_kernel(adj, f, walks_per_node=10, p_halt=0.2, max_walk_length=3, trace=trace)
        mats = SparseRandomWalk.on_normalized_laplacian(adj).get_random_walk_matrices(10, 0.2, 3, trace=trace)
        assert_same(got, scipy_kernel(mats, f))
        assert np.array_equal(got.toarray(), z[name + "_K_sparse"]), name


@pytest.mark.parametrize("f", [np.float32([1.0, -0.5, 0.25, 0.1, 2.0]), [1, 2, 0], [0.5] * 9, [], [0.0, 0.0]],
                         ids=["float32", "int_short", "long", "empty", "zeros"])
def test_grid_native(env, f):
    steps = _steps(env, grid_graph(40, 30), 100, 0.1, 5)
    _check(steps, f)


@pytest.mark.parametrize("load_mode,scale_mode", [(0, 1), (1, 0), (2, 1)])
def test_weighted_modes(env, load_mode, scale_mode):
    steps = _steps(env, random_graph(500, 1500, 3, weighted=True), 33, 0.2, 4, seed=7, load_mode=load_mode,
                   scale_mode=scale_mode)
    _check(steps, np.float32([0.9, -0.4, 0.3, 0.05]))


def test_powerlaw_hub_uses_global_table(env):
    steps = _steps(env, powerlaw_graph(3000, 20000, 1), 64, 0.1, 5, seed=99)
    names = _kernels(env, lambda: steps.kernel_matrix([1.0, 0.5, 0.25, 0.125, 0.0625]))
    assert any("kmat_rows_global_kernel<true>" in k for k in names), names
    k = _check(steps, [1.0, 0.5, 0.25, 0.125, 0.0625])
    assert np.diff(k.indptr).max() > 2048          # a hub row beyond the shared-memory bins


def test_L1_is_diagonal_and_isolated_nodes(env):
    adj = random_graph(300, 600, 5).tolil()
    adj[:, 7] = 0
    adj[7, :] = 0                                   # isolated node: a dead end, its Laplacian row is empty
    adj = adj.tocsr()
    adj.eliminate_zeros()
    steps = _steps(env, adj, 20, 0.1, 1)
    k = _check(steps, [1.5])
    assert np.array_equal(k.indices, np.repeat(np.arange(300), np.diff(k.indptr))) and np.all(k.data == 2.25)
    _check(_steps(env, adj, 20, 0.1, 4), [1.0, -0.3, 0.2, 0.1])


@pytest.mark.parametrize("coupling", ["antithetic", "repelling", "antithetic+repelling"])
def test_couplings_through_drop_in(env, coupling):
    from efficient_graph_gp_sparse.graph_kernels_sparse.fast_grf_kernel_general import fast_general_grf_kernel
    from efficient_graph_gp_sparse.random_walk_samplers_sparse import SparseRandomWalk

    adj = grid_graph(20, 15)
    f = [1.0, 0.6, 0.2, 0.1]
    got = fast_general_grf_kernel(adj, f, walks_per_node=16, p_halt=0.2, max_walk_length=4, coupling=coupling)
    mats = SparseRandomWalk.on_normalized_laplacian(adj).get_random_walk_matrices(16, 0.2, 4, coupling=coupling)
    assert_same(got, scipy_kernel(mats, f))


def test_config1_shape(env):
    steps = _steps(env, random_graph(2708, 5429, 11), 50, 0.1, 3)
    _check(steps, np.float32([1.0, 0.5, 0.25]))


def test_every_bin_and_repeatability(env):
    torch = env["torch"]
    cases = [(ring_graph(64), 8, 2), (grid_graph(40, 30), 100, 5), (random_graph(2000, 6000, 2), 50, 4),
             (powerlaw_graph(3000, 20000, 1), 64, 5)]
    names = set()
    for adj, W, L in cases:
        steps = _steps(env, adj, W, 0.1, L)
        f = [1.0 / (p + 1) for p in range(L)]
        names |= _kernels(env, lambda: steps.kernel_matrix(f))
        a, b = steps.kernel_matrix(f), steps.kernel_matrix(f)
        assert torch.equal(a.indptr, b.indptr) and torch.equal(a.indices, b.indices)
        assert torch.equal(a.data.view(torch.int64), b.data.view(torch.int64))
    for kern in ("kmat_phi_kernel", "kmat_tcount_kernel", "kmat_tfill_kernel", "kmat_size_kernel", "kmat_bin_kernel"):
        assert any(kern in k for k in names), kern
    for bin_ in ("warp", "cta", "global"):
        for mode in ("false", "true"):
            assert any(f"kmat_rows_{bin_}_kernel<{mode}>" in k for k in names), (bin_, mode, sorted(names))


def test_count_fill_through_lib(env):
    """grf_kmat_count / grf_kmat_fill on host-built operands: touched counts equal scipy's csr_matmat_maxnnz,
    the rows equal scipy's, and sentinels past the counted length stay untouched."""
    from scipy.sparse._sparsetools import csr_matmat_maxnnz

    torch, lib, eng = env["torch"], env["lib"], env["eng"]
    L = lib.lib()
    rng = np.random.default_rng(4)
    n = 3000
    phi = sp.random(n, n, density=0.004, format="csr", random_state=rng)
    phi = (phi + sp.csr_matrix((rng.standard_normal(400), (np.zeros(400, int), rng.choice(n, 400, replace=False))),
                               shape=(n, n))).tocsr()         # a dense row 0: a hub row of K
    phi.sort_indices()
    pt = phi.T.tocsr()
    want = phi @ phi.T
    dev = torch.device("cuda", torch.cuda.current_device())

    def up(a, dt):
        return torch.from_numpy(np.ascontiguousarray(a).astype(dt)).to(dev)

    ptr, col, val = up(phi.indptr, np.int64), up(phi.indices, np.int32), up(phi.data, np.float64)
    tptr, trow, tval = up(pt.indptr, np.int64), up(pt.indices, np.int32), up(pt.data, np.float64)
    st = eng._stream(dev)
    p = eng._ptr
    size = torch.empty(n, dtype=torch.int32, device=dev)
    lib.check(L.grf_kmat_row_sizes(p(ptr), p(col), p(tptr), n, p(size), st))
    rows, stats = env["km"]._bins(size, n, dev)
    assert stats[2] >= 1
    ctas = 3
    wsb = L.grf_kmat_workspace_bytes(stats[3], ctas)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    touched = torch.empty(n, dtype=torch.int32, device=dev)
    stored = torch.empty(n, dtype=torch.int32, device=dev)
    overflow = torch.empty(1, dtype=torch.int32, device=dev)
    ops = (p(ptr), p(col), p(val), p(tptr), p(trow), p(tval), n)
    lib.check(L.grf_kmat_count(*ops, p(size), p(rows), (ctypes.c_int64 * 3)(*stats[:3]), stats[3], ctas, p(ws), wsb,
                               p(touched), p(stored), p(overflow), st))
    assert int(overflow.item()) == 0
    ip = phi.indptr.astype(np.int32)
    ix = phi.indices.astype(np.int32)
    assert int(touched.sum()) == csr_matmat_maxnnz(n, n, ip, ix, pt.indptr.astype(np.int32),
                                                    pt.indices.astype(np.int32))
    assert np.array_equal(stored.cpu().numpy(), np.diff(want.indptr))
    kptr = torch.from_numpy(want.indptr.astype(np.int64)).to(dev)
    rows, stats = env["km"]._bins(touched, n, dev)
    wsb = L.grf_kmat_workspace_bytes(stats[3], ctas)
    ws = torch.empty(max(1, wsb), dtype=torch.uint8, device=dev)
    pad = 77
    kcol = torch.full((want.nnz + pad,), -5, dtype=torch.int32, device=dev)
    kval = torch.full((want.nnz + pad,), -7.5, dtype=torch.float64, device=dev)
    lib.check(L.grf_kmat_fill(*ops, p(touched), p(rows), (ctypes.c_int64 * 3)(*stats[:3]), stats[3], ctas, p(ws), wsb,
                              p(kptr), p(kcol), p(kval), p(overflow), st))
    assert int(overflow.item()) == 0
    kc, kv = kcol.cpu().numpy(), kval.cpu().numpy()
    assert np.all(kc[want.nnz:] == -5) and np.all(kv[want.nnz:] == -7.5)
    assert np.array_equal(kc[:want.nnz], want.indices)
    assert np.array_equal(kv[:want.nnz].view(np.int64), want.data.view(np.int64))


def test_too_large_k_raises_memory_error(env):
    torch = env["torch"]
    steps = _steps(env, grid_graph(40, 30), 100, 0.1, 5)
    f = [1.0, 0.5, 0.25, 0.1, 0.05]
    nnz = steps.kernel_matrix(f).nnz
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    with pytest.raises(MemoryError, match=f"nnz\\(K\\) = {nnz} ") as ei:
        steps.kernel_matrix(f, mem_limit=nnz * 12 - 1)
    del ei
    gc.collect()
    assert torch.cuda.memory_allocated() == before     # nothing of K was allocated, the temporaries are gone
