"""CPU tests of the host-side logic: the stand-in lazy-operator algebra (checked with a dense
backing operator), kernel / likelihood construction, Laplacians, modulators, CG restatement."""

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import load_golden
from grf_b200 import gp_compat, linop


def test_linop_algebra_against_dense():
    if linop.HAVE_UPSTREAM:
        pytest.skip("upstream linear_operator present")
    torch.manual_seed(0)
    a, b = torch.randn(7, 5), torch.randn(7, 5)
    A, B = linop.DenseLinearOperator(a), linop.DenseLinearOperator(b)
    v = torch.randn(5, 3)
    assert torch.allclose((A @ v), a @ v)
    assert torch.allclose((A.T @ torch.randn(7, 2)).shape == (5, 2) and (A.T).to_dense(), a.T)
    phi = sum(c * M for c, M in zip(torch.tensor([2.0, -1.0]), [A, B]))       # sparse_grf_kernel.py:59-61 idiom
    assert torch.allclose(phi.to_dense(), 2 * a - b)
    idx = torch.tensor([4, 0, 4, 6])
    assert torch.allclose(phi[idx].to_dense(), (2 * a - b)[idx])
    assert torch.allclose(phi[idx, :].to_dense(), (2 * a - b)[idx])
    K = phi[idx] @ phi[torch.tensor([1, 2])].transpose(-1, -2)                # Phi[x1] Phi[x2]^T
    want = (2 * a - b)[idx] @ (2 * a - b)[[1, 2]].T
    assert tuple(K.shape) == (4, 2) and torch.allclose(K.to_dense(), want, atol=1e-5)
    assert torch.allclose(K @ torch.ones(2), want @ torch.ones(2), atol=1e-5)
    eps = torch.randn(3, 5)
    assert torch.allclose(eps @ phi[idx].T, eps @ (2 * a - b)[idx].T, atol=1e-5)   # tensor @ operator
    S = (phi[idx] @ phi[idx].T) + 0.5 * linop.IdentityLinearOperator(4)
    assert torch.allclose(S.to_dense(), (2 * a - b)[idx] @ (2 * a - b)[idx].T + 0.5 * torch.eye(4), atol=1e-5)
    assert torch.allclose(S._matmul(torch.ones(4, 1)), S.to_dense() @ torch.ones(4, 1), atol=1e-5)
    assert torch.allclose((phi[idx] * phi[idx]).sum(dim=-1), ((2 * a - b)[idx] ** 2).sum(-1), atol=1e-5)


def test_kernels_construct_on_cpu_and_fail_loudly_without_gpu():
    from efficient_graph_gp_sparse.gptorch_kernels_sparse import SparseDiffusionKernel, SparseGRFKernel
    from efficient_graph_gp_sparse.preprocessor import GraphPreprocessor
    from efficient_graph_gp_sparse.utils_sparse import SparseLinearOperator

    eye = GraphPreprocessor.from_scipy_csr(sp.identity(4, format="csr"))
    ops = [SparseLinearOperator(eye) for _ in range(3)]
    torch.manual_seed(42)
    k = SparseGRFKernel(3, ops)
    torch.manual_seed(42)
    assert torch.equal(k.raw_modulator_vector.detach(), torch.randn(3))      # same init as the reference (:14-17)
    d = SparseDiffusionKernel(3, ops)
    assert float(d.beta) == pytest.approx(np.log1p(np.e), rel=1e-6)           # softplus(1.0)
    assert d.modulator_vector.shape == (3,)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            k(torch.tensor([0, 1]), torch.tensor([0, 1]))
    with pytest.raises(ValueError, match="CSR"):
        SparseLinearOperator(torch.eye(3))


def test_likelihood_and_settings_standins():
    if gp_compat.HAVE_GPYTORCH:
        pytest.skip("gpytorch present")
    lik = gp_compat.GaussianLikelihood()
    assert float(lik.noise) == pytest.approx(np.log(2.0) + 1e-4, rel=1e-5)    # gpytorch default
    lik.noise = 0.25
    assert float(lik.noise) == pytest.approx(0.25, rel=1e-5)
    gp_compat.settings.cg_tolerance._global_value = 1e-2
    assert gp_compat.settings.cg_tolerance.value() == 1e-2
    gp_compat.settings.cg_tolerance._global_value = 1.0


def test_laplacian_dropins_match_reference_golden():
    from efficient_graph_gp.graph_kernels.utils import get_normalized_laplacian as lap_dense
    from efficient_graph_gp.preprocessing import get_laplacian, get_normalized_laplacian as lap_np
    from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian as lap_sparse
    from conftest import golden_csr

    z = load_golden("kernels.npz")
    for name in ("cycle4", "grid6x4", "gnm40w"):
        adj = z[name + "_adj"]
        got = lap_sparse(sp.csr_matrix(adj))
        want = golden_csr(z, name + "_lap_sparse")
        assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
        assert np.array_equal(got.data, want.data)
        assert np.array_equal(lap_dense(adj), z[name + "_lap_dense"])
        lp = lap_np(adj)
        assert np.allclose(np.diag(lp), 1.0) and np.allclose(get_laplacian(adj).sum(1), 0)
    # self-checks the reference prints in graph_utils.py:58-65: symmetric, PSD, zero row sums on a regular graph
    ring = sp.csr_matrix(np.roll(np.eye(12), 1, 1) + np.roll(np.eye(12), -1, 1))
    lap = lap_sparse(ring).toarray()
    assert np.allclose(lap, lap.T) and np.allclose(lap.sum(1), 0) and np.linalg.eigvalsh(lap).min() > -1e-12


def test_modulators():
    from efficient_graph_gp.modulation_functions import diffusion_modulator
    from efficient_graph_gp_sparse.gptorch_kernels_sparse import diffusion_modulator_torch
    from oracle import grf_oracle as orc

    for l in range(6):
        assert diffusion_modulator(l, 1.7) == orc.diffusion_modulator(l, 1.7)
    got = diffusion_modulator_torch(torch.arange(6), torch.tensor(1.7, dtype=torch.float64)).numpy()
    assert np.allclose(got, [diffusion_modulator(l, 1.7) for l in range(6)], rtol=1e-12)


def test_cg_restatement_solves_spd_systems():
    from oracle import grf_oracle as orc
    from grf_b200.cg import linear_cg

    rng = np.random.default_rng(0)
    a = rng.standard_normal((40, 40))
    a = a @ a.T + 40 * np.eye(40)
    b = rng.standard_normal((40, 5))
    x = orc.linear_cg(lambda v: a @ v, b, tolerance=1e-10, eps=1e-30)
    assert np.allclose(x, np.linalg.solve(a, b), rtol=1e-7, atol=1e-9)
    x = orc.linear_cg(lambda v: a @ v, b, tolerance=1e-10)       # upstream's eps = 1e-10 guard stalls near 1e-5
    assert np.allclose(x, np.linalg.solve(a, b), rtol=1e-3, atol=1e-6)
    at = torch.tensor(a, dtype=torch.float32)
    xt, info = linear_cg(lambda v: at @ v, torch.tensor(b, dtype=torch.float32), tolerance=1e-6, return_info=True)
    assert np.allclose(xt.numpy(), np.linalg.solve(a, b), rtol=1e-3, atol=1e-4) and info["iterations"] >= 10
    x1 = linear_cg(lambda v: at @ v, torch.tensor(b[:, 0], dtype=torch.float32), tolerance=1e-6)
    assert x1.shape == (40,)


def test_walk_config_validation_and_row_chunks():
    """Host-side argument checks of the engine (no GPU needed) and the row chunking that keeps the
    staging of one walker launch under its byte budget."""
    from grf_b200 import engine

    for bad in (dict(walks_per_node=0, p_halt=0.1, max_walk_length=3),
                dict(walks_per_node=5, p_halt=0.1, max_walk_length=0),
                dict(walks_per_node=5, p_halt=1.5, max_walk_length=3),
                dict(walks_per_node=5, p_halt=-0.1, max_walk_length=3)):
        with pytest.raises(ValueError):
            engine.WalkConfig(**bad).validate()
    with pytest.raises(ValueError):
        engine.WalkConfig(5, 0.1, 3, draw_mode=engine._lib.DRAW_REPLAY).validate()   # replay without a trace
    engine.WalkConfig(5, 0.0, 1).validate()
    engine.WalkConfig(5, 1.0, 3).validate()

    stride = 401                                   # W = 100, L = 5
    chunks = list(engine._row_chunks(10, 1_000_010, stride, 6 << 30))
    assert chunks[0][0] == 10 and chunks[-1][1] == 1_000_010
    assert all(a[1] == b[0] for a, b in zip(chunks[:-1], chunks[1:]))
    assert all((hi - lo) * stride * 12 <= 6 << 30 for lo, hi in chunks)
    assert len(chunks) == 1
    chunks = list(engine._row_chunks(0, 4_194_304, stride, 6 << 30))
    assert len(chunks) > 1 and sum(hi - lo for lo, hi in chunks) == 4_194_304
    assert all((hi - lo) * stride * 12 <= 6 << 30 for lo, hi in chunks)
    assert list(engine._row_chunks(7, 7, stride, 6 << 30)) == [(7, 7)]       # empty shard: one empty chunk


def test_step_matrix_caches_plain_list_and_dict_keyed(tmp_path):
    """graph_preprocessor.py:142-165 pickles a plain list; the experiments wrap it in a dict
    (run_scaling_experiment.py:381-397 'step_matrices_torch' / 'step_matrices', data_utils.py:334-343)."""
    import pickle

    import scipy.sparse as sp
    from efficient_graph_gp_sparse.preprocessor import GraphPreprocessor

    mats = [sp.identity(5, format="csr"), sp.random(5, 5, 0.4, format="csr", random_state=1)]
    for name, payload in (("list.pkl", mats), ("bo.pkl", {"step_matrices_torch": mats, "metadata": {"n_nodes": 5}}),
                          ("dense.pkl", {"step_matrices": mats, "method": "dense"})):
        path = str(tmp_path / name)
        with open(path, "wb") as fh:
            pickle.dump(payload, fh)
        got = GraphPreprocessor.load_step_matrices(path)
        assert len(got) == 2 and all((a != b).nnz == 0 for a, b in zip(got, mats))
    with open(str(tmp_path / "other.pkl"), "wb") as fh:
        pickle.dump({"something": 1}, fh)
    with pytest.raises(KeyError):
        GraphPreprocessor.load_step_matrices(str(tmp_path / "other.pkl"))


def test_balanced_bounds_follow_the_cost_estimate():
    """sharding.balanced_bounds cuts contiguous start-node ranges at the equal-cost quantiles (host logic: plain
    torch ops, runs on CPU tensors): degree-only estimate, and a per-row cost such as pilot_row_cost's."""
    import types

    import torch
    from grf_b200 import sharding

    n = 1000
    deg = torch.ones(n, dtype=torch.int32)
    deg[600:] = 0                                             # the tail is isolated: 0.15 of a walking node each
    graph = types.SimpleNamespace(n_nodes=n, row_ptr=torch.cat([torch.zeros(1, dtype=torch.int32),
                                                                 torch.cumsum(deg, 0).to(torch.int32)]))
    b = sharding.balanced_bounds(graph, 4)
    assert b[0] == 0 and b[-1] == n and all(x <= y for x, y in zip(b, b[1:])) and len(b) == 5
    w = torch.where(deg > 0, 1.0, 0.15).double()
    loads = [float(w[x:y].sum()) for x, y in zip(b, b[1:])]
    assert max(loads) - min(loads) <= 1.0 + 1e-9              # within one node's weight of each other
    assert sharding.balanced_bounds(graph, 1) == [0, n]
    cost = torch.zeros(n, dtype=torch.float64)
    cost[:100] = 9.0                                          # a hub region: ten times the cost per row
    cost[100:] = 1.0
    b2 = sharding.balanced_bounds(graph, 2, row_cost=cost)
    assert b2[0] == 0 and b2[2] == n and 95 <= b2[1] <= 105   # half of the cost sits in the first 100 rows


def test_bench_dump_writes_the_last_steps_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: a fixed sample of the product's rows (the same rows on every run), its column sums
    over all rows and the two counts, as float32 / float64 .npy files of a few MB."""
    import bench

    t = 16
    assert bench.DUMP_ROWS * (t * 4 + 8) < 64 << 20
    monkeypatch.setattr(bench, "DUMP_ROWS", 512)
    n = 1500
    out = torch.randn(n, t, generator=torch.Generator().manual_seed(0))
    # one thread: indexing a CPU tensor would start torch's worker pool, and the oracle tests fork afterwards
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        for d in ("a", "b"):
            bench.dump_last_step(str(tmp_path / d), torch, None, 0, 1, n, 0, n, out, torch.tensor([4321]), 987)
    finally:
        torch.set_num_threads(threads)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["phi_nnz.npy", "product_colsum.npy", "product_row_ids.npy", "product_rows.npy", "walk_steps.npy"]
    for name in files:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype in (np.float32, np.float64) and a.tobytes() == b.tobytes(), name
    ids = np.load(tmp_path / "a" / "product_row_ids.npy")
    assert ids.shape == (bench.DUMP_ROWS,) and np.all(np.diff(ids) > 0) and ids[-1] < n
    assert np.array_equal(np.load(tmp_path / "a" / "product_rows.npy"), out.numpy()[ids.astype(np.int64)])
    assert np.allclose(np.load(tmp_path / "a" / "product_colsum.npy"), out.double().sum(0).numpy(), rtol=1e-12)
    assert np.load(tmp_path / "a" / "walk_steps.npy")[0] == 4321 and np.load(tmp_path / "a" / "phi_nnz.npy")[0] == 987
