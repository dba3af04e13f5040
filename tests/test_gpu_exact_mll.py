"""Exact marginal likelihood on the device: PhiBlocks.training_gram (csrc/grf_gram.cu) against a dense float64
A A^T, and ExactMLL's loss and closed-form gradients against dense float64 formulas, neg_mll_backward and an
L-BFGS run on the dense reference loss (tests/exact_mll_ref.py)."""

from __future__ import annotations

import numpy as np
import pytest

import exact_mll_ref as R
from gpu_util import grid_graph, powerlaw_graph, random_graph

pytestmark = pytest.mark.gpu


def _setup(adj, W, L, seed):
    import torch

    from efficient_graph_gp_sparse.preprocessor import GraphPreprocessor

    pp = GraphPreprocessor(adj, walks_per_node=W, p_halt=0.1, max_walk_length=L, random_walk_seed=seed,
                           use_tqdm=False)
    ops = pp.preprocess_graph()
    from grf_b200 import engine

    return dict(torch=torch, pp=pp, ops=ops, mats=pp.step_matrices_scipy,
                blocks=engine.phi_blocks_from_scipy(pp.step_matrices_scipy, "cuda"))


@pytest.fixture(scope="module")
def g400():
    return _setup(random_graph(400, 1300, 21), 30, 4, 7)


@pytest.fixture(scope="module")
def grid316():
    return _setup(grid_graph(316, 316), 100, 5, 3)


@pytest.fixture(scope="module")
def powerlaw():
    return _setup(powerlaw_graph(3000, 12000, 5), 40, 4, 11)


def _gram(setup, x, T, monkeypatch=None):
    from grf_b200 import engine

    old = engine.GRAM_HEAVY_THRESHOLD
    engine.GRAM_HEAVY_THRESHOLD = T
    try:
        E, stats = setup["blocks"]._training_gram(setup["torch"].as_tensor(x).cuda())
    finally:
        engine.GRAM_HEAVY_THRESHOLD = old
    return E, stats


def _check_gram(setup, x, T):
    from grf_b200 import engine

    T = engine.GRAM_HEAVY_THRESHOLD if T is None else T
    E, stats = _gram(setup, x, T)
    L, n = len(setup["mats"]), len(x)
    assert E.dtype == setup["torch"].float64 and tuple(E.shape) == (L, n, L, n)
    got = E.reshape(L * n, L * n).cpu().numpy()
    want = R.gram(setup["mats"], x)
    bound = R.gram_bound(setup["mats"], x)
    assert np.all(np.abs(got - want) <= bound), np.max(np.abs(got - want) / np.maximum(bound, 1e-300))
    assert np.array_equal(got, got.T)
    E2, _ = _gram(setup, x, T)
    assert setup["torch"].equal(E, E2)
    return stats


@pytest.mark.parametrize("T", [0, None, 10 ** 9])
def test_gram_g400(g400, T):
    rng = np.random.default_rng(1)
    x = np.r_[rng.permutation(400)[:150], [3, 3, 3, 17]]                   # repeated ids
    stats = _check_gram(g400, x, T)
    assert stats["nnz_train"] > 0 and stats["m"] > 0
    if T == 0:
        assert stats["p_light"] == 0 and stats["h"] == stats["m"]
    if T == 10 ** 9:
        assert stats["h"] == 0


@pytest.mark.parametrize("T", [0, None, 10 ** 9])
def test_gram_grid316(grid316, T):
    rng = np.random.default_rng(4)
    _check_gram(grid316, rng.choice(316 * 316, 600, replace=False), T)


def test_gram_powerlaw_both_paths_and_hub_row(powerlaw):
    """A hub training row (node 0 has the highest degree) and hub columns: at T = 32 both the light kernel and the
    dense H H^T run."""
    rng = np.random.default_rng(5)
    x = np.r_[[0, 1], rng.choice(np.arange(2, 3000), 400, replace=False)]
    stats = _check_gram(powerlaw, x, 32)
    assert stats["h"] > 0 and stats["p_light"] > 0
    for T in (0, None, 10 ** 9):
        _check_gram(powerlaw, x, T)


def test_gram_small_n_and_merged(g400):
    torch = g400["torch"]
    blocks = g400["blocks"]
    e0 = blocks.training_gram(torch.zeros(0, dtype=torch.int64).cuda())
    assert tuple(e0.shape) == (4, 0, 4, 0)
    _check_gram(g400, np.array([5]), None)
    _check_gram(g400, np.array([399]), 0)
    # merged blocks (L = 1): E is the Gram of the rows of Phi_f
    f = np.array([1.0, -0.5, 0.25, 0.125], np.float32)
    merged = blocks.merged(torch.tensor(f))
    x = np.arange(0, 400, 5)
    E = merged.training_gram(torch.tensor(x).cuda())
    assert tuple(E.shape) == (1, 80, 1, 80)
    phi = sum(float(fl) * m.astype(np.float32).astype(np.float64) for fl, m in zip(f, g400["mats"])).tocsr()
    a = phi[x]
    want = (a @ a.T).toarray()
    got = E.reshape(80, 80).cpu().numpy()
    assert np.all(np.abs(got - want) <= 1e-6 * np.abs(want).max())
    assert np.array_equal(got, got.T)


def test_gram_l32():
    s = _setup(random_graph(200, 600, 9), 8, 32, 2)
    _check_gram(s, np.random.default_rng(6).permutation(200)[:60], None)
    _check_gram(s, np.arange(0, 200, 4), 0)


def _kernels_run(setup, x, T):
    torch = setup["torch"]
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _gram(setup, x, T)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    light = any("gram_light_kernel" in nm for nm in names)
    mirror = any("gram_mirror_kernel" in nm for nm in names)
    gemm = any("gemm" in nm.lower() or "dmma" in nm.lower() for nm in names)
    return light, gemm, mirror


def test_gram_kernels_under_profiler(powerlaw):
    x = np.r_[[0], np.arange(10, 3000, 10)]
    assert _kernels_run(powerlaw, x, 10 ** 9) == (True, False, True)
    assert _kernels_run(powerlaw, x, 0) == (False, True, True)
    assert _kernels_run(powerlaw, x, 32) == (True, True, True)


# ---- ExactMLL ---------------------------------------------------------------------------------------------------
def _dense(setup, x, f, noise, y):
    """The dense float64 formulas of tests/test_gpu_gp.py::test_mll_gradient_matches_dense_float64."""
    mats = [m.astype(np.float32).astype(np.float64).tocsr()[x].toarray() for m in setup["mats"]]
    phi = sum(fl * m for fl, m in zip(f, mats))
    n = len(x)
    kh = phi @ phi.T + noise * np.eye(n)
    kinv = np.linalg.inv(kh)
    a = kinv @ y
    gf = [-(0.5 * a @ (m @ phi.T + phi @ m.T) @ a - 0.5 * np.trace(kinv @ (m @ phi.T + phi @ m.T))) / n
          for m in mats]
    gs = -(0.5 * a @ a - 0.5 * np.trace(kinv)) / n
    _, ld = np.linalg.slogdet(kh)
    loss = (0.5 * y @ a + 0.5 * ld + 0.5 * n * np.log(2 * np.pi)) / n
    return loss, np.array(gf), gs


@pytest.mark.parametrize("f", [[1.0, -0.4, 0.2, -0.05], [0.8, 0.0, 0.3, 0.1]])
def test_exact_mll_matches_dense(g400, f):
    torch = g400["torch"]
    from grf_b200.mll import ExactMLL

    rng = np.random.default_rng(11)
    x = np.sort(rng.permutation(400)[:120])
    y = np.sin(x / 15.0) + 0.1 * rng.standard_normal(120)
    ev = {}
    mll = ExactMLL(g400["blocks"], torch.tensor(x).cuda(), torch.tensor(y), events=ev)
    ft = torch.tensor(f, dtype=torch.float64, requires_grad=True)
    nt = torch.tensor(0.5, dtype=torch.float64, requires_grad=True)
    loss = mll.loss(ft, nt)
    loss.backward()
    assert {"start", "gather", "light", "heavy", "symmetrise", "eval_start", "kernel", "cholesky", "solve",
            "grad"} <= set(ev)
    want_loss, want_f, want_s = _dense(g400, x, np.array(f), 0.5, y)
    assert loss.dtype == torch.float64 and abs(loss.item() - want_loss) <= 1e-10 * abs(want_loss)
    got_f = ft.grad.numpy()
    assert np.all(np.abs(got_f - want_f) <= 1e-8 * np.abs(want_f).max()), (got_f, want_f)
    assert abs(nt.grad.item() - want_s) <= 1e-8 * abs(want_s)
    # repeated evaluations agree bit for bit
    l2 = mll.loss(torch.tensor(f, dtype=torch.float64), 0.5)
    assert l2.item() == loss.item() and torch.equal(mll.last["grad_f"].cpu(), torch.tensor(got_f))


def test_exact_mll_backward_matches_neg_mll_backward(g400):
    torch = g400["torch"]
    from efficient_graph_gp_sparse.gptorch_kernels_sparse import SparseGRFKernel
    from grf_b200.gp_compat import GaussianLikelihood
    from grf_b200.mll import ExactMLL, neg_mll_backward

    torch.manual_seed(1)
    rng = np.random.default_rng(11)
    kern = SparseGRFKernel(4, g400["ops"]).cuda()
    with torch.no_grad():
        kern.raw_modulator_vector.copy_(torch.tensor([1.0, -0.4, 0.2, -0.05]))
    lik = GaussianLikelihood()
    lik.noise = 0.5
    idx = np.sort(rng.permutation(400)[:120])
    y = np.sin(idx / 15.0) + 0.1 * rng.standard_normal(120)
    n = 120
    ref = neg_mll_backward(kern, lik, torch.tensor(idx), torch.tensor(y), probes=torch.eye(n) * np.sqrt(n),
                           cg_tolerance=1e-7, cg_eps=1e-30)
    want_f = kern.raw_modulator_vector.grad.cpu().numpy().copy()
    want_n = float(lik.raw_noise.grad)
    kern.raw_modulator_vector.grad = None
    lik.raw_noise.grad = None
    out = ExactMLL(kern.phi_blocks, torch.tensor(idx), torch.tensor(y).float()).backward(kern, lik)
    assert set(ref) <= set(out) and out["cg_iterations"] == 0 and "logdet" in out
    got_f = kern.raw_modulator_vector.grad.cpu().numpy()
    assert np.allclose(got_f, want_f, rtol=2e-3, atol=2e-3 * np.abs(want_f).max()), (got_f, want_f)
    assert abs(float(lik.raw_noise.grad) - want_n) <= 2e-3 * abs(want_n) + 1e-6
    assert abs(out["datafit"] - ref["datafit"]) <= 1e-3 * abs(ref["datafit"])
    assert np.allclose(out["grad_modulator"].numpy(), ref["grad_modulator"].numpy(), rtol=2e-3,
                       atol=2e-3 * np.abs(ref["grad_modulator"].numpy()).max())


def test_exact_mll_diffusion_modulator_finite_differences(g400):
    torch = g400["torch"]
    from efficient_graph_gp_sparse.gptorch_kernels_sparse import SparseDiffusionKernel
    from grf_b200.mll import ExactMLL

    kern = SparseDiffusionKernel(max_walk_length=4, step_matrices_torch=g400["ops"]).cuda().double()
    x = np.arange(0, 400, 3)
    y = np.cos(x / 20.0)
    mll = ExactMLL(kern.phi_blocks, torch.tensor(x).cuda(), torch.tensor(y))
    raw_noise = torch.tensor(-1.0, dtype=torch.float64, requires_grad=True)

    def loss():
        return mll.loss(kern.modulator_vector, torch.nn.functional.softplus(raw_noise))

    loss().backward()
    params = [kern.raw_beta, kern.raw_sigma_f, raw_noise]
    grads = [float(p.grad) for p in params]
    h = 1e-6
    for p, g in zip(params, grads):
        with torch.no_grad():
            p += h
            up = loss().item()
            p -= 2 * h
            dn = loss().item()
            p += h
        fd = (up - dn) / (2 * h)
        assert abs(g - fd) <= 1e-5 * max(abs(fd), 1e-3), (g, fd)


def test_exact_mll_lbfgs_matches_dense_reference(g400):
    torch = g400["torch"]
    from grf_b200.mll import ExactMLL

    rng = np.random.default_rng(12)
    x = np.sort(rng.permutation(400)[:100])
    y = np.sin(x / 15.0) + 0.1 * rng.standard_normal(100)
    mll = ExactMLL(g400["blocks"], torch.tensor(x).cuda(), torch.tensor(y))
    a = R.stacked_rows(g400["mats"], x).toarray()
    E = torch.tensor(a @ a.T).reshape(4, 100, 4, 100)
    yt = torch.tensor(y)

    def dense_loss(f, noise):
        k = torch.einsum("l,libj,b->ij", f, E, f) + noise * torch.eye(100, dtype=torch.float64)
        c = torch.linalg.cholesky(k)
        alpha = torch.cholesky_solve(yt[:, None], c)[:, 0]
        return (0.5 * yt @ alpha + torch.log(c.diagonal()).sum() + 50 * np.log(2 * np.pi)) / 100

    def fit(fn):
        theta = torch.tensor([1.0, 0.5, 0.2, 0.1, np.log(0.5)], dtype=torch.float64, requires_grad=True)
        opt = torch.optim.LBFGS([theta], lr=1, max_iter=200, tolerance_grad=1e-12, tolerance_change=1e-15,
                                line_search_fn="strong_wolfe")

        def closure():
            opt.zero_grad()
            v = fn(theta[:4], theta[4].exp())
            v.backward()
            return v

        opt.step(closure)
        return fn(theta[:4].detach(), theta[4].detach().exp()).item()

    got, want = fit(mll.loss), fit(dense_loss)
    assert abs(got - want) <= 1e-8 * abs(want), (got, want)


def test_exact_mll_model_and_errors(g400):
    torch = g400["torch"]
    from efficient_graph_gp_sparse.models import SparseGraphGP
    from grf_b200 import engine
    from grf_b200.gp_compat import GaussianLikelihood
    from grf_b200.mll import ExactMLL

    blocks = g400["blocks"]
    lik = GaussianLikelihood()
    lik.noise = 0.1
    x = torch.arange(0, 400, 7)
    model = SparseGraphGP(x.float()[:, None].cuda(), torch.sin(x / 9.0).cuda(), lik, g400["ops"], 4).cuda()
    mll = model.exact_mll()
    assert isinstance(mll, ExactMLL) and mll.n == x.numel()
    out = mll.backward(model.covar_module, lik)
    assert np.isfinite(out["loss"]) and model.covar_module.raw_modulator_vector.grad is not None
    y = torch.ones(3)
    with pytest.raises(IndexError):
        ExactMLL(blocks, torch.tensor([1, 2, 400]).cuda(), y)
    with pytest.raises(IndexError):
        blocks.training_gram(torch.tensor([-1]).cuda())
    shard = engine.phi_blocks_from_scipy([m[:200] for m in g400["mats"]], "cuda", transpose=False)
    with pytest.raises(ValueError):
        ExactMLL(shard, torch.tensor([1, 2, 3]).cuda(), y)
    with pytest.raises(ValueError):
        shard.training_gram(torch.tensor([1]).cuda())
    with pytest.raises(ValueError):
        ExactMLL(blocks, torch.tensor([1, 2]).cuda(), y)                      # y shape
    with pytest.raises(ValueError):
        ExactMLL(blocks, torch.tensor([1, 2, 3]).cuda(), torch.tensor([1.0, float("nan"), 0.0]))
    with pytest.raises(MemoryError):
        ExactMLL(blocks, torch.arange(300).cuda(), torch.ones(300), mem_limit=10 ** 6)
    with pytest.raises(MemoryError):
        blocks.training_gram(torch.arange(300).cuda(), mem_limit=10 ** 6)
    m3 = ExactMLL(blocks, torch.tensor([1, 2, 3]).cuda(), y)
    f = torch.ones(4)
    for bad in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError):
            m3.loss(f, bad)
    with pytest.raises(ValueError):
        m3.loss(torch.ones(3), 0.1)
    dup = ExactMLL(blocks, torch.tensor([5, 5]).cuda(), torch.ones(2))
    with pytest.raises(ValueError, match="sigma"):
        dup.loss(f, 1e-300)
