"""-m gpu tests of the exact posterior variance: grf_phi_row_quadform through _lib on synthetic Phi shards
(tests/matvec_abi_ref.py), ExactPosterior and SparseGraphGP.posterior_variance against float64 dense formulas.

q and d are held to the per-element bound of tests/posterior_ref.py, 2^-21 max(k, 1) sum_c (sum_e |w_e C_ec|)^2
(k = touched entries of the row), which holds for any summation order; the summation order is fixed, so repeated
calls must also agree bit for bit.  Columns [r, ldc) of C hold NaN and the tail of q and d a NaN sentinel, so a
kernel that read the padding into a result or wrote past n would fail."""

from __future__ import annotations

import ctypes

import numpy as np
import pytest

import matvec_abi_ref as R
import posterior_ref as P
from gpu_util import grid_graph, random_graph

pytestmark = pytest.mark.gpu


class Env:
    def __init__(self):
        import torch

        assert torch.cuda.is_available(), "these tests need a B200"
        from grf_b200 import _lib

        self.torch, self.m, self.lib = torch, _lib, _lib.lib()
        self._phis = {}

    def dev(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).cuda()

    def stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def phi(self, name):
        if name not in self._phis:
            hp = _profile(name)
            one = np.zeros((1, 2), np.int32)
            d = dict(blk_ptr=self.dev(hp.blk_ptr), entries=self.dev(hp.entries if hp.nnz else one))
            self._phis[name] = (hp, d)
        return self._phis[name]


def _profile(name):
    """qf    L = 3, 3000 x 2500: rows of 0..39 entries, empty rows, rows of exactly 255, 256, 257 and 2000 entries,
             hub column 0 holding {length 0, column 0, -0.0}
       l32   L = 32, 1200 x 1500: rows of 0..59 entries at all 32 lengths, rows of 257 and 600 entries
       heavy L = 3, 400 x 3000: positive values in [0.5, 1], rows of 20..39 entries and of 257, 700 and 2000 entries
             whose LAST entry weighs 64: a row that loses its last entry misses the bound by far"""
    if name == "qf":
        rng = np.random.default_rng(11)
        lens = rng.integers(0, 40, 3000)
        lens[rng.random(3000) < 0.05] = 0
        lens[R.SPECIAL_ROWS[:4]] = [255, 256, 257, 2000]
        return R.synth_phi(12, 3000, 2500, 3, lens, hub=0)
    if name == "l32":
        rng = np.random.default_rng(21)
        lens = rng.integers(0, 60, 1200)
        lens[R.SPECIAL_ROWS[:2]] = [257, 600]
        return R.synth_phi(22, 1200, 1500, 32, lens, hub=0, hub_len=np.full(1200, 2))
    if name == "heavy":
        rng = np.random.default_rng(31)
        lens = rng.integers(20, 40, 400)
        lens[R.SPECIAL_ROWS[:3]] = [257, 700, 2000]
        hp = R.synth_phi(32, 400, 3000, 3, lens, neg_zero=False)
        val = rng.uniform(0.5, 1.0, hp.nnz).astype(np.float32)
        last = np.r_[np.flatnonzero(np.diff(hp.row)), hp.nnz - 1]
        val[last] = 64.0
        hp.val = val
        return hp
    raise KeyError(name)


@pytest.fixture(scope="module")
def env():
    return Env()


def _vp(t, off=0):
    return None if t is None else ctypes.c_void_p(t.data_ptr() + 4 * off)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _slots(rng, n_cols, frac):
    touched = np.flatnonzero(rng.random(n_cols) < frac)
    slot = np.full(n_cols, -1, np.int32)
    slot[touched] = np.arange(touched.size, dtype=np.int32)
    return slot, touched.size


def _c_matrix(env, rng, m, r, lay, positive=False):
    """(device buffer, offset in floats, ldc, host C [m][r]): columns [r, ldc) are NaN; "tight" ldc = r, "pad"
    ldc = round_up(r, 4) + 4, "off1" the same ldc with the base one float past a 16-byte boundary."""
    ldc = r if lay == "tight" else (r + 3) // 4 * 4 + 4
    off = 1 if lay == "off1" else 0
    host = (rng.uniform(0.5, 1.0, (m, r)) if positive else rng.standard_normal((m, r))).astype(np.float32)
    full = np.full((max(1, m), max(1, ldc)), np.nan, np.float32)
    full[:m, :r] = host
    buf = np.r_[np.zeros(off, np.float32), full.ravel(), np.zeros(4, np.float32)]
    return env.dev(buf), off, ldc, host


def _call(env, hp, d, row_lo, f, x, n, slot, cbuf, coff, ldc, r, with_d=True):
    st = env.m.GrfPhi(hp.n_rows, hp.n_cols, row_lo, hp.L, d["blk_ptr"].data_ptr(), d["entries"].data_ptr(), None,
                      None, None, None, 0, 0, None, None, None, 0, hp.nnz, None)
    q = env.torch.full((n + 4,), float("nan"), dtype=env.torch.float32, device="cuda")
    dd = env.torch.full((n + 4,), float("nan"), dtype=env.torch.float32, device="cuda")
    xd = None if x is None else env.dev(x)
    fd, sd = env.dev(f), env.dev(slot)      # held until the call is queued: a freed block would be reused
    rc = env.lib.grf_phi_row_quadform(ctypes.byref(st), _vp(fd), _vp(xd), n, _vp(sd), _vp(cbuf, coff), ldc, r,
                                      _vp(q), _vp(dd) if with_d else None, env.stream())
    env.m.check(rc)
    env.torch.cuda.synchronize()
    return q.cpu().numpy(), dd.cpu().numpy()


def _ref(hp, f, ids, row_lo, slot, C):
    """q, d and bounds for the global ids (ids outside the shard select nothing)."""
    loc = np.asarray(ids, np.int64) - row_lo
    inside = (loc >= 0) & (loc < hp.n_rows)
    ptr = np.searchsorted(hp.row, np.arange(hp.n_rows + 1))
    w = np.asarray(f, np.float32).astype(np.float64)[hp.length] * hp.val.astype(np.float64)
    ti, col, wv = P.row_entries(ptr, hp.col, w, loc[inside])
    q, d, bq, bd = P.quadform(ti, col, wv, int(inside.sum()), slot, C)
    out = [np.zeros(loc.size) for _ in range(4)]
    for o, v in zip(out, (q, d, bq, bd)):
        o[inside] = v
    return (*out, inside)


def _check(got, want, bound, what):
    err = np.abs(got[:want.size].astype(np.float64) - want)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {bad.sum()} outside the bound, first {np.argmax(bad)}: "
                           f"got {got[np.argmax(bad)]!r} want {want[np.argmax(bad)]!r} bound {bound[np.argmax(bad)]!r}")


def _f(rng, L):
    f = (2.0 ** rng.uniform(-2, 1, L)).astype(np.float32)
    f[L - 1] = -f[L - 1]
    return f


# ---- grf_phi_row_quadform ----------------------------------------------------------------------------------
R_VALUES = (0, 1, 3, 4, 5, 127, 128, 129, 256, 600)


@pytest.mark.parametrize("lay", ["tight", "pad", "off1"])
@pytest.mark.parametrize("r", R_VALUES)
def test_row_quadform(env, r, lay):
    hp, d = env.phi("qf")
    rng = np.random.default_rng(r * 7 + len(lay))
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.5)
    slot[0] = m          # the hub column (and its -0.0 entry) is touched
    m += 1
    cbuf, coff, ldc, C = _c_matrix(env, rng, m, r, lay)
    row_lo = 0 if lay == "tight" else 700
    must = list(R.SPECIAL_ROWS[:4]) + [0, 1, 2]
    if lay == "tight":
        x, ids, n = None, np.arange(hp.n_rows), hp.n_rows
    else:   # ids below, inside and above the shard, the long rows first
        ids = np.r_[np.asarray(must) + row_lo, rng.integers(0, hp.n_rows + 2 * row_lo, 1500)].astype(np.int32)
        x, n = ids, ids.size
    q, dd = _call(env, hp, d, row_lo, f, x, n, slot, cbuf, coff, ldc, r)
    want_q, want_d, bq, bd, inside = _ref(hp, f, ids, row_lo, slot, C)
    _check(q, want_q, bq, "q")
    _check(dd, want_d, bd, "d")
    assert np.all(np.isnan(q[n:])) and np.all(np.isnan(dd[n:])), "wrote past n"
    if r == 0:
        assert np.all(_bits(q[:n]) == 0), "r = 0 must give q = +0"
    if (~inside).any():
        assert np.all(_bits(q[:n][~inside]) == 0) and np.all(_bits(dd[:n][~inside]) == 0), "outside: +0"
    q2, d2 = _call(env, hp, d, row_lo, f, x, n, slot, cbuf, coff, ldc, r)
    assert np.array_equal(_bits(q), _bits(q2)) and np.array_equal(_bits(dd), _bits(d2)), "not reproducible"


@pytest.mark.parametrize("r", [5, 129, 600])
def test_row_quadform_l32_and_no_d(env, r):
    hp, d = env.phi("l32")
    rng = np.random.default_rng(r)
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.3)
    cbuf, coff, ldc, C = _c_matrix(env, rng, m, r, "pad")
    q, dd = _call(env, hp, d, 0, f, None, hp.n_rows, slot, cbuf, coff, ldc, r, with_d=False)
    want_q, _, bq, _, _ = _ref(hp, f, np.arange(hp.n_rows), 0, slot, C)
    _check(q, want_q, bq, "q")
    assert np.all(np.isnan(dd)), "d = NULL must leave d alone"


@pytest.mark.parametrize("r", [3, 128, 129, 256])
def test_row_quadform_catches_lost_entries(env, r):
    """Positive weights and C, and a last entry of weight 64 per row: the 257-, 700- and 2000-entry rows take the
    chunked path, and losing their last entry (or the last partial panel) cannot stay inside the bound."""
    hp, d = env.phi("heavy")
    rng = np.random.default_rng(300 + r)
    f = np.array([1.0, 0.5, 0.75], np.float32)
    slot = np.arange(hp.n_cols, dtype=np.int32)           # every column touched
    cbuf, coff, ldc, C = _c_matrix(env, rng, hp.n_cols, r, "pad", positive=True)
    q, dd = _call(env, hp, d, 0, f, None, hp.n_rows, slot, cbuf, coff, ldc, r)
    want_q, want_d, bq, bd, _ = _ref(hp, f, np.arange(hp.n_rows), 0, slot, C)
    _check(q, want_q, bq, "q")
    _check(dd, want_d, bd, "d")
    # what the bound rules out: each long row without its last entry
    for row in R.SPECIAL_ROWS[:3]:
        e = np.flatnonzero(hp.row == row)
        w = f[hp.length[e]].astype(np.float64) * hp.val[e]
        short = np.sum((w[:-1] @ C[hp.col[e[:-1]]].astype(np.float64)) ** 2)
        assert abs(short - want_q[row]) > bq[row]


def test_row_quadform_no_touched_column_is_exactly_zero(env):
    hp, d = env.phi("qf")
    rng = np.random.default_rng(5)
    f = _f(rng, hp.L)
    slot = np.full(hp.n_cols, -1, np.int32)
    cbuf, coff, ldc, C = _c_matrix(env, rng, 4, 129, "pad")
    q, dd = _call(env, hp, d, 0, f, None, hp.n_rows, slot, cbuf, coff, ldc, 129)
    assert np.all(_bits(q[:hp.n_rows]) == 0)
    _, want_d, _, bd, _ = _ref(hp, f, np.arange(hp.n_rows), 0, slot, C)
    _check(dd, want_d, bd, "d")


def test_row_quadform_argument_errors(env):
    hp, d = env.phi("qf")
    st = env.m.GrfPhi(hp.n_rows, hp.n_cols, 0, hp.L, d["blk_ptr"].data_ptr(), d["entries"].data_ptr(), None, None,
                      None, None, 0, 0, None, None, None, 0, hp.nnz, None)
    buf = env.torch.zeros(64, dtype=env.torch.float32, device="cuda")
    out = env.torch.zeros(hp.n_rows, dtype=env.torch.float32, device="cuda")
    slot = env.torch.zeros(hp.n_cols, dtype=env.torch.int32, device="cuda")
    f = env.torch.ones(hp.L, dtype=env.torch.float32, device="cuda")
    ids = env.torch.zeros(4, dtype=env.torch.int32, device="cuda")
    fn, s = env.lib.grf_phi_row_quadform, env.stream()
    good = dict(phi=ctypes.byref(st), f=_vp(f), x=None, n=hp.n_rows, slot=_vp(slot), C=_vp(buf), ldc=4, r=4,
                q=_vp(out), d=None)
    env.m.check(fn(*good.values(), s))
    bad = [dict(phi=None), dict(f=None), dict(slot=None), dict(C=None), dict(q=None), dict(n=-1), dict(r=-1),
           dict(ldc=3), dict(n=5), dict(x=_vp(ids), n=-2)]
    for b in bad:
        args = dict(good, **b)
        with pytest.raises(ValueError):
            env.m.check(fn(*args.values(), s))
    for steps in (0, 33):
        st2 = env.m.GrfPhi(hp.n_rows, hp.n_cols, 0, steps, d["blk_ptr"].data_ptr(), d["entries"].data_ptr(), None,
                           None, None, None, 0, 0, None, None, None, 0, hp.nnz, None)
        with pytest.raises(ValueError):
            env.m.check(fn(ctypes.byref(st2), *list(good.values())[1:], s))


# ---- ExactPosterior / SparseGraphGP.posterior_variance ---------------------------------------------------------
def _phi_f(mats, f):
    return sum(float(np.float32(fl)) * m.astype(np.float32).astype(np.float64) for fl, m in zip(f, mats)).tocsr()


@pytest.fixture(scope="module")
def g400():
    import torch

    from efficient_graph_gp_sparse.preprocessor import GraphPreprocessor

    adj = random_graph(400, 1300, 21).tolil()
    adj[399, :] = 0          # an isolated node
    adj[:, 399] = 0
    adj = adj.tocsr()
    adj.eliminate_zeros()
    pp = GraphPreprocessor(adj, walks_per_node=30, p_halt=0.1, max_walk_length=4, random_walk_seed=7, use_tqdm=False)
    return dict(torch=torch, pp=pp, ops=pp.preprocess_graph())


@pytest.fixture(scope="module")
def grid316():
    import torch

    from efficient_graph_gp_sparse.preprocessor import GraphPreprocessor

    pp = GraphPreprocessor(grid_graph(316, 316), walks_per_node=100, p_halt=0.1, max_walk_length=5,
                           random_walk_seed=3, use_tqdm=False)
    return dict(torch=torch, pp=pp, ops=pp.preprocess_graph())


def _model(setup, train, noise, L, seed=0):
    torch = setup["torch"]
    from efficient_graph_gp_sparse.models import SparseGraphGP
    from grf_b200.gp_compat import GaussianLikelihood

    torch.manual_seed(seed)
    lik = GaussianLikelihood()
    lik.noise = noise
    y = torch.sin(torch.as_tensor(train, dtype=torch.float32) / 20.0)
    model = SparseGraphGP(torch.tensor(train, dtype=torch.float32)[:, None].cuda(), y.cuda(), lik, setup["ops"],
                          L).cuda()
    return model, float(lik.noise.item())


def _check_model(setup, model, noise, train, test):
    torch = setup["torch"]
    from grf_b200.posterior import ExactPosterior

    f = model.covar_module.modulator_vector.detach().cpu().numpy()
    phi = _phi_f(setup["pp"].step_matrices_scipy, f)
    want, prior = P.dense_variance(phi, train, test, noise)
    xt = torch.tensor(test, dtype=torch.float32)[:, None].cuda()
    got = model.posterior_variance(xt)
    assert got.dtype == torch.float32 and got.device.type == "cuda" and tuple(got.shape) == (len(test),)
    g = got.cpu().numpy()
    assert np.all(np.abs(g - want) <= 1e-4 * prior + 1e-30), np.max(np.abs(g - want) / np.maximum(prior, 1e-30))
    assert np.all(g >= 0) and np.all(g <= prior * (1 + 1e-5) + 1e-30)
    noisy = model.posterior_variance(xt, include_noise=True)
    assert torch.equal(noisy, got + torch.tensor(noise, dtype=torch.float32, device="cuda"))
    # nodes that share no column with the training rows: bit for bit the prior diagonal of the n = 0 call
    rows = phi[np.asarray(train)]
    touched = np.zeros(phi.shape[1], bool)
    touched[rows.indices] = True
    far = np.array([i for i, t in enumerate(test) if not touched[phi[t].indices].any()], np.int64)
    blocks = model.covar_module.phi_blocks
    prior_dev = ExactPosterior(blocks, f, np.zeros(0, np.int64), noise).variance(torch.tensor(test).cuda())
    if far.size:
        assert torch.equal(got[torch.tensor(far).cuda()], prior_dev[torch.tensor(far).cuda()])
    return got, far.size


def test_posterior_variance_g400(g400):
    rng = np.random.default_rng(3)
    for train in (rng.permutation(399)[:1], rng.permutation(400)[:240], np.arange(400),
                  np.r_[rng.permutation(400)[:100], [5, 5, 17, 17, 17, 399]]):      # duplicates, the isolated node
        model, noise = _model(g400, train, 0.1, 4)
        _check_model(g400, model, noise, train, np.arange(400))


def test_posterior_variance_grid316(grid316):
    rng = np.random.default_rng(4)
    train = rng.choice(316 * 316, 600, replace=False)
    test = np.r_[rng.choice(316 * 316, 2000, replace=False), train]
    model, noise = _model(grid316, train, 0.05, 5)
    _, n_far = _check_model(grid316, model, noise, train, test)
    assert n_far > 0


def test_exact_posterior_diffusion_modulator(g400):
    torch = g400["torch"]
    from efficient_graph_gp_sparse.gptorch_kernels_sparse import SparseDiffusionKernel
    from grf_b200.posterior import ExactPosterior

    kern = SparseDiffusionKernel(max_walk_length=4, step_matrices_torch=g400["ops"]).cuda()
    f = kern.modulator_vector.detach()
    train = np.arange(0, 400, 3)
    ev = {}
    post = ExactPosterior(kern.phi_blocks, f, torch.tensor(train).cuda(), 0.2, events=ev)
    got = post.variance(torch.arange(400).cuda()).cpu().numpy()
    assert {"start", "merge", "slots", "G", "gram", "cholesky", "solve", "quadform_start", "quadform"} <= set(ev)
    phi = _phi_f(g400["pp"].step_matrices_scipy, f.cpu().numpy())
    want, prior = P.dense_variance(phi, train, np.arange(400), 0.2)
    assert np.all(np.abs(got - want) <= 1e-4 * prior + 1e-30)
    assert post.variance(torch.zeros(0, dtype=torch.int64).cuda()).numel() == 0


def test_posterior_variance_matches_predict_samples(g400):
    torch = g400["torch"]
    rng = np.random.default_rng(5)
    train = rng.permutation(400)[:240]
    test = np.setdiff1d(np.arange(400), train)
    model, _ = _model(g400, train, 0.1, 4, seed=1)
    xt = torch.tensor(test).cuda()
    samples = torch.cat([model.predict(xt, n_samples=256, cg_tolerance=1e-6) for _ in range(4)])
    sv = samples.double().var(dim=0).cpu().numpy()
    pv = model.posterior_variance(xt).double().cpu().numpy()
    ok = np.abs(sv - pv) <= 5 * np.sqrt(2 / 1023) * pv
    assert ok.mean() >= 0.97, ok.mean()


def test_exact_posterior_errors(g400):
    torch = g400["torch"]
    from grf_b200 import engine
    from grf_b200.posterior import ExactPosterior

    model, _ = _model(g400, np.arange(10), 0.1, 4)
    blocks = model.covar_module.phi_blocks
    f = model.covar_module.modulator_vector.detach()
    with pytest.raises(IndexError):
        ExactPosterior(blocks, f, torch.tensor([1, 400]).cuda(), 0.1)
    post = ExactPosterior(blocks, f, torch.tensor([1, 2]).cuda(), 0.1)
    with pytest.raises(IndexError):
        post.variance(torch.tensor([-1]).cuda())
    with pytest.raises(IndexError):
        model.posterior_variance(torch.tensor([[400.0]]).cuda())
    shard = engine.phi_blocks_from_scipy([m[:200] for m in g400["pp"].step_matrices_scipy], "cuda", transpose=False)
    with pytest.raises(ValueError):
        ExactPosterior(shard, f, torch.tensor([1]).cuda(), 0.1)
    with pytest.raises(MemoryError):
        ExactPosterior(blocks, f, torch.arange(200).cuda(), 0.1, mem_limit=1000)
    with pytest.raises(ValueError):
        ExactPosterior(blocks, f, torch.tensor([1]).cuda(), 0.0)
