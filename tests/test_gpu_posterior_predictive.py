"""-m gpu tests of the exact posterior mean, joint covariance and samples: grf_phi_row_project through _lib on
synthetic Phi shards (tests/matvec_abi_ref.py), ExactPosterior and SparseGraphGP against the float64 dense formulas
of tests/predictive_ref.py.

Every projected element is held to the bound of tests/predictive_ref.py, 2^-22 max(k, 1) sum_e |w_e B_e,c| (k =
touched entries of the row), which holds for any summation order; the order is fixed, so repeated calls must also
agree bit for bit.  Columns [r, ldb) of B hold NaN, and columns [r, ldo) and the row after the last of out hold a NaN
sentinel that must come back bit for bit, so a kernel that read the padding into a result or wrote outside the
r x n block would fail."""

from __future__ import annotations

import ctypes

import numpy as np
import pytest

import matvec_abi_ref as R
import posterior_ref as P
import predictive_ref as Q
from gpu_util import grid_graph, random_graph

pytestmark = pytest.mark.gpu

SENTINEL = np.array([0x7FC0BEEF], np.uint32).view(np.float32)[0]


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
    """pj    L = 3, 3000 x 2500: rows of 0..39 entries, empty rows, rows of exactly 255, 256, 257 and 2000 entries,
             hub column 0 holding {length 0, column 0, -0.0}
       l32   L = 32, 1200 x 1500: rows of 0..59 entries at all 32 lengths, rows of 257 and 600 entries
       heavy L = 3, 400 x 3000: positive values in [0.5, 1], rows of 20..39 entries and of 257, 700 and 2000 entries
             whose LAST entry weighs 64: a row that loses its last entry misses the bound by far"""
    if name == "pj":
        rng = np.random.default_rng(41)
        lens = rng.integers(0, 40, 3000)
        lens[rng.random(3000) < 0.05] = 0
        lens[R.SPECIAL_ROWS[:4]] = [255, 256, 257, 2000]
        return R.synth_phi(42, 3000, 2500, 3, lens, hub=0)
    if name == "l32":
        rng = np.random.default_rng(51)
        lens = rng.integers(0, 60, 1200)
        lens[R.SPECIAL_ROWS[:2]] = [257, 600]
        return R.synth_phi(52, 1200, 1500, 32, lens, hub=0, hub_len=np.full(1200, 2))
    if name == "heavy":
        rng = np.random.default_rng(61)
        lens = rng.integers(20, 40, 400)
        lens[R.SPECIAL_ROWS[:3]] = [257, 700, 2000]
        hp = R.synth_phi(62, 400, 3000, 3, lens, neg_zero=False)
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


def _ld(r, lay):
    """"tight" ld = r, "pad" ld = round_up(r, 4) + 4, "off1" the same ld with the base one float past 16 bytes."""
    return (r if lay == "tight" else (r + 3) // 4 * 4 + 4), (1 if lay == "off1" else 0)


def _b_matrix(env, rng, m, r, lay, positive=False):
    """(device buffer, offset in floats, ldb, host B [m][r]); columns [r, ldb) are NaN."""
    ldb, off = _ld(r, lay)
    host = (rng.uniform(0.5, 1.0, (m, r)) if positive else rng.standard_normal((m, r))).astype(np.float32)
    full = np.full((max(1, m), max(1, ldb)), np.nan, np.float32)
    full[:m, :r] = host
    buf = np.r_[np.zeros(off, np.float32), full.ravel(), np.zeros(4, np.float32)]
    return env.dev(buf), off, ldb, host


def _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, lay="pad"):
    """out (host [n + 1][ldo] with the sentinel padding) after one call; lay sets ldo and the alignment of out."""
    st = env.m.GrfPhi(hp.n_rows, hp.n_cols, row_lo, hp.L, d["blk_ptr"].data_ptr(), d["entries"].data_ptr(), None,
                      None, None, None, 0, 0, None, None, None, 0, hp.nnz, None)
    ldo, ooff = _ld(r, lay)
    ldo = max(ldo, 1)
    out = env.dev(np.full(ooff + (n + 1) * ldo, SENTINEL, np.float32))
    xd = None if x is None else env.dev(x)
    fd, sd = env.dev(f), env.dev(slot)      # held until the call is queued: a freed block would be reused
    rc = env.lib.grf_phi_row_project(ctypes.byref(st), _vp(fd), _vp(xd), n, _vp(sd), _vp(bbuf, boff), ldb, r,
                                     _vp(out, ooff), ldo, env.stream())
    env.m.check(rc)
    env.torch.cuda.synchronize()
    return out.cpu().numpy()[ooff:].reshape(n + 1, ldo)


def _ref(hp, f, ids, row_lo, slot, B):
    loc = np.asarray(ids, np.int64) - row_lo
    inside = (loc >= 0) & (loc < hp.n_rows)
    ptr = np.searchsorted(hp.row, np.arange(hp.n_rows + 1))
    w = np.asarray(f, np.float32).astype(np.float64)[hp.length] * hp.val.astype(np.float64)
    ti, col, wv = P.row_entries(ptr, hp.col, w, loc[inside])
    o, b = Q.project(ti, col, wv, int(inside.sum()), slot, B)
    want, bound = np.zeros((loc.size, B.shape[1])), np.zeros((loc.size, B.shape[1]))
    want[inside], bound[inside] = o, b
    return want, bound, inside


def _check(out, n, r, want, bound, what):
    got = out[:n, :r].astype(np.float64)
    bad = ~(np.abs(got - want) <= bound)
    assert not bad.any(), (f"{what}: {bad.sum()} outside the bound, first {np.argwhere(bad)[0]}: "
                           f"got {got[bad][0]!r} want {want[bad][0]!r} bound {bound[bad][0]!r}")
    pad = np.r_[out[:n, r:].ravel(), out[n].ravel()]
    assert np.all(_bits(pad) == _bits(np.float32(SENTINEL))), f"{what}: wrote outside the r x n block"


def _f(rng, L):
    f = (2.0 ** rng.uniform(-2, 1, L)).astype(np.float32)
    f[L - 1] = -f[L - 1]
    return f


# ---- grf_phi_row_project ------------------------------------------------------------------------------------
R_VALUES = (0, 1, 2, 3, 4, 5, 8, 16, 17, 31, 32, 63, 64, 65, 100, 128, 129, 256, 600)


@pytest.mark.parametrize("lay", ["tight", "pad", "off1"])
@pytest.mark.parametrize("r", R_VALUES)
def test_row_project(env, r, lay):
    hp, d = env.phi("pj")
    rng = np.random.default_rng(r * 11 + len(lay))
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.5)
    slot[0] = m          # the hub column (and its -0.0 entry) is touched
    m += 1
    bbuf, boff, ldb, B = _b_matrix(env, rng, m, r, lay)
    row_lo = 0 if lay == "tight" else 700
    must = list(R.SPECIAL_ROWS[:4]) + [0, 1, 2]
    if lay == "tight":
        x, ids, n = None, np.arange(hp.n_rows), hp.n_rows
    else:   # ids below, inside and above the shard, the long rows first
        ids = np.r_[np.asarray(must) + row_lo, rng.integers(0, hp.n_rows + 2 * row_lo, 1500)].astype(np.int32)
        x, n = ids, ids.size
    out = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, lay)
    want, bound, inside = _ref(hp, f, ids, row_lo, slot, B)
    _check(out, n, r, want, bound, f"r={r} {lay}")
    if (~inside).any():
        assert np.all(_bits(out[:n, :r][~inside]) == 0), "rows outside the shard must be +0"
    out2 = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, lay)
    assert np.array_equal(_bits(out), _bits(out2)), "not reproducible"


@pytest.mark.parametrize("r", [3, 16, 129])
def test_row_project_l32(env, r):
    hp, d = env.phi("l32")
    rng = np.random.default_rng(r)
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.3)
    bbuf, boff, ldb, B = _b_matrix(env, rng, m, r, "pad")
    out = _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r)
    want, bound, _ = _ref(hp, f, np.arange(hp.n_rows), 0, slot, B)
    _check(out, hp.n_rows, r, want, bound, "l32")


@pytest.mark.parametrize("r", [1, 4, 16, 64, 128, 129, 256])
def test_row_project_catches_lost_entries(env, r):
    """Positive weights and B, and a last entry of weight 64 per row: the 257-, 700- and 2000-entry rows take the
    re-streamed path, and losing their last entry (or the last partial panel) cannot stay
    inside the bound."""
    hp, d = env.phi("heavy")
    rng = np.random.default_rng(400 + r)
    f = np.array([1.0, 0.5, 0.75], np.float32)
    slot = np.arange(hp.n_cols, dtype=np.int32)           # every column touched
    bbuf, boff, ldb, B = _b_matrix(env, rng, hp.n_cols, r, "pad", positive=True)
    out = _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r)
    want, bound, _ = _ref(hp, f, np.arange(hp.n_rows), 0, slot, B)
    _check(out, hp.n_rows, r, want, bound, "heavy")
    for row in R.SPECIAL_ROWS[:3]:      # what the bound rules out: each long row without its last entry
        e = np.flatnonzero(hp.row == row)
        w = f[hp.length[e]].astype(np.float64) * hp.val[e]
        short = w[:-1] @ B[hp.col[e[:-1]]].astype(np.float64)
        assert np.all(np.abs(short - want[row]) > bound[row])


def test_row_project_no_touched_column_is_exactly_zero(env):
    hp, d = env.phi("pj")
    rng = np.random.default_rng(5)
    f = _f(rng, hp.L)
    slot = np.full(hp.n_cols, -1, np.int32)
    for r in (1, 16, 129):
        bbuf, boff, ldb, _ = _b_matrix(env, rng, 4, r, "pad")
        out = _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r)
        assert np.all(_bits(out[:hp.n_rows, :r]) == 0)


def test_row_project_argument_errors(env):
    hp, d = env.phi("pj")
    st = env.m.GrfPhi(hp.n_rows, hp.n_cols, 0, hp.L, d["blk_ptr"].data_ptr(), d["entries"].data_ptr(), None, None,
                      None, None, 0, 0, None, None, None, 0, hp.nnz, None)
    buf = env.torch.zeros(64, dtype=env.torch.float32, device="cuda")
    out = env.torch.zeros(4 * hp.n_rows, dtype=env.torch.float32, device="cuda")
    slot = env.torch.zeros(hp.n_cols, dtype=env.torch.int32, device="cuda")
    f = env.torch.ones(hp.L, dtype=env.torch.float32, device="cuda")
    ids = env.torch.zeros(4, dtype=env.torch.int32, device="cuda")
    fn, s = env.lib.grf_phi_row_project, env.stream()
    good = dict(phi=ctypes.byref(st), f=_vp(f), x=None, n=hp.n_rows, slot=_vp(slot), B=_vp(buf), ldb=4, r=4,
                out=_vp(out), ldo=4)
    env.m.check(fn(*good.values(), s))
    bad = [dict(phi=None), dict(f=None), dict(slot=None), dict(B=None), dict(out=None), dict(n=-1), dict(r=-1),
           dict(ldb=3), dict(ldo=3), dict(n=5), dict(x=_vp(ids), n=-2)]
    for b in bad:
        args = dict(good, **b)
        with pytest.raises(ValueError, match="grf_phi_row_project"):
            env.m.check(fn(*args.values(), s))
    for steps in (0, 33):
        st2 = env.m.GrfPhi(hp.n_rows, hp.n_cols, 0, steps, d["blk_ptr"].data_ptr(), d["entries"].data_ptr(), None,
                           None, None, None, 0, 0, None, None, None, 0, hp.nnz, None)
        with pytest.raises(ValueError, match="grf_phi_row_project"):
            env.m.check(fn(ctypes.byref(st2), *list(good.values())[1:], s))
    st3 = env.m.GrfPhi(hp.n_rows, hp.n_cols, 0, hp.L, None, None, None, None, None, None, 0, 0, None, None, None, 0,
                       hp.nnz, None)
    with pytest.raises(ValueError, match="grf_phi_row_project"):
        env.m.check(fn(ctypes.byref(st3), *list(good.values())[1:], s))


def test_row_project_dispatch_reaches_each_shape(env):
    """torch.profiler sees the narrow kernel for r <= 4, the mid kernel for 4 < r <= 64 and the panels above."""
    from torch.profiler import ProfilerActivity, profile

    hp, d = env.phi("pj")
    rng = np.random.default_rng(9)
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.5)
    for r, name in ((1, "row_project_narrow_kernel"), (4, "row_project_narrow_kernel"),
                    (5, "row_project_mid_kernel"), (64, "row_project_mid_kernel"),
                    (65, "row_project_kernel"), (600, "row_project_kernel")):
        bbuf, boff, ldb, _ = _b_matrix(env, rng, m, r, "pad")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r)
        names = [e.name for e in prof.events() if "row_project" in e.name or "quadform" in e.name]
        assert names and all(name in n for n in names), (r, names)


def test_phi_blocks_row_project_operands(g400):
    """PhiBlocks.row_project: a B whose rows overlap (stride 0) is copied, not read past its end; a slot map that
    names a row B lacks, or an out whose rows overlap, is refused."""
    torch = g400["torch"]
    from grf_b200.posterior import ExactPosterior

    model, _, _ = _model(g400, np.arange(0, 400, 5), 0.1, 4)
    post = ExactPosterior(model.covar_module.phi_blocks, model.covar_module.modulator_vector.detach(),
                          torch.arange(0, 400, 5).cuda(), 0.1)
    one, xt = torch.ones(1, device="cuda"), torch.arange(400).cuda()
    row = torch.randn(1, 3, device="cuda")
    got = post.phi_f.row_project(one, xt, post.slot, row.expand(post.m, 3))
    assert torch.equal(got, post.phi_f.row_project(one, xt, post.slot, row.expand(post.m, 3).contiguous()))
    with pytest.raises(ValueError, match="col_slot"):
        post.phi_f.row_project(one, xt, post.slot, torch.zeros((post.m - 1, 3), device="cuda"))
    with pytest.raises(ValueError, match="out"):
        post.phi_f.row_project(one, xt, post.slot, row.expand(post.m, 3), out=torch.zeros(1, 3, device="cuda")
                               .expand(400, 3))


# ---- ExactPosterior / SparseGraphGP -------------------------------------------------------------------------
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
    return model, float(lik.noise.item()), y.numpy().astype(np.float64)


def _check_model(setup, train, test, noise, L, n_cov, s=8):
    torch = setup["torch"]
    model, noise, y = _model(setup, train, noise, L)
    f = model.covar_module.modulator_vector.detach().cpu().numpy()
    phi = _phi_f(setup["pp"].step_matrices_scipy, f)
    post = model.exact_posterior()
    xt = torch.tensor(test).cuda()

    mu = post.mean(xt)
    assert mu.dtype == torch.float32 and tuple(mu.shape) == (len(test),)
    want_mu, _ = Q.dense_mean(phi, train, y, test, noise)
    tol = 1e-4 * np.abs(want_mu).max()
    assert np.all(np.abs(mu.cpu().numpy() - want_mu) <= tol)
    cg = model.posterior_mean(torch.tensor(test, dtype=torch.float32)[:, None].cuda()).cpu().numpy()
    assert np.all(np.abs(mu.cpu().numpy() - cg) <= tol)

    ct = test[:n_cov]
    cov = post.covariance(torch.tensor(ct).cuda())
    assert cov.dtype == torch.float64 and torch.equal(cov, cov.T)
    want_c, kss = Q.dense_covariance(phi, train, ct, noise)
    scale = np.sqrt(np.outer(np.diag(kss), np.diag(kss)))
    assert np.all(np.abs(cov.cpu().numpy() - want_c) <= 1e-4 * scale + 1e-30)
    var = post.variance(torch.tensor(ct).cuda()).double()
    assert np.all(np.abs(torch.diagonal(cov).cpu().numpy() - var.cpu().numpy()) <= 1e-4 * np.diag(kss) + 1e-30)
    cov_m = model.posterior_covariance(torch.tensor(ct, dtype=torch.float32)[:, None].cuda(), include_noise=True)
    eye = torch.eye(len(ct), dtype=torch.float64, device="cuda")
    assert torch.equal(cov_m, cov_m.T)
    assert torch.allclose(cov_m - noise * eye, cov, rtol=1e-6, atol=1e-9 * float(np.diag(kss).max()))

    rng = np.random.default_rng(7)
    eps = rng.standard_normal((s, phi.shape[1])).astype(np.float32)
    eps_noise = rng.standard_normal((s, len(train))).astype(np.float32)
    got = post.sample(xt, s, eps=torch.tensor(eps).cuda(), eps_noise=torch.tensor(eps_noise).cuda())
    assert got.dtype == torch.float32 and tuple(got.shape) == (s, len(test))
    want_s = Q.dense_sample(phi, train, y, test, noise, eps, eps_noise)
    kdiag = np.asarray(phi[np.asarray(test)].multiply(phi[np.asarray(test)]).sum(axis=1)).ravel()
    assert np.all(np.abs(got.cpu().numpy() - want_s) <= 1e-3 * (np.sqrt(kdiag) + np.abs(want_s)) + 1e-6)
    return post, model


def test_posterior_predictive_g400(g400):
    rng = np.random.default_rng(3)
    for train in (rng.permutation(399)[:1], rng.permutation(400)[:240],
                  np.r_[rng.permutation(400)[:100], [5, 5, 17, 17, 17, 399]]):      # duplicates, the isolated node
        _check_model(g400, train, np.arange(400), 0.1, 4, 400)


def test_posterior_predictive_grid316(grid316):
    rng = np.random.default_rng(4)
    train = rng.choice(316 * 316, 600, replace=False)
    test = np.r_[rng.choice(316 * 316, 1500, replace=False), train[:100]]
    _check_model(grid316, train, test, 0.05, 5, 500)


def test_samples_match_the_exact_mean_and_variance(g400):
    torch = g400["torch"]
    rng = np.random.default_rng(5)
    train = rng.permutation(400)[:240]
    test = np.setdiff1d(np.arange(400), train)
    model, _, _ = _model(g400, train, 0.1, 4, seed=1)
    post = model.exact_posterior()
    xt = torch.tensor(test).cuda()
    gen = torch.Generator(device="cuda").manual_seed(11)
    s = 4096
    samples = post.sample(xt, s, generator=gen).double()
    mu, var = post.mean(xt).double(), post.variance(xt).double()
    ok_m = (samples.mean(0) - mu).abs() <= 5 * torch.sqrt(var / s)
    ok_v = (samples.var(0) - var).abs() <= 5 * np.sqrt(2 / (s - 1)) * var
    assert ok_m.double().mean() >= 0.97 and ok_v.double().mean() >= 0.97, (ok_m.double().mean(), ok_v.double().mean())
    noisy = post.sample(xt, s, generator=gen, include_noise=True).double()
    ok_n = (noisy.var(0) - var - 0.1).abs() <= 5 * np.sqrt(2 / (s - 1)) * (var + 0.1)
    assert ok_n.double().mean() >= 0.97


def test_variance_unchanged_by_y_train_and_the_prior(g400):
    torch = g400["torch"]
    from efficient_graph_gp_sparse.gptorch_kernels_sparse import SparseDiffusionKernel
    from grf_b200.posterior import ExactPosterior

    kern = SparseDiffusionKernel(max_walk_length=4, step_matrices_torch=g400["ops"]).cuda()
    f = kern.modulator_vector.detach()
    train = np.arange(0, 400, 3)
    y = np.cos(train / 30.0)
    xt = torch.arange(400).cuda()
    ev = {}
    post = ExactPosterior(kern.phi_blocks, f, torch.tensor(train).cuda(), 0.2, y_train=torch.tensor(y).cuda(),
                          events=ev)
    plain = ExactPosterior(kern.phi_blocks, f, torch.tensor(train).cuda(), 0.2)
    assert torch.equal(post.variance(xt), plain.variance(xt)) and torch.equal(post.C, plain.C)
    phi = _phi_f(g400["pp"].step_matrices_scipy, f.cpu().numpy())
    want, _ = Q.dense_mean(phi, train, y, np.arange(400), 0.2)
    assert np.all(np.abs(post.mean(xt).cpu().numpy() - want) <= 1e-4 * np.abs(want).max())
    assert {"project_start", "project", "quadform_start", "quadform", "solve"} <= set(ev)
    # n = 0: mean 0, covariance K**, samples from the prior
    empty = torch.zeros(0, dtype=torch.int64).cuda()
    prior = ExactPosterior(kern.phi_blocks, f, empty, 0.2, y_train=torch.zeros(0).cuda())
    assert torch.equal(prior.mean(xt), torch.zeros(400, device="cuda"))
    ids = np.arange(0, 400, 7)
    _, kss = Q.dense_covariance(phi, np.zeros(0, np.int64), ids, 0.2)
    cov = prior.covariance(torch.tensor(ids).cuda()).cpu().numpy()
    assert np.all(np.abs(cov - kss) <= 1e-5 * np.sqrt(np.outer(np.diag(kss), np.diag(kss))) + 1e-30)
    eps = np.random.default_rng(2).standard_normal((3, 400)).astype(np.float32)
    got = prior.sample(torch.tensor(ids).cuda(), 3, eps=torch.tensor(eps).cuda(),
                       eps_noise=torch.zeros((3, 0)).cuda()).cpu().numpy()
    want_s = Q.dense_sample(phi, np.zeros(0, np.int64), np.zeros(0), ids, 0.2, eps, np.zeros((3, 0)))
    assert np.allclose(got, want_s, rtol=1e-4, atol=1e-4)
    assert post.covariance(empty).shape == (0, 0) and post.mean(empty).numel() == 0
    assert tuple(post.sample(empty, 2).shape) == (2, 0)


def test_posterior_predictive_errors(g400):
    torch = g400["torch"]
    from grf_b200 import engine
    from grf_b200.posterior import ExactPosterior

    model, _, _ = _model(g400, np.arange(10), 0.1, 4)
    blocks = model.covar_module.phi_blocks
    f = model.covar_module.modulator_vector.detach()
    x = torch.tensor([1, 2]).cuda()
    plain = ExactPosterior(blocks, f, x, 0.1)
    with pytest.raises(ValueError):
        plain.mean(x)
    with pytest.raises(ValueError):
        plain.sample(x, 4)
    with pytest.raises(ValueError):
        ExactPosterior(blocks, f, x, 0.1, y_train=torch.zeros(3).cuda())
    post = ExactPosterior(blocks, f, x, 0.1, y_train=torch.zeros(2).cuda())
    for bad in (torch.tensor([-1]).cuda(), torch.tensor([400]).cuda()):
        with pytest.raises(IndexError):
            post.mean(bad)
        with pytest.raises(IndexError):
            post.covariance(bad)
        with pytest.raises(IndexError):
            post.sample(bad, 2)
    with pytest.raises(IndexError):
        model.posterior_covariance(torch.tensor([[400.0]]).cuda())
    for n_samples in (0, -3):
        with pytest.raises(ValueError):
            post.sample(x, n_samples)
    with pytest.raises(ValueError):
        post.sample(x, 2, eps=torch.zeros((2, 399)).cuda())
    with pytest.raises(ValueError):
        post.sample(x, 2, eps_noise=torch.zeros((2, 3)).cuda())
    post.mem_limit = 1000
    with pytest.raises(MemoryError, match="bytes"):
        post.covariance(torch.arange(200).cuda())
    with pytest.raises(MemoryError, match="bytes"):
        post.sample(torch.arange(200).cuda(), 64)
    shard = engine.phi_blocks_from_scipy([m[:200] for m in g400["pp"].step_matrices_scipy], "cuda", transpose=False)
    with pytest.raises(ValueError):
        ExactPosterior(shard, f, torch.tensor([1]).cuda(), 0.1, y_train=torch.zeros(1).cuda())
