"""-m gpu tests of conditioning the exact posterior on new observations: grf_phi_row_condition through _lib on the
synthetic Phi shards of tests/test_gpu_posterior_predictive.py, and ExactPosterior.condition_on / PosteriorMarginals
against a posterior constructed from scratch on the union, within the derived bound of tests/condition_ref.py.

Kernel checks: p is held to the projection bound of tests/predictive_ref.py (2^-22 max(k, 1) sum_e |w_e B_e,c|), so
q to q0 + sum_c p_c^2 within sum_c (2 |p_c| + b_c) b_c, var to max(d - q, 0) within that plus one float32 rounding,
and the mean to the bound of column r.  Columns [k, ldb) of B hold NaN; element n of q, var and mean holds a
sentinel that must come back bit for bit.

The file name sorts after test_gpu_coupled.py on purpose: a torch.profiler session that runs before that file's tests
in the same process leaves later sessions without kernel events (the parent's own profiler tests fail that way when
test_gpu_exact_mll.py's profiler test is run first), and this file has a profiler test."""

from __future__ import annotations

import ctypes

import numpy as np
import pytest

import condition_ref as CR
import matvec_abi_ref as R
import posterior_ref as P
import predictive_ref as Q
from test_gpu_posterior_predictive import (SENTINEL, Env, _b_matrix, _bits, _f, _model, _phi_f, _slots, _vp,  # noqa: F401
                                           g400, grid316)

pytestmark = pytest.mark.gpu

QSENT = np.array([0x7FF8DEADBEEF0001], np.uint64).view(np.float64)[0]


@pytest.fixture(scope="module")
def env():
    return Env()


def _st(env, hp, d, row_lo, L=None, blk=True):
    return env.m.GrfPhi(hp.n_rows, hp.n_cols, row_lo, hp.L if L is None else L,
                        d["blk_ptr"].data_ptr() if blk else None, d["entries"].data_ptr() if blk else None, None,
                        None, None, None, 0, 0, None, None, None, 0, hp.nnz, None)


def _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, q0, d0):
    """(q, var, mean) as host arrays of n + 1 elements (the last one a sentinel) after one call."""
    st = _st(env, hp, d, row_lo)
    q = env.dev(np.r_[q0, QSENT].astype(np.float64))
    dd = env.dev(np.r_[d0, SENTINEL].astype(np.float32))
    var = env.dev(np.full(n + 1, SENTINEL, np.float32))
    mean = env.dev(np.full(n + 1, SENTINEL, np.float32))
    xd = None if x is None else env.dev(x)
    fd, sd = env.dev(f), env.dev(slot)
    rc = env.lib.grf_phi_row_condition(ctypes.byref(st), _vp(fd), _vp(xd), n, _vp(sd), _vp(bbuf, boff), ldb, r, wm,
                                       _vp(q), _vp(dd), _vp(var), _vp(mean) if wm else None, env.stream())
    env.m.check(rc)
    env.torch.cuda.synchronize()
    return q.cpu().numpy(), var.cpu().numpy(), mean.cpu().numpy()


def _check(hp, f, ids, row_lo, slot, B, r, wm, q0, d0, got, what):
    q, var, mean = got
    n = len(q0)
    loc = np.asarray(ids, np.int64) - row_lo
    inside = (loc >= 0) & (loc < hp.n_rows)
    ptr = np.searchsorted(hp.row, np.arange(hp.n_rows + 1))
    w = np.asarray(f, np.float32).astype(np.float64)[hp.length] * hp.val.astype(np.float64)
    ti, col, wv = P.row_entries(ptr, hp.col, w, loc[inside])
    p_in, b_in = Q.project(ti, col, wv, int(inside.sum()), slot, B)
    p, pb = np.zeros((n, B.shape[1])), np.zeros((n, B.shape[1]))
    p[inside], pb[inside] = p_in, b_in
    want_q = q0 + np.sum(p[:, :r] ** 2, axis=1)
    qb = np.sum((2 * np.abs(p[:, :r]) + pb[:, :r]) * pb[:, :r], axis=1) + 2.0 ** -45 * want_q
    assert np.all(np.abs(q[:n] - want_q) <= qb), what
    assert np.array_equal(q[:n][~inside].view(np.int64), np.asarray(q0, np.float64)[~inside].view(np.int64)), \
        f"{what}: q of ids outside the shard changed"
    diff = d0.astype(np.float64) - want_q
    want_v = np.where(np.isnan(diff), diff, np.maximum(diff, 0))
    vb = qb + 2.0 ** -23 * np.abs(want_v)
    ok = (np.abs(var[:n] - want_v) <= vb) | (np.isnan(want_v) & np.isnan(var[:n]))
    assert ok.all(), f"{what}: var, first {np.flatnonzero(~ok)[:3]}"
    assert not np.any(_bits(var[:n]) == _bits(np.float32(-0.0))), f"{what}: var clamps to +0"
    if wm:
        assert np.all(np.abs(mean[:n] - p[:, r]) <= pb[:, r]), f"{what}: mean"
        assert np.all(_bits(mean[:n][~inside]) == 0), f"{what}: mean outside the shard is +0"
        assert _bits(mean[n:]) == _bits(np.float32(SENTINEL))
    else:
        assert np.all(_bits(mean) == _bits(np.float32(SENTINEL))), f"{what}: mean written without with_mean"
    assert np.array_equal(q[n:].view(np.int64), np.array([QSENT]).view(np.int64)), f"{what}: q past n"
    assert _bits(var[n:]) == _bits(np.float32(SENTINEL)), f"{what}: var past n"


K_VALUES = [(1, 0), (0, 1), (2, 1), (3, 1), (4, 0), (4, 1), (5, 0), (7, 1), (8, 0), (16, 1), (17, 0), (31, 1),
            (33, 0), (63, 1), (64, 0)]


@pytest.mark.parametrize("lay", ["tight", "pad", "off1"])
@pytest.mark.parametrize("r,wm", K_VALUES)
def test_row_condition(env, r, wm, lay):
    hp, d = env.phi("pj")
    rng = np.random.default_rng(100 * r + 7 * wm + len(lay))
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.5)
    slot[0] = m
    m += 1
    k = r + wm
    bbuf, boff, ldb, B = _b_matrix(env, rng, m, k, lay)
    row_lo = 0 if lay == "tight" else 700
    if lay == "tight":
        x, ids, n = None, np.arange(hp.n_rows), hp.n_rows
    else:
        must = np.r_[list(R.SPECIAL_ROWS[:4]), [0, 1, 2]] + row_lo
        ids = np.r_[must, rng.integers(0, hp.n_rows + 2 * row_lo, 1500)].astype(np.int32)
        x, n = ids, ids.size
    q0 = rng.uniform(0, 2, n)
    d0 = (q0 + rng.uniform(-1, 40, n)).astype(np.float32)
    d0[5] = np.nan
    got = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, q0, d0)
    _check(hp, f, ids, row_lo, slot, B, r, wm, q0, d0, got, f"r={r} wm={wm} {lay}")
    assert np.isnan(got[1][5])
    again = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, q0, d0)
    for a, b in zip(got, again):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), "not reproducible"
    # q accumulates: a second call from the returned q adds the same squares again
    q1 = got[0][:n]
    got2 = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, q1, d0)
    inc = got[0][:n] - q0
    assert np.all(np.abs(got2[0][:n] - (q1 + inc)) <= 2.0 ** -45 * (q1 + 2 * inc))


@pytest.mark.parametrize("r,wm", [(3, 1), (20, 1)])
def test_row_condition_l32(env, r, wm):
    hp, d = env.phi("l32")
    rng = np.random.default_rng(r)
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.3)
    bbuf, boff, ldb, B = _b_matrix(env, rng, m, r + wm, "pad")
    q0 = np.zeros(hp.n_rows)
    d0 = np.full(hp.n_rows, 1e3, np.float32)
    got = _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r, wm, q0, d0)
    _check(hp, f, np.arange(hp.n_rows), 0, slot, B, r, wm, q0, d0, got, "l32")


def test_row_condition_long_rows_and_all_minus_one(env):
    hp, d = env.phi("heavy")
    rng = np.random.default_rng(3)
    f = np.array([1.0, 0.5, 0.75], np.float32)
    slot = np.arange(hp.n_cols, dtype=np.int32)
    for r, wm in ((3, 1), (40, 1)):
        bbuf, boff, ldb, B = _b_matrix(env, rng, hp.n_cols, r + wm, "pad", positive=True)
        q0, d0 = np.zeros(hp.n_rows), np.full(hp.n_rows, 1e12, np.float32)
        got = _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r, wm, q0, d0)
        _check(hp, f, np.arange(hp.n_rows), 0, slot, B, r, wm, q0, d0, got, "heavy")
    none = np.full(hp.n_cols, -1, np.int32)
    q0 = rng.uniform(0, 1, hp.n_rows)
    got = _call(env, hp, d, 0, f, None, hp.n_rows, none, bbuf, boff, ldb, r, wm, q0, np.ones(hp.n_rows, np.float32))
    assert np.array_equal(got[0][:hp.n_rows], q0 + 0.0) and np.all(_bits(got[2][:hp.n_rows]) == 0)


def test_row_condition_argument_errors(env):
    hp, d = env.phi("pj")
    st = _st(env, hp, d, 0)
    t = env.torch
    buf = t.zeros(64 * 70, dtype=t.float32, device="cuda")
    q = t.zeros(hp.n_rows, dtype=t.float64, device="cuda")
    v = [t.zeros(hp.n_rows, dtype=t.float32, device="cuda") for _ in range(3)]
    slot = t.zeros(hp.n_cols, dtype=t.int32, device="cuda")
    f = t.ones(hp.L, dtype=t.float32, device="cuda")
    ids = t.zeros(4, dtype=t.int32, device="cuda")
    fn, s = env.lib.grf_phi_row_condition, env.stream()
    good = dict(phi=ctypes.byref(st), f=_vp(f), x=None, n=hp.n_rows, slot=_vp(slot), B=_vp(buf), ldb=4, r=3, wm=1,
                q=_vp(q), d=_vp(v[0]), var=_vp(v[1]), mean=_vp(v[2]))
    env.m.check(fn(*good.values(), s))
    bad = [dict(phi=None), dict(f=None), dict(slot=None), dict(B=None), dict(q=None), dict(d=None), dict(var=None),
           dict(mean=None), dict(r=0, wm=0), dict(r=64, wm=1, ldb=70), dict(r=-1), dict(wm=2), dict(ldb=3),
           dict(n=5), dict(x=_vp(ids), n=-2)]
    for b in bad:
        with pytest.raises(ValueError, match="grf_phi_row_condition"):
            env.m.check(fn(*dict(good, **b).values(), s))
    env.m.check(fn(*dict(good, wm=0, mean=None).values(), s))      # mean may be NULL without the mean column
    for steps in (0, 33):
        st2 = _st(env, hp, d, 0, L=steps)
        with pytest.raises(ValueError, match="grf_phi_row_condition"):
            env.m.check(fn(ctypes.byref(st2), *list(good.values())[1:], s))
    st3 = _st(env, hp, d, 0, blk=False)
    with pytest.raises(ValueError, match="grf_phi_row_condition"):
        env.m.check(fn(ctypes.byref(st3), *list(good.values())[1:], s))


def test_row_condition_dispatch_reaches_each_shape(env):
    from torch.profiler import ProfilerActivity, profile

    hp, d = env.phi("pj")
    rng = np.random.default_rng(9)
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.5)
    for r, wm, name in ((1, 0, "row_condition_narrow_kernel"), (3, 1, "row_condition_narrow_kernel"),
                        (4, 1, "row_condition_mid_kernel"), (63, 1, "row_condition_mid_kernel")):
        bbuf, boff, ldb, _ = _b_matrix(env, rng, m, r + wm, "pad")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r, wm, np.zeros(hp.n_rows),
                  np.ones(hp.n_rows, np.float32))
        names = [e.name for e in prof.events() if "row_condition" in e.name]
        assert names and all(name in n for n in names), (r, wm, names)


# ---- ExactPosterior.condition_on / PosteriorMarginals ----------------------------------------------------------
def _union_ref(phi, x0, batches, noise):
    """Fresh (ascending) slot map, C*, the error bounds and L of the union, in training order."""
    x = np.r_[x0, *batches].astype(np.int64)
    slot, G, _ = P.exact_cache(phi, x, noise)
    L, C, E_c, E_f, kappa = CR.chain(G, len(x0), [len(b) for b in batches], noise)
    assert kappa <= CR.KAPPA_MAX
    return x, slot, G, L, C, E_c, E_f


def _compare(setup, post, fresh, x0, batches, y, noise, cand, n_cov=60, s=4):
    """Every output of the conditioned posterior against the fresh one, within the bounds of condition_ref."""
    torch = setup["torch"]
    f = fresh.f.cpu().numpy()
    phi = _phi_f(setup["pp"].step_matrices_scipy, f)
    x, slot, G, L, C, E_c, E_f = _union_ref(phi, x0, batches, noise)
    xt = torch.tensor(cand).cuda()
    ti, col, w = P.row_entries(phi.indptr, phi.indices, phi.data.astype(np.float32), cand)
    nq = len(cand)
    A, dc = CR.proj_delta(ti, col, w, nq, slot, C, E_c)
    _, df = CR.proj_delta(ti, col, w, nq, slot, C, E_f)
    var_f = fresh.variance(xt).double().cpu().numpy()
    q = np.sum(Q.project(ti, col, w, nq, slot, C)[0] ** 2, axis=1)
    vb = CR.var_bound(A, dc, df, q, var_f)
    var_c = post.variance(xt).double().cpu().numpy()
    assert np.all(np.abs(var_c - var_f) <= vb), np.max(np.abs(var_c - var_f) / vb)
    out = dict(var=var_c, vb=vb)
    if y is not None:
        a = CR.weights(G, L, y)
        mb = CR.mean_bound(ti, col, w, nq, slot, a)
        mu_c, mu_f = post.mean(xt).double().cpu().numpy(), fresh.mean(xt).double().cpu().numpy()
        assert np.all(np.abs(mu_c - mu_f) <= mb)
        out.update(mean=mu_c, mb=mb)
        rng = np.random.default_rng(len(x))
        eps = rng.standard_normal((s, phi.shape[1])).astype(np.float32)
        en = rng.standard_normal((s, len(x))).astype(np.float32)
        e_t, en_t = torch.tensor(eps).cuda(), torch.tensor(en).cuda()
        sc = post.sample(xt, s, eps=e_t, eps_noise=en_t).double().cpu().numpy()
        sf = fresh.sample(xt, s, eps=e_t, eps_noise=en_t).double().cpu().numpy()
        prior_x = (phi[x] @ eps.astype(np.float64).T)
        v = y[:, None] - prior_x - np.sqrt(noise) * en.astype(np.float64).T
        import scipy.linalg as sla
        z = sla.solve_triangular(L, v, lower=True)
        sb = CR.sample_bound(ti, col, w, nq, slot, C, E_c, E_f, z, len(x)).T
        assert np.all(np.abs(sc - sf) <= sb), np.max(np.abs(sc - sf) / sb)
    ct = cand[:n_cov]
    tic, colc, wc = P.row_entries(phi.indptr, phi.indices, phi.data.astype(np.float32), ct)
    Pm = Q.project(tic, colc, wc, len(ct), slot, C)[0]
    _, dcc = CR.proj_delta(tic, colc, wc, len(ct), slot, C, E_c)
    _, dfc = CR.proj_delta(tic, colc, wc, len(ct), slot, C, E_f)
    cb = CR.cov_bound(Pm, dcc, dfc)
    cov_c, cov_f = post.covariance(torch.tensor(ct).cuda()), fresh.covariance(torch.tensor(ct).cuda())
    assert torch.equal(cov_c, cov_c.T)
    assert np.all(np.abs(cov_c.cpu().numpy() - cov_f.cpu().numpy()) <= cb)
    return out


def _fresh(setup, model, x, y, noise):
    torch = setup["torch"]
    from grf_b200.posterior import ExactPosterior

    return ExactPosterior(model.covar_module.phi_blocks, model.covar_module.modulator_vector.detach(),
                          torch.tensor(x).cuda(), noise, y_train=None if y is None else torch.tensor(y).cuda())


def _run_chain(setup, train, batches, cand, noise, L):
    torch = setup["torch"]
    model, noise, y0 = _model(setup, train, noise, L)
    post = model.exact_posterior()
    marg = post.marginals(torch.tensor(cand).cuda())
    assert torch.equal(marg.variance(), post.variance(torch.tensor(cand).cuda()))
    ys = [y0]
    rng = np.random.default_rng(17)
    done = []
    for xb in batches:
        yb = rng.standard_normal(len(xb))
        ev = {}
        post.events = ev
        v0 = post.version
        assert post.condition_on(torch.tensor(xb).cuda(), torch.tensor(yb).cuda()) is post
        assert post.version == v0 + 1 and marg.stale
        assert {"condition_start", "cross", "factor", "append", "weights"} <= set(ev)
        assert post.ldc == (post.n + 3) // 4 * 4
        ys.append(yb)
        done.append(xb)
        y = np.concatenate(ys)
        fresh = _fresh(setup, model, np.r_[train, *done], y, noise)
        out = _compare(setup, post, fresh, train, done, y, noise, cand)
        vm = marg.variance().double().cpu().numpy()
        assert not marg.stale
        assert np.all(np.abs(vm - out["var"]) <= out["vb"])
        assert np.all(np.abs(marg.mean.double().cpu().numpy() - out["mean"]) <= out["mb"])
    return post, marg, model, noise


def test_condition_on_g400(g400):
    rng = np.random.default_rng(3)
    perm = rng.permutation(400)
    train = perm[:120]
    batches = [perm[120:121], perm[121:128], np.r_[perm[128:170], train[:5], train[:3]]]   # b = 1, 7, 50
    _run_chain(g400, train, batches, np.arange(400), 0.1, 4)


def test_condition_on_grid316(grid316):
    rng = np.random.default_rng(4)
    nodes = rng.choice(316 * 316, 700, replace=False)
    train = nodes[:600]
    batches = [nodes[600:601], nodes[601:608], nodes[608:658]]
    cand = np.r_[rng.choice(316 * 316, 2000, replace=False), nodes[600:658]]
    _run_chain(grid316, train, batches, cand, 0.05, 5)


def test_marginals_both_refresh_paths_and_staleness(g400):
    """k + 1 <= 64 columns since the last refresh take row_condition; 100 take row_quadform + row_project."""
    torch = g400["torch"]
    rng = np.random.default_rng(5)
    perm = rng.permutation(400)
    train = perm[:100]
    model, noise, y0 = _model(g400, train, 0.1, 4)
    post = model.exact_posterior()
    cand = torch.arange(400).cuda()
    marg = post.marginals(cand)
    assert not marg.stale and marg.refresh() is marg
    ys, done = [y0], []
    for sizes in ((63,), (50, 50)):       # one refresh over 63 columns (+ a), one over 100
        for b in sizes:
            xb = perm[100 + sum(len(d) for d in done):][:b]
            yb = rng.standard_normal(b)
            post.condition_on(torch.tensor(xb).cuda(), torch.tensor(yb).cuda())
            done.append(xb)
            ys.append(yb)
        assert marg.stale
        y = np.concatenate(ys)
        fresh = _fresh(g400, model, np.r_[train, *done], y, noise)
        out = _compare(g400, post, fresh, train, done, y, noise, np.arange(400))
        assert np.all(np.abs(marg.variance().double().cpu().numpy() - out["var"]) <= out["vb"])
        assert np.all(np.abs(marg.mean.double().cpu().numpy() - out["mean"]) <= out["mb"])
        assert torch.equal(marg.variance(include_noise=True), marg.variance() + torch.tensor(noise).float().cuda())


def test_condition_on_diffusion_prior_without_y(g400):
    torch = g400["torch"]
    from efficient_graph_gp_sparse.gptorch_kernels_sparse import SparseDiffusionKernel
    from grf_b200.posterior import ExactPosterior

    kern = SparseDiffusionKernel(max_walk_length=4, step_matrices_torch=g400["ops"]).cuda()
    f = kern.modulator_vector.detach()
    x0 = np.arange(0, 400, 7)
    xb = np.r_[np.arange(3, 400, 11), 0, 0]
    for start in (x0, np.zeros(0, np.int64)):           # n = 0 start too
        post = ExactPosterior(kern.phi_blocks, f, torch.tensor(start).cuda(), 0.2)
        marg = post.marginals(torch.arange(400).cuda())
        with pytest.raises(ValueError):
            post.condition_on(torch.tensor(xb).cuda(), torch.zeros(len(xb)).cuda())
        with pytest.raises(ValueError):
            marg.mean
        post.condition_on(torch.tensor(xb).cuda())
        fresh = ExactPosterior(kern.phi_blocks, f, torch.tensor(np.r_[start, xb]).cuda(), 0.2)
        out = _compare(g400, post, fresh, start, [xb], None, 0.2, np.arange(400))
        assert np.all(np.abs(marg.variance().double().cpu().numpy() - out["var"]) <= out["vb"])


def test_condition_on_errors(g400):
    torch = g400["torch"]
    model, noise, y0 = _model(g400, np.arange(10), 0.1, 4)
    post = model.exact_posterior()
    xb = torch.tensor([20, 21]).cuda()
    with pytest.raises(ValueError):
        post.condition_on(xb)                                   # y_new required
    with pytest.raises(ValueError):
        post.condition_on(xb, torch.zeros(3).cuda())
    for bad in (torch.tensor([-1]).cuda(), torch.tensor([400]).cuda()):
        with pytest.raises(IndexError):
            post.condition_on(bad, torch.zeros(1).cuda())
    state = lambda p: (p.n, p.m, p.version, p.ldc, p.C.clone(), p.L.clone(), p.slot.clone(), p.a.clone())
    before = state(post)
    assert post.condition_on(torch.zeros(0, dtype=torch.int64).cuda(), torch.zeros(0).cuda()) is post
    post.mem_limit = 1000
    with pytest.raises(MemoryError, match="bytes"):
        post.condition_on(xb, torch.zeros(2).cuda())
    post.mem_limit = None
    post.noise = -1e6                                           # K_22 + sigma^2 I - L_21 L_21^T is not PD
    with pytest.raises(ValueError, match="sigma"):
        post.condition_on(xb, torch.zeros(2).cuda())
    post.noise = noise
    after = state(post)
    for a, b in zip(before, after):
        assert (torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b)
    post.condition_on(xb, torch.zeros(2).cuda())                # still usable
    assert post.n == 12 and post.version == 1
