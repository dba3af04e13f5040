"""-m gpu tests of removing observations from the exact posterior and replacing its targets: grf_phi_row_downdate
through _lib on the synthetic Phi shards of tests/test_gpu_posterior_predictive.py, and ExactPosterior.forget /
set_targets / PosteriorMarginals against a posterior constructed from scratch on the kept rows, within the bound of
tests/downdate_ref.py.

Kernel checks as in tests/test_gpu_posterior_condition.py with the sign flipped: q against q0 - sum_c p_c^2 within
sum_c (2 |p_c| + b_c) b_c (+ 2^-45 of the magnitudes), var against max(d - q, 0) and the mean against the
projection bound; columns [k, ldb) of B hold NaN and element n of q, var and mean a sentinel.

The file name sorts after test_gpu_coupled.py on purpose (see tests/test_gpu_posterior_condition.py): it has a
torch.profiler test."""

from __future__ import annotations

import ctypes

import numpy as np
import pytest
import scipy.linalg as sla

import condition_ref as CR
import downdate_ref as DR
import matvec_abi_ref as R
import posterior_ref as P
import predictive_ref as Q
from test_gpu_posterior_condition import QSENT, _st
from test_gpu_posterior_predictive import (SENTINEL, Env, _b_matrix, _bits, _f, _model, _phi_f, _slots, _vp,  # noqa: F401
                                           g400, grid316)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    return Env()


def _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, q0, d0, fn="grf_phi_row_downdate"):
    """(q, var, mean) as host arrays of n + 1 elements (the last one a sentinel) after one call."""
    st = _st(env, hp, d, row_lo)
    q = env.dev(np.r_[q0, QSENT].astype(np.float64))
    dd = env.dev(np.r_[d0, SENTINEL].astype(np.float32))
    var = env.dev(np.full(n + 1, SENTINEL, np.float32))
    mean = env.dev(np.full(n + 1, SENTINEL, np.float32))
    xd = None if x is None else env.dev(x)
    fd, sd = env.dev(f), env.dev(slot)
    rc = getattr(env.lib, fn)(ctypes.byref(st), _vp(fd), _vp(xd), n, _vp(sd), _vp(bbuf, boff), ldb, r, wm, _vp(q),
                              _vp(dd), _vp(var), _vp(mean) if wm else None, env.stream())
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
    sq = np.sum(p[:, :r] ** 2, axis=1)
    want_q = q0 - sq
    qb = np.sum((2 * np.abs(p[:, :r]) + pb[:, :r]) * pb[:, :r], axis=1) + 2.0 ** -45 * (np.abs(q0) + sq)
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


K_VALUES = [(1, 0), (0, 1), (2, 1), (3, 1), (4, 0), (4, 1), (5, 0), (8, 0), (16, 1), (31, 1), (33, 0), (63, 1),
            (64, 0)]


@pytest.mark.parametrize("lay", ["tight", "pad", "off1"])
@pytest.mark.parametrize("r,wm", K_VALUES)
def test_row_downdate(env, r, wm, lay):
    hp, d = env.phi("pj")
    rng = np.random.default_rng(100 * r + 7 * wm + len(lay) + 1)
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
    q0 = rng.uniform(0, 2, n) + 40.0
    d0 = (q0 + rng.uniform(-1, 40, n)).astype(np.float32)
    d0[5] = np.nan
    got = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, q0, d0)
    _check(hp, f, ids, row_lo, slot, B, r, wm, q0, d0, got, f"r={r} wm={wm} {lay}")
    assert np.isnan(got[1][5])
    again = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, q0, d0)
    for a, b in zip(got, again):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), "not reproducible"
    # the same B through row_condition, then row_downdate, returns to q0 (the p are the same bits)
    up = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, q0, d0, fn="grf_phi_row_condition")
    back = _call(env, hp, d, row_lo, f, x, n, slot, bbuf, boff, ldb, r, wm, up[0][:n], d0)
    inc = up[0][:n] - q0
    assert np.all(np.abs(back[0][:n] - q0) <= 2.0 ** -45 * (q0 + 2 * inc))
    if wm:
        assert np.array_equal(_bits(back[2]), _bits(up[2]))


@pytest.mark.parametrize("r,wm", [(3, 1), (20, 1)])
def test_row_downdate_l32(env, r, wm):
    hp, d = env.phi("l32")
    rng = np.random.default_rng(r + 1)
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.3)
    bbuf, boff, ldb, B = _b_matrix(env, rng, m, r + wm, "pad")
    q0 = np.full(hp.n_rows, 1e4)
    d0 = np.full(hp.n_rows, 1e3, np.float32)
    got = _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r, wm, q0, d0)
    _check(hp, f, np.arange(hp.n_rows), 0, slot, B, r, wm, q0, d0, got, "l32")


def test_row_downdate_long_rows_and_all_minus_one(env):
    hp, d = env.phi("heavy")
    rng = np.random.default_rng(4)
    f = np.array([1.0, 0.5, 0.75], np.float32)
    slot = np.arange(hp.n_cols, dtype=np.int32)
    for r, wm in ((3, 1), (40, 1)):
        bbuf, boff, ldb, B = _b_matrix(env, rng, hp.n_cols, r + wm, "pad", positive=True)
        q0, d0 = np.full(hp.n_rows, 1e12), np.full(hp.n_rows, 2e12, np.float32)
        got = _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r, wm, q0, d0)
        _check(hp, f, np.arange(hp.n_rows), 0, slot, B, r, wm, q0, d0, got, "heavy")
    none = np.full(hp.n_cols, -1, np.int32)
    q0 = rng.uniform(0, 1, hp.n_rows)
    got = _call(env, hp, d, 0, f, None, hp.n_rows, none, bbuf, boff, ldb, r, wm, q0, np.ones(hp.n_rows, np.float32))
    assert np.array_equal(got[0][:hp.n_rows], q0 - 0.0) and np.all(_bits(got[2][:hp.n_rows]) == 0)


def test_row_downdate_argument_errors(env):
    hp, d = env.phi("pj")
    st = _st(env, hp, d, 0)
    t = env.torch
    buf = t.zeros(64 * 70, dtype=t.float32, device="cuda")
    q = t.zeros(hp.n_rows, dtype=t.float64, device="cuda")
    v = [t.zeros(hp.n_rows, dtype=t.float32, device="cuda") for _ in range(3)]
    slot = t.zeros(hp.n_cols, dtype=t.int32, device="cuda")
    f = t.ones(hp.L, dtype=t.float32, device="cuda")
    ids = t.zeros(4, dtype=t.int32, device="cuda")
    fn, s = env.lib.grf_phi_row_downdate, env.stream()
    good = dict(phi=ctypes.byref(st), f=_vp(f), x=None, n=hp.n_rows, slot=_vp(slot), B=_vp(buf), ldb=4, r=3, wm=1,
                q=_vp(q), d=_vp(v[0]), var=_vp(v[1]), mean=_vp(v[2]))
    env.m.check(fn(*good.values(), s))
    bad = [dict(phi=None), dict(f=None), dict(slot=None), dict(B=None), dict(q=None), dict(d=None), dict(var=None),
           dict(mean=None), dict(r=0, wm=0), dict(r=64, wm=1, ldb=70), dict(r=-1), dict(wm=2), dict(ldb=3),
           dict(n=5), dict(x=_vp(ids), n=-2)]
    for b in bad:
        with pytest.raises(ValueError, match="grf_phi_row_downdate"):
            env.m.check(fn(*dict(good, **b).values(), s))
    env.m.check(fn(*dict(good, wm=0, mean=None).values(), s))
    for steps in (0, 33):
        st2 = _st(env, hp, d, 0, L=steps)
        with pytest.raises(ValueError, match="grf_phi_row_downdate"):
            env.m.check(fn(ctypes.byref(st2), *list(good.values())[1:], s))
    st3 = _st(env, hp, d, 0, blk=False)
    with pytest.raises(ValueError, match="grf_phi_row_downdate"):
        env.m.check(fn(ctypes.byref(st3), *list(good.values())[1:], s))


DISPATCH = ((1, 0, "row_downdate_narrow_kernel"), (3, 1, "row_downdate_narrow_kernel"),
            (4, 1, "row_downdate_mid_kernel"), (63, 1, "row_downdate_mid_kernel"))


def _dispatch_names():
    """For each (r, with_mean) of DISPATCH, the names of the kernels torch.profiler saw in one call."""
    from torch.profiler import ProfilerActivity, profile

    env = Env()
    hp, d = env.phi("pj")
    rng = np.random.default_rng(10)
    f = _f(rng, hp.L)
    slot, m = _slots(rng, hp.n_cols, 0.5)
    seen = []
    for r, wm, _ in DISPATCH:
        bbuf, boff, ldb, _ = _b_matrix(env, rng, m, r + wm, "pad")
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _call(env, hp, d, 0, f, None, hp.n_rows, slot, bbuf, boff, ldb, r, wm, np.zeros(hp.n_rows),
                  np.ones(hp.n_rows, np.float32))
        seen.append([e.name for e in prof.events() if "row_downdate" in e.name or "row_condition" in e.name])
    return seen


def test_row_downdate_dispatch_reaches_each_shape():
    """Run in a child process: a torch.profiler session in this process would leave the sessions of the profiler
    tests in later files without kernel events."""
    import json
    import os
    import subprocess
    import sys

    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    code = ("import json, sys; sys.path[:0] = {!r}; import test_gpu_posterior_downdate as T; "
            "print('NAMES' + json.dumps(T._dispatch_names()))").format(
        [here, root, os.path.join(root, "efficient-gaussian-process-on-graphs_b200")])
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable, *flags, "-c", code], capture_output=True, text=True, cwd=here,
                         timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    seen = json.loads(res.stdout.split("NAMES")[-1])
    for (r, wm, name), names in zip(DISPATCH, seen):
        assert names and all(name in n for n in names), (r, wm, names)


def test_phi_blocks_row_downdate_operands(g400):
    torch = g400["torch"]
    model, _, _ = _model(g400, np.arange(20), 0.1, 4)
    post = model.exact_posterior()
    phi = post.phi_f
    x = torch.arange(10).cuda()
    q = torch.zeros(10, dtype=torch.float64).cuda()
    d, var, mean = (torch.ones(10).cuda() for _ in range(3))
    B = torch.zeros((post.m, 2)).cuda()
    phi.row_downdate(torch.ones(1).cuda(), x, post.slot, B, 1, True, q, d, var, mean)
    for bad in (dict(B=B.double()), dict(B=torch.zeros((post.m, 1)).cuda()), dict(q=q.float()),
                dict(r=64), dict(var=var[:5]), dict(B=torch.zeros((post.m - 1, 2)).cuda())):
        kw = dict(B=B, r=1, q=q, var=var)
        kw.update(bad)
        with pytest.raises(ValueError, match="row_downdate"):
            phi.row_downdate(torch.ones(1).cuda(), x, post.slot, kw["B"], kw["r"], True, kw["q"], d, kw["var"], mean)


# ---- ExactPosterior.forget / set_targets / PosteriorMarginals ---------------------------------------------------
class Hist:
    """A posterior driven through appends and removals next to its float64 Track: every row of the history is a
    column of G_all over the union slots."""

    def __init__(self, setup, model, x_all, n0, noise, y_all=None):
        self.setup, self.model, self.noise = setup, model, noise
        self.x_all = np.asarray(x_all, np.int64)
        self.y_all = y_all
        f = model.covar_module.modulator_vector.detach().cpu().numpy()
        self.phi = _phi_f(setup["pp"].step_matrices_scipy, f)
        rows = self.phi[self.x_all]
        cols = np.unique(rows.indices)
        self.slot = np.full(self.phi.shape[1], -1, np.int64)
        self.slot[cols] = np.arange(cols.size)
        self.tr = DR.Track(rows[:, cols].T.toarray(), np.arange(n0), noise)
        self.margs = []                      # (PosteriorMarginals, blocks)

    def add(self, post, idx, y=None):
        torch = self.setup["torch"]
        post.condition_on(torch.tensor(self.x_all[idx]).cuda(),
                          None if y is None else torch.tensor(y).cuda())
        self.tr.append(idx)

    def remove(self, post, positions):
        post.forget(self.setup["torch"].tensor(positions).cuda())
        self.tr.remove(positions)

    def marginal(self, post, cand):
        m = post.marginals(self.setup["torch"].tensor(cand).cuda())
        self.margs.append((m, self.tr.marginal()))
        return m

    def fresh(self, y):
        torch = self.setup["torch"]
        from grf_b200.posterior import ExactPosterior

        return ExactPosterior(self.model.covar_module.phi_blocks, self.model.covar_module.modulator_vector.detach(),
                              torch.tensor(self.x_all[self.tr.order]).cuda(), self.noise,
                              y_train=None if y is None else torch.tensor(y).cuda())

    def compare(self, post, y, cand, n_cov=60, s=4):
        """Every output of the changed posterior and of its marginals against a fresh one, within the bounds."""
        torch = self.setup["torch"]
        tr, phi, slot = self.tr, self.phi, self.slot
        assert max(tr.kappa) <= CR.KAPPA_MAX
        assert post.n == len(tr.order) and np.array_equal(post.x.cpu().numpy(), self.x_all[tr.order])
        fresh = self.fresh(y)
        C, E_c, E_f = tr.C, tr.E, CR.U * np.abs(tr.C)
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
        fb = DR.side_bound(A, df, q, var_f)
        for m, blocks in self.margs:
            if not np.array_equal(m.x.cpu().numpy(), cand):
                continue
            mb_v = DR.marginal_bound(ti, col, w, nq, slot, blocks, var_f) + fb
            vm = m.variance().double().cpu().numpy()
            assert not m.stale
            assert np.all(np.abs(vm - var_f) <= mb_v), np.max(np.abs(vm - var_f) / mb_v)
        if y is not None:
            a = CR.weights(tr.G[:, tr.order], tr.L, y)
            mb = CR.mean_bound(ti, col, w, nq, slot, a)
            mu_c, mu_f = post.mean(xt).double().cpu().numpy(), fresh.mean(xt).double().cpu().numpy()
            assert np.all(np.abs(mu_c - mu_f) <= mb)
            for m, _ in self.margs:
                if np.array_equal(m.x.cpu().numpy(), cand):
                    assert np.all(np.abs(m.mean.double().cpu().numpy() - mu_f) <= mb)
            if len(tr.order):
                rng = np.random.default_rng(len(tr.order))
                eps = rng.standard_normal((s, phi.shape[1])).astype(np.float32)
                en = rng.standard_normal((s, len(tr.order))).astype(np.float32)
                e_t, en_t = torch.tensor(eps).cuda(), torch.tensor(en).cuda()
                sc = post.sample(xt, s, eps=e_t, eps_noise=en_t).double().cpu().numpy()
                sf = fresh.sample(xt, s, eps=e_t, eps_noise=en_t).double().cpu().numpy()
                prior_x = phi[self.x_all[tr.order]] @ eps.astype(np.float64).T
                v = y[:, None] - prior_x - np.sqrt(self.noise) * en.astype(np.float64).T
                z = sla.solve_triangular(tr.L, v, lower=True)
                sb = CR.sample_bound(ti, col, w, nq, slot, C, E_c, E_f, z, len(tr.order)).T
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
        # columns no kept row touches: their rows of C are exactly zero
        live = np.zeros(post.m, bool)
        xs = self.x_all[tr.order]
        if xs.size:
            live[post.slot.cpu().numpy()[np.unique(phi[xs].indices)]] = True
        assert torch.all(post.C[torch.tensor(~live).cuda()] == 0)
        return fresh


def _state(post):
    t = post.a.clone() if post.a is not None else None
    return (post.n, post.m, post.version, post.ldc, post.C.clone(), post.L.clone(), post.slot.clone(), t,
            post.x.clone(), None if post.y is None else post.y.clone(), post.nnz_train)


def _same(a, b):
    import torch

    for u, v in zip(a, b):
        assert (torch.equal(u, v) if isinstance(u, torch.Tensor) else u == v)


def test_forget_g400(g400):
    """Front, middle, end and random removals, with repeated ids in x, against fresh posteriors."""
    torch = g400["torch"]
    rng = np.random.default_rng(11)
    train = rng.permutation(400)[:160]
    train[20:23] = train[5]                             # repeated ids
    model, noise, y0 = _model(g400, train, 0.1, 4)
    post = model.exact_posterior()
    h = Hist(g400, model, train, len(train), noise)
    cand = np.arange(400)
    h.marginal(post, cand)
    y = y0.copy()
    picks = (lambda n: [0], lambda n: np.arange(0, 16), lambda n: [21, 5, 60], lambda n: np.arange(40, 56),
             lambda n: [n - 1, n - 2, 3], lambda n: rng.choice(n, 30, replace=False))
    for pick in picks:
        pos = np.asarray(pick(post.n))
        ev = {}
        post.events = ev
        v0 = post.version
        h.remove(post, pos)
        assert post.version == v0 + 1
        assert {"downdate_start", "downdate_factor", "downdate_columns", "downdate_weights"} <= set(ev)
        assert post.ldc == (post.n + 3) // 4 * 4
        y = np.delete(y, pos)
        h.compare(post, y, cand)


def test_chain_grid316(grid316):
    """condition_on -> forget -> condition_on -> forget (a sliding window), marginals made at the start and
    mid-chain."""
    torch = grid316["torch"]
    rng = np.random.default_rng(12)
    nodes = rng.choice(316 * 316, 760, replace=False)
    model, noise, y0 = _model(grid316, nodes[:600], 0.05, 5)
    post = model.exact_posterior()
    ys = np.r_[y0, rng.standard_normal(160)]
    h = Hist(grid316, model, nodes, 600, noise)
    cand = np.r_[rng.choice(316 * 316, 2000, replace=False), nodes[550:700]]
    h.marginal(post, cand)
    y = y0.copy()
    h.add(post, np.arange(600, 650), ys[600:650])
    y = np.r_[y, ys[600:650]]
    h.remove(post, np.arange(0, 50))                    # the oldest 50 rows
    y = y[50:]
    h.compare(post, y, cand)
    h.marginal(post, cand)                              # a second one, mid-chain
    h.add(post, np.arange(650, 651), ys[650:651])
    y = np.r_[y, ys[650:651]]
    h.remove(post, [0])
    y = y[1:]
    h.add(post, np.arange(651, 667), ys[651:667])
    y = np.r_[y, ys[651:667]]
    h.remove(post, np.r_[np.arange(0, 16), [post.n - 1]])
    y = np.r_[y[16:-1]]
    h.compare(post, y, cand)


def test_marginals_across_mixed_histories_and_both_paths(g400):
    """Runs of more than 64 columns (row_quadform + row_project) and at most 64 (the fused passes), removals of
    rows appended after the marginals were made, and a stale marginal that skips several changes."""
    torch = g400["torch"]
    rng = np.random.default_rng(13)
    perm = rng.permutation(400)
    model, noise, y0 = _model(g400, perm[:120], 0.1, 4)
    post = model.exact_posterior()
    ys = np.r_[y0, rng.standard_normal(280)]
    h = Hist(g400, model, perm[:300], 120, noise)
    cand = np.arange(400)
    m1 = h.marginal(post, cand)
    y = y0.copy()
    h.remove(post, np.arange(0, 70))                    # 70 + 1 columns: the fallback
    y = y[70:]
    h.compare(post, y, cand)
    h.add(post, np.arange(120, 190), ys[120:190])       # 70 appended columns
    y = np.r_[y, ys[120:190]]
    h.remove(post, np.arange(50, 60))                   # rows appended after m1 was made
    y = np.delete(y, np.arange(50, 60))
    h.compare(post, y, cand)
    h.marginal(post, cand)
    for k in range(3):                                   # several changes between refreshes
        h.add(post, np.arange(190 + 5 * k, 195 + 5 * k), ys[190 + 5 * k:195 + 5 * k])
        y = np.r_[y, ys[190 + 5 * k:195 + 5 * k]]
        h.remove(post, [2 * k])
        y = np.delete(y, 2 * k)
    assert m1.stale
    h.compare(post, y, cand)
    assert len(post._log) == 0                           # every marginal is current: the log is trimmed
    del h.margs[:]
    m1 = None
    h.add(post, np.arange(205, 210), ys[205:210])
    assert len(post._log) == 0 and len(post._watchers) == 0


def test_append_only_marginals_unchanged(g400):
    """With appends alone the refresh is the single pass over [C[:, n_seen:n] | a] it always was: bit for bit."""
    torch = g400["torch"]
    rng = np.random.default_rng(14)
    perm = rng.permutation(400)
    model, noise, _ = _model(g400, perm[:100], 0.1, 4)
    post = model.exact_posterior()
    cand = torch.arange(400).cuda()
    marg = post.marginals(cand)
    one = torch.ones(1).cuda()
    q, d = marg.q.clone(), marg.d.clone()
    var, mean = marg._var.clone(), marg._mean.clone()
    n0 = post.n
    for b in (1, 7, 20):
        xb = perm[100 + post.n - n0:][:b]
        post.condition_on(torch.tensor(xb).cuda(), torch.tensor(rng.standard_normal(b)).cuda())
    n = post.n
    B = torch.empty((post.m, n - n0 + 1), dtype=torch.float32, device="cuda")
    B[:, :n - n0] = post.C[:, n0:n]
    B[:, n - n0] = post.a[:, 0]
    post.phi_f.row_condition(one, cand, post.slot, B, n - n0, True, q, d, var, mean)
    assert torch.equal(marg.variance(), var) and torch.equal(marg.mean, mean) and torch.equal(marg.q, q)
    for b in (40, 30):                                   # 70 columns: row_quadform + row_project
        xb = perm[100 + post.n - n0:][:b]
        post.condition_on(torch.tensor(xb).cuda(), torch.tensor(rng.standard_normal(b)).cuda())
    dq, _ = post.phi_f.row_quadform(one, cand, post.slot, post.C[:, n:post.n])
    q += dq.to(torch.float64)
    var = torch.clamp_min((d.to(torch.float64) - q).to(torch.float32), 0.0)
    mean = post.phi_f.row_project(one, cand, post.slot, post.a)[:, 0]
    assert torch.equal(marg.variance(), var) and torch.equal(marg.mean, mean)


def test_gp_bucb_round_trip(g400):
    """Hallucinate a batch with condition_on(x, mean(x)), then set_targets with the real values: the posterior of
    the real targets."""
    torch = g400["torch"]
    rng = np.random.default_rng(15)
    perm = rng.permutation(400)
    train = perm[:150]
    model, noise, y0 = _model(g400, train, 0.1, 4)
    post = model.exact_posterior()
    h = Hist(g400, model, perm[:158], 150, noise)
    cand = np.arange(400)
    marg = h.marginal(post, cand)
    for i in range(150, 158):                            # greedy batch: one at a time, mean as the target
        xb = torch.tensor(perm[i:i + 1]).cuda()
        h.add(post, [i], post.mean(xb).double().cpu().numpy())
        marg.variance()
    real = rng.standard_normal(8)
    v0 = post.version
    assert post.set_targets(torch.tensor(real).cuda(), positions=torch.arange(150, 158)) is post
    assert post.version == v0 + 1 and marg.stale
    y = np.r_[y0, real]
    fresh = h.compare(post, y, cand)
    assert torch.equal(post.y, torch.tensor(y).cuda())
    # all targets at once; variance and C stay bit for bit
    C, L, var = post.C.clone(), post.L.clone(), marg.variance()
    y2 = rng.standard_normal(158)
    post.set_targets(torch.tensor(y2).cuda())
    assert torch.equal(post.C, C) and torch.equal(post.L, L) and torch.equal(marg.variance(), var)
    h.compare(post, y2, cand)
    assert post.set_targets([], positions=[]) is post and post.version == v0 + 2


def test_forget_everything_and_the_diffusion_prior(g400):
    torch = g400["torch"]
    from efficient_graph_gp_sparse.gptorch_kernels_sparse import SparseDiffusionKernel
    from grf_b200.posterior import ExactPosterior

    kern = SparseDiffusionKernel(max_walk_length=4, step_matrices_torch=g400["ops"]).cuda()
    f = kern.modulator_vector.detach()
    x0 = np.r_[np.arange(0, 400, 7), 0, 0]
    post = ExactPosterior(kern.phi_blocks, f, torch.tensor(x0).cuda(), 0.2)
    cand = torch.arange(400).cuda()
    marg = post.marginals(cand)
    post.forget(torch.arange(10, 20))
    want = ExactPosterior(kern.phi_blocks, f, torch.tensor(np.delete(x0, np.arange(10, 20))).cuda(), 0.2)
    assert torch.allclose(post.variance(cand), want.variance(cand), rtol=1e-4, atol=1e-5)
    post.forget(np.random.default_rng(0).permutation(post.n))     # every row: the prior
    prior = ExactPosterior(kern.phi_blocks, f, torch.zeros(0, dtype=torch.int64).cuda(), 0.2)
    assert post.n == 0 and post.L.shape == (0, 0) and post.C.shape[1] == 0 and post.nnz_train == 0
    assert torch.equal(post.variance(cand), prior.variance(cand))
    assert torch.equal(post.covariance(cand[:30]), prior.covariance(cand[:30]))
    assert torch.allclose(marg.variance(), prior.variance(cand), rtol=1e-4, atol=1e-4)
    with pytest.raises(ValueError):
        post.set_targets(torch.zeros(0).cuda())
    post.condition_on(torch.tensor([3, 5, 3]).cuda())             # grows again from n = 0
    again = ExactPosterior(kern.phi_blocks, f, torch.tensor([3, 5, 3]).cuda(), 0.2)
    assert torch.allclose(post.variance(cand), again.variance(cand), rtol=1e-4, atol=1e-5)
    assert torch.allclose(marg.variance(), again.variance(cand), rtol=1e-4, atol=1e-4)


def test_retired_slots_match_a_fresh_posterior(g400):
    """Candidates that touch only columns of removed rows get exactly the prior variance, as from a posterior that
    never saw those rows; a later append reuses the retired slots."""
    torch = g400["torch"]
    model, noise, y0 = _model(g400, np.r_[np.arange(0, 40), 399], 0.1, 4)
    post = model.exact_posterior()
    m0 = post.m
    post.forget([40])                                    # the isolated node 399: its own column only
    from grf_b200.posterior import ExactPosterior

    fresh = ExactPosterior(model.covar_module.phi_blocks, model.covar_module.modulator_vector.detach(),
                           torch.arange(40).cuda(), noise, y_train=torch.tensor(y0[:40]).cuda())
    c = torch.tensor([399]).cuda()
    assert torch.equal(post.variance(c), fresh.variance(c))
    assert torch.equal(post.mean(c), torch.zeros(1).cuda()) and torch.equal(fresh.mean(c), torch.zeros(1).cuda())
    post.condition_on(c, torch.ones(1).cuda())
    assert post.m == m0                                  # the slot came back
    want = ExactPosterior(model.covar_module.phi_blocks, model.covar_module.modulator_vector.detach(),
                          torch.tensor(np.r_[np.arange(40), 399]).cuda(), noise,
                          y_train=torch.tensor(np.r_[y0[:40], 1.0]).cuda())
    assert torch.allclose(post.variance(torch.arange(400).cuda()), want.variance(torch.arange(400).cuda()),
                          rtol=1e-4, atol=1e-5)


def test_forget_and_set_targets_errors(g400):
    torch = g400["torch"]
    model, noise, y0 = _model(g400, np.arange(30), 0.1, 4)
    post = model.exact_posterior()
    marg = post.marginals(torch.arange(400).cuda())
    before = _state(post)
    for bad in ([30], [-1], [0, 31]):
        with pytest.raises(IndexError):
            post.forget(bad)
    with pytest.raises(ValueError, match="repeat"):
        post.forget([3, 4, 3])
    assert post.forget([]) is post and post.forget(torch.zeros(0, dtype=torch.int64)) is post
    post.mem_limit = 1000
    with pytest.raises(MemoryError, match="bytes"):
        post.forget([0])
    post.mem_limit = None
    L_saved = post.L.clone()
    post.L[10, 5:] = 0.0                                 # T = L[R2, j0:] gets a zero row: T T^T is singular
    tampered = _state(post)
    with pytest.raises(ValueError, match="positive definite"):
        post.forget([5])
    _same(tampered, _state(post))
    post.L.copy_(L_saved)
    for y, pos, exc in ((torch.zeros(29), None, ValueError), (torch.zeros(2), [1], ValueError),
                        (torch.tensor([float("nan")]), [1], ValueError), (torch.tensor([float("inf")] * 30), None,
                                                                         ValueError),
                        (torch.zeros(1), [30], IndexError), (torch.zeros(2), [1, 1], ValueError)):
        with pytest.raises(exc):
            post.set_targets(y.cuda(), positions=pos)
    _same(before, _state(post))
    assert not marg.stale
    post.forget([0, 29])                                 # still usable
    assert post.n == 28 and post.version == 1
    from grf_b200.posterior import ExactPosterior

    no_y = ExactPosterior(model.covar_module.phi_blocks, model.covar_module.modulator_vector.detach(),
                          torch.arange(5).cuda(), noise)
    with pytest.raises(ValueError, match="y_train"):
        no_y.set_targets(torch.zeros(5).cuda())
