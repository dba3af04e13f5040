"""-m gpu tests of the matvec-layer C entry points, called directly through grf_b200._lib.

Every test builds its inputs on the host (tests/matvec_abi_ref.py: synthetic Phi in both block layouts, no walker
and no grf_transpose_*), calls one entry point on torch's current stream, synchronises once and compares with a
float64 reference under a per-element bound.  For the product out = Phi_f[x1] (Phi_f[x2]^T V):

    |got - want|_ij <= 2^-22 * ( len(Phi[x1_i]) * A_ij + (|Phi_f[x1]| (n o (|Phi_f[x2]|^T |V|)))_ij ),
    A = |Phi_f[x1]| (|Phi_f[x2]|^T |V|),   |Phi_f| = sum_l |f_l| |M_l|,   n_c = summands of column c of U,

the float32 summation bound with a factor-4 margin (n_c <= max_c len(Phi^T_c), so it is at most
2^-22 (len(Phi[x1_i]) + max_c len(Phi^T_c)) A_ij).  It holds for any summation order; where the order is fixed
(all but the atomic scatter) repeated calls must also agree bit for bit.  Memory the kernels must leave alone
(rows of `out` for ids outside the shard, columns [t, ldo) of `out`, the tail of partial buffers) is checked bit
for bit against a sentinel; columns [t, ldu) of U and vfull are scratch and hold NaN beforehand, so that a
kernel that read them into a result would fail.  Each row of the grf_phi_matvec table names the kernels it
reaches, and the first call of each row runs under torch.profiler to confirm them."""

from __future__ import annotations

import ctypes
import zlib
from dataclasses import dataclass, fields
from typing import Optional

import numpy as np
import pytest

import matvec_abi_ref as R

pytestmark = pytest.mark.gpu

SENT = np.float32(-1234.5)       # sentinel of memory that must stay untouched


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

    def sync(self):
        self.torch.cuda.synchronize()

    def phi(self, name):
        """(HostPhi, device arrays) of a profile, built once per module."""
        if name not in self._phis:
            hp = R.profile(name)
            tptr, tent = hp.transpose()
            one = np.zeros((1, 2), np.int32)
            d = dict(blk_ptr=self.dev(hp.blk_ptr), entries=self.dev(hp.entries if hp.nnz else one),
                     tblk_ptr=self.dev(tptr), tentries=self.dev(tent if hp.nnz else one))
            self._phis[name] = (hp, d)
        return self._phis[name]


@pytest.fixture(scope="module")
def env():
    return Env()


def _vp(t, off=0):
    return None if t is None else ctypes.c_void_p(t.data_ptr() + 4 * off)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


# ---- strided operands -------------------------------------------------------------------------------------
def _ld(lay, t):
    return {"tight": t, "pad4": (t + 3) // 4 * 4, "plus7": t + 7, "off1": (t + 3) // 4 * 4}[lay]


class Mat:
    """A rows x t float32 matrix inside a larger buffer: leading dimension and base offset by layout
    ("off1": the base pointer is one float past a 16-byte boundary), a guard tail of 3 floats."""

    def __init__(self, env, rows, t, lay, fill):
        self.env, self.rows, self.t = env, rows, t
        self.ld, self.off = _ld(lay, t), 1 if lay == "off1" else 0
        self.buf = env.torch.full((rows * self.ld + self.off + 3,), float(fill), dtype=env.torch.float32,
                                  device="cuda")

    @property
    def ptr(self):
        return _vp(self.buf, self.off)

    def view(self):
        return self.buf[self.off:self.off + self.rows * self.ld].view(self.rows, self.ld)

    def set(self, a):
        self.view()[:, :self.t] = self.env.torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()

    def get(self):
        return self.view()[:, :self.t].cpu().numpy()

    def raw(self):
        return self.buf.cpu().numpy().copy()

    def cells(self, rows):
        """mask over raw(): the [0, t) columns of the given rows."""
        m = np.zeros(self.buf.numel(), bool)
        for r in np.flatnonzero(rows):
            b = self.off + r * self.ld
            m[b:b + self.t] = True
        return m


def _check_close(got, want, bound, what):
    err = np.abs(got.astype(np.float64) - want)
    bad = ~(err <= bound)
    if bad.any():
        i = np.argwhere(bad)[0]
        raise AssertionError(f"{what}: {bad.sum()} elements outside the bound, first {tuple(i)}: got {got[tuple(i)]!r} "
                             f"want {want[tuple(i)]!r} bound {bound[tuple(i)]!r}")


def _kernels(env, fn):
    """Run fn() under torch.profiler; the names of the CUDA kernels it launched (spaces removed)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        env.sync()
    return {e.key.replace(" ", "") for e in prof.key_averages()}


def _f(rng, L):
    """Modulator with a zero and a negative entry."""
    f = (2.0 ** rng.uniform(-2, 1, L)).astype(np.float32)
    f[1] = 0.0
    f[L - 1] = -f[L - 1]
    return f


def _ids(rng, k, row_lo, n_rows, *, uniq=False, must=()):
    """k global row ids from [row_lo - 200, row_lo + n_rows + 200): ids below and above the shard, `must` (local
    rows) first; unless uniq, about a tenth of them twice (never more than twice, so that atomic sums of repeats
    stay order independent)."""
    lo, hi = max(0, row_lo - 200), row_lo + n_rows + 200
    base = rng.choice(np.arange(lo, hi), size=min(k, hi - lo), replace=False)
    base = np.r_[np.asarray(must, np.int64) + row_lo, base[~np.isin(base, np.asarray(must) + row_lo)]][:k]
    if not uniq:
        base = np.r_[base, rng.choice(base, size=max(1, k // 10), replace=False)]
    return rng.permutation(base).astype(np.int32)


# ---- long-row tables, tcols, windows ------------------------------------------------------------------------
def _long(env, hp, d, side, chunk, ordered, ld, rng, keep, checks):
    """GrfLongRows of one side from grf_row_census + grf_long_rows_build (threshold 256, chunks of `chunk`),
    checked against the host; chunk_order = a random permutation when `ordered`."""
    torch, lib = env.torch, env.lib
    ptr, ent, n = ((d["blk_ptr"], d["entries"], hp.n_rows) if side == "fwd"
                   else (d["tblk_ptr"], d["tentries"], hp.n_cols))
    lens = hp.row_len if side == "fwd" else hp.col_len
    census = torch.full((3,), -1, dtype=torch.int32, device="cuda")
    env.m.check(lib.grf_row_census(_vp(ptr), n, hp.L, R.THRESHOLD, _vp(census), env.stream()))
    n_long, n_chunks, n_full = census.tolist()
    host = hp.census()[0:3] if side == "fwd" else hp.census()[3:6]
    assert [n_long, n_chunks, n_full] == host
    if n_long == 0:
        return None
    long_lens = lens[lens > R.THRESHOLD]
    n_chunks = int(((long_lens + chunk - 1) // chunk).sum())
    rows = torch.empty(n_long, dtype=torch.int32, device="cuda")
    chunk_ptr = torch.empty(n_long + 1, dtype=torch.int32, device="cuda")
    bounds = torch.empty((n_chunks, 2), dtype=torch.int32, device="cuda")
    ticket = torch.empty(1, dtype=torch.int64, device="cuda")
    env.m.check(lib.grf_long_rows_build(_vp(ptr), _vp(ent), n, hp.L, R.THRESHOLD, chunk, n_long, n_chunks,
                                        _vp(ticket), _vp(rows), _vp(chunk_ptr), _vp(bounds), None, env.stream()))

    def check_table():
        """every long row once, its chunks of `chunk` entries tiling its entry run in order (checked after the
        product, so that a wrong table is first seen by the product's bound)"""
        hptr = (hp.blk_ptr if side == "fwd" else hp.transpose()[0]).astype(np.int64)
        r, cp, bd = rows.cpu().numpy(), chunk_ptr.cpu().numpy(), bounds.cpu().numpy()
        assert sorted(r.tolist()) == np.flatnonzero(lens > R.THRESHOLD).tolist()
        for i, row in enumerate(r):
            b, e = hptr[row * hp.L], hptr[(row + 1) * hp.L]
            want = np.arange(b, e, chunk)
            assert np.array_equal(bd[cp[i]:cp[i + 1], 0], want) and np.array_equal(bd[cp[i]:cp[i + 1], 1],
                                                                                    np.minimum(want + chunk, e))

    checks.append(check_table)
    order = env.dev(rng.permutation(n_chunks).astype(np.int32)) if ordered else None
    partial = torch.full((n_chunks, ld), float("nan"), dtype=torch.float32, device="cuda")
    keep += [rows, chunk_ptr, bounds, ticket, order, partial]
    return env.m.GrfLongRows(R.THRESHOLD, n_long, n_chunks, rows.data_ptr(), chunk_ptr.data_ptr(),
                             bounds.data_ptr(), partial.data_ptr(), ld, None if order is None else order.data_ptr())


def _windows(env, hp, d, side, keep):
    ptr, ent, n = ((d["blk_ptr"], d["entries"], hp.n_rows) if side == "fwd"
                   else (d["tblk_ptr"], d["tentries"], hp.n_cols))
    win = env.torch.empty(((n + 31) // 32, 2), dtype=env.torch.int32, device="cuda")
    mw = env.torch.empty(1, dtype=env.torch.int32, device="cuda")
    env.m.check(env.lib.grf_block_windows(_vp(ptr), _vp(ent), n, hp.L, _vp(win), _vp(mw), env.stream()))
    env.sync()
    hptr, hent = (hp.blk_ptr, hp.entries) if side == "fwd" else hp.transpose()
    hwin, hmw = R.windows(hptr, hent, n, hp.L)
    assert np.array_equal(win.cpu().numpy(), hwin) and int(mw.item()) == hmw
    keep.append(win)
    return win, hmw, hwin


# ---- the grf_phi_matvec table -------------------------------------------------------------------------------
@dataclass(frozen=True)
class C:
    phi: str
    t: int
    which: int = 3                 # 1 / 2 / 3 plus the +4 / +8 / +16 / +32 flags
    lay: str = "pad4"              # V and out: tight (ld = t), pad4 (round_up(t, 4)), plus7 (t + 7), off1
    ulay: str = "pad4"             # U and vfull
    vfull: bool = False
    x1: bool = False               # a row selection with ids outside the shard and repeats
    x2: Optional[str] = None       # None | "sel" (>= 1/16 of the rows) | "few" (< 1/16: scatter half) | "uniq"
    long: Optional[int] = None     # chunk size of the long-row split (None: no split)
    order: bool = False            # random chunk_order
    tcols: Optional[str] = None    # None | "all" | "used" (strict subset) | "none" (n_tcols = 0)
    sched: bool = False
    row_lo: int = 0
    win: bool = False
    k: tuple = ()                  # kernels the call must launch

    def id(self):
        parts = [self.phi, f"t{self.t}", f"w{self.which}", self.lay]
        for fld in fields(self)[4:-1]:
            v = getattr(self, fld.name)
            if v not in (None, False, 0, "pad4"):
                parts.append(fld.name if v is True else f"{fld.name}{v}")
        return "-".join(parts)


B, CO, TI = "spmm_blocks_kernel", "spmv_coop_kernel", "spmm_tiled_kernel"
LR, PAD, SCU, SCA, SCT = ("long_reduce_kernel", "pad_copy_kernel", "scatter_rows_unique_kernel", "scatter_rows_kernel",
                          "spmm_scatter_kernel")


def b(tpr, vec, stream=False):
    return f"{B}<{tpr},{vec},{'true' if stream else 'false'}>"


CASES = [
    # ---- pl: avg 19 entries per row, so the one-row-per-lane-group kernel also at t <= 4 ----
    C("pl", 1, lay="tight", k=(b(1, 1),)),                                     # VEC=1 TPR=1 both halves
    C("pl", 2, lay="tight", k=(b(2, 1),)),                                     # VEC=1 TPR=2
    C("pl", 3, lay="tight", k=(b(4, 1), b(1, 4))),                             # Phi^T V scalar (ldv = 3), Phi U float4
    C("pl", 3, k=(b(1, 4),)),                                                  # float4 TPR=1; ldo = 4 > t
    C("pl", 4, lay="tight", sched=True, k=(b(1, 4),)),                         # TPR=1 with the ticket scheduler
    C("pl", 5, lay="tight", k=(b(8, 1), b(2, 4))),                             # VEC=1 TPR=8 / float4 TPR=2
    C("pl", 5, vfull=True, x1=True, x2="sel", row_lo=1000, k=(SCA, b(2, 4))),  # vfull + atomic scatter of x2
    C("pl", 8, which=3 + 32, k=(b(2, 4, True),)),                              # streaming gathers TPR=2
    C("pl", 8, lay="plus7", k=(b(8, 1), b(2, 4))),                             # ldv = 15: scalar first half
    C("pl", 8, lay="plus7", vfull=True, k=(PAD, b(2, 4))),                     # V staged into vfull
    C("pl", 12, lay="tight", long=256, k=(b(4, 4), LR)),                       # long rows both sides, chunk = 256
    C("pl", 12, lay="off1", k=(b(16, 1), b(4, 4))),                            # unaligned V: VEC=1 TPR=16
    C("pl", 12, lay="off1", vfull=True, k=(PAD, b(4, 4))),                     # unaligned V staged
    C("pl", 16, lay="tight", long=100, order=True, k=(b(4, 4), LR)),           # chunk < threshold, ordered
    C("pl", 16, which=3 + 32, lay="tight", sched=True, k=(b(4, 4, True),)),    # streaming + scheduler
    C("pl", 16, which=3 + 8, lay="tight", x1=True, x2="uniq", row_lo=1000, vfull=True, k=(SCU, b(4, 4))),
    C("pl", 16, which=1 + 16, long=256, k=(b(4, 4), LR)),                      # U += on the split-row path
    C("pl", 17, lay="tight", vfull=True, k=(PAD, b(8, 4))),                    # t = 17 staged, TPR=8
    C("pl", 17, long=256, order=True, k=(b(8, 4), LR)),                        # ldo = 20: padding columns of out
    C("pl", 17, lay="tight", k=(b(32, 1), b(8, 4))),                           # VEC=1 TPR=32
    C("pl", 32, long=256, tcols="all", k=(b(8, 4), LR)),                       # tcols = every column
    C("pl", 32, which=3 + 32, lay="tight", tcols="used", k=(b(8, 4, True),)),  # tcols = the non-empty columns
    C("pl", 64, long=100, k=(b(16, 4), LR)),                                   # TPR=16, chunk < threshold
    C("pl", 64, which=3 + 32, k=(b(16, 4, True),)),
    C("pl", 65, k=(b(32, 4),)),                                                # TPR=32 float4
    C("pl", 65, lay="tight", k=(b(32, 1), b(32, 4))),                          # VEC=1 with 3 column tiles
    C("pl", 128, which=3 + 32, k=(b(32, 4, True),)),
    C("pl", 128, lay="tight", x1=True, row_lo=1000, k=(b(32, 4),)),
    C("pl", 130, long=256, k=(b(32, 4), LR)),                                  # 2 column tiles, ldo = 132
    C("pl", 130, lay="plus7", k=(b(32, 1), b(32, 4))),                         # VEC=1, 5 column tiles
    C("pl", 16, lay="tight", x1=True, x2="few", row_lo=1000, k=(SCT, b(4, 4))),  # scatter half (atomics)
    C("pl", 3, x1=True, x2="few", row_lo=1000, k=(SCT, b(1, 4))),
    C("pl", 16, which=2, lay="tight", x1=True, row_lo=1000, k=(b(4, 4),)),     # second half only
    C("pl", 16, which=1, lay="tight", k=(b(4, 4),)),                           # first half only
    C("pl", 16, which=1, ulay="off1", k=(b(16, 1),)),                          # unaligned U: VEC=1
    # ---- dense: avg 100 entries per row -> CSR-vector kernel at t <= 4 ----
    C("dense", 1, lay="tight", long=256, k=(f"{CO}<32,1>", LR)),                # coop T=1 + split rows both sides
    C("dense", 2, lay="tight", k=(f"{CO}<32,2>",)),
    C("dense", 3, long=256, k=(f"{CO}<32,3>", LR)),
    C("dense", 4, lay="tight", x1=True, x2="sel", vfull=True, row_lo=300, k=(SCA, f"{CO}<32,4>")),
    C("dense", 4, which=1 + 16, lay="tight", long=256, k=(f"{CO}<32,4>", LR)),  # U += on the coop split path
    C("dense", 2, which=1 + 16, lay="tight", k=(f"{CO}<32,2>",)),             # U += on the coop path
    C("dense", 8, k=(b(2, 4),)),
    # ---- l32: length 31 sets bit 31 of the packed column ----
    C("l32", 16, long=256, k=(b(4, 4), LR)),
    C("l32", 3, lay="tight", k=(b(4, 1), b(1, 4))),
    C("l32", 1, lay="tight", x1=True, x2="sel", vfull=True, row_lo=500, k=(SCA, b(1, 1))),
    # ---- band: column windows -> shared-memory tiles ----
    C("band", 16, win=True, k=(f"{TI}<4>",)),                                  # tiled both halves
    C("band", 64, win=True, k=(f"{TI}<16>",)),                                 # + Phi chunks that do not fit
    C("band", 4, lay="tight", win=True, k=(f"{TI}<1>",)),
    C("band", 128, win=True, k=(f"{TI}<32>", b(32, 4))),                       # Phi^T declines the tiles
    C("band", 16, which=3 + 4, win=True, k=(b(4, 4),)),                        # +4: global gathers
    C("band", 16, which=1 + 16, win=True, k=(b(4, 4),)),                       # U += never tiles
    # ---- shards without entries / without rows ----
    C("empty", 16, tcols="none", k=(b(4, 4),)),                                # n_tcols = 0: U zero-filled
    C("empty", 3, tcols="all", k=(b(1, 4),)),
    C("noshard", 16, x1=True, x2="sel", vfull=True, row_lo=100, k=(b(4, 4),)),  # n_rows = 0
    C("noshard", 5, which=1, lay="tight"),                                     # memset of U only
]


class Run:
    """One grf_phi_matvec configuration: inputs, buffers and the call."""

    def __init__(self, env, c: C):
        torch = env.torch
        self.env, self.c = env, c
        self.hp, d = env.phi(c.phi)
        hp, t = self.hp, c.t
        self.rng = rng = np.random.default_rng(zlib.crc32(c.id().encode()))
        self.keep = []
        self.f = _f(rng, hp.L)
        self.f_dev = env.dev(self.f)
        must = [r for r in list(R.SPECIAL_ROWS) + [0, 1, 2, 3, 4, 5] if r < hp.n_rows]
        self.x1 = _ids(rng, max(8, hp.n_rows // 12), c.row_lo, hp.n_rows, must=must) if c.x1 else None
        n2k = {"sel": max(5, hp.n_rows // 7), "uniq": max(5, hp.n_rows // 7), "few": max(1, hp.n_rows // 40)}
        self.x2 = (_ids(rng, n2k[c.x2], c.row_lo, hp.n_rows, uniq=c.x2 == "uniq", must=must) if c.x2 else None)
        if c.x2 == "few":
            assert len(self.x2) * 16 < hp.n_rows
        elif c.x2:
            assert len(self.x2) * 16 >= hp.n_rows
        self.n1 = hp.n_rows if self.x1 is None else len(self.x1)
        self.n2 = hp.n_rows if self.x2 is None else len(self.x2)
        ld4 = (t + 3) // 4 * 4
        self.table_checks = []
        lf = _long(env, hp, d, "fwd", c.long, c.order, ld4, rng, self.keep, self.table_checks) if c.long else None
        lt = _long(env, hp, d, "t", c.long, c.order, ld4, rng, self.keep, self.table_checks) if c.long else None
        if c.long:
            assert lf is not None and lt is not None, "the profile should split rows on both sides"
        tcols, n_tcols = None, 0
        if c.tcols:
            ids = {"all": np.arange(hp.n_cols), "used": np.flatnonzero(hp.col_len > 0), "none": np.zeros(0)}[c.tcols]
            if c.tcols == "used":
                assert 0 < ids.size < hp.n_cols
            tcols, n_tcols = env.dev(np.r_[ids, 0].astype(np.int32)), ids.size
        self.sched = torch.zeros(2, dtype=torch.int32, device="cuda") if c.sched else None
        win = twin = None
        mw = tmw = 0
        if c.win:
            win, mw, hwin = _windows(env, hp, d, "fwd", self.keep)
            twin, tmw, htwin = _windows(env, hp, d, "t", self.keep)
            self.plans = (R.tiled_plan(hwin, mw, hp.n_rows, t), R.tiled_plan(htwin, tmw, hp.n_cols, t))
        self.keep += [tcols, d]
        self.phi = env.m.GrfPhi(hp.n_rows, hp.n_cols, c.row_lo, hp.L, d["blk_ptr"].data_ptr(),
                                d["entries"].data_ptr(), d["tblk_ptr"].data_ptr(), d["tentries"].data_ptr(),
                                None if win is None else win.data_ptr(), None if twin is None else twin.data_ptr(),
                                mw, tmw, None if lf is None else ctypes.pointer(lf),
                                None if lt is None else ctypes.pointer(lt), None if tcols is None else tcols.data_ptr(),
                                n_tcols, hp.nnz, None if self.sched is None else self.sched.data_ptr())
        self.keep += [lf, lt]
        # operands
        self.v = Mat(env, self.n2, t, c.lay, SENT)
        self.out = Mat(env, self.n1, t, c.lay, SENT)
        self.u = Mat(env, hp.n_cols, t, c.ulay, np.nan)
        self.vfull = Mat(env, hp.n_rows, t, c.ulay, 0.0 if c.which & 8 else np.nan) if c.vfull else None
        self.u0 = None
        if c.which & 16:
            self.u0 = rng.standard_normal((hp.n_cols, t)).astype(np.float32)
        if (c.which & 3) == 2:       # the second half reads a given U
            self.u0 = rng.standard_normal((hp.n_cols, t)).astype(np.float32)
        self.new_v()

    def new_v(self):
        self.vh = self.rng.standard_normal((self.n2, self.c.t)).astype(np.float32)
        self.v.set(self.vh)

    def prepare(self):
        if self.u0 is not None:
            self.u.set(self.u0)

    def call(self):
        c, hp, env = self.c, self.hp, self.env
        self.prepare()
        rc = env.lib.grf_phi_matvec(ctypes.byref(self.phi), _vp(self.f_dev),
                                    None if self.x1 is None else _vp(self._x1d()), self.n1,
                                    None if self.x2 is None else _vp(self._x2d()), self.n2, self.v.ptr, self.v.ld,
                                    self.out.ptr, self.out.ld, self.u.ptr, self.u.ld,
                                    None if self.vfull is None else self.vfull.ptr, c.t, c.which, env.stream())
        env.m.check(rc)

    def _x1d(self):
        if not hasattr(self, "_x1_dev"):
            self._x1_dev = self.env.dev(self.x1)
        return self._x1_dev

    def _x2d(self):
        if not hasattr(self, "_x2_dev"):
            self._x2_dev = self.env.dev(self.x2)
        return self._x2_dev

    def check(self):
        """Compare with the float64 reference; sentinels of out; the scheduler's ints."""
        c, hp = self.c, self.hp
        env = self.env
        env.sync()
        which = c.which & 3
        if which == 2:
            u, ua, n_c = self.u0.astype(np.float64), np.abs(self.u0.astype(np.float64)), np.zeros(hp.n_cols)
        else:
            u, ua, n_c = R.ref_first_half(hp, self.f, self.x2, self.vh, c.row_lo, self.u0)
        if which == 1:
            _check_close(self.u.get(), u, R.UB * n_c[:, None] * ua, f"{c.id()} U")
        else:
            want, bound = R.ref_second_half(hp, self.f, self.x1, u, ua, n_c, c.row_lo)
            mine = np.ones(self.n1, bool) if self.x1 is None else R.in_shard(self.x1, c.row_lo, hp.n_rows)
            got = self.out.get()
            _check_close(got[mine], want[mine], bound[mine], f"{c.id()} out")
            raw = self.out.raw()
            keep = ~self.out.cells(mine)
            assert np.array_equal(_bits(raw[keep]), _bits(np.full(keep.sum(), SENT))), \
                f"{c.id()}: out was written outside rows of the shard x columns [0, t)"
        if self.sched is not None:
            assert self.sched.tolist() == [0, 0]

    def result_bits(self):
        return _bits(self.out.raw() if (self.c.which & 3) != 1 else self.u.get())


@pytest.mark.parametrize("c", CASES, ids=[c.id() for c in CASES])
def test_phi_matvec(env, c):
    r = Run(env, c)
    names = _kernels(env, r.call)
    for k in c.k:
        assert any(k in n for n in names), f"{c.id()}: expected {k} among {sorted(n for n in names if 'grf' in n)}"
    r.check()
    for check_table in r.table_checks:
        check_table()
    if c.win:
        fwd, tside = r.plans
        if c.t == 64:
            assert fwd is not None and 0 < sum(fwd) < len(fwd), "some chunks of Phi should fall back"
        if c.t == 128:
            assert fwd is not None and tside is None
        if c.t in (4, 16) and not c.which & 20:
            assert fwd is not None and all(fwd) and tside is not None and all(tside)
    if c.which & 8:
        # vfull was zeroed once; a second call with the same x2 and a new V needs no memset
        r.new_v()
        r.call()
        r.check()
        return
    if c.x2 == "few":
        return                                  # fp32 atomics: the summation order is not fixed
    first = r.result_bits()
    for _ in range(2 if c.sched else 1):
        r.call()
        r.check()
        assert np.array_equal(r.result_bits(), first), f"{c.id()}: repeated call differs"


# ---- grf_phi_fgrad ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("phi,t,lay,sel", [
    ("pl", 1, "pad4", False),     # VEC=1 TPR=1, all rows
    ("pl", 4, "pad4", True),      # VEC=4 TPR=1
    ("pl", 16, "off1", True),     # unaligned left / P: VEC=1 TPR=16
    ("pl", 17, "pad4", True),     # t % 4 != 0: VEC=1 TPR=32
    ("pl", 128, "pad4", True),    # VEC=4 TPR=32
    ("pl", 130, "plus7", True),   # VEC=1, 5 column passes per lane
    ("l32", 3, "tight", False),
    ("l32", 64, "pad4", True),
    ("l32", 130, "off1", True),
])
def test_phi_fgrad(env, phi, t, lay, sel):
    hp, d = env.phi(phi)
    rng = np.random.default_rng(t * 7 + len(phi))
    row_lo = 700 if sel else 0
    x = _ids(rng, 300, row_lo, hp.n_rows, must=list(R.SPECIAL_ROWS[:2])) if sel else None
    n = hp.n_rows if x is None else len(x)
    left, p = Mat(env, n, t, lay, np.nan), Mat(env, hp.n_cols, t, lay, np.nan)
    lh = rng.standard_normal((n, t)).astype(np.float32)
    ph = rng.standard_normal((hp.n_cols, t)).astype(np.float32)
    left.set(lh)
    p.set(ph)
    g0 = rng.standard_normal(hp.L).astype(np.float32)
    grad = env.dev(np.r_[g0, np.full(4, SENT, np.float32)])
    st = env.m.GrfPhi(hp.n_rows, hp.n_cols, row_lo, hp.L, d["blk_ptr"].data_ptr(), d["entries"].data_ptr(), None,
                      None, None, None, 0, 0, None, None, None, 0, hp.nnz, None)
    xd = None if x is None else env.dev(x)
    env.m.check(env.lib.grf_phi_fgrad(ctypes.byref(st), _vp(xd), n, left.ptr, left.ld, p.ptr, p.ld, t, _vp(grad),
                                      env.stream()))
    env.sync()
    got = grad.cpu().numpy()
    want, bound = R.ref_fgrad(hp, x, lh, ph, row_lo)
    _check_close(got[:hp.L], g0 + want, bound + R.UB * np.abs(g0), "grad (accumulated onto its prior contents)")
    assert np.array_equal(_bits(got[hp.L:]), _bits(np.full(4, SENT)))


# ---- grf_phi_row_dots ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("phi,mode", [("pl", "null"), ("pl", "pairs"), ("pl", "x1"), ("l32", "null"),
                                      ("l32", "pairs")])
def test_phi_row_dots(env, phi, mode):
    hp, d = env.phi(phi)
    rng = np.random.default_rng(len(mode) * 31 + hp.L)
    f = _f(rng, hp.L)
    row_lo = 0 if mode == "null" else 500
    must = [r for r in list(R.SPECIAL_ROWS) + [0, 1, 2, 3, 4, 5] if r < hp.n_rows]
    x1 = x2 = None
    n = hp.n_rows
    if mode == "pairs":
        x1 = _ids(rng, 900, row_lo, hp.n_rows, must=must)
        x2 = rng.permutation(x1).astype(np.int32)
        x2[:len(must)] = x1[:len(must)]        # long rows against themselves
        n = len(x1)
    elif mode == "x1":
        x1 = rng.permutation(np.arange(hp.n_rows) + row_lo - 100).astype(np.int32)
    dots = env.torch.full((n * hp.L + 4,), float("nan"), dtype=env.torch.float32, device="cuda")
    st = env.m.GrfPhi(hp.n_rows, hp.n_cols, row_lo, hp.L, d["blk_ptr"].data_ptr(), d["entries"].data_ptr(), None,
                      None, None, None, 0, 0, None, None, None, 0, hp.nnz, None)
    x1d = None if x1 is None else env.dev(x1)
    x2d = None if x2 is None else env.dev(x2)
    fd = env.dev(f)
    env.m.check(env.lib.grf_phi_row_dots(ctypes.byref(st), _vp(fd), _vp(x1d), _vp(x2d), n, _vp(dots), env.stream()))
    env.sync()
    raw = dots.cpu().numpy()
    got = raw[:n * hp.L].reshape(n, hp.L)
    want, bound, both = R.ref_row_dots(hp, f, x1, x2, n, row_lo)
    assert (~both).any() or mode == "null"
    assert np.all(_bits(got[~both]) == 0), "pairs outside the shard must be exactly +0"
    _check_close(got, want, bound, "row dots")
    assert np.all(np.isnan(raw[n * hp.L:]))


# ---- CG vector kernels --------------------------------------------------------------------------------------
CG_SHAPES = [(n, t) for n in (1, 7, 1000) for t in (1, 3, 4, 16, 17, 64, 256)] + [(2 ** 20 + 3, 4), (2 ** 20 + 3, 17)]


@pytest.mark.parametrize("off", [0, 1], ids=["aligned", "offset1"])
@pytest.mark.parametrize("n,t", CG_SHAPES)
def test_cg_vector_kernels(env, n, t, off):
    """grf_cg_dot, grf_cg_update and grf_cg_direction one by one against float64 (VEC=4 when t % 4 == 0 and the
    base pointers are 16-byte aligned, VEC=1 otherwise)."""
    torch, lib = env.torch, env.lib
    rng = np.random.default_rng(n * 1000 + t * 2 + off)
    P = lib.grf_cg_num_partials(n, t)
    eps = 1e-10

    def mat(a):
        buf = torch.full((n * t + off + 4,), float(SENT), dtype=torch.float32, device="cuda")
        buf[off:off + n * t] = torch.from_numpy(np.ascontiguousarray(a, np.float32).ravel()).cuda()
        return buf

    def get(buf):
        return buf[off:off + n * t].view(n, t).cpu().numpy()

    def vec(a, extra=4):
        return env.dev(np.r_[np.asarray(a, np.float32).ravel(), np.full(extra, SENT, np.float32)])

    def partial_buf():
        return torch.full(((P + 2) * t,), float("nan"), dtype=torch.float32, device="cuda")

    def totals(buf):
        raw = buf.cpu().numpy()
        assert np.all(np.isfinite(raw[:P * t])), "every partial row must be written"
        assert np.all(np.isnan(raw[P * t:])), "only grf_cg_num_partials rows may be written"
        return raw[:P * t].reshape(P, t).astype(np.float64).sum(axis=0)

    s = env.stream()
    d0 = rng.standard_normal((n, t)).astype(np.float32)
    kd = rng.standard_normal((n, t)).astype(np.float32)
    sigma2 = np.float32(0.37)

    # --- grf_cg_dot: ad = Kd + sigma2 d in place, partials of <d, ad> ---
    runs = []
    for _ in range(2):
        ad, d, part = mat(kd), mat(d0), partial_buf()
        env.m.check(lib.grf_cg_dot(_vp(ad, off), t, _vp(d, off), t, ctypes.c_float(sigma2), n, t, _vp(part), s))
        env.sync()
        runs.append((get(ad), part.cpu().numpy()))
    assert np.array_equal(_bits(runs[0][0]), _bits(runs[1][0])) and np.array_equal(_bits(runs[0][1]),
                                                                                     _bits(runs[1][1]))
    ad_got = runs[0][0]
    want = kd.astype(np.float64) + np.float64(sigma2) * d0
    _check_close(ad_got, want, 2.0 ** -23 * np.abs(want), "cg_dot ad")
    prod = d0.astype(np.float64) * ad_got
    _check_close(totals(part), prod.sum(0), R.UB * (n + 1) * np.abs(prod).sum(0), "cg_dot <d, ad>")

    # --- grf_cg_update: alpha = rs / <d, ad>; x += alpha d; r -= alpha ad; partials of <r, r> ---
    x0 = rng.standard_normal((n, t)).astype(np.float32)
    r0 = rng.standard_normal((n, t)).astype(np.float32)
    rs = rng.uniform(0.5, 2.0, t).astype(np.float32)
    dad = (rng.uniform(0.5, 1.5, (P, t)) / P).astype(np.float32)
    if t > 1:
        dad[:, 0] = 0.0                       # <d, Ad> = 0: alpha = 0, the column is left as it is
    runs = []
    for _ in range(2):
        x, r, d, ad, rr = mat(x0), mat(r0), mat(d0), mat(ad_got), partial_buf()
        rs_d, dad_d = vec(rs), env.dev(dad)
        env.m.check(lib.grf_cg_update(_vp(x, off), t, _vp(r, off), t, _vp(d, off), t, _vp(ad, off), t, _vp(rs_d),
                                      _vp(dad_d), n, t, ctypes.c_float(eps), _vp(rr), s))
        env.sync()
        runs.append((get(x), get(r), rr.cpu().numpy()))
        assert np.array_equal(_bits(rs_d.cpu().numpy()[:t]), _bits(rs))
    for a, b_ in zip(runs[0], runs[1]):
        assert np.array_equal(_bits(a), _bits(b_))
    x_got, r_got, _ = runs[0]
    tot = dad.astype(np.float64).sum(0)
    alpha = np.where(tot > eps, rs / np.where(tot > 0, tot, 1.0), 0.0)
    ad64 = ad_got.astype(np.float64)
    _check_close(x_got, x0 + alpha * d0, R.UB * (np.abs(x0) + (P + 2) * np.abs(alpha * d0)), "cg_update x")
    _check_close(r_got, r0 - alpha * ad64, R.UB * (np.abs(r0) + (P + 2) * np.abs(alpha * ad64)), "cg_update r")
    if t > 1:
        assert np.array_equal(_bits(x_got[:, 0]), _bits(x0[:, 0])) and np.array_equal(_bits(r_got[:, 0]),
                                                                                        _bits(r0[:, 0]))
    rr_host = r_got.astype(np.float64) ** 2
    _check_close(totals(rr), rr_host.sum(0), R.UB * (n + 1) * rr_host.sum(0), "cg_update <r, r>")

    # --- grf_cg_direction: rs_out = <r, r>; d = r + (rs_out / rs) d ---
    rs_old = rng.uniform(0.5, 2.0, t).astype(np.float32)
    if t > 1:
        rs_old[0] = 0.0                        # rs_old = 0: beta = 0, d = r
    rrp = (rng.uniform(0.5, 1.5, (P, t)) / P).astype(np.float32)
    runs = []
    for _ in range(2):
        d, r = mat(d0), mat(r0)
        rs_d, rrp_d, rs_out = vec(rs_old), env.dev(rrp), vec(np.full(t, np.nan))
        env.m.check(lib.grf_cg_direction(_vp(d, off), t, _vp(r, off), t, _vp(rs_d), _vp(rrp_d), n, t,
                                         ctypes.c_float(eps), _vp(rs_out), s))
        env.sync()
        runs.append((get(d), rs_out.cpu().numpy()))
        assert np.array_equal(_bits(rs_d.cpu().numpy()), _bits(np.r_[rs_old, np.full(4, SENT, np.float32)]))
    assert np.array_equal(_bits(runs[0][0]), _bits(runs[1][0])) and np.array_equal(_bits(runs[0][1]),
                                                                                     _bits(runs[1][1]))
    d_got, rs_out_got = runs[0]
    rs_new = rrp.astype(np.float64).sum(0)
    _check_close(rs_out_got[:t], rs_new, R.UB * P * rs_new, "cg_direction rs_out")
    assert np.array_equal(_bits(rs_out_got[t:]), _bits(np.full(4, SENT))), "rs_out holds t floats"
    beta = np.where(rs_old > eps, rs_new / np.where(rs_old > 0, rs_old, 1.0), 0.0)
    _check_close(d_got, r0 + beta * d0, R.UB * (np.abs(r0) + (P + 2) * np.abs(beta * d0)), "cg_direction d")
    if t > 1:
        assert np.array_equal(_bits(d_got[:, 0]), _bits(r0[:, 0]))


def test_cg_refuses_more_than_256_columns(env):
    lib, torch = env.lib, env.torch
    buf = torch.zeros(257 * 4, dtype=torch.float32, device="cuda")
    p, s = _vp(buf), env.stream()
    t = 257
    assert lib.grf_cg_dot(p, t, p, t, ctypes.c_float(0.0), 1, t, p, s) == env.m.GRF_ERR_INVALID
    assert lib.grf_cg_update(p, t, p, t, p, t, p, t, p, p, 1, t, ctypes.c_float(0.0), p, s) == env.m.GRF_ERR_INVALID
    assert lib.grf_cg_direction(p, t, p, t, p, p, 1, t, ctypes.c_float(0.0), _vp(buf, 4), s) == env.m.GRF_ERR_INVALID


# ---- Phi^T bit for bit --------------------------------------------------------------------------------------
def _transpose(env, hp, d, r0=0, r1=None, col_counts=False, census=False):
    torch, lib = env.torch, env.lib
    r1 = hp.n_rows if r1 is None else r1
    L, n_cols = hp.L, hp.n_cols
    hptr = hp.blk_ptr.astype(np.int64)
    entry_lo, nnz = int(hptr[r0 * L]), int(hptr[r1 * L] - hptr[r0 * L])
    blk = _vp(d["blk_ptr"], r0 * L)
    ws = torch.empty(lib.grf_transpose_workspace_bytes(n_cols, L, nnz), dtype=torch.uint8, device="cuda")
    tptr = torch.full((n_cols * L + 1,), -7, dtype=torch.int32, device="cuda")
    tent = torch.full((max(1, nnz) + 1, 2), -7, dtype=torch.int32, device="cuda")
    sub = R.HostPhi(r1 - r0, n_cols, L, *(a[(hp.row >= r0) & (hp.row < r1)] for a in (hp.row - r0, hp.length, hp.col,
                                                                                      hp.val)))
    cc = env.dev(sub.col_counts()) if col_counts else None
    ch = torch.full((6,), -1, dtype=torch.int32).pin_memory() if census else None
    s = env.stream()
    env.m.check(lib.grf_transpose_offsets(blk, _vp(d["entries"]), r1 - r0, n_cols, L, _vp(cc), _vp(tptr), _vp(ws),
                                          R.THRESHOLD, None if ch is None else ctypes.c_void_p(ch.data_ptr()), s))
    env.m.check(lib.grf_transpose_fill(blk, _vp(d["entries"]), r1 - r0, n_cols, L, entry_lo, nnz, _vp(ws),
                                       _vp(tent), s))
    env.sync()
    want_ptr, want_ent = sub.transpose()
    assert np.array_equal(tptr.cpu().numpy(), want_ptr)
    got = tent.cpu().numpy()
    assert np.array_equal(got[:nnz], want_ent)
    assert np.all(got[max(1, nnz):] == -7), "tentries written past nnz"
    if census:
        assert ch.tolist() == sub.census()


def _upload(env, hp):
    return dict(blk_ptr=env.dev(hp.blk_ptr), entries=env.dev(hp.entries if hp.nnz else np.zeros((1, 2), np.int32)))


@pytest.mark.parametrize("phi,rows,col_counts", [
    ("pl", None, False), ("pl", None, True), ("pl", (3001, 9000), False), ("pl", (3001, 9000), True),
    ("l32", None, False), ("l32", (1000, 2500), True), ("dense", None, False), ("band", None, True)])
def test_transpose_bit_exact(env, phi, rows, col_counts):
    hp, d = env.phi(phi)
    r0, r1 = rows or (0, hp.n_rows)
    _transpose(env, hp, d, r0, r1, col_counts=col_counts, census=True)


def test_transpose_bit_exact_many_tiles_per_cta(env):
    """2.4 M entries: more than 296 CTAs x 4096 items, so every CTA walks several tiles."""
    rng = np.random.default_rng(9)
    hp = R.synth_phi(10, 40000, 30000, 3, rng.integers(40, 80, 40000), hub=0)
    _transpose(env, hp, _upload(env, hp), census=True)


def _key_width_cases():
    """n_cols * L on both sides of every key width 1 .. 25 bits: 2^k and 2^k + 1 (passes of at most 10 bits:
    the pass count changes at 1024 | 1025 and 2^20 | 2^20 + 1, the digit split at every width)."""
    out = []
    for k in range(0, 25):
        for nk in (2 ** k, 2 ** k + 1):
            L = next(L for L in (32, 5, 4, 3, 1) if nk % L == 0)
            out.append((nk // L, L))
    return list(dict.fromkeys(out))


@pytest.mark.parametrize("n_cols,L", _key_width_cases())
def test_transpose_key_widths(env, n_cols, L):
    hp = R.random_phi(n_cols * 7 + L, 300, n_cols, L, 5000)
    _transpose(env, hp, _upload(env, hp), col_counts=n_cols % 2 == 1, census=True)
