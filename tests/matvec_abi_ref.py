"""Host-side Phi builder and float64 references for the matvec-layer C entry points.

``synth_phi`` makes the per-length matrices M_l (float32, canonical CSR: columns sorted and unique per row and
length) from a row-length profile and packs them into BOTH block layouts of include/grf_b200.h on the host:
Phi blocks (row-major over (row, length), ``length << 27 | column``) and Phi^T blocks (row-major over (column,
length), every segment sorted by row, ``length << 27 | local row``).  Tests of grf_phi_matvec therefore depend
neither on the walker nor on grf_transpose_*, and the transpose can be checked bit for bit against this one.

Error bound of the references.  With u = 2^-24, a float32 sum of n products (each rounded once) is within
(n + 1) u  sum |terms|  of the exact sum, whatever the summation order.  Two chained sums give, for
out = Phi_f[x1] (Phi_f[x2]^T V),

    |got - want|_ij <= 2^-22 * ( len(Phi[x1_i]) * A_ij + (|Phi_f[x1]| (n o (|Phi_f[x2]|^T |V|)))_ij ),
    A = |Phi_f[x1]| (|Phi_f[x2]|^T |V|)   (float64),

where |Phi_f| = sum_l |f_l| |M_l| (the magnitudes of the summands, not of their sum), len counts the stored
entries of a row over all lengths and n_c is the number of summands of column c of U (len(Phi^T_c), counting a
repeated x2 id once per repeat).  Since n_c <= max_c len(Phi^T_c), this is at most the classic
2^-22 (len(Phi[x1_i]) + max_c len(Phi^T_c)) A_ij: the summation bound with a factor-4 margin.  It holds for any
summation order, so the atomic paths are held to it too."""

from __future__ import annotations

import numpy as np
import scipy.sparse as sp

SHIFT = 27                       # GRF_ENTRY_STEP_SHIFT
COL_MASK = (1 << SHIFT) - 1
THRESHOLD = 256                  # long-row split threshold used by the tests (the engine's LONG_ROW_THRESHOLD)
UB = 2.0 ** -22                  # 4 u, u = 2^-24


def pack(length, col):
    """int32 words ``length << 27 | col`` (length 31 sets bit 31: the word is negative as an int32)."""
    return ((np.asarray(length, np.uint32) << np.uint32(SHIFT)) | np.asarray(col, np.uint32)).view(np.int32)


class HostPhi:
    """One row shard of Phi: entries (row, length, col, val) sorted by (row, length, col)."""

    def __init__(self, n_rows, n_cols, L, row, length, col, val):
        self.n_rows, self.n_cols, self.L = int(n_rows), int(n_cols), int(L)
        order = np.lexsort((col, length, row))
        self.row = np.asarray(row, np.int64)[order]
        self.length = np.asarray(length, np.int64)[order]
        self.col = np.asarray(col, np.int64)[order]
        self.val = np.asarray(val, np.float32)[order]
        self.nnz = self.row.size
        key = self.row * (self.L * self.n_cols) + self.length * self.n_cols + self.col
        assert np.all(np.diff(key) > 0), "(row, length, col) must be unique"

    # ---- Phi blocks ------------------------------------------------------------------------------------
    @property
    def blk_ptr(self):
        cnt = np.bincount(self.row * self.L + self.length, minlength=self.n_rows * self.L)
        return np.r_[0, np.cumsum(cnt)].astype(np.int32)

    @property
    def entries(self):
        e = np.empty((max(1, self.nnz), 2), np.int32)
        e[:self.nnz, 0] = pack(self.length, self.col)
        e[:self.nnz, 1] = self.val.view(np.int32)
        return e[:self.nnz] if self.nnz else e

    @property
    def row_len(self):
        return np.bincount(self.row, minlength=self.n_rows).astype(np.int64)

    # ---- Phi^T blocks, transposed here -----------------------------------------------------------------
    def transpose(self, r0=0, r1=None):
        """(tblk_ptr, tentries) of rows [r0, r1), local rows counted from r0."""
        r1 = self.n_rows if r1 is None else r1
        m = (self.row >= r0) & (self.row < r1)
        row, length, col, val = self.row[m] - r0, self.length[m], self.col[m], self.val[m]
        order = np.lexsort((row, length, col))
        cnt = np.bincount(col * self.L + length, minlength=self.n_cols * self.L)
        tptr = np.r_[0, np.cumsum(cnt)].astype(np.int32)
        tent = np.empty((row.size, 2), np.int32)
        tent[:, 0] = pack(length[order], row[order])
        tent[:, 1] = val[order].view(np.int32)
        return tptr, tent

    @property
    def col_len(self):
        return np.bincount(self.col, minlength=self.n_cols).astype(np.int64)

    def col_counts(self):
        return np.bincount(self.col * self.L + self.length, minlength=self.n_cols * self.L).astype(np.int32)

    def census(self, threshold=THRESHOLD):
        """grf_row_census of both sides: [long rows, chunks, non-empty rows] of Phi, then of Phi^T."""
        out = []
        for lens in (self.row_len, self.col_len):
            lng = lens[lens > threshold]
            out += [lng.size, int(((lng + threshold - 1) // threshold).sum()), int((lens > 0).sum())]
        return out

    # ---- float64 matrices -------------------------------------------------------------------------------
    def mat(self, l):
        m = self.length == l
        return sp.csr_matrix((self.val[m].astype(np.float64), (self.row[m], self.col[m])),
                             shape=(self.n_rows, self.n_cols))

    def phi_f(self, f32):
        """sum_l f_l M_l and sum_l |f_l| |M_l| in float64 (f and the values float32-rounded)."""
        w = np.asarray(f32, np.float32).astype(np.float64)[self.length]
        v = self.val.astype(np.float64)
        shape = (self.n_rows, self.n_cols)
        p = sp.coo_matrix((w * v, (self.row, self.col)), shape=shape).tocsr()
        pa = sp.coo_matrix((np.abs(w * v), (self.row, self.col)), shape=shape).tocsr()
        return p, pa

    def count_mat(self):
        return sp.csr_matrix((np.ones(self.nnz), (self.row, self.col)), shape=(self.n_rows, self.n_cols))


def _distinct(rng, lens, space, draw):
    """Per row r, lens[r] distinct keys in [0, space) drawn by draw(rows) -> keys; returns (rows, keys)."""
    lens = np.asarray(lens, np.int64)
    have = np.empty(0, np.int64)
    for _ in range(60):
        cnt = np.bincount(have // space, minlength=lens.size)
        short = np.flatnonzero(cnt < lens)
        if short.size == 0:
            break
        rows = np.repeat(short, 2 * (lens[short] - cnt[short]) + 2)
        have = np.unique(np.r_[have, rows * space + draw(rows)])
    else:
        raise AssertionError("row profile asks for more distinct keys than the draw can give")
    rows = have // space
    order = np.lexsort((rng.random(have.size), rows))      # random subset of exactly lens[r] per row
    have, rows = have[order], rows[order]
    start = np.r_[0, np.cumsum(np.bincount(rows, minlength=lens.size))][rows]
    keep = np.arange(have.size) - start < lens[rows]
    return rows[keep], have[keep] % space


def values(rng, n):
    """Both signs, magnitudes 2^-20 .. 2^4 (log-uniform), float32."""
    return (rng.choice([-1.0, 1.0], n) * 2.0 ** rng.uniform(-20, 4, n)).astype(np.float32)


def synth_phi(seed, n_rows, n_cols, L, lens, *, hub=None, hub_len=None, pool=None, draw=None, neg_zero=True):
    """Phi with row r holding exactly lens[r] entries.

    hub: a column that every row with lens[r] >= 1 and hub_len[r] (default 1) reaches -- at hub_len[r] distinct
    lengths, counted in lens[r] -- so that hub column holds up to sum(hub_len) entries.  pool: the columns the
    other entries draw from (default: all but the hub; columns outside it and the hub stay empty).  draw(rows,
    rng) -> columns overrides the uniform draw from the pool.  neg_zero: the hub entry at length 0 of the first
    row that has one becomes -0.0 (with hub = 0 that is the entry {length 0, column 0, -0.0})."""
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, np.int64).copy()
    hrow = np.empty(0, np.int64)
    hlen = np.empty(0, np.int64)
    if hub is not None:
        hk = np.minimum(lens, 1 if hub_len is None else np.asarray(hub_len, np.int64))
        hk = np.minimum(hk, L)
        hrow, hlen = _distinct(rng, hk, L, lambda rows: rng.integers(0, L, rows.size))
        lens = lens - hk
    if pool is None:
        pool = np.setdiff1d(np.arange(n_cols), [] if hub is None else [hub])
    if draw is None:
        def draw(rows, rng):
            return pool[rng.integers(0, pool.size, rows.size)]
    rows, keys = _distinct(rng, lens, L * n_cols,
                           lambda rows: rng.integers(0, L, rows.size) * n_cols + draw(rows, rng))
    row = np.r_[rows, hrow]
    length = np.r_[keys // n_cols, hlen]
    col = np.r_[keys % n_cols, np.full(hrow.size, -1 if hub is None else hub, np.int64)]
    val = values(rng, row.size)
    if hub is not None and neg_zero:
        z = np.flatnonzero((col == hub) & (length == 0) & (np.arange(row.size) >= rows.size))
        if z.size:
            val[z[np.argmin(row[z])]] = np.float32(-0.0)
    return HostPhi(n_rows, n_cols, L, row, length, col, val)


# ---- selections and references ------------------------------------------------------------------------
def selection(ids, row_lo, n_rows):
    """0/1 matrix [len(ids)][n_rows] picking local row ids[k] - row_lo (rows outside the shard: zero rows);
    None = identity."""
    if ids is None:
        return sp.identity(n_rows, format="csr")
    loc = np.asarray(ids, np.int64) - row_lo
    k = np.flatnonzero((loc >= 0) & (loc < n_rows))
    return sp.csr_matrix((np.ones(k.size), (k, loc[k])), shape=(len(ids), n_rows))


def in_shard(ids, row_lo, n_rows):
    loc = np.asarray(ids, np.int64) - row_lo
    return (loc >= 0) & (loc < n_rows)


def ref_first_half(hp, f32, x2, v, row_lo=0, u0=None):
    """U = Phi_f[x2]^T V (+ U0): value, |summands| and the number of summands per column."""
    p, pa = hp.phi_f(f32)
    s2 = selection(x2, row_lo, hp.n_rows)
    v = np.asarray(v, np.float64)
    u = (s2 @ p).T @ v
    ua = (s2 @ pa).T @ np.abs(v)
    n_c = np.asarray((s2 @ hp.count_mat()).sum(axis=0)).ravel()
    if u0 is not None:
        u = u + u0
        ua = ua + np.abs(u0)
        n_c = n_c + 1
    return u, ua, n_c


def ref_second_half(hp, f32, x1, u, ua, n_c, row_lo=0):
    """out = Phi_f[x1] U with its per-element bound (see the module docstring)."""
    p, pa = hp.phi_f(f32)
    s1 = selection(x1, row_lo, hp.n_rows)
    out = s1 @ (p @ u)
    a = s1 @ (pa @ ua)
    b = s1 @ (pa @ (n_c[:, None] * ua))
    len1 = s1 @ hp.row_len.astype(np.float64)
    return out, UB * (len1[:, None] * a + b)


def ref_matvec(hp, f32, x1, x2, v, row_lo=0, u0=None):
    u, ua, n_c = ref_first_half(hp, f32, x2, v, row_lo, u0)
    return ref_second_half(hp, f32, x1, u, ua, n_c, row_lo)


def ref_fgrad(hp, x, left, p, row_lo=0):
    """sum_k sum_c left[k, c] (M_l[x_k] P)[c] per length l, and the any-order bound per length:
    2^-22 (max_k len_l(x_k) + n t + 2) sum |summands|."""
    s = selection(x, row_lo, hp.n_rows)
    left, p = np.asarray(left, np.float64), np.asarray(p, np.float64)
    want, bound = np.zeros(hp.L), np.zeros(hp.L)
    n, t = left.shape
    for l in range(hp.L):
        m = s @ hp.mat(l)
        want[l] = np.sum(left * (m @ p))
        a = np.sum(np.abs(left) * (abs(m) @ np.abs(p)))
        max_len = np.diff(m.indptr).max() if m.shape[0] else 0
        bound[l] = UB * (max_len + n * t + 2) * a
    return want, bound


def ref_row_dots(hp, f32, x1, x2, n, row_lo=0):
    """dots[i][l] = sum over the length-l entries e of row x1[i] of e.val * Phi_f[x2[i], col(e)], with the bound
    2^-22 (L + 2) sum |e.val| |Phi_f|[x2[i], col(e)] (Phi_f[b, c] is an L-term float32 sum)."""
    ids1 = np.arange(n) + row_lo if x1 is None else np.asarray(x1)
    ids2 = np.arange(n) + row_lo if x2 is None else np.asarray(x2)
    both = in_shard(ids1, row_lo, hp.n_rows) & in_shard(ids2, row_lo, hp.n_rows)
    ids1 = np.where(both, ids1, -1)     # a pair outside the shard selects nothing on either side
    ids2 = np.where(both, ids2, -1)
    s1, s2 = selection(ids1, row_lo, hp.n_rows), selection(ids2, row_lo, hp.n_rows)
    p, pa = hp.phi_f(f32)
    pb, pab = s2 @ p, s2 @ pa
    want, bound = np.zeros((n, hp.L)), np.zeros((n, hp.L))
    for l in range(hp.L):
        m = s1 @ hp.mat(l)
        want[:, l] = np.asarray(m.multiply(pb).sum(axis=1)).ravel()
        bound[:, l] = UB * (hp.L + 2) * np.asarray(abs(m).multiply(pab).sum(axis=1)).ravel()
    return want, bound, both


# ---- the shared-memory-tiled kernel's plan (host copy of try_launch_tiled in csrc/grf_matvec.cu) ---------
SM_COUNT = 148
TILE_SMEM = 224 * 1024


def windows(ptr, ent, n_rows, L):
    """grf_block_windows on the host: {min col, max col} of every 32 consecutive rows, and the widest."""
    ptr = np.asarray(ptr, np.int64)
    cols = np.asarray(ent)[:, 0].view(np.uint32) & np.uint32(COL_MASK) if len(ent) else np.empty(0, np.uint32)
    n_groups = (n_rows + 31) // 32
    win = np.empty((n_groups, 2), np.int64)
    for g in range(n_groups):
        b, e = ptr[32 * g * L], ptr[min(n_rows, 32 * g + 32) * L]
        win[g] = (cols[b:e].min(), cols[b:e].max()) if e > b else (2 ** 31 - 1, -1)
    width = win[:, 1] - win[:, 0] + 1
    return win, int(max(0, width[win[:, 1] >= win[:, 0]].max(initial=0)))


def tiled_plan(win, max_width, n_rows, t):
    """None if try_launch_tiled declines, else one flag per chunk: True = its window fits in shared memory."""
    if max_width <= 0 or t % 4 or t > 128 or n_rows < 64:
        return None
    cap = TILE_SMEM // (t * 4)
    chunk = 0
    for k in range(1, 65):
        r = -(-n_rows // (SM_COUNT * k))
        r = -(-r // 32) * 32
        if r + max_width + 64 <= cap:
            chunk = r
            break
    if chunk < 64 or max_width > 6 * chunk:
        return None
    flags = []
    for r0 in range(0, n_rows, chunk):
        w = win[r0 // 32:(min(n_rows, r0 + chunk) - 1) // 32 + 1]
        w = w[w[:, 1] >= w[:, 0]]
        width = (w[:, 1].max() - w[:, 0].min() + 1) if len(w) else 0
        flags.append(bool(0 < width <= cap))
    return flags


# ---- the synthetic Phi of the tests ---------------------------------------------------------------------
SPECIAL_ROWS = np.arange(10, 18)                                      # rows with fixed lengths (see profile)
BAND_SHIFTED = ((3200, -400), (3328, 400), (12800, -400), (12928, 400))   # (first row of 32, column shift)


def profile(name):
    """The Phi shards of the matvec tests.

    pl     L = 3, 12000 x 5000, rows of 2..39 entries (avg ~21: the one-row-per-lane-group kernels even at
           t <= 4), 5 % empty rows, 5 % rows of one entry, rows of exactly 255, 256 (= threshold), 257, 512,
           513, 769, 1100 and 2000 entries, 400 empty columns and hub column 0 with ~11400 entries (one per
           non-empty row), holding {length 0, column 0, -0.0}
    dense  L = 3, 1500 x 2000, rows of 60..139 entries (avg > 64: the CSR-vector kernels at t <= 4), rows of 300
           and 700 entries, a few empty rows, hub column 0 (1500 entries)
    l32    L = 32, 3000 x 2500, rows of 0..59 entries at all 32 lengths, rows of 257 and 600 entries, hub column
           0 reached at 2 lengths per row (~5900 entries)
    band   L = 3, 20000 x 20000, columns within +-8 of the row; four groups of 32 rows shifted by +-400 columns, so
           that two chunks of 160 rows of the tiled kernel at t = 64 do not fit in shared memory
    empty  L = 3, 64 x 100 without entries
    noshard  L = 3, 0 x 100 (a GPU without rows)"""
    if name == "pl":
        rng = np.random.default_rng(101)
        n, m = 12000, 5000
        lens = rng.integers(2, 40, n)
        lens[rng.random(n) < 0.05] = 0
        lens[rng.random(n) < 0.05] = 1
        lens[SPECIAL_ROWS] = [255, 256, 257, 512, 513, 769, 1100, 2000]
        pool = np.setdiff1d(np.arange(1, m), rng.choice(np.arange(1, m), 400, replace=False))
        return synth_phi(102, n, m, 3, lens, hub=0, pool=pool)
    if name == "dense":
        rng = np.random.default_rng(201)
        n, m = 1500, 2000
        lens = rng.integers(60, 140, n)
        lens[[3, 4, 5]] = 0
        lens[SPECIAL_ROWS[:2]] = [300, 700]
        pool = np.setdiff1d(np.arange(1, m), rng.choice(np.arange(1, m), 100, replace=False))
        return synth_phi(202, n, m, 3, lens, hub=0, pool=pool)
    if name == "l32":
        rng = np.random.default_rng(301)
        n, m = 3000, 2500
        lens = rng.integers(0, 60, n)
        lens[SPECIAL_ROWS[:2]] = [257, 600]
        pool = np.setdiff1d(np.arange(1, m), rng.choice(np.arange(1, m), 50, replace=False))
        return synth_phi(302, n, m, 32, lens, hub=0, hub_len=np.full(n, 2), pool=pool)
    if name == "band":
        rng = np.random.default_rng(401)
        n = 20000
        shift = np.zeros(n, np.int64)
        for r0, s in BAND_SHIFTED:
            shift[r0:r0 + 32] = s

        def draw(rows, rng):
            return np.clip(rows + shift[rows] + rng.integers(-8, 9, rows.size), 0, n - 1)

        return synth_phi(402, n, n, 3, rng.integers(4, 20, n), draw=draw)
    if name == "empty":
        return synth_phi(501, 64, 100, 3, np.zeros(64, np.int64))
    if name == "noshard":
        return synth_phi(601, 0, 100, 3, np.zeros(0, np.int64))
    raise KeyError(name)


def random_phi(seed, n_rows, n_cols, L, nnz):
    """~nnz uniformly spread (row, length, col) entries plus the first and the last key of the (column,
    length) key space -- for the transpose at a given key width."""
    rng = np.random.default_rng(seed)
    key = rng.integers(0, n_rows * L * n_cols, nnz)
    key = np.unique(np.r_[key, 0, n_rows * L * n_cols - 1])
    row, rest = key // (L * n_cols), key % (L * n_cols)
    return HostPhi(n_rows, n_cols, L, row, rest // n_cols, rest % n_cols, values(rng, key.size))
