"""Exact GP posterior on the GRF features from one float64 factor: variance, mean, joint covariance and pathwise
samples (no reference counterpart for the first three: the reference's users estimate them from ``predict``
samples, whose relative error is sqrt(2 / (s - 1)) for s samples, and ``predict`` itself solves by CG).

For a whole Phi, a modulator f, training ids x (n of them, repeats allowed), noise sigma^2 > 0 and test ids x*:

    K = Phi_f[x] Phi_f[x]^T + sigma^2 I,   k_i = Phi_f[x] Phi_f[x*_i]^T,
    var_i = Phi_f[x*_i] . Phi_f[x*_i] - k_i^T K^-1 k_i          (+ sigma^2 with include_noise)

The n training rows touch only a set S of m columns (m <= nnz(Phi_f[x]), far below N in the BO setting), so:

    slot[c]   rank of column c in S (ascending), or -1 (int32 [N])
    G         m x n, G[slot[c], j] = Phi_f[x_j, c]       (float64; the merged Phi_f holds one entry per (row, col),
                                                           so plain assignment fills it deterministically)
    L         Cholesky factor of G^T G + sigma^2 I         (float64, cuBLAS / cuSOLVER through torch; kept)
    C         G L^-T, m x n, stored as float32 with leading dimension ldc
    q_i       sum_c (sum_{e in row x*_i, slot >= 0} w_e C[slot(e), c])^2,  d_i = sum_e w_e^2
    var_i     max(d_i - q_i, 0)

q and d are one pass over the test rows of Phi_f (``grf_phi_row_quadform``, csrc/grf_posterior.cu); entries whose
column is not in S cost one 4-byte lookup.  With s_i = row x*_i of Phi_f restricted to S (indexed by slot), the rest
of the posterior is the projection S* B = [s_i . B[:, c]] for a dense B (``grf_phi_row_project``):

    mean        mu_i  = s_i . a,                          a = G K^-1 y       (float64, stored as float32 [m, 1])
    covariance  Sigma = K** - P P^T,                      P = S* C           (q x n; P P^T in float64)
    samples     f*    = Phi_f[x*] eps + S* B,             B = C (L^-1 V),    V = y 1^T - Phi_f[x] eps - sigma E

the samples being pathwise conditioning (``SparseGraphGP.predict``) with an exact solve: eps ~ N(0, I_N) and
E ~ N(0, I_n) per sample, L^-1 V a float64 triangular solve and B a float32 GEMM.

Between refits of f and sigma^2 a BO loop only appends observations: ``condition_on`` extends L and C by block
Cholesky (C keeps its old columns and gains b), and ``PosteriorMarginals`` keeps the mean and variance at a fixed
candidate set current with one pass over the candidate rows per update (``grf_phi_row_condition``: q grows by the
squares of the projections onto the new columns of C, the mean is the projection onto the new a).

``forget`` removes training rows (the positions B in the current training order, R the kept ones, j0 = min B):

    Z  = L^-1 E_B (n x b; its rows before j0 are zero),  Z^T Z = (K^-1)_BB = R_B^T R_B   (b x b Cholesky)
    U  = C Z R_B^-1 (m x b):  C C^T - U U^T = G_R K_RR^-1 G_R^T,  so at every candidate  q' = q - |S* U|^2
    L' = [[L[:j0, :j0], 0], [L[R2, :j0], chol(T T^T)]],  T = L[R2, j0:]  (R2: the kept rows after j0)
    C' = [C[:, :j0] | C[:, j0:] T^T L'_22^-T]              (the right factor has orthonormal columns)

(removing the trailing positions truncates L and C), a is recomputed from L' in float64, and the rows of C' of
columns that only removed rows touched are set to exactly zero: those columns keep their slots (m never shrinks; a
later append that touches one reuses it) and give candidates the contribution of a posterior built without them,
none.  ``set_targets`` replaces y and recomputes a; L and C stay.  ``PosteriorMarginals`` replays any mix of these
changes from the posterior's change log: the appended columns of C through ``grf_phi_row_condition``, U through
``grf_phi_row_downdate`` (q shrinks by the same squares), and the mean once, onto the current a.
"""

from __future__ import annotations

import weakref
from typing import Dict, Optional

import torch

from .engine import PhiBlocks
from .kernel_matrix import _free_bytes


def _condition_chunk(n: int, m: int) -> int:
    """Rows of C_old converted to float64 at a time by condition_on: 256 MiB of them."""
    return max(1, min(m, (1 << 28) // (8 * max(n, 1))))


def condition_bytes(n: int, b: int, m: int, nnz_old: int) -> int:
    """Device bytes ExactPosterior.condition_on allocates to append b rows to n rows (nnz_old entries of Phi_f)
    that touch m columns afterwards: the new C (float32, ldc = round_up(n + b, 4)) and L (float64), G_new^T (float64
    [b, m]), one float64 row chunk of C_old and its product, and the K_21 products (two float64 [entries, b]
    buffers over at most the nnz_old old entries)."""
    nb = n + b
    ldc = (nb + 3) // 4 * 4
    chunk = _condition_chunk(n, m)
    return 4 * m * ldc + 8 * nb * nb + 8 * b * m + 8 * chunk * (n + 2 * b) + 16 * nnz_old * b


def downdate_bytes(n: int, b: int, j0: int, m: int, nnz: int, logged: bool = True) -> int:
    """Device bytes ExactPosterior.forget allocates to remove b of n rows, the first at position j0, from a
    posterior whose C has m rows and whose training rows hold nnz entries of Phi_f: the new C (float32, ldc =
    round_up(n - b, 4)) and L (float64); T = L[R2, j0:], T T^T, L'_22 and the right factor M (float64); one float64 row
    chunk of C[:, j0:] and its product; the gather of the kept rows' entries (int64 row, column and index, float32
    value); and with ``logged`` (a PosteriorMarginals is alive) E_B, Z, Z^T Z, R_B, Z R_B^-1 and [M | Z R_B^-1]
    (float64) and U (float32 [m, b])."""
    nn, nt = n - b, n - j0
    n2 = nn - j0
    ldc = (nn + 3) // 4 * 4
    chunk = _condition_chunk(nt, m)
    need = 4 * m * ldc + 8 * nn * nn + 16 * n2 * nt + 16 * n2 * n2 + 8 * chunk * (nt + n2 + b) + 28 * nnz
    if logged:
        need += 24 * nt * b + 16 * b * b + 8 * nt * (n2 + b) + 4 * m * b
    return need


class ExactPosterior:
    """The training-side cache (slots, L, C and, with ``y_train``, a = G K^-1 y) of the exact posterior, built once
    per (Phi, f, x, sigma^2, y).

    ``mem_limit``: bytes G, K, L and C (and a covariance's P and K**) may take instead of the free device memory;
    MemoryError (naming the bytes) is raised before they are allocated when they do not fit.  ``events``: CUDA
    events recorded at the stage boundaries ("start", "merge", "slots", "G", "gram", "cholesky", "solve";
    ``variance`` adds "quadform_start" and "quadform"; every projection, of ``mean``, ``covariance`` and ``sample``,
    "project_start" and "project"; ``sample`` also "sample_start", "prior", "triangular" and "gemm";
    ``condition_on`` "condition_start", "cross", "factor", "append" and "weights"; ``forget`` "downdate_start",
    "downdate_factor", "downdate_columns" and "downdate_weights"; a PosteriorMarginals refresh "refresh_start" and
    "refresh")."""

    def __init__(self, blocks: PhiBlocks, f, x_train, noise, mem_limit: Optional[int] = None,
                 events: Optional[Dict[str, torch.cuda.Event]] = None, *, y_train=None):
        if blocks.is_shard:
            raise ValueError("ExactPosterior needs the whole Phi; a row shard holds only some of the training rows")
        noise = float(noise)
        if not noise > 0.0 or noise == float("inf"):
            raise ValueError(f"ExactPosterior: the noise variance must be positive and finite, got {noise}")
        dev = blocks.device
        self.blocks, self.noise, self.events, self.device = blocks, noise, events, dev
        self.mem_limit = mem_limit
        x = PhiBlocks._ids(x_train, dev)
        blocks.check_ids(x)
        n = int(x.numel())
        self.n, self.x, self.f = n, x, blocks._f(f)
        self.y = None
        if y_train is not None:
            self.y = torch.as_tensor(y_train, device=dev).detach().flatten().to(torch.float64)
            if self.y.numel() != n:
                raise ValueError(f"ExactPosterior: y_train has {self.y.numel()} values for {n} training ids")

        with torch.cuda.device(dev):
            self._mark("start")
            self.phi_f = blocks.merged(f)                 # Phi_f: one length, one entry per (row, col)
            self._mark("merge")
            j, cols, vals = self._gather(x)
            total = int(j.numel())
            self.nnz_train = total
            cols_s = torch.unique(cols)                  # S, ascending
            m = int(cols_s.numel())
            self.m = m
            self.slot = torch.full((blocks.n_cols,), -1, dtype=torch.int32, device=dev)
            self.slot[cols_s] = torch.arange(m, dtype=torch.int32, device=dev)
            self._mark("slots")

            self.ldc = (n + 3) // 4 * 4
            need = 16 * m * n + 16 * n * n + 4 * m * self.ldc   # G^T and L^-1 G^T (float64), K and L, C (float32)
            budget = _free_bytes(dev) if mem_limit is None else int(mem_limit)
            if need > budget:
                raise MemoryError(f"exact posterior: G, K, L and C of {n} training rows touching {m} columns need "
                                  f"{need} bytes, {budget} bytes of device memory are free")
            gt = torch.zeros((n, m), dtype=torch.float64, device=dev)           # G^T
            if total:
                gt[j, self.slot[cols].to(torch.int64)] = vals.to(torch.float64)
            del j, cols, vals
            self._mark("G")
            k = gt @ gt.T
            k.diagonal().add_(noise)
            self._mark("gram")
            chol, info = torch.linalg.cholesky_ex(k)
            del k
            self._mark("cholesky")
            if n and int(info.item()) > 0:
                raise ValueError(f"exact posterior: G^T G + sigma^2 I is not positive definite in float64 "
                                 f"(sigma^2 = {noise}, n = {n}, leading minor {int(info.item())})")
            self.a = None
            if self.y is not None:                                              # a = G K^-1 y
                alpha = torch.cholesky_solve(self.y[:, None], chol) if n else self.y[:, None]
                self.a = (gt.T @ alpha).to(torch.float32)
                del alpha
            ct = torch.linalg.solve_triangular(chol, gt, upper=False)           # L^-1 G^T = C^T
            del gt
            self.L = chol
            self.C = torch.zeros((m, self.ldc), dtype=torch.float32, device=dev)
            self.C[:, :n] = ct.T
            del ct
            self._mark("solve")
        self.version = 0
        # (version, "append" / "remove" / "targets", float32 block) of every change a live PosteriorMarginals has
        # not seen yet: the appended columns of C, or U of a removal (see PosteriorMarginals.refresh)
        self._log = []
        self._watchers = weakref.WeakSet()

    def _gather(self, x):
        """(row index j, column, value) of every entry of the rows x of the merged Phi_f, row by row in entry
        order: int64, int64 and float32 device tensors."""
        dev = self.device
        ptr = self.phi_f.blk_ptr.to(torch.int64)
        ent = self.phi_f.entries
        xl = x.to(torch.int64)
        start = ptr[xl]
        lens = ptr[xl + 1] - start
        total = int(lens.sum().item()) if xl.numel() else 0
        j = torch.repeat_interleave(torch.arange(xl.numel(), device=dev), lens, output_size=total)
        first = torch.cumsum(lens, 0) - lens
        idx = start[j] + torch.arange(total, device=dev) - first[j]
        cols = ent[idx, 0].to(torch.int64)           # length 0: the packed word is the column
        vals = ent[idx, 1].view(torch.float32)
        return j, cols, vals

    def _mark(self, name: str) -> None:
        if self.events is not None:
            self.events[name] = torch.cuda.Event(enable_timing=True)
            self.events[name].record(torch.cuda.current_stream(self.device))

    def variance(self, x_test, include_noise: bool = False) -> torch.Tensor:
        """Posterior variance at the test ids (float32 device tensor [len(x_test)]); ``include_noise`` adds sigma^2
        (the predictive variance of a noisy observation).  IndexError for ids outside Phi."""
        dev = self.device
        xt = PhiBlocks._ids(x_test, dev)
        self.blocks.check_ids(xt)
        with torch.cuda.device(dev):
            self._mark("quadform_start")
            q, d = self.phi_f.row_quadform(torch.ones(1, device=dev), xt, self.slot, self.C[:, :self.n])
            self._mark("quadform")
            var = torch.clamp_min(d - q, 0.0)
            if include_noise:
                var = var + torch.tensor(self.noise, dtype=torch.float32, device=dev)
        return var

    def _test_ids(self, x_test):
        xt = PhiBlocks._ids(x_test, self.device)
        self.blocks.check_ids(xt)
        return xt

    def _need_y(self, what: str) -> None:
        if self.y is None:
            raise ValueError(f"ExactPosterior.{what} needs the training targets: construct it with y_train=")

    def _project(self, xt, B) -> torch.Tensor:
        self._mark("project_start")
        out = self.phi_f.row_project(torch.ones(1, device=self.device), xt, self.slot, B)
        self._mark("project")
        return out

    def mean(self, x_test) -> torch.Tensor:
        """Posterior mean k(x*, X) (K(X, X) + sigma^2 I)^-1 y at the test ids (float32 device tensor
        [len(x_test)]): one projection of the rows of Phi_f onto a = G K^-1 y, no solve.  ValueError without
        ``y_train``; IndexError for ids outside Phi."""
        self._need_y("mean")
        xt = self._test_ids(x_test)
        with torch.cuda.device(self.device):
            return self._project(xt, self.a)[:, 0]

    def covariance(self, x_test, include_noise: bool = False) -> torch.Tensor:
        """Joint posterior covariance K** - K*x K^-1 Kx* between the test ids (float64 device tensor [q, q],
        exactly symmetric); ``include_noise`` adds sigma^2 I.  K** is ``row_dots`` over the q (q + 1) / 2 pairs of
        the merged Phi_f, K*x K^-1 Kx* = P P^T with P = S* C one projection.  MemoryError (naming the bytes) before
        P or K** is allocated when they do not fit; IndexError for ids outside Phi."""
        xt = self._test_ids(x_test)
        dev, n = self.device, self.n
        q = int(xt.numel())
        pairs = q * (q + 1) // 2
        # P (float32 and float64), Sigma and P P^T (float64), per pair: the index pair (int64 and int32), K** dots
        # (float32 and float64) and the difference
        need = 12 * q * n + 16 * q * q + 44 * pairs
        budget = _free_bytes(dev) if self.mem_limit is None else int(self.mem_limit)
        if need > budget:
            raise MemoryError(f"exact posterior covariance: P and K** of {q} test nodes and {n} training rows need "
                              f"{need} bytes, {budget} bytes of device memory are free")
        with torch.cuda.device(dev):
            cov = torch.zeros((q, q), dtype=torch.float64, device=dev)
            if q == 0:
                return cov
            iu = torch.triu_indices(q, q, device=dev)
            vals = self.phi_f.row_dots(torch.ones(1, device=dev), xt[iu[0]], xt[iu[1]])[:, 0].to(torch.float64)
            if n:
                p = self._project(xt, self.C[:, :n]).to(torch.float64)
                vals -= (p @ p.T)[iu[0], iu[1]]
                del p
            cov[iu[0], iu[1]] = vals
            cov[iu[1], iu[0]] = vals
            if include_noise:
                cov.diagonal().add_(self.noise)
        return cov

    def sample(self, x_test, n_samples: int, generator: Optional[torch.Generator] = None,
               include_noise: bool = False, eps=None, eps_noise=None) -> torch.Tensor:
        """Joint posterior samples at the test ids (float32 device tensor [n_samples, len(x_test)]) by pathwise
        conditioning with an exact solve: f* = Phi_f[x*] eps + S* C L^-1 (y - Phi_f[x] eps - sigma E).  ``eps``
        (float32 [n_samples, N]) and ``eps_noise`` (float32 [n_samples, n]) replace the standard normal draws of
        eps and E; otherwise they come from ``generator`` (a generator on Phi's device, or the default one).
        ``include_noise`` adds sigma times a standard normal draw per test node: samples of noisy observations.
        ValueError without ``y_train`` or for n_samples < 1; IndexError for ids outside Phi; MemoryError (naming the
        bytes) before the draws are allocated when they do not fit."""
        self._need_y("sample")
        s = int(n_samples)
        if s < 1:
            raise ValueError(f"ExactPosterior.sample: n_samples must be at least 1, got {n_samples}")
        xt = self._test_ids(x_test)
        dev, n, N = self.device, self.n, self.blocks.n_cols
        q = int(xt.numel())
        sigma = self.noise ** 0.5
        # eps and its transposed copy, E, the prior at x and x*, V and L^-1 V (float64 and float32), B, the projection,
        # the sum and its transpose, the noise draws
        need = 8 * s * N + 4 * s * n + 4 * s * (n + q) + 20 * s * n + 4 * s * self.m + 16 * s * q
        budget = _free_bytes(dev) if self.mem_limit is None else int(self.mem_limit)
        if need > budget:
            raise MemoryError(f"exact posterior samples: {s} samples at {q} test nodes over {N} nodes need {need} "
                              f"bytes, {budget} bytes of device memory are free")

        def draws(given, shape, what):
            if given is None:
                return torch.randn(shape, generator=generator, device=dev)
            t = torch.as_tensor(given, device=dev).detach().to(torch.float32)
            if tuple(t.shape) != shape:
                raise ValueError(f"ExactPosterior.sample: {what} must have shape {shape}, got {tuple(t.shape)}")
            return t

        with torch.cuda.device(dev):
            eps = draws(eps, (s, N), "eps")
            eps_noise = draws(eps_noise, (s, n), "eps_noise")
            if q == 0:
                return torch.zeros((s, 0), dtype=torch.float32, device=dev)
            self._mark("sample_start")
            prior = self.blocks.apply(self.f, eps.T, rows=torch.cat([self.x, xt]))       # [n + q, s]
            self._mark("prior")
            fs = prior[n:]
            if n:
                v = self.y[:, None] - prior[:n].to(torch.float64) - sigma * eps_noise.T.to(torch.float64)
                z = torch.linalg.solve_triangular(self.L, v, upper=False).to(torch.float32)   # L^-1 V
                del v
                self._mark("triangular")
                b = self.C[:, :n] @ z                                                   # G K^-1 V, float32
                del z
                self._mark("gemm")
                fs = fs + self._project(xt, b)
            if include_noise:
                fs = fs + sigma * torch.randn((q, s), generator=generator, device=dev)
        return fs.T.contiguous()

    def condition_on(self, x_new, y_new=None) -> "ExactPosterior":
        """Append b training rows in place (f and sigma^2 stay): afterwards every method answers as a posterior
        constructed on x + x_new (and y + y_new) does, within float32 round-off.  Returns self.

        With K_21 = G_new^T G and K_22 = G_new^T G_new (float64 sums of the exact products of the gathered entries):
            L_21 = (L_11^-1 K_21^T)^T,   L_22 = chol(K_22 + sigma^2 I - L_21 L_21^T),
            C    = [C_old | C_new],      C_new = (G_new - C_old L_21^T) L_22^-T     (float64 in row chunks, stored
                                                                                     as float32; ldc = round_up(n + b, 4))
        and, with y, a = G K^-1 y from the new factor (float64).  Columns of the new rows outside S get the slots
        m, m + 1, .. in ascending column order, so after a call the slots are no longer ascending over S (the
        kernels do not care).  C and L are reallocated at their new size.

        ``y_new`` is required exactly when the posterior has y (``y_new = mean(x_new)`` gives the "hallucinated"
        conditioning of batch UCB selection).  Ids may repeat or be in x already.  An empty x_new is a no-op; each
        call that adds rows increments ``version``.  IndexError for ids outside Phi; ValueError for a y_new of the
        wrong length, or when the extended K is not positive definite in float64 (the posterior is then left as it
        was); MemoryError (naming the bytes) before anything is allocated.  Events: "condition_start", "cross",
        "factor", "append" and "weights"."""
        dev, n = self.device, self.n
        xn = self._test_ids(x_new)
        b = int(xn.numel())
        yn = None
        if (y_new is None) != (self.y is None):
            raise ValueError("ExactPosterior.condition_on: y_new is required exactly when the posterior has "
                             "training targets")
        if y_new is not None:
            yn = torch.as_tensor(y_new, device=dev).detach().flatten().to(torch.float64)
            if yn.numel() != b:
                raise ValueError(f"ExactPosterior.condition_on: y_new has {yn.numel()} values for {b} new ids")
        if b == 0:
            return self
        nb = n + b
        with torch.cuda.device(dev):
            self._mark("condition_start")
            jn, cn, vn = self._gather(xn)
            cols_n = torch.unique(cn)
            fresh = cols_n[self.slot[cols_n] < 0]             # ascending
            m0, m1 = self.m, self.m + int(fresh.numel())
            ldc = (nb + 3) // 4 * 4
            chunk = _condition_chunk(n, m1)
            need = condition_bytes(n, b, m1, self.nnz_train)
            budget = _free_bytes(dev) if self.mem_limit is None else int(self.mem_limit)
            if need > budget:
                raise MemoryError(f"exact posterior condition_on: C and L of {nb} training rows touching {m1} "
                                  f"columns need {need} bytes, {budget} bytes of device memory are free")
            slot = self.slot.clone()
            slot[fresh] = torch.arange(m0, m1, dtype=torch.int32, device=dev)
            sn = slot[cn].to(torch.int64)
            gnt = torch.zeros((b, m1), dtype=torch.float64, device=dev)            # G_new^T
            gnt[jn, sn] = vn.to(torch.float64)
            k22 = gnt @ gnt.T
            k21 = torch.zeros((b, n), dtype=torch.float64, device=dev)
            if n:                       # K_21[:, j] = sum over the entries of old row j of val * G_new^T[:, slot]
                jo, co, vo = self._gather(self.x)
                so = slot[co].to(torch.int64)
                hit = torch.zeros(m1, dtype=torch.bool, device=dev)
                hit[sn] = True
                keep = hit[so]
                jo, so, vo = jo[keep], so[keep], vo[keep]
                prod = gnt[:, so].T * vo.to(torch.float64)[:, None]             # exact products, [entries, b]
                k21 = torch.segment_reduce(prod, "sum", lengths=torch.bincount(jo, minlength=n), axis=0).T
                del jo, co, vo, so, keep, hit, prod
            self._mark("cross")
            l21t = torch.linalg.solve_triangular(self.L, k21.T, upper=False) if n else k21.T   # L_21^T, [n, b]
            s22 = k22 - l21t.T @ l21t
            s22.diagonal().add_(self.noise)
            l22, info = torch.linalg.cholesky_ex(s22)
            if int(info.item()) > 0:
                raise ValueError(f"exact posterior: G^T G + sigma^2 I is not positive definite in float64 "
                                 f"(sigma^2 = {self.noise}, n = {nb}, leading minor {n + int(info.item())})")
            del k21, k22, s22
            self._mark("factor")
            C = torch.zeros((m1, ldc), dtype=torch.float32, device=dev)
            C[:m0, :n] = self.C[:, :n]
            for r0 in range(0, m1, chunk):                   # C_new = (G_new - C_old L_21^T) L_22^-T, by rows
                r1 = min(m1, r0 + chunk)
                t = gnt[:, r0:r1].T.contiguous()
                if n and r0 < m0:
                    t[:min(r1, m0) - r0] -= self.C[r0:min(r1, m0), :n].to(torch.float64) @ l21t
                C[r0:r1, n:nb] = torch.linalg.solve_triangular(l22.T, t, upper=True, left=False).to(torch.float32)
                del t
            L = torch.zeros((nb, nb), dtype=torch.float64, device=dev)
            L[:n, :n] = self.L
            L[n:, :n] = l21t.T
            L[n:, n:] = l22
            del l21t, l22
            self._mark("append")
            x_all = torch.cat([self.x, xn])
            a = None
            if yn is not None:
                y = torch.cat([self.y, yn])
                a = self._weights(x_all, y, L, slot, m1)
            # nothing above changed the posterior (a failed factor leaves it as it was); now it takes the new state
            self.slot, self.m, self.C, self.L, self.ldc = slot, m1, C, L, ldc
            self.x, self.n = x_all, nb
            self.nnz_train += int(jn.numel())
            if yn is not None:
                self.y, self.a = y, a
            self.version += 1
            self._record("append", C[:, n:nb])
            self._mark("weights")
        return self

    def _weights(self, x, y, L, slot, m: int) -> torch.Tensor:
        """a = G K^-1 y (float32 [m, 1]) from the factor L of K over the training ids x: float64 sums over the
        slot-sorted entries (slots no training row touches get exactly 0)."""
        n = int(x.numel())
        if n == 0:
            return torch.zeros((m, 1), dtype=torch.float32, device=self.device)
        alpha = torch.cholesky_solve(y[:, None], L)[:, 0]
        ja, ca, va = self._gather(x)
        sa = slot[ca].to(torch.int64)
        order = torch.argsort(sa * n + ja)
        contrib = (va.to(torch.float64) * alpha[ja])[order]
        a = torch.segment_reduce(contrib, "sum", lengths=torch.bincount(sa, minlength=m), axis=0)
        return a.to(torch.float32)[:, None]

    def _record(self, kind: str, block: Optional[torch.Tensor]) -> None:
        """Log a change (made as ``version``) for the live PosteriorMarginals; nothing is kept when there is none."""
        self._trim()
        if len(self._watchers):
            self._log.append((self.version, kind, None if block is None else block.clone()))

    def _trim(self) -> None:
        """Drop the log entries every live PosteriorMarginals has already seen."""
        seen = [w.version for w in self._watchers]
        oldest = min(seen) if seen else self.version
        self._log = [e for e in self._log if e[0] > oldest]

    def _positions(self, positions, what: str) -> torch.Tensor:
        """Positions into the current training order as an int64 host tensor (in the given order); IndexError
        outside [0, n), ValueError for a repeated position."""
        pos = torch.as_tensor(positions).detach().flatten()
        if pos.numel() and (pos.dtype.is_floating_point or pos.dtype.is_complex or pos.dtype == torch.bool):
            raise ValueError(f"ExactPosterior.{what}: positions must be integers, got {pos.dtype}")
        pos = pos.cpu().to(torch.int64)
        if pos.numel() and (int(pos.min()) < 0 or int(pos.max()) >= self.n):
            bad = pos[(pos < 0) | (pos >= self.n)][0]
            raise IndexError(f"ExactPosterior.{what}: position {int(bad)} is outside the {self.n} training rows")
        if torch.unique(pos).numel() != pos.numel():
            raise ValueError(f"ExactPosterior.{what}: positions repeat")
        return pos

    def forget(self, positions) -> "ExactPosterior":
        """Remove the training rows at ``positions`` (indices into the current training order; ids may repeat in x,
        so rows are named by position) in place: afterwards every method answers as a posterior constructed on the
        kept rows, in their order, does, within float32 round-off.  Returns self.

        With B the removed positions, R2 the kept positions after j0 = min B and T = L[R2, j0:]:
            L' = [[L[:j0, :j0], 0], [L[R2, :j0], chol(T T^T)]],   C' = [C[:, :j0] | C[:, j0:] T^T L'_22^-T]
        (the product in float64 row chunks, stored as float32; ldc = round_up(n - b, 4)), and, with y, a = G K^-1 y
        from L' (float64).  Rows of C' whose column no kept row touches are set to exactly zero; the slots stay.
        While a PosteriorMarginals is alive, the same chunks also form U = C Z R_B^-1 for its refresh (module
        docstring).  C and L are reallocated at their new size.

        An empty call is a no-op; removing every row leaves the prior (n = 0); each call that removes rows
        increments ``version``.  IndexError for a position outside [0, n); ValueError for a repeated position, or
        when chol(T T^T) fails in float64 (the posterior is then left as it was); MemoryError (naming the bytes)
        before anything is allocated.  Events: "downdate_start", "downdate_factor", "downdate_columns" and
        "downdate_weights"."""
        pos = torch.sort(self._positions(positions, "forget")).values
        b = int(pos.numel())
        if b == 0:
            return self
        dev, n, m = self.device, self.n, self.m
        j0 = int(pos[0])
        keep = torch.ones(n, dtype=torch.bool)
        keep[pos] = False
        kept = torch.nonzero(keep).flatten()
        nn, nt = n - b, n - j0
        n2 = nn - j0
        logged = len(self._watchers) > 0
        need = downdate_bytes(n, b, j0, m, self.nnz_train, logged)
        budget = _free_bytes(dev) if self.mem_limit is None else int(self.mem_limit)
        if need > budget:
            raise MemoryError(f"exact posterior forget: C and L of {nn} training rows touching {m} columns need "
                              f"{need} bytes, {budget} bytes of device memory are free")
        with torch.cuda.device(dev):
            self._mark("downdate_start")
            r2 = (kept[j0:] - j0).to(dev)                      # the kept rows after j0, in the trailing block
            L22 = self.L[j0:, j0:]
            T = L22[r2]                                        # [n2, nt]
            l22 = torch.zeros((0, 0), dtype=torch.float64, device=dev)
            if n2:
                l22, info = torch.linalg.cholesky_ex(T @ T.T)
                if int(info.item()) > 0:
                    raise ValueError(f"exact posterior forget: the trailing factor T T^T of the {n2} kept rows after "
                                     f"position {j0} is not positive definite in float64 (leading minor "
                                     f"{int(info.item())})")
            L = torch.zeros((nn, nn), dtype=torch.float64, device=dev)
            L[:j0, :j0] = self.L[:j0, :j0]
            L[j0:, :j0] = self.L[j0:, :j0][r2]
            L[j0:, j0:] = l22
            self._mark("downdate_factor")
            rhs = torch.linalg.solve_triangular(l22, T, upper=False).T if n2 else T.T    # M = T^T L'_22^-T
            del T
            if logged:                                         # Z R_B^-1, Z = L^-1 E_B (rows >= j0)
                eb = torch.zeros((nt, b), dtype=torch.float64, device=dev)
                eb[(pos - j0).to(dev), torch.arange(b, device=dev)] = 1.0
                z = torch.linalg.solve_triangular(L22, eb, upper=False)
                del eb
                rb, info = torch.linalg.cholesky_ex(z.T @ z)
                if int(info.item()) > 0:
                    raise ValueError(f"exact posterior forget: (K^-1)_BB of the {b} removed rows is not positive "
                                     f"definite in float64 (leading minor {int(info.item())})")
                w = torch.linalg.solve_triangular(rb.T, z, upper=True, left=False)
                rhs = torch.cat([rhs, w], 1)
                del z, rb, w
            ldc = (nn + 3) // 4 * 4
            C = torch.zeros((m, ldc), dtype=torch.float32, device=dev)
            C[:, :j0] = self.C[:, :j0]
            U = torch.empty((m, b), dtype=torch.float32, device=dev) if logged else None
            chunk = _condition_chunk(nt, m)
            for r0 in range(0, m, chunk):                     # C[:, j0:] [M | Z R_B^-1], by rows
                r1 = min(m, r0 + chunk)
                prod = self.C[r0:r1, j0:n].to(torch.float64) @ rhs
                C[r0:r1, j0:nn] = prod[:, :n2].to(torch.float32)
                if logged:
                    U[r0:r1] = prod[:, n2:].to(torch.float32)
                del prod
            del rhs
            x_kept = self.x[kept.to(dev)]
            jk, ck, _ = self._gather(x_kept)
            live = torch.zeros(m, dtype=torch.bool, device=dev)
            live[self.slot[ck].to(torch.int64)] = True
            C[~live] = 0.0                                     # columns only the removed rows touched
            nnz = int(jk.numel())
            del jk, ck, live
            self._mark("downdate_columns")
            y, a = None, None
            if self.y is not None:
                y = self.y[kept.to(dev)]
                a = self._weights(x_kept, y, L, self.slot, m)
            # nothing above changed the posterior; now it takes the new state
            self.C, self.L, self.ldc = C, L, ldc
            self.nnz_train = nnz
            self.x, self.n = x_kept, nn
            if y is not None:
                self.y, self.a = y, a
            self.version += 1
            self._record("remove", U)
            self._mark("downdate_weights")
        return self

    def set_targets(self, y, positions=None) -> "ExactPosterior":
        """Replace the training targets: all of them (``positions`` None; y has n values), or those at
        ``positions`` (indices into the current training order; y has one value per position).  a = G K^-1 y is
        recomputed from L in float64; L and C stay.  Each call that changes targets increments ``version``; an empty
        ``positions`` is a no-op.  With ``condition_on(x, mean(x))`` for a batch of hallucinated observations, this
        swaps in the real targets once they arrive.  Returns self.  ValueError on a posterior built without y, for
        a y of the wrong length or with non-finite values, or for a repeated position; IndexError for a position
        outside [0, n)."""
        self._need_y("set_targets")
        dev = self.device
        yv = torch.as_tensor(y, device=dev).detach().flatten().to(torch.float64)
        if positions is None:
            if yv.numel() != self.n:
                raise ValueError(f"ExactPosterior.set_targets: y has {yv.numel()} values for {self.n} training rows")
            pos = None
        else:
            pos = self._positions(positions, "set_targets")
            if yv.numel() != pos.numel():
                raise ValueError(f"ExactPosterior.set_targets: y has {yv.numel()} values for {pos.numel()} "
                                 "positions")
        if not bool(torch.isfinite(yv).all()):
            raise ValueError("ExactPosterior.set_targets: y must be finite")
        if pos is not None and pos.numel() == 0:
            return self
        with torch.cuda.device(dev):
            if pos is None:
                y_all = yv.clone()
            else:
                y_all = self.y.clone()
                y_all[pos.to(dev)] = yv
            self.a = self._weights(self.x, y_all, self.L, self.slot, self.m)
            self.y = y_all
            self.version += 1
            self._record("targets", None)
        return self

    def marginals(self, x_cand) -> "PosteriorMarginals":
        """The mean and variance at a fixed candidate set, kept current across ``condition_on``, ``forget`` and
        ``set_targets`` calls at the cost of one pass over the candidate rows per kind of change (see
        PosteriorMarginals).  IndexError for ids outside Phi."""
        return PosteriorMarginals(self, x_cand)


class PosteriorMarginals:
    """Mean and variance of an ExactPosterior at fixed candidate ids, brought up to date after the posterior gained
    or lost training rows, or changed targets, without redoing the pass over all n columns of C.

    It keeps d (float32) and q (float64) of var = max(d - q, 0).  ``refresh`` replays the posterior's change log
    since the last refresh, consecutive changes of one kind together: appends add the squares of the candidates'
    projections onto the appended columns of C to q, removals subtract those onto U (module docstring), and the mean
    is recomputed once from the current a.  For k columns of one kind, with_mean = 1 on the last of them:
      k + with_mean <= 64   one ``row_condition`` (appends) or ``row_downdate`` (removals) pass with B = [blocks | a]
                            (the blocks, and a in the last column, copied into an m x (k + with_mean) buffer)
      k + with_mean > 64    ``row_quadform`` on the blocks (q rounded to float32 once) plus one ``row_project`` onto a
    A history of appends alone is one block of the columns C gained, so it refreshes exactly as the posterior's
    columns would.  The posterior keeps the blocks only while a PosteriorMarginals that has not seen them is alive.
    ``mean`` and ``variance`` refresh when the posterior has changed since the last refresh."""

    def __init__(self, post: ExactPosterior, x_cand):
        self.post = post
        self.x = post._test_ids(x_cand)
        dev = post.device
        with torch.cuda.device(dev):
            q, self.d = post.phi_f.row_quadform(torch.ones(1, device=dev), self.x, post.slot, post.C[:, :post.n])
            self.q = q.to(torch.float64)
            self._var = torch.clamp_min(self.d - q, 0.0)      # = post.variance(x_cand)
            self._mean = post._project(self.x, post.a)[:, 0].contiguous() if post.y is not None else None
        self.version, self.n_seen = post.version, post.n
        post._watchers.add(self)

    @property
    def stale(self) -> bool:
        return self.version != self.post.version

    def refresh(self) -> "PosteriorMarginals":
        """Bring q, the variance and the mean up to date with the posterior (a no-op when it is current)."""
        post = self.post
        if not self.stale:
            return self
        dev, wm, m = post.device, post.y is not None, post.m
        runs = []                                     # [kind, [blocks]]: consecutive changes of one kind
        for v, kind, block in post._log:
            if v <= self.version or kind == "targets":
                continue
            if runs and runs[-1][0] == kind:
                runs[-1][1].append(block)
            else:
                runs.append([kind, [block]])
        if not runs:                                  # only the targets changed
            runs.append(["append", []])
        one = torch.ones(1, device=dev)
        with torch.cuda.device(dev):
            post._mark("refresh_start")
            for i, (kind, blocks) in enumerate(runs):
                mean_here = int(wm and i == len(runs) - 1)
                k = sum(int(blk.shape[1]) for blk in blocks)
                B = torch.empty((m, k + mean_here), dtype=torch.float32, device=dev)
                c = 0
                for blk in blocks:                    # blocks logged before C gained slots: zero in the new rows
                    B[:blk.shape[0], c:c + blk.shape[1]] = blk
                    B[blk.shape[0]:, c:c + blk.shape[1]] = 0.0
                    c += blk.shape[1]
                if k + mean_here <= 64:
                    if mean_here:
                        B[:, k] = post.a[:, 0]
                    update = post.phi_f.row_condition if kind == "append" else post.phi_f.row_downdate
                    update(one, self.x, post.slot, B, k, mean_here, self.q, self.d, self._var,
                           self._mean if mean_here else None)
                else:
                    dq, _ = post.phi_f.row_quadform(one, self.x, post.slot, B[:, :k])
                    if kind == "append":
                        self.q += dq.to(torch.float64)
                    else:
                        self.q -= dq.to(torch.float64)
                    self._var = torch.clamp_min((self.d.to(torch.float64) - self.q).to(torch.float32), 0.0)
                    if mean_here:
                        self._mean = post.phi_f.row_project(one, self.x, post.slot, post.a)[:, 0].contiguous()
                del B
            post._mark("refresh")
        self.version, self.n_seen = post.version, post.n
        post._trim()
        return self

    @property
    def mean(self) -> torch.Tensor:
        """Posterior mean at the candidates (float32 [len(x_cand)]); ValueError without training targets."""
        self.post._need_y("mean")
        return self.refresh()._mean.clone()

    def variance(self, include_noise: bool = False) -> torch.Tensor:
        """Posterior variance at the candidates (float32 [len(x_cand)]); ``include_noise`` adds sigma^2."""
        var = self.refresh()._var.clone()
        if include_noise:
            var = var + torch.tensor(self.post.noise, dtype=torch.float32, device=self.post.device)
        return var
