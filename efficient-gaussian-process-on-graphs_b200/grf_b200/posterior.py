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
"""

from __future__ import annotations

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


class ExactPosterior:
    """The training-side cache (slots, L, C and, with ``y_train``, a = G K^-1 y) of the exact posterior, built once
    per (Phi, f, x, sigma^2, y).

    ``mem_limit``: bytes G, K, L and C (and a covariance's P and K**) may take instead of the free device memory;
    MemoryError (naming the bytes) is raised before they are allocated when they do not fit.  ``events``: CUDA
    events recorded at the stage boundaries ("start", "merge", "slots", "G", "gram", "cholesky", "solve";
    ``variance`` adds "quadform_start" and "quadform"; every projection, of ``mean``, ``covariance`` and ``sample``,
    "project_start" and "project"; ``sample`` also "sample_start", "prior", "triangular" and "gemm";
    ``condition_on`` "condition_start", "cross", "factor", "append" and "weights"; a PosteriorMarginals refresh
    "refresh_start" and "refresh")."""

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
            if yn is not None:                               # a = G K^-1 y, float64 sums over slot-sorted entries
                y = torch.cat([self.y, yn])
                alpha = torch.cholesky_solve(y[:, None], L)[:, 0]
                ja, ca, va = self._gather(x_all)
                sa = slot[ca].to(torch.int64)
                order = torch.argsort(sa * nb + ja)
                contrib = (va.to(torch.float64) * alpha[ja])[order]
                a = torch.segment_reduce(contrib, "sum", lengths=torch.bincount(sa, minlength=m1), axis=0)
                a = a.to(torch.float32)[:, None]
                del alpha, ja, ca, va, sa, order, contrib
            # nothing above changed the posterior (a failed factor leaves it as it was); now it takes the new state
            self.slot, self.m, self.C, self.L, self.ldc = slot, m1, C, L, ldc
            self.x, self.n = x_all, nb
            self.nnz_train += int(jn.numel())
            if yn is not None:
                self.y, self.a = y, a
            self.version += 1
            self._mark("weights")
        return self

    def marginals(self, x_cand) -> "PosteriorMarginals":
        """The mean and variance at a fixed candidate set, kept current across ``condition_on`` calls at the cost
        of one pass over the candidate rows per refresh (see PosteriorMarginals).  IndexError for ids outside Phi."""
        return PosteriorMarginals(self, x_cand)


class PosteriorMarginals:
    """Mean and variance of an ExactPosterior at fixed candidate ids, brought up to date after the posterior is
    conditioned on new rows without redoing the pass over all n columns of C.

    It keeps d (float32) and q (float64) of var = max(d - q, 0).  After ``condition_on`` appended k = n - n_seen
    columns to C, ``refresh`` adds the squares of the candidates' projections onto those columns to q and recomputes
    the mean from the new a:
      k + with_mean <= 64   one ``row_condition`` pass with B = [C[:, n_seen:n] | a] (a copied into the last
                            column of an m x (k + 1) buffer)
      k + with_mean > 64    ``row_quadform`` on C[:, n_seen:n] (q rounded to float32 once) plus one ``row_project``
                            onto a
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

    @property
    def stale(self) -> bool:
        return self.version != self.post.version

    def refresh(self) -> "PosteriorMarginals":
        """Bring q, the variance and the mean up to date with the posterior (a no-op when it is current)."""
        post = self.post
        if not self.stale:
            return self
        dev, n0, n = post.device, self.n_seen, post.n
        k, wm = n - n0, post.y is not None
        one = torch.ones(1, device=dev)
        with torch.cuda.device(dev):
            post._mark("refresh_start")
            if k + wm <= 64:
                B = torch.empty((post.m, k + wm), dtype=torch.float32, device=dev)
                B[:, :k] = post.C[:, n0:n]
                if wm:
                    B[:, k] = post.a[:, 0]
                post.phi_f.row_condition(one, self.x, post.slot, B, k, wm, self.q, self.d, self._var,
                                         self._mean if wm else None)
            else:
                dq, _ = post.phi_f.row_quadform(one, self.x, post.slot, post.C[:, n0:n])
                self.q += dq.to(torch.float64)
                self._var = torch.clamp_min((self.d.to(torch.float64) - self.q).to(torch.float32), 0.0)
                if wm:
                    self._mean = post.phi_f.row_project(one, self.x, post.slot, post.a)[:, 0].contiguous()
            post._mark("refresh")
        self.version, self.n_seen = post.version, n
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
