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
"""

from __future__ import annotations

from typing import Dict, Optional

import torch

from .engine import PhiBlocks
from .kernel_matrix import _free_bytes


class ExactPosterior:
    """The training-side cache (slots, L, C and, with ``y_train``, a = G K^-1 y) of the exact posterior, built once
    per (Phi, f, x, sigma^2, y).

    ``mem_limit``: bytes G, K, L and C (and a covariance's P and K**) may take instead of the free device memory;
    MemoryError (naming the bytes) is raised before they are allocated when they do not fit.  ``events``: CUDA
    events recorded at the stage boundaries ("start", "merge", "slots", "G", "gram", "cholesky", "solve";
    ``variance`` adds "quadform_start" and "quadform"; every projection, of ``mean``, ``covariance`` and ``sample``,
    "project_start" and "project"; ``sample`` also "sample_start", "prior", "triangular" and "gemm")."""

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
            ptr = self.phi_f.blk_ptr.to(torch.int64)
            ent = self.phi_f.entries
            xl = x.to(torch.int64)
            start = ptr[xl]
            lens = ptr[xl + 1] - start
            total = int(lens.sum().item()) if n else 0
            self.nnz_train = total
            j = torch.repeat_interleave(torch.arange(n, device=dev), lens, output_size=total)
            first = torch.cumsum(lens, 0) - lens
            idx = start[j] + torch.arange(total, device=dev) - first[j]
            cols = ent[idx, 0].to(torch.int64)           # length 0: the packed word is the column
            vals = ent[idx, 1].view(torch.float32)
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
            del j, first, idx, cols, vals
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
