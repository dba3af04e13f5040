"""Exact GP posterior variance on the GRF features (no reference counterpart: the reference's users estimate it
from ``predict`` samples, whose relative error is sqrt(2 / (s - 1)) for s samples).

For a whole Phi, a modulator f, training ids x (n of them, repeats allowed), noise sigma^2 > 0 and test ids x*:

    K = Phi_f[x] Phi_f[x]^T + sigma^2 I,   k_i = Phi_f[x] Phi_f[x*_i]^T,
    var_i = Phi_f[x*_i] . Phi_f[x*_i] - k_i^T K^-1 k_i          (+ sigma^2 with include_noise)

The n training rows touch only a set S of m columns (m <= nnz(Phi_f[x]), far below N in the BO setting), so:

    slot[c]   rank of column c in S (ascending), or -1 (int32 [N])
    G         m x n, G[slot[c], j] = Phi_f[x_j, c]       (float64; the merged Phi_f holds one entry per (row, col),
                                                           so plain assignment fills it deterministically)
    L         Cholesky factor of G^T G + sigma^2 I         (float64, cuBLAS / cuSOLVER through torch)
    C         G L^-T, m x n, stored as float32 with leading dimension ldc
    q_i       sum_c (sum_{e in row x*_i, slot >= 0} w_e C[slot(e), c])^2,  d_i = sum_e w_e^2
    var_i     max(d_i - q_i, 0)

q and d are one pass over the test rows of Phi_f (``grf_phi_row_quadform``, csrc/grf_posterior.cu); entries whose
column is not in S cost one 4-byte lookup.
"""

from __future__ import annotations

from typing import Dict, Optional

import torch

from .engine import PhiBlocks
from .kernel_matrix import _free_bytes


class ExactPosterior:
    """The training-side cache (slots, C) of the exact posterior variance, built once per (Phi, f, x, sigma^2).

    ``mem_limit``: bytes G, K, L and C may take instead of the free device memory; MemoryError (naming the bytes)
    is raised before they are allocated when they do not fit.  ``events``: CUDA events recorded at the stage
    boundaries ("start", "merge", "slots", "G", "gram", "cholesky", "solve"; ``variance`` adds "quadform_start"
    and "quadform")."""

    def __init__(self, blocks: PhiBlocks, f, x_train, noise, mem_limit: Optional[int] = None,
                 events: Optional[Dict[str, torch.cuda.Event]] = None):
        if blocks.is_shard:
            raise ValueError("ExactPosterior needs the whole Phi; a row shard holds only some of the training rows")
        noise = float(noise)
        if not noise > 0.0 or noise == float("inf"):
            raise ValueError(f"ExactPosterior: the noise variance must be positive and finite, got {noise}")
        dev = blocks.device
        self.blocks, self.noise, self.events, self.device = blocks, noise, events, dev
        x = PhiBlocks._ids(x_train, dev)
        blocks.check_ids(x)
        n = int(x.numel())
        self.n = n

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
            ct = torch.linalg.solve_triangular(chol, gt, upper=False)           # L^-1 G^T = C^T
            del gt, chol
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
