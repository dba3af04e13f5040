"""Exact-GP marginal log-likelihood gradients with CG + stochastic trace estimation.

This is what the reference gets from upstream GPyTorch when its training loops call
``loss = -mll(model(X), y); loss.backward()`` (run_scaling_experiment.py:603-612,
graph_bo/utils/bo_utils.py:244-251) with ``max_cholesky_size = 0`` and
``num_trace_samples`` probe vectors (SURVEY.md 3.3): one batched CG solve
``(K + s2 I)^-1 [y | z_1 .. z_p]`` and, per hyper-parameter,

    dL/dtheta = 1/2 a^T (dK/dtheta) a  -  1/2 * mean_j  w_j^T (dK/dtheta) z_j ,   a = Khat^-1 y, w_j = Khat^-1 z_j.

Here the solve is the fused CUDA CG on the Phi(Phi^T V) matvec and, for the modulator f
(K = Phi_f Phi_f^T, Phi_f = sum_l f_l M_l), the bilinear forms are the per-length reductions of
``grf_phi_fgrad``; the chain to the raw parameters (softplus constraints, the diffusion
formula) is left to autograd through ``modulator_vector`` / ``likelihood.noise``.
gpytorch is not installed in this image, so parity is against a float64 dense evaluation
(tests/test_gpu_gp.py), not against upstream.
"""

from __future__ import annotations

import math
from typing import Dict, Optional

import torch

from .engine import PhiBlocks, _free_bytes


def lanczos_logdet(matmul, probes: torch.Tensor, iterations: int = 1) -> float:
    """log|A| by stochastic Lanczos quadrature: mean_j ||z_j||^2 e_1^T log(T_j) e_1 with T_j the
    ``iterations`` x ``iterations`` Lanczos tridiagonal of A started at z_j / ||z_j||.

    The reference sets ``max_lanczos_quadrature_iterations = 1`` (run_scaling_experiment.py:133,
    graph_bo/utils/gpytorch_config.py:8), for which T_j is the Rayleigh quotient z^T A z / z^T z --
    one batched matvec.  More iterations run the three-term recurrence with full
    re-orthogonalisation (small k)."""
    z = probes.to(torch.float32)
    norms2 = (z * z).sum(dim=0)
    q = z / norms2.sqrt()
    qs = [q]
    alphas, betas = [], []
    beta_prev, q_prev = None, None
    for k in range(iterations):
        w = matmul(q)
        if q_prev is not None:
            w = w - beta_prev * q_prev
        alpha = (w * q).sum(dim=0)
        w = w - alpha * q
        for qq in qs:                                   # re-orthogonalise (k is small)
            w = w - (w * qq).sum(dim=0) * qq
        alphas.append(alpha)
        beta = w.norm(dim=0)
        if k + 1 < iterations:
            betas.append(beta)
            q_prev, beta_prev = q, beta
            q = w / beta.clamp_min(1e-20)
            qs.append(q)
    a = torch.stack(alphas, dim=1).double().cpu()                      # [p, k]
    p, k = a.shape
    T = torch.diag_embed(a)
    if k > 1:
        b = torch.stack(betas, dim=1).double().cpu()                   # [p, k-1]
        T = T + torch.diag_embed(b, offset=1) + torch.diag_embed(b, offset=-1)
    evals, evecs = torch.linalg.eigh(T)
    quad = (evecs[:, 0, :] ** 2 * torch.log(evals.clamp_min(1e-30))).sum(dim=1)   # e_1^T log(T) e_1
    return float((norms2.double().cpu() * quad).mean())


def neg_mll_backward(kernel, likelihood, x_train: torch.Tensor, y_train: torch.Tensor, num_probes: int = 16,
                     cg_tolerance: float = 1e-2, max_cg_iterations: int = 1000, probes: Optional[torch.Tensor] = None,
                     generator: Optional[torch.Generator] = None, cg_eps: float = 1e-10,
                     lanczos_iterations: int = 1):
    """Accumulate d(-mll/n)/dtheta into ``.grad`` of the kernel's and the likelihood's parameters.

    Returns a dict with the loss estimate (-mll/n, log-determinant by ``lanczos_iterations`` steps of
    stochastic Lanczos quadrature on the same probes; 0 skips it), the CG iteration count and the gradients.
    ``probes`` ([n, p]) overrides the Gaussian probe vectors (used by the exactness test)."""
    blocks = kernel.phi_blocks
    dev = blocks.device
    x = x_train.long().flatten().to(dev)
    y = y_train.to(dev).to(torch.float32).reshape(-1)
    n = y.numel()
    f = kernel.modulator_vector            # differentiable function of the raw parameters
    noise = likelihood.noise               # idem
    s2 = float(noise.detach())
    if probes is None:
        probes = torch.randn(n, num_probes, device=dev, generator=generator)
    probes = probes.to(dev).to(torch.float32)
    p = probes.shape[1]
    rhs = torch.cat([y[:, None], probes], dim=1).contiguous()

    K = kernel(x, x)
    sol, info = K.solve(rhs, s2, tolerance=cg_tolerance, max_iter=max_cg_iterations, eps=cg_eps, return_info=True)
    alpha, w = sol[:, :1].contiguous(), sol[:, 1:].contiguous()

    fd = f.detach()
    with torch.no_grad():
        # d/df_l of a^T K a and of sum_j w_j^T K z_j
        g_fit = blocks.fgrad(fd, alpha, alpha, x1=x, x2=x)
        g_tr = blocks.fgrad(fd, w, probes, x1=x, x2=x)
        dL_df = 0.5 * g_fit - 0.5 * g_tr / p
        dL_ds2 = 0.5 * float((alpha * alpha).sum()) - 0.5 * float((w * probes).sum()) / p
        datafit = 0.5 * float((y * alpha[:, 0]).sum())
        loss = None
        if lanczos_iterations > 0:
            plan = K.plan(p)
            logdet = lanczos_logdet(lambda v: plan(v.contiguous()) + s2 * v, probes, lanczos_iterations)
            loss = (datafit + 0.5 * logdet + 0.5 * n * 1.8378770664093453) / n
    # loss = -mll / n  (gpytorch's ExactMarginalLogLikelihood divides by the number of data points)
    f.backward((-dL_df / n).to(f.dtype).to(f.device), retain_graph=True)
    noise.backward(torch.as_tensor([-dL_ds2 / n], dtype=noise.dtype, device=noise.device).reshape(noise.shape))
    return {"loss": loss, "datafit": datafit, "cg_iterations": info["iterations"],
            "grad_modulator": (-dL_df / n).cpu(), "grad_noise": -dL_ds2 / n}


class _ExactLoss(torch.autograd.Function):
    """-mll/n as a function of (f, sigma^2); the backward is the closed form of ExactMLL._evaluate, not autograd
    through the Cholesky factor."""

    @staticmethod
    def forward(ctx, f, noise, mll):
        out = mll._evaluate(f.detach(), noise.detach())
        ctx.grads = [(g, t.shape, t.dtype, t.device) for g, t in ((out["grad_f"], f), (out["grad_noise"], noise))]
        return out["loss"]

    @staticmethod
    def backward(ctx, g):
        (gf, *f_meta), (gn, *n_meta) = ctx.grads

        def like(v, shape, dtype, device):
            return (g.to(v.device) * v).to(device=device, dtype=dtype).reshape(shape)

        return like(gf, *f_meta), like(gn, *n_meta), None


class ExactMLL:
    """Exact negative log-marginal likelihood -mll/n of the GRF GP and its closed-form gradients in the modulator f
    and the noise sigma^2, for fitting them on BO-sized training sets (hundreds to a few thousand nodes).

    The constructor builds the per-length Gram E = PhiBlocks.training_gram(x) once (float64 [L, n, L, n]; E does
    not depend on f or sigma^2).  Every evaluation is then dense float64 n x n work, with no pass over Phi:

        K = sum_{l, b} f_l f_b E[l, :, b, :] + sigma^2 I = L_K L_K^T,       alpha = K^-1 y,   W = alpha alpha^T - K^-1
        -mll/n = (1/2 y^T alpha + sum log diag L_K + n/2 log 2 pi) / n
        d mll / d f_l = sum_b f_b <W, E[l, :, b, :]>_F,                      d mll / d sigma^2 = (alpha^T alpha - tr K^-1) / 2

    ``loss(f, noise)`` is differentiable in both (``loss.backward()`` reaches the raw parameters behind them), and
    ``backward(kernel, likelihood)`` is the drop-in for ``neg_mll_backward``.  Evaluations are deterministic: the
    same (f, sigma^2) gives the same bits, so L-BFGS line searches and early stopping on the loss work.

    ``y_train`` is held in float64; ValueError for non-finite values, a length other than len(x_train), an empty
    training set or a row shard; IndexError for ids outside Phi.  ``mem_limit``: bytes E, the hub columns' dense H
    and the n x n work arrays may take instead of the free device memory (MemoryError, naming the bytes, before they
    are allocated).  ``events``: CUDA events at the stage boundaries ("start", then training_gram's "gather",
    "light", "heavy", "symmetrise"; every evaluation "eval_start", "kernel", "cholesky", "solve", "grad")."""

    def __init__(self, blocks: PhiBlocks, x_train, y_train, mem_limit: Optional[int] = None,
                 events: Optional[Dict[str, torch.cuda.Event]] = None):
        if blocks.is_shard:
            raise ValueError("ExactMLL needs the whole Phi; a row shard holds only some of the training rows")
        dev = blocks.device
        self.blocks, self.events, self.device = blocks, events, dev
        x = PhiBlocks._ids(x_train, dev)
        blocks.check_ids(x)
        n, L = int(x.numel()), blocks.n_steps
        if n == 0:
            raise ValueError("ExactMLL: the training set is empty")
        y = torch.as_tensor(y_train, device=dev).detach().flatten().to(torch.float64)
        if y.numel() != n:
            raise ValueError(f"ExactMLL: y_train has {y.numel()} values for {n} training ids")
        if not bool(torch.isfinite(y).all()):
            raise ValueError("ExactMLL: y_train holds non-finite values")
        self.n, self.L, self.x, self.y = n, L, x, y
        work = exact_mll_work_bytes(n, L)
        budget = _free_bytes(dev) if mem_limit is None else int(mem_limit)
        if work > budget:
            raise MemoryError(f"ExactMLL: the n x n work arrays of {n} training rows and {L} lengths need {work} "
                              f"bytes, {budget} bytes of device memory are free")
        with torch.cuda.device(dev):
            self._mark("start")
            self.E, self.gram_stats = blocks._training_gram(x, budget - work, events)
        self.last = None

    def _mark(self, name: str) -> None:
        if self.events is not None:
            self.events[name] = torch.cuda.Event(enable_timing=True)
            self.events[name].record(torch.cuda.current_stream(self.device))

    def _evaluate(self, f: torch.Tensor, noise: torch.Tensor) -> dict:
        n, L, dev = self.n, self.L, self.device
        fv = f.to(device=dev, dtype=torch.float64).flatten()
        if fv.numel() != L:
            raise ValueError(f"ExactMLL: the modulator has {fv.numel()} entries, Phi has {L} walk lengths")
        s2 = float(noise)
        if not s2 > 0.0 or s2 == float("inf"):
            raise ValueError(f"ExactMLL: the noise variance must be positive and finite, got {s2}")
        fh = fv.tolist()
        with torch.cuda.device(dev):
            self._mark("eval_start")
            eb = torch.zeros((L, n, n), dtype=torch.float64, device=dev)    # eb[l] = sum_b f_b E[l, :, b, :]
            for b in range(L):
                eb.add_(self.E[:, :, b, :], alpha=fh[b])
            k = torch.zeros((n, n), dtype=torch.float64, device=dev)
            for l in range(L):
                k.add_(eb[l], alpha=fh[l])
            k.diagonal().add_(s2)
            self._mark("kernel")
            chol, info = torch.linalg.cholesky_ex(k)
            del k
            self._mark("cholesky")
            if int(info.item()) > 0:
                raise ValueError(f"ExactMLL: K = sum f_l f_b E_lb + sigma^2 I is not positive definite in float64 "
                                 f"(sigma^2 = {s2}, n = {n}, leading minor {int(info.item())})")
            alpha = torch.cholesky_solve(self.y[:, None], chol)[:, 0]
            w = torch.cholesky_inverse(chol)
            self._mark("solve")
            tr_inv = w.diagonal().sum()
            w.neg_().add_(torch.outer(alpha, alpha))                         # W = alpha alpha^T - K^-1
            g_f = eb.reshape(L, n * n) @ w.reshape(n * n)                    # d mll / d f
            del w, eb
            g_s2 = 0.5 * (alpha @ alpha - tr_inv)
            datafit = 0.5 * (self.y @ alpha)
            logdet = 2.0 * torch.log(chol.diagonal()).sum()
            loss = (datafit + 0.5 * logdet + 0.5 * n * math.log(2.0 * math.pi)) / n
            self._mark("grad")
        self.last = {"loss": loss, "datafit": datafit, "logdet": logdet, "grad_f": -g_f / n, "grad_noise": -g_s2 / n}
        return self.last

    def loss(self, f, noise) -> torch.Tensor:
        """-mll/n at the modulator f (length L) and noise variance sigma^2 (> 0), a float64 scalar on Phi's device,
        differentiable in ``f`` and ``noise`` when they are tensors that require grad.  ValueError for a modulator
        of the wrong length, sigma^2 <= 0 or non-finite, or a K that is not positive definite in float64."""
        f = f if torch.is_tensor(f) else torch.as_tensor(f, dtype=torch.float64)
        noise = noise if torch.is_tensor(noise) else torch.as_tensor(noise, dtype=torch.float64)
        return _ExactLoss.apply(f, noise, self)

    def backward(self, kernel, likelihood) -> dict:
        """Accumulate d(-mll/n)/dtheta into ``.grad`` of the kernel's and the likelihood's parameters (through
        ``kernel.modulator_vector`` and ``likelihood.noise``), as ``neg_mll_backward`` does, exactly.  Returns its
        keys (``loss``, ``datafit``, ``cg_iterations`` = 0, ``grad_modulator``, ``grad_noise``) and ``logdet``."""
        loss = self.loss(kernel.modulator_vector, likelihood.noise)
        loss.backward()
        out = self.last
        return {"loss": loss.item(), "datafit": float(out["datafit"]), "cg_iterations": 0,
                "grad_modulator": out["grad_f"].cpu(), "grad_noise": float(out["grad_noise"]),
                "logdet": float(out["logdet"])}


def exact_mll_work_bytes(n: int, L: int) -> int:
    """Bytes of one ExactMLL evaluation's float64 work arrays: sum_b f_b E[:, :, b, :] (L n^2), K, its factor and
    K^-1 (or W) and alpha alpha^T (4 n^2)."""
    return 8 * n * n * (L + 4)
