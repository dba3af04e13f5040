"""Drop-in for ``models/sparse_grf_model.py:10-45``: zero-mean exact GP with the sparse GRF
kernel and pathwise-conditioning ``predict`` (the CG solve runs on the fused CUDA matvec)."""

import torch

from grf_b200.cg import linear_cg
from grf_b200.gp_compat import HAVE_GPYTORCH, ExactGP, settings
from ..gptorch_kernels_sparse.sparse_grf_kernel import SparseGRFKernel

if HAVE_GPYTORCH:  # pragma: no cover
    import gpytorch


class SparseGraphGP(ExactGP):
    def __init__(self, x_train, y_train, likelihood, step_matrices, max_walk_length):
        super().__init__(x_train, y_train, likelihood)
        self.x_train, self.y_train = x_train, y_train
        self.covar_module = SparseGRFKernel(max_walk_length=max_walk_length, step_matrices_torch=step_matrices)
        if HAVE_GPYTORCH:  # pragma: no cover
            self.mean_module = gpytorch.means.ZeroMean()
        self.num_nodes = step_matrices[0].shape[0]

    def forward(self, x):
        covar = self.covar_module(x)
        if HAVE_GPYTORCH:  # pragma: no cover
            return gpytorch.distributions.MultivariateNormal(self.mean_module(x), covar)
        return torch.zeros(x.numel(), device=covar.device), covar

    def posterior_mean(self, x_test, cg_tolerance=1e-6, max_cg_iterations=1000, return_info=False):
        """K_test,train (K_train,train + sigma^2 I)^-1 y -- the noise-free limit of ``predict``
        (what its samples average to); used for the posterior-mean parity check."""
        train_indices = self.x_train.int().flatten()
        test_indices = x_test.int().flatten()
        dev = self.covar_module.phi_blocks.device
        phi = self.covar_module._get_feature_matrix()
        phi_train = phi[train_indices, :]
        K_train_train = phi_train @ phi_train.T
        K_test_train = phi[test_indices, :] @ phi_train.T
        noise_variance = float(self.likelihood.noise.item())
        with torch.no_grad():
            y = self.y_train.to(dev).to(torch.float32).reshape(-1, 1)
            alpha, info = K_train_train.solve(y, noise_variance, tolerance=cg_tolerance,
                                              max_iter=max_cg_iterations, eps=1e-30, return_info=True)
            out = K_test_train._matmul(alpha)[:, 0]
        return (out, info) if return_info else out

    def posterior_variance(self, x_test, include_noise=False):
        """Exact posterior variance k(x*, x*) - k(x*, X) (K(X, X) + sigma^2 I)^-1 k(X, x*) at every test node
        (float32 device tensor), with sigma^2 added when ``include_noise``.  No sampling: a float64 Cholesky factor
        on the columns the training rows touch, then one CUDA pass over the test rows (grf_b200/posterior.py)."""
        from grf_b200.posterior import ExactPosterior

        blocks = self.covar_module.phi_blocks
        f = self.covar_module.modulator_vector.detach()
        train_indices = self.x_train.long().flatten()
        test_indices = torch.as_tensor(x_test).long().flatten()
        post = ExactPosterior(blocks, f, train_indices, float(self.likelihood.noise.item()))
        return post.variance(test_indices, include_noise=include_noise)

    def posterior_covariance(self, x_test, include_noise=False):
        """Exact joint posterior covariance K** - K*X (K(X, X) + sigma^2 I)^-1 KX* between the test nodes (float64
        device tensor [q, q], exactly symmetric), with sigma^2 I added when ``include_noise``
        (grf_b200/posterior.py)."""
        from grf_b200.posterior import ExactPosterior

        blocks = self.covar_module.phi_blocks
        f = self.covar_module.modulator_vector.detach()
        train_indices = self.x_train.long().flatten()
        test_indices = torch.as_tensor(x_test).long().flatten()
        post = ExactPosterior(blocks, f, train_indices, float(self.likelihood.noise.item()))
        return post.covariance(test_indices, include_noise=include_noise)

    def exact_posterior(self):
        """The exact posterior (grf_b200.posterior.ExactPosterior) for the current modulator, noise, x_train and
        y_train: factor once per refit, then ``mean``, ``variance``, ``covariance`` and ``sample`` at any test
        nodes without a further solve."""
        from grf_b200.posterior import ExactPosterior

        blocks = self.covar_module.phi_blocks
        f = self.covar_module.modulator_vector.detach()
        return ExactPosterior(blocks, f, self.x_train.long().flatten(), float(self.likelihood.noise.item()),
                              y_train=self.y_train.flatten())

    def exact_mll(self):
        """The exact -mll/n and its closed-form gradients (grf_b200.mll.ExactMLL) for x_train and y_train: the
        per-length Gram of the training rows is built once, then ``loss(f, noise)`` / ``backward(kernel,
        likelihood)`` cost dense n x n float64 work per evaluation.  A drop-in for ``neg_mll_backward`` in a refit
        loop, deterministic, so L-BFGS can run on it."""
        from grf_b200.mll import ExactMLL

        return ExactMLL(self.covar_module.phi_blocks, self.x_train.long().flatten(), self.y_train.flatten())

    def predict(self, x_test, n_samples=64, cg_tolerance=None, max_cg_iterations=1000, return_info=False):
        """Posterior samples at ``x_test`` by pathwise conditioning (sparse_grf_model.py:21-45):
        f_test_prior + K_test,train (K_train,train + sigma^2 I)^-1 (y - f_train_prior - eps)."""
        train_indices = self.x_train.int().flatten()
        test_indices = x_test.int().flatten()
        dev = self.covar_module.phi_blocks.device

        phi = self.covar_module._get_feature_matrix()
        phi_train = phi[train_indices, :]
        phi_test = phi[test_indices, :]
        K_train_train = phi_train @ phi_train.T
        K_test_train = phi_test @ phi_train.T

        noise_variance = float(self.likelihood.noise.item())
        noise_std = noise_variance ** 0.5

        eps1_batch = torch.randn(n_samples, self.num_nodes, device=dev)
        eps2_batch = noise_std * torch.randn(n_samples, len(train_indices), device=dev)

        with torch.no_grad():
            f_test_prior = eps1_batch @ phi_test.T            # (n_samples, n_test)
            f_train_prior = eps1_batch @ phi_train.T          # (n_samples, n_train)
            b_batch = self.y_train.to(dev).unsqueeze(0) - (f_train_prior + eps2_batch)

            tol = settings.cg_tolerance.value() if cg_tolerance is None else cg_tolerance
            v_batch, info = K_train_train.solve(b_batch.T.contiguous(), noise_variance, tolerance=tol,
                                                max_iter=max_cg_iterations, return_info=True)
            out = f_test_prior + K_test_train._matmul(v_batch).T
        return (out, info) if return_info else out
