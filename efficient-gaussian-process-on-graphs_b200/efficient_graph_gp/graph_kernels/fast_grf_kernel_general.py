"""Drop-in for ``graph_kernels/fast_grf_kernel_general.py:11-39`` (dense API).

Same signature, returns the dense ``(N, N)`` float64 kernel ``Phi Phi^T``.
The walks run on the GPU; ``Phi = sum_l f_l M_l`` is assembled from the sparse
step matrices (the reference materialises an ``(N, N, L)`` tensor first, :38)
and the one dense contraction of this small-graph API, ``Phi @ Phi.T`` in
float64, is a plain library GEMM on the device.
"""

from typing import Sequence

import numpy as np
import torch

from efficient_graph_gp.random_walk_samplers import Graph, RandomWalk
from efficient_graph_gp.graph_kernels.utils import get_normalized_laplacian


def _phi_from_steps(steps, modulator_vector) -> torch.Tensor:
    """Dense float64 Phi on the device: sum_l f_l M_l, added in order of l like ``F @ f``."""
    n_rows, n_cols, L = steps.n_rows, steps.n_cols, steps.n_steps
    dev = steps.device
    phi = torch.zeros((n_rows, n_cols), dtype=torch.float64, device=dev)
    off = steps.offsets
    for l in range(L):
        ip = off[l * n_rows:(l + 1) * n_rows + 1]
        b, e = int(ip[0]), int(ip[-1])
        rows = torch.repeat_interleave(torch.arange(n_rows, device=dev), (ip[1:] - ip[:-1]))
        cols = steps.col[b:e].long()
        phi[rows, cols] += float(modulator_vector[l]) * steps.val[b:e]
    return phi


def fast_general_grf_kernel(
    adj_matrix: np.ndarray,
    modulator_vector: Sequence[float],
    walks_per_node: int = 50,
    p_halt: float = 0.1,
    max_walk_length: int = 10,
    *,
    trace=None,
    coupling: str = "iid",
) -> np.ndarray:
    """GRF kernel estimate K ~ Phi Phi^T using importance-sampled random walks.  ``coupling``: how the walks
    of one start node share their draws (``grf_b200.engine.COUPLINGS``; "iid" = independent, as the reference)."""
    modulator_vector = np.asarray(modulator_vector, dtype=float)
    if modulator_vector.shape[0] != max_walk_length:
        # the reference fails inside ``feature_matrices @ modulator`` with a shape error (:38)
        raise ValueError("The length of the modulator vector must be equal to the max_walk_length.")
    laplacian = get_normalized_laplacian(adj_matrix)
    random_walk = RandomWalk(Graph(laplacian), seed=42)
    steps = random_walk.get_step_matrices_device(walks_per_node, p_halt, max_walk_length, trace=trace,
                                                   coupling=coupling)
    phi = _phi_from_steps(steps, modulator_vector)
    return (phi @ phi.T).cpu().numpy()
