"""Drop-in for ``graph_kernels_sparse/fast_grf_kernel_general.py:20-55``.

Same signature and return type (scipy CSR kernel ``K = Phi Phi^T``); the
Laplacian, the walks and the per-length accumulation run on
the GPU, ``Phi = sum_p f_p M_p`` and the final sparse-sparse product stay in
scipy exactly as in the reference (:48-55) -- they are a one-off on this
small-graph API, not part of the CG loop.
"""

from typing import Sequence

import scipy.sparse as sp

from efficient_graph_gp_sparse.random_walk_samplers_sparse import SparseRandomWalk
from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian  # noqa: F401 (API)


def fast_general_grf_kernel(
    adj_matrix,
    modulator_vector: Sequence[float],
    walks_per_node: int = 50,
    p_halt: float = 0.1,
    max_walk_length: int = 10,
    *,
    trace=None,
    coupling: str = "iid",
):
    """Sparse GRF kernel estimate K ~ Phi Phi^T on the normalized Laplacian.  ``coupling``: how the walks of
    one start node share their draws (``grf_b200.engine.COUPLINGS``; "iid" = independent, as the reference)."""
    # the Laplacian (graph_utils.py:5-30) is formed on the device, bit-identical to the host one
    random_walk = SparseRandomWalk.on_normalized_laplacian(adj_matrix, seed=None)
    step_matrices = random_walk.get_random_walk_matrices(walks_per_node, p_halt, max_walk_length, trace=trace,
                                                           coupling=coupling)

    num_nodes = adj_matrix.shape[0]
    Phi = sp.csr_matrix((num_nodes, num_nodes))
    for step, f_p in enumerate(modulator_vector):
        if step < len(step_matrices):
            Phi += f_p * step_matrices[step]
    return Phi @ Phi.T
