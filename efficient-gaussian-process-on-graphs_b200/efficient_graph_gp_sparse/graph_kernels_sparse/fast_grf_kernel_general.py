"""Drop-in for ``graph_kernels_sparse/fast_grf_kernel_general.py:20-55``.

Same signature and return type (scipy CSR kernel ``K = Phi Phi^T``).  The
Laplacian, the walks, the per-length accumulation, ``Phi = sum_p f_p M_p`` and
the sparse-sparse product ``Phi @ Phi.T`` all run on the GPU
(``StepMatrices.kernel_matrix``, csrc/grf_kernel_matrix.cu); only K itself is
copied to the host.  The result equals the reference's scipy result (:48-55)
in ``indptr``, ``indices`` and ``data``, dtypes included -- rows are in scipy's
(unsorted) order.
"""

from typing import Sequence

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
    neighbour_sampling: str = "uniform",
):
    """Sparse GRF kernel estimate K ~ Phi Phi^T on the normalized Laplacian, as a scipy csr_matrix.
    ``modulator_vector``: f_p for p < min(len, max_walk_length), real scalars that widen to float64.
    ``coupling``: how the walks of one start node share their draws (``grf_b200.engine.COUPLINGS``; "iid" =
    independent, as the reference).  ``neighbour_sampling``: "uniform" (as the reference) or "weighted" (neighbour k
    with probability |w_k| / sum |w|: bounded importance weights on the normalized Laplacian).  Raises MemoryError, naming nnz(K), when K does not fit on the device."""
    # the Laplacian (graph_utils.py:5-30) is formed on the device, bit-identical to the host one
    random_walk = SparseRandomWalk.on_normalized_laplacian(adj_matrix, seed=None)
    step_matrices = random_walk.get_step_matrices_device(walks_per_node, p_halt, max_walk_length, trace=trace,
                                                          coupling=coupling, neighbour_sampling=neighbour_sampling)
    return step_matrices.kernel_matrix(modulator_vector).to_scipy()
