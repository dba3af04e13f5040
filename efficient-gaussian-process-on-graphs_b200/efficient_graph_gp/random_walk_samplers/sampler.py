"""Drop-in for the reference's dense sampler (``random_walk_samplers/sampler.py:63-203``).

``Graph`` and ``RandomWalk`` keep their signatures; ``get_random_walk_matrices``
still returns the dense ``(N, N, L)`` float64 tensor the GPflow kernels consume
(general_kernel_fast_grf.py:44-59), but the walks run in the grf_b200 CUDA
walker over a CSR view of the dense matrix (``np.flatnonzero(row)`` order ==
sorted CSR columns, sampler.py:22-24) instead of an O(N) row scan per step.

Load semantics (DESIGN.md, SURVEY.md 8c): the estimator is the cumulative one
(``load *= deg*w/(1-p)``, sampler.py:58) regardless of ``n_processes``.  The
reference's ``_sequential_walks`` (taken when ``n_processes == 1`` or the graph
is tiny) assigns instead of multiplying (sampler.py:183), which biases every
length >= 2; it is reproduced only on request (``sequential_semantics=True``)
so that it can be parity-tested.  ``ablation=True`` means ``load = w``
(sampler.py:180-181) on every path.
"""

from typing import Optional

import numpy as np
import scipy.sparse as sp

from grf_b200 import _lib
from grf_b200.engine import DeviceGraph, WalkConfig, build_step_matrices


class Graph:
    """Minimal dense graph wrapper exposing adjacency, degree, and edge weights."""

    def __init__(self, adjacency_matrix: Optional[np.ndarray] = None) -> None:
        if adjacency_matrix is not None:
            self.adjacency_matrix = adjacency_matrix
            self.num_nodes = adjacency_matrix.shape[0]
        else:
            self.adjacency_matrix = None
            self.num_nodes = 0

    def get_neighbors(self, node: int) -> np.ndarray:
        return np.flatnonzero(self.adjacency_matrix[node])

    def get_num_nodes(self) -> int:
        return self.num_nodes

    def get_edge_weight(self, node1: int, node2: int) -> float:
        return self.adjacency_matrix[node1, node2]

    def to_csr(self) -> sp.csr_matrix:
        a = sp.csr_matrix(np.asarray(self.adjacency_matrix, dtype=float))
        a.eliminate_zeros()
        a.sort_indices()
        return a


class RandomWalk:
    """Random-walk generator producing step-conditioned feature tensors (GPU)."""

    def __init__(self, graph: Graph, seed: Optional[int] = None, device=None) -> None:
        self.graph = graph
        self.rng = np.random.default_rng(seed)
        self.seed = seed or 42
        self._device = device

    def get_step_matrices_device(self, num_walks, p_halt, max_walk_length, ablation=False,
                                 sequential_semantics=False, trace=None, *, coupling="iid"):
        csr = self.graph.to_csr()
        dg = DeviceGraph(csr.indptr, csr.indices, csr.data, self.graph.get_num_nodes(), self._device)
        if ablation:
            load_mode = _lib.LOAD_ABLATION
        elif sequential_semantics:
            load_mode = _lib.LOAD_LAST_STEP
        else:
            load_mode = _lib.LOAD_CUMULATIVE
        cfg = WalkConfig(int(num_walks), float(p_halt), int(max_walk_length), seed=self.seed,
                         draw_mode=_lib.DRAW_PHILOX if trace is None else _lib.DRAW_REPLAY,
                         load_mode=load_mode, trace=trace, coupling=coupling)
        return build_step_matrices(dg, cfg, scale_mode=_lib.SCALE_DIV)  # value / num_walks, sampler.py:201

    def get_random_walk_matrices(
        self,
        num_walks: int,
        p_halt: float,
        max_walk_length: int,
        use_tqdm: bool = False,
        n_processes: Optional[int] = None,
        ablation: bool = False,
        *,
        sequential_semantics: bool = False,
        trace=None,
        coupling: str = "iid",
    ) -> np.ndarray:
        """(num_nodes, num_nodes, max_walk_length) float64; [i, j, l] estimates (A^l)[i, j].  ``coupling``:
        how the walks of one start node share their draws (``grf_b200.engine.COUPLINGS``; "iid" = independent)."""
        del use_tqdm, n_processes
        steps = self.get_step_matrices_device(num_walks, p_halt, max_walk_length, ablation,
                                              sequential_semantics, trace, coupling=coupling)
        return steps.to_dense_tensor()
