"""Drop-in for the reference's ``SparseRandomWalk`` (sparse_sampler.py:59-132),
running on a B200 through ``grf_b200``.

Same constructor and ``get_random_walk_matrices`` signature and return type
(a list of ``max_walk_length`` scipy CSR matrices, float64, sorted int32
columns, ``M_0 = I``).  Differences, all deliberate (DESIGN.md):

* the walks run in one CUDA kernel, not in a fork pool: ``n_processes`` is
  accepted and ignored (it never changed the estimator, only the PCG64
  streams), ``use_tqdm`` is accepted and ignored (in the reference it raises
  NameError, sparse_sampler.py:34);
* native draws are Philox4x32-10 keyed by ``seed or 42`` (same seed rule as
  sparse_sampler.py:65) with counter (start*W + walk, step), so the result does
  not depend on how start nodes are sharded;
* ``trace=(trace_u, trace_k)`` replays recorded draws of the reference's own
  PCG64 streams instead -- the output is then bit-identical to the reference;
* ``coupling=`` (keyword only, default ``"iid"``: the independent draws above)
  couples the walks of one start node for a lower-variance estimate:
  ``"antithetic"``, ``"repelling"`` or ``"antithetic+repelling"``
  (``grf_b200.engine.COUPLINGS``; native draws only);
* ``neighbour_sampling=`` (keyword only, default ``"uniform"``: the reference's
  rule) with ``"weighted"`` picks neighbour k with probability |w_k| / sum |w|
  and multiplies the load by sign(w_k) * sum |w| / (1 - p_halt): still
  unbiased, and far less variance on graphs with hubs (native draws only, not
  with repelling neighbours).
"""

from typing import List, Optional

import scipy.sparse as sp

from grf_b200 import _lib
from grf_b200.engine import DeviceGraph, PhiBlocks, StepMatrices, WalkConfig, build_phi_blocks, build_step_matrices


class SparseRandomWalk:
    """Sparse random-walk generator on CSR adjacency matrices (GPU)."""

    def __init__(self, adjacency_matrix: sp.spmatrix, seed: Optional[int] = None, device=None) -> None:
        self.adjacency = adjacency_matrix.tocsr()
        self.num_nodes = self.adjacency.shape[0]
        self.seed = seed or 42
        self.indptr = self.adjacency.indptr
        self.indices = self.adjacency.indices
        self.data = self.adjacency.data.astype(float, copy=False)
        self._device = device
        self._graph = None

    @classmethod
    def on_normalized_laplacian(cls, adjacency_matrix: sp.spmatrix, seed: Optional[int] = None,
                                device=None) -> "SparseRandomWalk":
        """Walker on D^-1/2 (D - A) D^-1/2 of ``adjacency_matrix``, normalised on the device
        (same values and structure as ``get_normalized_laplacian``, graph_utils.py:5-30)."""
        self = cls.__new__(cls)
        self._graph = DeviceGraph.laplacian_of(adjacency_matrix, device)
        self.adjacency = None
        self.num_nodes = adjacency_matrix.shape[0]
        self.seed = seed or 42
        self.indptr = self.indices = self.data = None
        self._device = device
        return self

    @property
    def graph(self) -> DeviceGraph:
        if self._graph is None:
            self._graph = DeviceGraph(self.indptr, self.indices, self.data, self.num_nodes, self._device)
        return self._graph

    def _config(self, num_walks, p_halt, max_walk_length, trace, trace_start=0, coupling="iid",
                neighbour_sampling="uniform") -> WalkConfig:
        return WalkConfig(
            walks_per_node=int(num_walks), p_halt=float(p_halt), max_walk_length=int(max_walk_length),
            seed=self.seed, draw_mode=_lib.DRAW_PHILOX if trace is None else _lib.DRAW_REPLAY, trace=trace,
            trace_start=int(trace_start), coupling=coupling, neighbour_sampling=neighbour_sampling)

    def get_step_matrices_device(self, num_walks, p_halt, max_walk_length, start_lo=0, start_hi=None,
                                 trace=None, trace_start=0, *, coupling="iid",
                                 neighbour_sampling="uniform") -> StepMatrices:
        """The step matrices left in HBM (rows [start_lo, start_hi) only).  ``trace_start``: the first start
        node the replayed trace covers (a trace recorded for a row slice is indexed from there)."""
        cfg = self._config(num_walks, p_halt, max_walk_length, trace, trace_start, coupling, neighbour_sampling)
        return build_step_matrices(self.graph, cfg, start_lo, start_hi, scale_mode=_lib.SCALE_MUL_RECIP)

    def get_phi_blocks(self, num_walks, p_halt, max_walk_length, start_lo=0, start_hi=None, trace=None,
                       trace_start=0, *, coupling="iid", neighbour_sampling="uniform") -> PhiBlocks:
        """Phi in the matvec layout, built without leaving the device."""
        cfg = self._config(num_walks, p_halt, max_walk_length, trace, trace_start, coupling, neighbour_sampling)
        return build_phi_blocks(self.graph, cfg, start_lo, start_hi)

    def get_random_walk_matrices(
        self,
        num_walks: int,
        p_halt: float,
        max_walk_length: int,
        use_tqdm: bool = False,
        n_processes: Optional[int] = None,
        *,
        trace=None,
        coupling: str = "iid",
        neighbour_sampling: str = "uniform",
    ) -> List[sp.csr_matrix]:
        del use_tqdm, n_processes
        return self.get_step_matrices_device(num_walks, p_halt, max_walk_length, trace=trace,
                                             coupling=coupling, neighbour_sampling=neighbour_sampling).to_scipy()
