"""Drop-in for ``preprocessor/graph_preprocessor.py:10-165``.

Same constructor, attributes (``step_matrices_scipy``, ``step_matrices_torch``),
``preprocess_graph``, ``from_scipy_csr`` and pickle cache format.  Everything
between the adjacency and the operators stays on the GPU: the normalized
Laplacian (``grf_laplacian_*``, bit-identical to graph_utils.py:5-30), the walks,
the step matrices and the torch CSR tensors wrapped by the
``SparseLinearOperator``s (int64 indices, float32 values, as :117-139).
``step_matrices_scipy`` is copied to the host only when it is read (or saved);
``step_matrices_torch`` additionally carries the fused Phi blocks
(``.phi_blocks``) so that the kernels never rebuild them.
"""

import hashlib
import os
import pickle
from typing import List, Optional

import scipy.sparse as sp
import torch

from grf_b200 import _lib
from grf_b200.engine import DeviceGraph, PhiBlocks, WalkConfig, build_step_matrices
from efficient_graph_gp_sparse.utils_sparse import SparseLinearOperator


class StepOperatorList(list):
    """``list[SparseLinearOperator]`` that remembers the fused device layout."""

    phi_blocks: Optional[PhiBlocks] = None

    def to(self, device):
        out = StepOperatorList(op.to(device) for op in self)
        if self.phi_blocks is not None and self.phi_blocks.device == torch.device(device):
            out.phi_blocks = self.phi_blocks
        return out


class GraphPreprocessor:
    """Computes the GRF step matrices of a graph (random walks on its normalized Laplacian)."""

    def __init__(self, adjacency_matrix: sp.csr_matrix,
                 walks_per_node: int = 10,
                 p_halt: float = 0.5,
                 max_walk_length: int = 10,
                 random_walk_seed: int = 42,
                 load_from_disk: bool = False,
                 use_tqdm: bool = True,
                 cache_filename: Optional[str] = None,
                 n_processes: int = None,
                 device=None,
                 *,
                 coupling: str = "iid",
                 neighbour_sampling: str = "uniform") -> None:
        if adjacency_matrix.shape[0] != adjacency_matrix.shape[1]:
            raise ValueError("Adjacency matrix must be square.")

        self.adj_matrix = adjacency_matrix
        self.walks_per_node = walks_per_node
        self.p_halt = p_halt
        self.max_walk_length = max_walk_length
        self.random_walk_seed = random_walk_seed
        self.use_tqdm = use_tqdm
        self._cache_filename = cache_filename      # default name: hashed from the graph on first use (see below)
        self.n_processes = n_processes
        self.device = device
        self.coupling = coupling   # grf_b200.engine.COUPLINGS: how the walks of one start node share their draws
        self.neighbour_sampling = neighbour_sampling   # grf_b200.engine.NEIGHBOUR_SAMPLINGS: how a walk moves on
        self._scipy = None
        self._steps_device = None

        if load_from_disk:
            if os.path.exists(self.cache_filename):
                self.step_matrices_scipy = self.load_step_matrices(self.cache_filename)
                self.step_matrices_torch = self._wrap(self.step_matrices_scipy, None)
            else:
                raise FileNotFoundError(f"Cache file {self.cache_filename} not found.")

    @property
    def cache_filename(self) -> str:
        """Same default as the reference (an md5 over the adjacency arrays, graph_preprocessor.py:64,75-83), but
        computed when a cache file is first named rather than in the constructor: hashing the 2 GB of a
        70 M-edge adjacency takes 3 s on the host -- 50x the whole Phi build it would precede."""
        if self._cache_filename is None:
            self._cache_filename = self._generate_cache_filename()
        return self._cache_filename

    @cache_filename.setter
    def cache_filename(self, value) -> None:
        self._cache_filename = value

    def _generate_cache_filename(self) -> str:
        """Same key as the reference (graph_preprocessor.py:75-83), so caches are interchangeable; coupled
        draws append the coupling and weighted neighbour draws append "_weighted", so that such a cache never answers a
        request for the reference's draws."""
        adj_hash = hashlib.md5(self.adj_matrix.data.tobytes() +
                               self.adj_matrix.indices.tobytes() +
                               self.adj_matrix.indptr.tobytes()).hexdigest()[:8]
        graph_size = self.adj_matrix.shape[0]
        params = f"{graph_size}_{self.walks_per_node}_{self.p_halt}_{self.max_walk_length}_{self.random_walk_seed}"
        if self.coupling != "iid":
            params += f"_{self.coupling}"
        if self.neighbour_sampling != "uniform":
            params += f"_{self.neighbour_sampling}"
        return f"experiments_sparse/step_matrices/step_matrices_{adj_hash}_{params}.pkl"

    def _target_device(self) -> torch.device:
        if self.device is not None:
            return torch.device(self.device)
        return (torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available()
                else torch.device("cpu"))

    def _wrap(self, mats, blocks) -> StepOperatorList:
        dev = self._target_device()
        ops = StepOperatorList(SparseLinearOperator(self.from_scipy_csr(m).to(dev)) for m in mats)
        ops.phi_blocks = blocks
        return ops

    def _wrap_device(self, steps, blocks) -> StepOperatorList:
        """torch sparse-CSR tensors straight from the device step matrices (no host round trip)."""
        n, L = steps.n_rows, steps.n_steps
        bounds = steps.offsets[0:n * L + 1:max(1, n)][:L + 1].cpu().tolist() if n else [0] * (L + 1)
        ops = StepOperatorList()
        for s in range(L):
            b, e = bounds[s], bounds[s + 1]
            crow = (steps.offsets[s * n:(s + 1) * n + 1] - b) if n else torch.zeros(1, dtype=torch.int64,
                                                                                   device=steps.device)
            t = torch.sparse_csr_tensor(crow, steps.col[b:e].long(), steps.val[b:e].float(),
                                        (n, steps.n_cols), dtype=torch.float32)
            ops.append(SparseLinearOperator(t))
        ops.phi_blocks = blocks
        return ops

    @property
    def step_matrices_scipy(self) -> List[sp.csr_matrix]:
        if self._scipy is None and self._steps_device is not None:
            self._scipy = self._steps_device.to_scipy()
        return self._scipy

    @step_matrices_scipy.setter
    def step_matrices_scipy(self, mats) -> None:
        self._scipy = mats

    def preprocess_graph(self, save_to_disk: bool = False, *, trace=None) -> List[SparseLinearOperator]:
        graph = DeviceGraph.laplacian_of(self.adj_matrix, self.device)
        cfg = WalkConfig(int(self.walks_per_node), float(self.p_halt), int(self.max_walk_length),
                         seed=self.random_walk_seed or 42,
                         draw_mode=_lib.DRAW_PHILOX if trace is None else _lib.DRAW_REPLAY, trace=trace,
                         coupling=self.coupling, neighbour_sampling=self.neighbour_sampling)
        self._steps_device = build_step_matrices(graph, cfg, scale_mode=_lib.SCALE_MUL_RECIP)
        self._scipy = None
        if save_to_disk:
            self.save_step_matrices(self.step_matrices_scipy, self.cache_filename)
        self.step_matrices_torch = self._wrap_device(self._steps_device,
                                                     PhiBlocks.from_step_matrices(self._steps_device))
        return self.step_matrices_torch

    def preprocess_phi(self, start_lo: int = 0, start_hi: Optional[int] = None, *, trace=None,
                       group=None) -> PhiBlocks:
        """The pipeline of ``preprocess_graph`` kept in the matvec layout only: host adjacency -> device
        Laplacian -> walks -> Phi blocks (+ Phi^T) for the start nodes ``[start_lo, start_hi)`` -- what a
        row-sharded run (one process per GPU) or a graph whose float64 step matrices are not wanted
        calls.  No host copy, no torch CSR tensors; ``SparseGRFKernel`` accepts the result's operators.
        ``group`` (torch.distributed group or True): the ranks hold the same adjacency -- each uploads a slice of it
        and NCCL all-gathers the rest (``DeviceGraph.__init__``)."""
        from grf_b200.engine import build_phi_blocks

        graph = DeviceGraph.laplacian_of(self.adj_matrix, self.device, group=group)
        cfg = WalkConfig(int(self.walks_per_node), float(self.p_halt), int(self.max_walk_length),
                         seed=self.random_walk_seed or 42,
                         draw_mode=_lib.DRAW_PHILOX if trace is None else _lib.DRAW_REPLAY, trace=trace,
                         coupling=self.coupling, neighbour_sampling=self.neighbour_sampling)
        return build_phi_blocks(graph, cfg, start_lo, start_hi)

    @staticmethod
    def from_scipy_csr(scipy_csr: sp.csr_matrix) -> torch.Tensor:
        """scipy CSR -> torch sparse CSR (int64 indices, float32 values), as graph_preprocessor.py:117-139."""
        if not isinstance(scipy_csr, sp.csr_matrix):
            raise ValueError("Input must be a scipy CSR matrix.")
        crow_indices = torch.from_numpy(scipy_csr.indptr).long()
        col_indices = torch.from_numpy(scipy_csr.indices).long()
        values = torch.from_numpy(scipy_csr.data).float()
        return torch.sparse_csr_tensor(crow_indices, col_indices, values,
                                       (scipy_csr.shape[0], scipy_csr.shape[1]), dtype=torch.float32)

    @staticmethod
    def save_step_matrices(step_matrices: List[sp.csr_matrix], filename: str) -> None:
        d = os.path.dirname(filename)
        if d:
            os.makedirs(d, exist_ok=True)
        with open(filename, "wb") as f:
            pickle.dump(step_matrices, f)

    @staticmethod
    def load_step_matrices(filename: str) -> List[sp.csr_matrix]:
        """The reference's pickle (a plain list, graph_preprocessor.py:154-165) and the dict-keyed caches its
        experiments write: ``{'step_matrices_torch': [scipy CSR, ...], ...}``
        (experiments/sparse/scaling_exp/run_scaling_experiment.py:381-397 and
        experiments/sparse/scalable_bo/bo_utils/data_utils.py:311-343; despite the key the values are scipy
        matrices) or ``{'step_matrices': ...}`` for the dense method."""
        with open(filename, "rb") as f:
            payload = pickle.load(f)
        if isinstance(payload, dict):
            for key in ("step_matrices_torch", "step_matrices", "step_matrices_scipy"):
                if key in payload:
                    payload = payload[key]
                    break
            else:
                raise KeyError(f"{filename}: no step matrices in a cache with keys {sorted(payload)}")
        return payload

    @classmethod
    def load_step_operators(cls, filename: str, device=None) -> "StepOperatorList":
        """A cache file -> the operators ``SparseGRFKernel`` takes, on ``device``: what
        ``load_step_matrices_from_file`` (run_scaling_experiment.py:550-562) and ``convert_to_device``
        (data_utils.py:346-351) do with ``from_scipy_csr`` + ``SparseLinearOperator``."""
        mats = cls.load_step_matrices(filename)
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        ops = StepOperatorList(SparseLinearOperator(cls.from_scipy_csr(sp.csr_matrix(m)).to(device)) for m in mats)
        return ops
