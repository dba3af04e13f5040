"""Device pipeline of the GRF hot path: walker -> staging -> CSR / Phi blocks -> matvec.

Everything here is plumbing around the C ABI (``include/grf_b200.h``): torch
allocates the buffers and provides the stream, the CUDA library does the work.
No CPU fallback -- a missing library or a non-CUDA device raises.

Reference call stack this replaces (SURVEY.md 3.1-3.3):
  SparseRandomWalk.get_random_walk_matrices   sparse_sampler.py:72-132
  RandomWalk.get_random_walk_matrices         sampler.py:93-203
  GraphPreprocessor.from_scipy_csr            graph_preprocessor.py:117-139
  SparseLinearOperator._matmul / transpose    sparse_lo.py:16-25
  SparseGRFKernel.forward                     sparse_grf_kernel.py:24-62
"""

from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import GrfGraph, GrfLongRows, GrfPhi, GrfWalkCfg, check

LONG_ROW_THRESHOLD = 256   # rows of Phi / Phi^T with more entries are split into chunks of this size
# line-pair entries for the merged t = 16 product (csrc/grf_pairs.cu).  Opt-in: on config 2 the pair kernel halves
# the gather wavefronts (L1 data stage 77 % -> 46 % busy) but not the time -- 44 us per half against 26 us for the
# tuned 64-byte-row kernel, which it would have to beat by instruction count as well (profiles/README.md)
PAIR_LAYOUT = os.environ.get("GRF_PAIR_LAYOUT", "0") == "1"
PAIR_MAX_RATIO = 0.8       # ... when pairing leaves at most this share of the union entries
UNION_CHUNK = 1024         # rows with more entries are merged (union layout) chunk by chunk
# entries per chunk of a long COLUMN (<= LONG_ROW_THRESHOLD).  Smaller chunks span fewer rows of V but cost a
# partial-sum row each: config 4 Phi^T V 5.41 ms at 256, 5.49 at 128, 6.10 at 64
T_CHUNK = int(os.environ.get("GRF_T_CHUNK", str(LONG_ROW_THRESHOLD)))
CHUNK_ORDER = os.environ.get("GRF_CHUNK_ORDER", "1") != "0"   # issue the chunks by the first row they gather
_MAX_STAGE_BYTES = 16 << 30  # staging budget per walker launch; larger shards are walked in row chunks
_LAZY_ENTRY_BYTES = 1 << 30  # up to this bound the Phi entries are allocated by capacity (no host wait for the count)
# Rows per Phi^T block.  Transposing a shard in row blocks bounds the sort workspace (24 bytes per entry of a
# block) and lets a shard exceed 2^31 entries on the Phi^T side; it does NOT pay as cache blocking of V: with 2^19-row
# blocks the first half of the config-4 product went from 7.4 to 12.8 ms (every block re-reads the 21 M segment
# pointers and read-modify-writes all of U, and most columns hold ~1 entry per block).  Hence one block up to 2^22 rows.
T_BLOCK_ROWS = 1 << 22


def _device(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("grf_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError(f"grf_b200 needs a CUDA device, got {device}; there is no CPU fallback")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


_pending_host = []
_free_small_pinned = []


def _small_pinned() -> torch.Tensor:
    """64 bytes of pinned host memory for a count / census that the GPU copies back asynchronously.  Recycled
    (``_recycle_pinned``, by the reader once it has the value): cudaHostAlloc costs ~0.1 ms and serialises with
    the device, and every Phi build needs two or three."""
    if not _free_small_pinned:
        # one cudaHostAlloc (milliseconds, and it serialises with the device) serves 64 buffers: a caller that keeps
        # many Phi alive with their counts unread would otherwise pay it once per build
        slab = torch.empty(16 * 64, dtype=torch.int32, pin_memory=True)
        _free_small_pinned.extend(slab[i * 16:(i + 1) * 16] for i in range(64))
    return _free_small_pinned.pop()


def _recycle_pinned(buf: Optional[torch.Tensor]) -> None:
    if buf is not None and len(_free_small_pinned) < 256 and not any(b is buf for b in _free_small_pinned):
        _free_small_pinned.append(buf)


def _keep_until_done(buf: torch.Tensor, event: torch.cuda.Event) -> None:
    """The C library copies into ``buf`` (pinned) asynchronously, which torch's host allocator does
    not see: hold a reference until the copy's event has completed, whoever drops the owner first."""
    _pending_host[:] = [(b, e) for b, e in _pending_host if not e.query()]
    _pending_host.append((buf, event))


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream(device: torch.device):
    """cudaStream_t of torch's current stream on ``device`` (every C call is asynchronous on it)."""
    if _raw_stream is not None:
        return ctypes.c_void_p(_raw_stream(device.index))   # same handle, without building a Stream object
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


# WalkConfig.coupling -> GRF_DRAW_COUPLE_* bits (definitions at GrfWalkCfg.seed in include/grf_b200.h):
# "antithetic" pairs the halting draws of walks (2q, 2q+1), "repelling" spreads the walks of a start node that
# stand on the same node over its neighbours.  Every walk keeps its marginal law: M_l stays unbiased.
COUPLINGS = {
    "iid": 0,
    "antithetic": _lib.DRAW_COUPLE_HALT,
    "repelling": _lib.DRAW_COUPLE_NEIGHBOURS,
    "antithetic+repelling": _lib.DRAW_COUPLE_HALT | _lib.DRAW_COUPLE_NEIGHBOURS,
}


@dataclass
class WalkConfig:
    """Arguments of the reference's walk loop (sparse_sampler.py:26-31) + draw source."""

    walks_per_node: int
    p_halt: float
    max_walk_length: int
    seed: int = 42
    draw_mode: int = _lib.DRAW_PHILOX
    load_mode: int = _lib.LOAD_CUMULATIVE
    trace: Optional[Tuple] = None  # (trace_u float64, trace_k int32), [(walk_id - trace_start*W)*L + step]
    trace_start: int = 0           # first start node the trace covers (a trace recorded for a row slice)
    coupling: str = "iid"          # one of COUPLINGS: how the W walks of a start node share their draws

    def validate(self):
        if int(self.walks_per_node) < 1:
            raise ValueError("walks_per_node must be >= 1")
        if int(self.max_walk_length) < 1:
            raise ValueError("max_walk_length must be >= 1")
        if not (0.0 <= float(self.p_halt) <= 1.0):
            raise ValueError("p_halt must be in [0, 1]")
        if self.draw_mode == _lib.DRAW_REPLAY and self.trace is None:
            raise ValueError("replay mode needs trace=(trace_u, trace_k)")
        if self.coupling not in COUPLINGS:
            raise ValueError(f"coupling must be one of {sorted(COUPLINGS)}, not {self.coupling!r}")
        if COUPLINGS[self.coupling] and (self.draw_mode != _lib.DRAW_PHILOX or self.trace is not None):
            raise ValueError("coupled draws need native Philox draws (no replayed trace)")

    def draw_flags(self) -> int:
        """draw_mode of GrfWalkCfg: the draw source with the coupling bits OR-ed in."""
        return int(self.draw_mode) | COUPLINGS[self.coupling]


def _to_host_pinned(t: torch.Tensor) -> torch.Tensor:
    """Device tensor -> pinned host tensor (pageable destinations run at ~2 GB/s)."""
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return host


_UPLOAD_CHUNK = 32 << 20      # bytes per pinned staging slot
_UPLOAD_THREADS = int(os.environ.get("GRF_UPLOAD_THREADS", "4"))
_UPLOAD_MIN = 64 << 20        # smaller arrays take torch's own pageable copy
_upload_state = {}            # device index -> (executor, [(stream, [pinned slots], [events])] per thread)


def _upload(arr: np.ndarray, dev: torch.device) -> torch.Tensor:
    """A large pageable host array -> a device tensor, ordered on torch's current stream.

    torch's pageable copy stages through one pinned buffer on one host thread (~10 GB/s: the 2 GB adjacency of a
    70 M-edge graph took 0.2 s, five times the whole Phi build).  Here a few host threads fill pinned slots in
    parallel (numpy copies release the GIL) and every slot goes out as its own asynchronous copy on the thread's
    stream, so the host memcpy of one chunk overlaps the DMA of the others."""
    arr = np.ascontiguousarray(arr)
    if arr.nbytes < _UPLOAD_MIN or not arr.flags.c_contiguous:
        return torch.from_numpy(arr).to(dev, non_blocking=True)
    from concurrent.futures import ThreadPoolExecutor

    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _upload_state:
        with torch.cuda.device(dev):
            lanes = [(torch.cuda.Stream(dev), [torch.empty(_UPLOAD_CHUNK, dtype=torch.uint8, pin_memory=True)
                                               for _ in range(2)], [torch.cuda.Event(), torch.cuda.Event()])
                     for _ in range(_UPLOAD_THREADS)]
        _upload_state[key] = (ThreadPoolExecutor(_UPLOAD_THREADS, thread_name_prefix="grf-upload"), lanes)
    pool, lanes = _upload_state[key]
    out = torch.empty(arr.shape, dtype=torch.from_numpy(arr[:0]).dtype, device=dev)
    src = arr.reshape(-1).view(np.uint8)
    dst = out.reshape(-1).view(torch.uint8)
    n = src.shape[0]
    n_chunks = (n + _UPLOAD_CHUNK - 1) // _UPLOAD_CHUNK
    ready = torch.cuda.Event()
    ready.record(torch.cuda.current_stream(dev))      # `out` exists on the current stream from here on

    def lane_work(t):
        stream, slots, events = lanes[t]
        with torch.cuda.device(dev):
            stream.wait_event(ready)
            for k, c in enumerate(range(t, n_chunks, _UPLOAD_THREADS)):
                lo, hi = c * _UPLOAD_CHUNK, min(n, (c + 1) * _UPLOAD_CHUNK)
                j = k & 1
                events[j].synchronize()               # the copy that last used this slot has left it
                np.copyto(slots[j].numpy()[: hi - lo], src[lo:hi])
                with torch.cuda.stream(stream):
                    dst[lo:hi].copy_(slots[j][: hi - lo], non_blocking=True)
                    events[j].record(stream)

    for fut in [pool.submit(lane_work, t) for t in range(_UPLOAD_THREADS)]:
        fut.result()
    cur = torch.cuda.current_stream(dev)
    for stream, _, _ in lanes:
        cur.wait_stream(stream)
    return out


def _upload_shared(arr: np.ndarray, dev: torch.device, group) -> torch.Tensor:
    """``_upload`` of an array that every rank of ``group`` holds identically: rank r uploads slice r, then one
    all-gather (NCCL over NVLink) completes every rank's copy."""
    import torch.distributed as dist

    pg = None if group is True else group
    world = dist.get_world_size(pg)
    arr = np.ascontiguousarray(arr)
    if world == 1 or arr.ndim != 1 or arr.nbytes < _UPLOAD_MIN:
        return _upload(arr, dev)
    rank = dist.get_rank(pg)
    n = arr.shape[0]
    per = (n + world - 1) // world
    lo, hi = min(n, rank * per), min(n, (rank + 1) * per)
    piece = torch.zeros(per, dtype=torch.from_numpy(arr[:0]).dtype, device=dev)
    if hi > lo:
        piece[: hi - lo].copy_(_upload(arr[lo:hi], dev))
    out = torch.empty(per * world, dtype=piece.dtype, device=dev)
    dist.all_gather_into_tensor(out, piece, group=pg)
    return out[:n]


class DeviceGraph:
    """The walk graph resident in HBM: CSR row_ptr/col_idx int32, val float64
    (what SparseRandomWalk.__init__ keeps, sparse_sampler.py:62-70)."""

    def __init__(self, indptr, indices, data, n_nodes: int, device=None, group=None):
        """``group`` (a torch.distributed group, or True for the default one): every rank of the group holds the
        SAME host arrays and wants the same replicated graph -- each then uploads one 1/world slice over its own
        PCIe link and the slices are all-gathered over NVLink (8 ranks pushing the whole 2 GB adjacency through
        one host's memory system took longer than the Phi build they feed)."""
        self.device = _device(device)
        indptr = np.ascontiguousarray(indptr)
        if indptr.shape[0] != n_nodes + 1:
            raise ValueError("indptr must have n_nodes + 1 entries")
        nnz = int(indptr[-1]) if n_nodes > 0 else 0
        if nnz >= 2 ** 31 or n_nodes >= 2 ** 31:
            raise ValueError("graph exceeds int32 index range")
        self.n_nodes = int(n_nodes)
        self.nnz = nnz
        self._scaled = {}
        self._shared = {}
        up = (lambda a: _upload(a, self.device)) if group is None else (lambda a: _upload_shared(a, self.device, group))
        self.row_ptr = up(indptr.astype(np.int32, copy=False))
        self.col_idx = up(np.ascontiguousarray(indices[:nnz]).astype(np.int32, copy=False))
        self.val = up(np.ascontiguousarray(data[:nnz]).astype(np.float64, copy=False))

    @classmethod
    def from_scipy(cls, adj, device=None) -> "DeviceGraph":
        if adj.shape[0] != adj.shape[1]:
            raise ValueError("Adjacency matrix must be square.")
        a = adj.tocsr()
        return cls(a.indptr, a.indices, a.data.astype(float, copy=False), a.shape[0], device)

    def c_struct(self) -> GrfGraph:
        return GrfGraph(self.n_nodes, self.nnz, self.row_ptr.data_ptr(), self.col_idx.data_ptr(),
                        self.val.data_ptr())

    @classmethod
    def _from_device(cls, row_ptr, col_idx, val, n_nodes) -> "DeviceGraph":
        g = cls.__new__(cls)
        g.device = row_ptr.device
        g.n_nodes, g.nnz = int(n_nodes), int(col_idx.numel())
        g._scaled = {}
        g._shared = {}
        g.row_ptr, g.col_idx, g.val = row_ptr, col_idx, val
        return g

    @classmethod
    def laplacian_of(cls, adj, device=None, group=None) -> "DeviceGraph":
        """The walk graph D^-1/2 (D - A) D^-1/2 of a scipy adjacency, normalised on the device
        (graph_utils.py:5-30, bit-identical values and structure).  ``group``: see ``__init__``."""
        if adj.shape[0] != adj.shape[1]:
            raise ValueError("Adjacency matrix must be square.")
        a = adj.tocsr()
        if not a.has_canonical_format:
            a = a.copy()
            a.sum_duplicates()
        return cls(a.indptr, a.indices, a.data.astype(float, copy=False), a.shape[0], device, group).laplacian()

    def laplacian(self) -> "DeviceGraph":
        """D^-1/2 (D - A) D^-1/2 of this graph read as a canonical CSR adjacency (sorted columns, no
        duplicates), on the device -- no host round trip (graph_utils.py:5-30)."""
        L = _lib.lib()
        dev, n = self.device, self.n_nodes
        with torch.cuda.device(dev):
            deg = torch.empty(max(1, n), dtype=torch.float64, device=dev)
            dis = torch.empty(max(1, n), dtype=torch.float64, device=dev)
            cnt = torch.empty(max(1, n), dtype=torch.int32, device=dev)
            g = self.c_struct()
            check(L.grf_laplacian_count(ctypes.byref(g), _ptr(deg), _ptr(dis), _ptr(cnt), _stream(dev)))
            ptr = scan_counts(cnt, n, 1, _lib.ORDER_ROW_MAJOR, i64=False)
            total = int(ptr[-1].item()) if n else 0
            col = torch.empty(max(1, total), dtype=torch.int32, device=dev)[:total]
            val = torch.empty(max(1, total), dtype=torch.float64, device=dev)[:total]
            check(L.grf_laplacian_fill(ctypes.byref(g), _ptr(deg), _ptr(dis), _ptr(ptr), _ptr(col), _ptr(val),
                                       _stream(dev)))
        return DeviceGraph._from_device(ptr, col, val, n)

    def to_scipy(self):
        import scipy.sparse as sp

        return sp.csr_matrix((self.val.cpu().numpy(), self.col_idx.cpu().numpy(), self.row_ptr.cpu().numpy()),
                             shape=(self.n_nodes, self.n_nodes))

    def shared_columns(self, bounds: Sequence[int], max_walk_length: int, max_fraction: float = 0.5):
        """Columns that the Phi blocks of two or more row shards can touch: nodes reachable within
        ``max_walk_length - 1`` hops from start nodes of >= 2 of the shards ``bounds[g] .. bounds[g+1]``.
        Depends on the graph and the sharding only (cached), needs no collective, and is a superset
        of what any draw touches -- assign it to ``PhiBlocks.shared_hint`` and the sharded matvec
        exchanges just these rows of Phi^T V.  Returns "all" when they exceed ``max_fraction`` of the
        nodes (then a plain all-reduce is cheaper)."""
        key = (tuple(int(b) for b in bounds), int(max_walk_length))
        if key not in self._shared:
            world = len(key[0]) - 1
            if world > 64:
                return None             # no bound: the plan falls back to exchanging the touched columns
            b = torch.tensor(key[0], dtype=torch.int64, device=self.device)
            mask = torch.empty(max(1, self.n_nodes), dtype=torch.int64, device=self.device)
            scratch = torch.empty_like(mask)
            g = self.c_struct()
            check(_lib.lib().grf_shard_reach(ctypes.byref(g), _ptr(b), world, max(0, key[1] - 1), _ptr(mask),
                                             _ptr(scratch), _stream(self.device)))
            mask = mask[: self.n_nodes]
            shared = torch.nonzero((mask & (mask - 1)) != 0).flatten()
            self._shared = {key: "all" if shared.numel() > max_fraction * self.n_nodes else shared}
        return self._shared[key]

    def edge_records(self, p_halt: float) -> torch.Tensor:
        """{(deg * w) / (1 - p_halt), neighbour} per edge, 16 bytes each (cached per p_halt): what the walker
        gathers per step."""
        key = float(p_halt)
        if key not in self._scaled:
            out = torch.empty((max(1, self.nnz), 2), dtype=torch.float64, device=self.device)
            g = self.c_struct()
            check(_lib.lib().grf_edge_records(ctypes.byref(g), key, _ptr(out), _stream(self.device)))
            self._scaled = {key: out}
        return self._scaled[key]


@dataclass
class Staging:
    stage_col: Optional[torch.Tensor]   # int32 [n_rows * stride]      (reference layout: column + float64 sum)
    stage_sum: Optional[torch.Tensor]   # float64 [n_rows * stride]
    row_cnt: torch.Tensor     # int32 [n_rows * L]
    stride: int
    n_rows: int
    row_lo: int
    visits: torch.Tensor      # int64 [1] walk-steps executed
    col_counts: Optional[torch.Tensor] = None   # int32 [n_nodes * L] entries per (column, length), if counted
    stage_ent: Optional[torch.Tensor] = None    # int32 [n_rows * stride, 2]: finished Phi entries (matvec layout)


def scan_counts(row_cnt: torch.Tensor, n_rows: int, n_steps: int, order: int, i64: bool,
                with_total: bool = False):
    """Exclusive prefix sum of the counts ([n + 1], last = total).  ``with_total``: also return the
    device int64[1] grand total (exact even when an int32 output wrapped)."""
    dev = row_cnt.device
    n = n_rows * n_steps
    out = torch.empty(n + 1, dtype=torch.int64 if i64 else torch.int32, device=dev)
    ws = torch.empty(_lib.lib().grf_scan_workspace_bytes(n) // 8, dtype=torch.int64, device=dev)
    check(_lib.lib().grf_scan_counts(_ptr(row_cnt), n_rows, n_steps, order, _ptr(out), int(i64), _ptr(ws),
                                     _stream(dev)))
    return (out, ws[:1]) if with_total else out


def run_walker(graph: DeviceGraph, cfg: WalkConfig, start_lo: int = 0, start_hi: Optional[int] = None,
               visits: Optional[torch.Tensor] = None, col_counts: Optional[torch.Tensor] = None,
               count_columns: bool = False, entries_scale_mode: Optional[int] = None) -> Staging:
    """One grf_walk launch over start nodes [start_lo, start_hi).  ``count_columns`` (or a zeroed /
    partially accumulated ``col_counts`` int32 [n_nodes * L]) also counts the entries per (column,
    length) while they are emitted: the segment sizes of the Phi^T blocks, for free.
    ``entries_scale_mode`` (SCALE_*): the walker leaves finished float32 Phi entries in staging
    (8 bytes per record instead of 12) -- the matvec layout needs nothing else."""
    cfg.validate()
    L = _lib.lib()
    dev = graph.device
    start_hi = graph.n_nodes if start_hi is None else start_hi
    n_rows = start_hi - start_lo
    stride = L.grf_walk_stage_stride(cfg.walks_per_node, cfg.max_walk_length)
    stage_col = stage_sum = stage_ent = None
    if entries_scale_mode is None:
        stage_col = torch.empty(max(1, n_rows * stride), dtype=torch.int32, device=dev)
        stage_sum = torch.empty(max(1, n_rows * stride), dtype=torch.float64, device=dev)
    else:
        stage_ent = torch.empty((max(1, n_rows * stride), 2), dtype=torch.int32, device=dev)
    row_cnt = torch.empty(max(1, n_rows * cfg.max_walk_length), dtype=torch.int32, device=dev)
    if visits is None:
        visits = torch.zeros(1, dtype=torch.int64, device=dev)
    if col_counts is None and count_columns:
        col_counts = torch.zeros(max(1, graph.n_nodes * cfg.max_walk_length), dtype=torch.int32, device=dev)
    tu = tk = None
    trace_base = 0
    if cfg.draw_mode == _lib.DRAW_REPLAY:
        tu = torch.as_tensor(cfg.trace[0], dtype=torch.float64).to(dev).contiguous()
        tk = torch.as_tensor(cfg.trace[1], dtype=torch.int32).to(dev).contiguous()
        if start_lo < cfg.trace_start and n_rows > 0:
            raise ValueError("trace starts after the first start node of this launch")
        trace_base = int(cfg.trace_start) * cfg.walks_per_node
        need = (start_hi - int(cfg.trace_start)) * cfg.walks_per_node * cfg.max_walk_length
        if n_rows > 0 and (tu.numel() < need or tk.numel() < need):
            raise ValueError("trace arrays must cover the walks of start nodes trace_start .. start_hi - 1 "
                             "((start_hi - trace_start) * W * L entries)")
    g = graph.c_struct()
    edges = None
    if cfg.load_mode != _lib.LOAD_ABLATION and cfg.max_walk_length > 1 and graph.nnz > 0 and cfg.p_halt < 1.0:
        edges = graph.edge_records(cfg.p_halt)
    c = GrfWalkCfg(start_lo, start_hi, cfg.walks_per_node, cfg.max_walk_length, float(cfg.p_halt), cfg.draw_flags(),
                   cfg.load_mode, int(cfg.seed) & 0xFFFFFFFFFFFFFFFF,
                   None if tu is None else tu.data_ptr(), None if tk is None else tk.data_ptr(),
                   None if edges is None else edges.data_ptr(),
                   None if col_counts is None else col_counts.data_ptr(), trace_base,
                   None if stage_ent is None else stage_ent.data_ptr(),
                   _lib.SCALE_MUL_RECIP if entries_scale_mode is None else int(entries_scale_mode))
    check(L.grf_walk(ctypes.byref(g), ctypes.byref(c), stride, _ptr(stage_col), _ptr(stage_sum), _ptr(row_cnt),
                     _ptr(visits), _stream(dev)))
    return Staging(stage_col, stage_sum, row_cnt, stride, n_rows, start_lo, visits, col_counts, stage_ent)


def _row_chunks(start_lo: int, start_hi: int, stride: int, max_stage_bytes: int, slot_bytes: int = 12):
    rows_per = max(1, max_stage_bytes // (stride * slot_bytes))
    lo = start_lo
    while lo < start_hi:
        hi = min(start_hi, lo + rows_per)
        yield lo, hi
        lo = hi
    if start_lo == start_hi:
        yield start_lo, start_hi


class StepMatrices:
    """The reference's output layout on device: L CSR matrices (rows = this
    shard's start nodes), concatenated step-major.  ``offsets[s*n_rows + r]`` is
    the position of (step s, row r); float64 values, int32 sorted columns."""

    def __init__(self, offsets, col, val, n_rows, n_cols, n_steps, row_lo, visits=0):
        self.offsets, self.col, self.val = offsets, col, val
        self.n_rows, self.n_cols, self.n_steps, self.row_lo = n_rows, n_cols, n_steps, row_lo
        self.visits = visits

    @property
    def device(self):
        return self.col.device

    def nnz_per_step(self) -> List[int]:
        off = self.offsets[:: max(1, self.n_rows)][: self.n_steps + 1].cpu().tolist() if self.n_rows else [0] * (
            self.n_steps + 1)
        return [off[s + 1] - off[s] for s in range(self.n_steps)]

    def to_scipy(self):
        """list[scipy.sparse.csr_matrix] of shape (n_rows, n_cols) -- what
        get_random_walk_matrices returns (sparse_sampler.py:117-132).

        One device->host copy per array into pinned memory (pageable destinations ran at
        ~2 GB/s), and the matrices are assembled around views of those buffers without
        scipy re-validating or copying the index arrays."""
        import scipy.sparse as sp

        n, L = self.n_rows, self.n_steps
        dev = self.device
        # per-step row pointers, rebased to 0, as int32 (scipy's index dtype for nnz < 2^31)
        starts = self.offsets[0:n * L + 1:max(1, n)][:L + 1] if n else torch.zeros(L + 1, dtype=torch.int64,
                                                                                   device=dev)
        bounds = starts.cpu().tolist()
        big = any(bounds[s + 1] - bounds[s] >= 2 ** 31 for s in range(L))
        idx_dtype = torch.int64 if big else torch.int32
        ip_dev = torch.empty((L, n + 1), dtype=idx_dtype, device=dev)
        for s in range(L):
            ip_dev[s] = (self.offsets[s * n:(s + 1) * n + 1] - bounds[s]).to(idx_dtype) if n else 0

        def fetch(t):
            host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            host.copy_(t, non_blocking=True)
            return host

        ip_h, col_h, val_h = fetch(ip_dev), fetch(self.col), fetch(self.val)
        torch.cuda.current_stream(dev).synchronize()
        ip, col, val = ip_h.numpy(), col_h.numpy(), val_h.numpy()
        if big:
            col = col.astype(np.int64)
        mats = []
        for s in range(L):
            b, e = bounds[s], bounds[s + 1]
            m = sp.csr_matrix((n, self.n_cols), dtype=np.float64)
            m.data, m.indices, m.indptr = val[b:e], col[b:e], ip[s]
            m.has_sorted_indices = True
            mats.append(m)
        return mats

    def kernel_matrix(self, f, **kwargs):
        """K = Phi_f Phi_f^T with Phi_f = sum_p f_p M_p (p < min(len(f), L)), formed on the device: a
        ``kernel_matrix.KernelMatrix`` (device indptr / indices / data, ``.to_scipy()``) equal to the reference's
        scipy ``Phi @ Phi.T`` (fast_grf_kernel_general.py:48-55) in every array.  Raises MemoryError, naming
        nnz(K), when K does not fit in free device memory."""
        from .kernel_matrix import kernel_matrix

        return kernel_matrix(self, f, **kwargs)

    def to_dense_tensor(self) -> np.ndarray:
        """(n_rows, n_cols, L) float64 -- RandomWalk's output layout (sampler.py:196-201)."""
        return self.to_dense_device().cpu().numpy() if self.n_rows * self.n_cols * self.n_steps < (1 << 22) \
            else _to_host_pinned(self.to_dense_device()).numpy()

    def to_dense_device(self) -> torch.Tensor:
        """The (n_rows, n_cols, L) float64 tensor assembled on the device: one scatter of the merged records
        (every (row, column, length) occurs once), no host loop over scipy matrices."""
        n, m, L, dev = self.n_rows, self.n_cols, self.n_steps, self.device
        out = torch.zeros((n, m, L), dtype=torch.float64, device=dev)
        if n and self.col.numel():
            counts = self.offsets[1:] - self.offsets[:-1]                       # [L * n], step-major
            seg = torch.repeat_interleave(torch.arange(L * n, device=dev), counts, output_size=self.col.numel())
            step = torch.div(seg, n, rounding_mode="floor")
            row = seg - step * n
            out.view(-1)[(row * m + self.col.long()) * L + step] = self.val
        return out

    @staticmethod
    def concat_rows(parts: Sequence["StepMatrices"]) -> "StepMatrices":
        if len(parts) == 1:
            return parts[0]
        L, n_cols = parts[0].n_steps, parts[0].n_cols
        dev = parts[0].device
        cols, vals, cnts = [], [], []
        for s in range(L):
            for p in parts:
                o = p.offsets[s * p.n_rows: (s + 1) * p.n_rows + 1]
                b, e = int(o[0]), int(o[-1])
                cols.append(p.col[b:e])
                vals.append(p.val[b:e])
                cnts.append(o[1:] - o[:-1])
        counts = torch.cat(cnts) if cnts else torch.zeros(0, dtype=torch.int64, device=dev)
        offsets = torch.zeros(counts.numel() + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=offsets[1:])
        n_rows = sum(p.n_rows for p in parts)
        return StepMatrices(offsets, torch.cat(cols), torch.cat(vals), n_rows, n_cols, L, parts[0].row_lo,
                            sum(p.visits for p in parts))


def _steps_from_staging(st: Staging, cfg: WalkConfig, n_cols: int, scale_mode: int) -> StepMatrices:
    L = cfg.max_walk_length
    dev = st.stage_col.device
    offsets = scan_counts(st.row_cnt, st.n_rows, L, _lib.ORDER_STEP_MAJOR, i64=True)
    total = int(offsets[-1].item())
    col = torch.empty(max(1, total), dtype=torch.int32, device=dev)[:total]
    val = torch.empty(max(1, total), dtype=torch.float64, device=dev)[:total]
    check(_lib.lib().grf_compact_steps(_ptr(st.stage_col), _ptr(st.stage_sum), _ptr(st.row_cnt), _ptr(offsets),
                                       st.n_rows, L, st.stride, cfg.walks_per_node, scale_mode, _ptr(col), _ptr(val),
                                       _stream(dev)))
    return StepMatrices(offsets, col, val, st.n_rows, n_cols, L, st.row_lo)


def build_step_matrices(graph: DeviceGraph, cfg: WalkConfig, start_lo: int = 0, start_hi: Optional[int] = None,
                        scale_mode: int = _lib.SCALE_MUL_RECIP,
                        max_stage_bytes: int = _MAX_STAGE_BYTES) -> StepMatrices:
    """Walker + compaction into the reference's per-length CSR layout (on device)."""
    cfg.validate()
    start_hi = graph.n_nodes if start_hi is None else start_hi
    stride = _lib.lib().grf_walk_stage_stride(cfg.walks_per_node, cfg.max_walk_length)
    visits = torch.zeros(1, dtype=torch.int64, device=graph.device)
    parts = []
    for lo, hi in _row_chunks(start_lo, start_hi, stride, max_stage_bytes):
        st = run_walker(graph, cfg, lo, hi, visits=visits)
        parts.append(_steps_from_staging(st, cfg, graph.n_nodes, scale_mode))
        del st
    out = StepMatrices.concat_rows(parts)
    out.visits = int(visits.item())
    return out


class TBlock:
    """Phi^T of the rows [r0, r0 + n_rows) of a shard: block CSR over (column, walk length), entries
    {length << 27 | row - r0, value}, every segment ordered by row.  A large shard keeps one per
    T_BLOCK_ROWS rows (the first half of the product then gathers V one L2-sized row block at a time)."""

    def __init__(self, r0: int, n_rows: int, nnz: int, tblk_ptr: torch.Tensor, tentries: torch.Tensor):
        self.r0, self.n_rows, self.nnz = int(r0), int(n_rows), int(nnz)
        self.tblk_ptr, self.tentries = tblk_ptr, tentries
        self.census = None      # (pinned int32[6], event): rows of Phi in this block [0:3], of this Phi^T [3:6]
        self.long = None        # chunk table of the columns longer than LONG_ROW_THRESHOLD (dict) or None
        self.long_c = {}        # ld -> (GrfLongRows, partial buffer)
        self.tcols = None       # non-empty columns (int32) when they are a small fraction of N (single block only)
        self.touched = None     # int32 0/1 per column, set together with tcols
        self.tcols_cap = None


class PhiBlocks:
    """Phi in the matvec layout: block CSR over (row, walk length) with
    {int32 col, float32 val} entries, plus the same for Phi^T (built once --
    the reference re-sorts every M_l on every forward, sparse_lo.py:23-25).

    ``matvec`` is the kernel matvec ``Phi[x1] (Phi[x2]^T V)`` with
    ``Phi = sum_l f[l] M_l`` (sparse_grf_kernel.py:24-62); f is applied at
    matvec time so it can be a learnable parameter."""

    def __init__(self, blk_ptr, entries, n_rows, n_cols, n_steps, row_lo=0, visits=0):
        if max(n_rows, n_cols) > (1 << _lib.ENTRY_STEP_SHIFT) or n_steps > (1 << (32 - _lib.ENTRY_STEP_SHIFT)):
            raise ValueError("Phi blocks hold at most 2^27 rows/columns per GPU and 32 walk lengths")
        self.blk_ptr, self._entries = blk_ptr, entries
        self._nnz_pending = None   # (pinned int64[1], event): `_entries` has spare capacity until this resolves
        self.n_rows, self.n_cols, self.n_steps, self.row_lo = n_rows, n_cols, n_steps, row_lo
        self.tblocks: Optional[List[TBlock]] = None   # Phi^T, one block per T_BLOCK_ROWS rows (build_transpose)
        self.win = self.twin = None
        self.win_max_width = self.twin_max_width = 0
        # shared-memory-tiled matvec for banded Phi: correct and tested, but measured equal to the
        # global-gather kernel at config 2 (both are bound by L1 wavefronts per entry), so opt-in
        self.use_tiles = False
        # hand the last rows of every matvec pass out by ticket (GrfPhi.sched); env GRF_B200_DYNAMIC=0
        # keeps the fixed stride (for A/B timing)
        self.dynamic_rows = os.environ.get("GRF_B200_DYNAMIC", "1") != "0"
        # gather the right-hand side with L1::no_allocate loads, per half (Phi^T V, Phi U).  Opt-in experiment
        # (env GRF_B200_STREAM=11): measured 3-5x SLOWER on the power-law Phi (40.6 / 26.3 ms against 12.8 / 5.0),
        # so the cached loads stay the default; MatvecPlan._tune_gathers() measures both on request.
        env = os.environ.get("GRF_B200_STREAM", "00")
        self.stream_gather = (env[0] == "1", env[-1] == "1")
        self._sched = None
        self._col_counts = None  # int32 [n_cols * L] from the walker (GrfWalkCfg.col_counts), used once by build_transpose
        self.visits = visits
        self._union = None
        self._pairs = None      # per side: pair row pointers / slot of every union entry (build_pairs)
        self._pent = None       # on a merged PhiBlocks: the pair entries of (Phi_f, Phi_f^T)
        # sharded matvec: columns to exchange between the ranks, if known up front (tensor of ids or
        # "all"; DeviceGraph.shared_columns); None = the plan finds them with one all-reduce
        self.shared_hint = None
        self._long_fwd = None   # chunk table of the rows of Phi longer than LONG_ROW_THRESHOLD
        self._long_built = False
        self._long_fwd_c = {}   # ld -> (GrfLongRows, partial buffer) kept alive for the calls
        self._ws = {}

    @property
    def device(self):
        return self.blk_ptr.device

    @property
    def entries(self) -> torch.Tensor:
        """[nnz, 2] int32 view of the {length << 27 | col, value bits} pairs.  A Phi built straight from
        staging holds a capacity-sized buffer until the entry count -- copied to pinned host memory behind
        the offset scan -- is first needed; by then the compaction kernel is already queued, so reading
        it does not idle the GPU."""
        if self._nnz_pending is not None:
            host, arrived, base = self._nnz_pending
            arrived.synchronize()
            self._nnz_pending = None
            self._entries = self._entries[: int(host[0])]
            _recycle_pinned(base)
        return self._entries

    @entries.setter
    def entries(self, value: torch.Tensor) -> None:
        self._entries, self._nnz_pending = value, None

    @property
    def nnz(self) -> int:
        return int(self.entries.shape[0])

    # ---- the transposed side: one block, or one per T_BLOCK_ROWS rows -----------------------------
    def _tb0(self) -> Optional[TBlock]:
        if self.tblocks is None:
            return None
        if len(self.tblocks) != 1:
            raise ValueError("this Phi^T is stored in several row blocks; the single-block view does not exist")
        return self.tblocks[0]

    @property
    def tblk_ptr(self):
        tb = self._tb0()
        return None if tb is None else tb.tblk_ptr

    @property
    def tentries(self):
        tb = self._tb0()
        return None if tb is None else tb.tentries

    @property
    def _tcols(self):
        return self.tblocks[0].tcols if self.tblocks is not None and len(self.tblocks) == 1 else None

    @_tcols.setter
    def _tcols(self, value):
        self._tb0().tcols = value

    @property
    def _touched(self):
        return self.tblocks[0].touched if self.tblocks is not None and len(self.tblocks) == 1 else None

    @property
    def _long(self):
        """[long rows of Phi, long columns of the (single) Phi^T block] once build_long_rows() has run."""
        if not self._long_built:
            return None
        return [self._long_fwd, self.tblocks[0].long if self.tblocks else None]

    @_long.setter
    def _long(self, value):
        self._long_built = value is not None
        self._long_fwd = None if value is None else value[0]
        if self.tblocks:
            for tb in self.tblocks:
                tb.long = None
            if value is not None:
                self.tblocks[0].long = value[1]

    @property
    def _long_c(self):
        return self._long_fwd_c

    @_long_c.setter
    def _long_c(self, value):
        self._long_fwd_c = value
        for tb in self.tblocks or []:
            tb.long_c = {}

    def build_transpose(self, block_rows: Optional[int] = None) -> "PhiBlocks":
        """Phi^T blocks (once per Phi): per row block, two C calls on one workspace -- segment offsets, then
        a stable radix sort of the block's entries by (column, length).  The row census of both sides is
        copied to pinned host memory behind the offsets, so build_long_rows() reads it while the sort
        still runs instead of draining the GPU."""
        if self.tblocks is not None:
            return self
        block_rows = T_BLOCK_ROWS if block_rows is None else int(block_rows)
        n_blocks = 1 if self.n_rows <= block_rows + block_rows // 2 else -(-self.n_rows // block_rows)
        rows = [self.n_rows * b // n_blocks for b in range(n_blocks + 1)]
        if n_blocks == 1:
            bounds = [0, self.nnz]
        else:
            idx = torch.tensor([r * self.n_steps for r in rows], dtype=torch.int64, device=self.device)
            bounds = self.blk_ptr[idx].cpu().tolist()
        counts = self._col_counts if n_blocks == 1 else None   # the walker's counts cover the whole shard
        self._col_counts = None
        self.tblocks = [self._build_tblock(rows[b], rows[b + 1], bounds[b], bounds[b + 1], counts)
                        for b in range(n_blocks)]
        tb = self.tblocks[0]
        if n_blocks == 1 and tb.nnz and self.n_rows < self.n_cols:
            # a row shard: list its non-empty columns now (capacity n_cols, the census gives the length
            # later), while the host would otherwise wait for the sort
            self._list_nonempty_columns(tb, self.n_cols)
        return self

    def _build_tblock(self, r0: int, r1: int, e0: int, e1: int, col_counts) -> TBlock:
        L = _lib.lib()
        dev, st = self.device, _stream(self.device)
        n_seg = self.n_cols * self.n_steps
        nnz = e1 - e0
        ws = torch.empty(L.grf_transpose_workspace_bytes(self.n_cols, self.n_steps, nnz), dtype=torch.uint8, device=dev)
        tblk_ptr = torch.empty(n_seg + 1, dtype=torch.int32, device=dev)
        tentries = torch.empty((max(1, nnz), 2), dtype=torch.int32, device=dev)[:nnz]
        tb = TBlock(r0, r1 - r0, nnz, tblk_ptr, tentries)
        base = _small_pinned() if nnz else None
        host = None if base is None else base[:6]
        ptr = ctypes.c_void_p(self.blk_ptr.data_ptr() + 4 * r0 * self.n_steps)
        ent = _ptr(self.entries) if self.nnz else None
        check(L.grf_transpose_offsets(ptr, ent, r1 - r0, self.n_cols, self.n_steps, _ptr(col_counts), _ptr(tblk_ptr),
                                      _ptr(ws), LONG_ROW_THRESHOLD, _ptr(host), st))
        if host is not None:
            arrived = torch.cuda.Event()
            arrived.record(torch.cuda.current_stream(dev))
            tb.census = (host, arrived, base)
            _keep_until_done(base, arrived)
        check(L.grf_transpose_fill(ptr, ent, r1 - r0, self.n_cols, self.n_steps, e0, nnz, _ptr(ws), _ptr(tentries), st))
        return tb

    def _list_nonempty_columns(self, tb: TBlock, capacity: int) -> None:
        lib, dev = _lib.lib(), self.device
        tb.touched = torch.empty(self.n_cols, dtype=torch.int32, device=dev)
        pos = torch.empty(self.n_cols + 1, dtype=torch.int32, device=dev)
        ws = torch.empty(lib.grf_scan_workspace_bytes(self.n_cols), dtype=torch.uint8, device=dev)
        tb.tcols_cap = torch.empty(max(1, capacity), dtype=torch.int32, device=dev)
        check(lib.grf_nonempty_rows(_ptr(tb.tblk_ptr), self.n_cols, self.n_steps, _ptr(tb.touched), _ptr(pos),
                                    _ptr(ws), _ptr(tb.tcols_cap), _stream(dev)))

    def _start_census(self, tb: TBlock) -> None:
        """Row statistics of both sides for a block that did not come through _build_tblock()."""
        if tb.nnz == 0 or tb.census is not None:
            return
        lib, dev, L = _lib.lib(), self.device, self.n_steps
        census = torch.empty(6, dtype=torch.int32, device=dev)
        ptr = ctypes.c_void_p(self.blk_ptr.data_ptr() + 4 * tb.r0 * L)
        check(lib.grf_row_census(ptr, tb.n_rows, L, LONG_ROW_THRESHOLD, _ptr(census[0:3]), _stream(dev)))
        check(lib.grf_row_census(_ptr(tb.tblk_ptr), self.n_cols, L, LONG_ROW_THRESHOLD, _ptr(census[3:6]),
                                 _stream(dev)))
        base = _small_pinned()
        host = base[:6]
        host.copy_(census, non_blocking=True)
        arrived = torch.cuda.Event()
        arrived.record(torch.cuda.current_stream(dev))
        tb.census = (host, arrived, base)
        _keep_until_done(base, arrived)

    def build_windows(self) -> "PhiBlocks":
        """Column windows per 32 rows of Phi and Phi^T (lets a banded Phi use the tiled matvec)."""
        self.build_transpose()
        if self.win is not None or self.nnz == 0 or not self.use_tiles or len(self.tblocks) != 1:
            return self
        L = _lib.lib()
        dev = self.device
        widths = torch.zeros(2, dtype=torch.int32, device=dev)
        self.win = torch.empty(((self.n_rows + 31) // 32, 2), dtype=torch.int32, device=dev)
        self.twin = torch.empty(((self.n_cols + 31) // 32, 2), dtype=torch.int32, device=dev)
        check(L.grf_block_windows(_ptr(self.blk_ptr), _ptr(self.entries), self.n_rows, self.n_steps, _ptr(self.win),
                                  ctypes.c_void_p(widths.data_ptr()), _stream(dev)))
        check(L.grf_block_windows(_ptr(self.tblk_ptr), _ptr(self.tentries), self.n_cols, self.n_steps,
                                  _ptr(self.twin), ctypes.c_void_p(widths.data_ptr() + 4), _stream(dev)))
        self.win_max_width, self.twin_max_width = (int(x) for x in widths.cpu().tolist())
        return self

    # ---- union rows: Phi_f = sum_l f[l] M_l materialised on the union pattern ------------
    def build_union(self) -> "PhiBlocks":
        """Merge the per-length segments of every row of Phi and Phi^T (once per Phi)."""
        if self._union is not None:
            return self
        self.build_transpose()
        if len(self.tblocks) != 1:
            raise ValueError("the union layout needs a single-block Phi^T (shards beyond ~T_BLOCK_ROWS rows multiply "
                             "the per-length blocks)")
        L = _lib.lib()
        dev = self.device
        sides = []
        for ptr, ent, n in ((self.blk_ptr, self.entries, self.n_rows), (self.tblk_ptr, self.tentries, self.n_cols)):
            # tasks: a row, or one UNION_CHUNK-entry chunk of a long row's flat run (hub columns must not
            # serialise one warp); listed row by row, so a scan over the tasks is a scan over the rows
            nL = self.n_steps
            row_b = ptr[0:n * nL:nL].to(torch.int64)
            row_e = ptr[nL:n * nL + 1:nL].to(torch.int64)
            nch = torch.clamp((row_e - row_b + UNION_CHUNK - 1) // UNION_CHUNK, min=1)
            task_ptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            torch.cumsum(nch, 0, out=task_ptr[1:])
            n_tasks = int(task_ptr[-1].item())
            if n_tasks == n:
                task_row = torch.arange(n, dtype=torch.int32, device=dev)
                task_b, task_e = row_b.to(torch.int32), row_e.to(torch.int32)
            else:
                rows = torch.repeat_interleave(torch.arange(n, device=dev), nch, output_size=n_tasks)
                local = torch.arange(n_tasks, device=dev) - task_ptr[rows]
                tb = row_b[rows] + local * UNION_CHUNK
                task_b = tb.to(torch.int32)
                task_e = torch.minimum(tb + UNION_CHUNK, row_e[rows]).to(torch.int32)
                task_row = rows.to(torch.int32)
                del rows, local, tb
            mkey = torch.empty(max(1, self.nnz), dtype=torch.int32, device=dev)
            mval = torch.empty(max(1, self.nnz), dtype=torch.float32, device=dev)
            tcnt = torch.empty(max(1, n_tasks), dtype=torch.int32, device=dev)
            check(L.grf_union_rank(_ptr(ptr), _ptr(ent), nL, _ptr(task_row), _ptr(task_b), _ptr(task_e), n_tasks,
                                   _ptr(mkey), _ptr(mval), _ptr(tcnt), _stream(dev)))
            task_u0 = scan_counts(tcnt, n_tasks, 1, _lib.ORDER_ROW_MAJOR, i64=False)
            n_union = int(task_u0[-1].item())
            uhdr = torch.empty((max(1, n_union), 2), dtype=torch.int32, device=dev)[:n_union]
            task_v0 = torch.empty(max(1, n_tasks), dtype=torch.int32, device=dev)
            check(L.grf_union_fill(_ptr(ptr), _ptr(mkey), nL, _ptr(task_row), _ptr(task_b), _ptr(task_e), n_tasks,
                                   _ptr(task_u0), _ptr(uhdr), _ptr(task_v0), _stream(dev)))
            uptr = task_u0[task_ptr].contiguous()
            sides.append(dict(n=n, uptr=uptr, uhdr=uhdr, mval=mval, n_union=n_union, n_tasks=n_tasks,
                              task_u0=task_u0, task_v0=task_v0))
            del mkey, task_row, task_b, task_e, tcnt
        self._union = sides
        return self

    def build_pairs(self) -> "PhiBlocks":
        """Line pairs of the union rows (csrc/grf_pairs.cu): once per Phi, per side the pair row pointers and the
        pair slot of every union entry."""
        self.build_union()
        if self._pairs is None:
            L = _lib.lib()
            dev = self.device
            out = []
            for side in self._union:
                n, n_union = side["n"], side["n_union"]
                pcnt = torch.empty(max(1, n), dtype=torch.int32, device=dev)
                check(L.grf_pairs_count(_ptr(side["uptr"]), _ptr(side["uhdr"]), n, _ptr(pcnt), _stream(dev)))
                pptr = scan_counts(pcnt, n, 1, _lib.ORDER_ROW_MAJOR, i64=False)
                n_pairs = int(pptr[-1].item())
                pidx = torch.empty(max(1, n_union), dtype=torch.int32, device=dev)
                check(L.grf_pairs_index(_ptr(side["uptr"]), _ptr(side["uhdr"]), n, _ptr(pptr), _ptr(pidx),
                                        _stream(dev)))
                out.append(dict(pptr=pptr, pidx=pidx, n_pairs=n_pairs, n_union=n_union, n=n))
            self._pairs = out
        return self

    @property
    def pair_ratio(self) -> float:
        """Pair entries / union entries over both sides (1.0 = no column has its line partner)."""
        self.build_pairs()
        return sum(p["n_pairs"] for p in self._pairs) / max(1, sum(p["n_union"] for p in self._pairs))

    @property
    def nnz_union(self) -> int:
        self.build_union()
        return self._union[0]["n_union"]

    def merged(self, f, into: Optional["PhiBlocks"] = None, pairs: bool = False) -> "PhiBlocks":
        """Phi_f as a single-length PhiBlocks (multiply it with f = [1]).  ``into`` re-uses the
        buffers of an earlier result (same Phi) when the modulator changed.  ``pairs``: also fill the line-pair
        entries (``into._pent``) that ``grf_pairs_spmm`` multiplies."""
        self.build_union()
        L = _lib.lib()
        dev = self.device
        f = self._f(f)
        fwd, tr = self._union
        if into is None:
            ent = torch.empty((max(1, fwd["n_union"]), 2), dtype=torch.int32, device=dev)[:fwd["n_union"]]
            tent = torch.empty((max(1, tr["n_union"]), 2), dtype=torch.int32, device=dev)[:tr["n_union"]]
            into = PhiBlocks(fwd["uptr"], ent, self.n_rows, self.n_cols, 1, self.row_lo)
            into.tblocks = [TBlock(0, self.n_rows, tr["n_union"], tr["uptr"], tent)]
        for side, ent in ((fwd, into.entries), (tr, into.tentries)):
            check(L.grf_union_materialize(_ptr(side["task_u0"]), _ptr(side["task_v0"]), side["n_tasks"],
                                          _ptr(side["uhdr"]), _ptr(side["mval"]), _ptr(f), self.n_steps, _ptr(ent),
                                          _stream(dev)))
        if pairs:
            self.build_pairs()
            if into._pent is None:
                into._pent = [torch.empty((max(1, p["n_pairs"]), 4), dtype=torch.int32, device=dev)
                              for p in self._pairs]
            for p, ent, pent in zip(self._pairs, (into.entries, into.tentries), into._pent):
                check(L.grf_pairs_fill(_ptr(ent), _ptr(p["pidx"]), p["n_union"], p["n_pairs"], _ptr(pent),
                                       _stream(dev)))
        return into

    def _long_rows_of(self, ptr: torch.Tensor, n: int, ent: Optional[torch.Tensor], n_long: int, n_chunks: int,
                      chunk: int = LONG_ROW_THRESHOLD):
        """Chunk table for the rows of one side that are longer than LONG_ROW_THRESHOLD (or None), built on the
        device from the census counts (``grf_long_rows_build``: no host round trip, two launches).  With the
        side's entries the chunks also get an issue order: by the first X row they gather (segments are sorted,
        so a chunk reads an ascending run of rows) -- the chunks in flight then share a window of X in L2."""
        if n == 0 or self.nnz == 0 or n_long == 0:
            return None
        dev = ptr.device
        if chunk != LONG_ROW_THRESHOLD:        # the census counted chunks of LONG_ROW_THRESHOLD entries
            nL = self.n_steps
            lens = (ptr[nL:n * nL + 1:nL] - ptr[0:n * nL:nL]).to(torch.int64)
            n_chunks = int(((lens[lens > LONG_ROW_THRESHOLD] + chunk - 1) // chunk).sum().item())
        rows = torch.empty(n_long, dtype=torch.int32, device=dev)
        chunk_ptr = torch.empty(n_long + 1, dtype=torch.int32, device=dev)
        bounds = torch.empty((n_chunks, 2), dtype=torch.int32, device=dev)
        ordered = ent is not None and CHUNK_ORDER and n_chunks > 1
        first = torch.empty(n_chunks, dtype=torch.int32, device=dev) if ordered else None
        ticket = torch.empty(1, dtype=torch.int64, device=dev)
        check(_lib.lib().grf_long_rows_build(_ptr(ptr), _ptr(ent), n, self.n_steps, LONG_ROW_THRESHOLD, chunk, n_long,
                                             n_chunks, _ptr(ticket), _ptr(rows), _ptr(chunk_ptr), _ptr(bounds),
                                             _ptr(first), _stream(dev)))
        order = torch.argsort(first).to(torch.int32) if ordered else None
        return dict(rows=rows, chunk_ptr=chunk_ptr, bounds=bounds, n_long=n_long, n_chunks=n_chunks, order=order)

    def build_long_rows(self) -> "PhiBlocks":
        """One-off matvec preparation: which rows / columns need the long-row split, and the list of
        non-empty columns when this shard touches few of them.  Reads the census that
        build_transpose() started; the chunk tables are only built when a long row exists."""
        if not self._long_built:
            self.build_transpose()
            self._long_built = True
            self._long_fwd = None
            if self.nnz == 0:
                return self
            fwd_long = fwd_chunks = 0      # rows of Phi: summed over the row blocks of Phi^T
            for tb in self.tblocks:
                if tb.nnz == 0:
                    continue
                self._start_census(tb)
                host, done, base = tb.census
                done.synchronize()
                long_f, chunks_f, _, long_t, chunks_t, cols_used = host.tolist()
                tb.census = (host.clone(), done, None)      # the values stay; the pinned buffer goes back to the pool
                _recycle_pinned(base)
                fwd_long, fwd_chunks = fwd_long + long_f, fwd_chunks + chunks_f
                tb.long = self._long_rows_of(tb.tblk_ptr, self.n_cols, tb.tentries, long_t, chunks_t, T_CHUNK)
                if len(self.tblocks) == 1:
                    # columns this (row) shard touches: worth a list when most of the N columns are empty
                    if cols_used < 0.75 * self.n_cols:
                        if tb.tcols_cap is None:
                            self._list_nonempty_columns(tb, cols_used)
                        tb.tcols = tb.tcols_cap[:cols_used]
                    else:
                        tb.touched = None
                    tb.tcols_cap = None
            self._long_fwd = self._long_rows_of(self.blk_ptr, self.n_rows, self.entries, fwd_long, fwd_chunks)
        return self

    def _long_struct(self, side: Optional[dict], cache: dict, ld: int):
        """ctypes GrfLongRows of one side with a partial buffer of leading dimension ``ld`` (cached per ld)."""
        if side is None or ld <= 0:
            return None
        if ld not in cache:
            partial = torch.empty((side["n_chunks"], ld), dtype=torch.float32, device=self.device)
            cache.clear()
            cache[ld] = (GrfLongRows(LONG_ROW_THRESHOLD, side["n_long"], side["n_chunks"], side["rows"].data_ptr(),
                                     side["chunk_ptr"].data_ptr(), side["bounds"].data_ptr(), partial.data_ptr(), ld,
                                     side["order"].data_ptr() if side.get("order") is not None else None),
                         partial)
        return cache[ld][0]

    def c_struct(self, ld: int = 0, block: Optional[int] = None) -> GrfPhi:
        """The GrfPhi argument block.  ``block`` = None: all rows of Phi with the (single) Phi^T block -- both
        halves of a product; ``block`` = b: the view of row block b for the first half (its rows of Phi, its
        Phi^T)."""
        tb = None
        if self.tblocks:
            tb = self.tblocks[0 if block is None else block]
            if block is None and len(self.tblocks) != 1:
                tb = None     # second half only: the forward side does not need Phi^T
        whole = block is None
        tiles = whole and self.use_tiles and self.win is not None
        fwd = self._long_struct(self._long_fwd, self._long_fwd_c, ld) if (whole and self._long_built) else None
        tr = self._long_struct(tb.long, tb.long_c, ld) if (tb is not None and self._long_built) else None
        r0 = 0 if whole else tb.r0
        n_rows = self.n_rows if whole else tb.n_rows
        nnz = self.nnz if whole else tb.nnz
        tcols = tb.tcols if tb is not None else None
        return GrfPhi(n_rows, self.n_cols, self.row_lo + r0, self.n_steps,
                      self.blk_ptr.data_ptr() + 4 * r0 * self.n_steps,
                      self.entries.data_ptr() if self.nnz else None,
                      None if tb is None else tb.tblk_ptr.data_ptr(),
                      None if tb is None or not tb.nnz else tb.tentries.data_ptr(),
                      self.win.data_ptr() if tiles else None, self.twin.data_ptr() if tiles else None,
                      self.win_max_width if tiles else 0, self.twin_max_width if tiles else 0,
                      ctypes.pointer(fwd) if fwd is not None else None,
                      ctypes.pointer(tr) if tr is not None else None,
                      None if tcols is None else tcols.data_ptr(),
                      0 if tcols is None else tcols.numel(), nnz, self._sched_ptr())

    def _gather_flags(self):
        sg = self.stream_gather or (False, False)
        return (32 if sg[0] else 0), (32 if sg[1] else 0)

    def _first_half(self, f, rows, n2, v, ldv, u, ldu, vfull, t, flags, structs=None):
        """U = Phi[rows]^T V block by block (the second and later row blocks add to U)."""
        fn, st = _lib.lib().grf_phi_matvec, _stream(self.device)
        for b, tb in enumerate(self.tblocks):
            c = structs[b] if structs is not None else self.c_struct((t + 3) // 4 * 4, block=b)
            vb, nb = v, n2
            if rows is None:
                vb, nb = (None if v is None else v + 4 * tb.r0 * ldv), tb.n_rows
            vf = None if vfull is None else vfull + 4 * tb.r0 * ldu
            rc = fn(ctypes.byref(c), _ptr(f), None, tb.n_rows, _ptr(rows), nb,
                    None if vb is None else ctypes.c_void_p(vb), ldv, None, 0, ctypes.c_void_p(u), ldu,
                    None if vf is None else ctypes.c_void_p(vf), t, 1 | flags | (16 if b else 0), st)
            if rc:
                check(rc)

    def _sched_ptr(self):
        # ticket scratch of the matvec kernels (GrfPhi.sched): zero between launches
        if not self.dynamic_rows:
            return None
        if getattr(self, "_sched", None) is None:
            self._sched = torch.zeros(4, dtype=torch.int32, device=self.device)
        return self._sched.data_ptr()

    @staticmethod
    def _ids(x, dev):
        if x is None:
            return None
        x = torch.as_tensor(x, device=dev)
        return x.flatten().to(torch.int32).contiguous()

    @property
    def is_shard(self) -> bool:
        """True when these blocks hold the rows of a slice of the start nodes (ids outside it belong to a peer)."""
        return self.row_lo != 0 or self.n_rows != self.n_cols

    def check_ids(self, x) -> None:
        """Raise IndexError for row ids outside Phi, as ``phi[idx]`` does in the reference
        (sparse_grf_kernel.py:32-41).  The kernels themselves skip ids outside the local rows -- that is what a
        row shard needs -- so on the whole Phi an out-of-range id would otherwise come back as a zero row.  One
        min/max (a device sync): called where an operator or a plan is built, not per product."""
        if x is None:
            return
        x = torch.as_tensor(x, device=self.device).flatten()
        if x.numel() == 0:
            return
        lo, hi = (int(v) for v in torch.aminmax(x))
        n = self.n_cols if self.is_shard else self.n_rows
        if lo < 0 or hi >= n:
            raise IndexError(f"row index {lo if lo < 0 else hi} is out of bounds for Phi with {n} rows")

    def row_dots(self, f, x1=None, x2=None) -> torch.Tensor:
        """dots[i, l] = <M_l[x1[i], :], Phi_f[x2[i], :]> (float32 [n, L]); ``dots @ f`` is diag(K[x1, x2]).
        No densification: a warp per pair (``grf_phi_row_dots``)."""
        dev = self.device
        f = self._f(f)
        a, b = self._ids(x1, dev), self._ids(x2, dev)
        if (a is None) != (b is None):      # one side indexed: the other is the identity list
            ident = torch.arange(self.row_lo, self.row_lo + self.n_rows, dtype=torch.int32, device=dev)
            a, b = (ident if a is None else a), (ident if b is None else b)
        n = self.n_rows if a is None else a.numel()
        if a is not None and b.numel() != n:
            raise ValueError("row_dots: x1 and x2 must have the same length")
        dots = torch.zeros((n, self.n_steps), dtype=torch.float32, device=dev)
        phi = self.c_struct()
        check(_lib.lib().grf_phi_row_dots(ctypes.byref(phi), _ptr(f), _ptr(a), _ptr(b), n, _ptr(dots), _stream(dev)))
        return dots

    def _f(self, f) -> torch.Tensor:
        f = torch.as_tensor(f, device=self.device).detach().to(torch.float32).contiguous()
        if f.numel() != self.n_steps:
            raise ValueError(f"modulator has {f.numel()} entries, Phi has {self.n_steps} walk lengths")
        return f

    @staticmethod
    def _rhs(x, dev) -> torch.Tensor:
        x = torch.as_tensor(x, device=dev).detach()
        if x.dim() != 2:
            raise ValueError("right-hand side must be 2-D [rows, t]")
        x = x.to(torch.float32)
        if (x.stride(1) != 1 and x.shape[1] != 1) or (x.shape[0] > 1 and x.stride(0) < x.shape[1]):
            x = x.contiguous()
        return x

    def apply_t(self, f, v, rows=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """U = Phi[rows]^T v: v [n2, t] -> U [n_cols, t] (this GPU's partial sum
        when Phi is row-sharded).  ``out`` may be a [n_cols, >=t] float32 buffer."""
        dev = self.device
        self.build_windows()
        self.build_long_rows()
        f = self._f(f)
        v = self._rhs(v, dev)
        rows = self._ids(rows, dev)
        n2, t = v.shape
        if n2 != (self.n_rows if rows is None else rows.numel()):
            raise ValueError("rhs has the wrong number of rows")
        if out is None:
            ldu = (t + 3) // 4 * 4
            out = torch.empty((self.n_cols, ldu), dtype=torch.float32, device=dev)
        u = out
        vfull = None
        if rows is not None or t % 4 != 0 or v.stride(0) % 4 != 0:
            # scatter target for a row subset / staging buffer for a V that is not 16-byte friendly
            vfull = torch.zeros((max(1, self.n_rows), u.stride(0)), dtype=torch.float32, device=dev)
        if self.n_rows == 0 or not self.tblocks:
            u[:, :t].zero_()
            return u[:, :t]
        self._first_half(f, rows, n2, v.data_ptr(), v.stride(0), u.data_ptr(), u.stride(0),
                         None if vfull is None else vfull.data_ptr(), t, self._gather_flags()[0])
        return u[:, :t]

    def apply(self, f, u, rows=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """out = Phi[rows] u: u [n_cols, t] -> [n1, t]."""
        dev = self.device
        self.build_windows()
        self.build_long_rows()
        f = self._f(f)
        u = self._rhs(u, dev)
        rows = self._ids(rows, dev)
        if u.shape[0] != self.n_cols:
            raise ValueError("rhs has the wrong number of rows")
        t = u.shape[1]
        n1 = self.n_rows if rows is None else rows.numel()
        if out is None:
            out = torch.zeros((n1, t), dtype=torch.float32, device=dev)
        elif out.shape != (n1, t) or out.dtype != torch.float32 or out.stride(1) != 1:
            raise ValueError("out must be a float32 [n1, t] tensor with unit column stride")
        phi = self.c_struct((t + 3) // 4 * 4)
        check(_lib.lib().grf_phi_matvec(
            ctypes.byref(phi), _ptr(f), _ptr(rows), n1, None, self.n_rows, None, 0, _ptr(out), out.stride(0),
            _ptr(u), u.stride(0), None, t, 2 | self._gather_flags()[1], _stream(dev)))
        return out

    def matvec(self, f, v, x1=None, x2=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """out[n1, t] = Phi[x1] (Phi[x2]^T v);  v is [n2, t] (or [n2]) on this device."""
        v = torch.as_tensor(v, device=self.device)
        squeeze = v.dim() == 1
        if squeeze:
            v = v[:, None]
        t = v.shape[1]
        ldu = (t + 3) // 4 * 4
        key = ("u", ldu)
        if key not in self._ws:
            self._ws[key] = torch.empty((self.n_cols, ldu), dtype=torch.float32, device=self.device)
        u = self.apply_t(f, v, rows=x2, out=self._ws[key])
        res = self.apply(f, u, rows=x1, out=out)
        return res[:, 0] if squeeze else res

    def plan(self, f, t: int, x1=None, x2=None, group=None, merged: bool = True, exchange=None) -> "MatvecPlan":
        """Pre-validated kernel matvec for a CG loop: one C call (two launches) per product.  ``exchange``
        (sharding.Exchange, with ``group``): the sum of the ranks' partials runs through it -- the plan writes its
        partial straight into the exchange's (peer-mapped) U."""
        return MatvecPlan(self, f, t, x1, x2, group, merged, exchange)

    def t_matvec(self, f, v, x2=None) -> torch.Tensor:
        """U = Phi[x2]^T v  ([n_cols, t]) in a fresh buffer."""
        return self.apply_t(f, v, rows=x2)

    def fgrad_half(self, rows, left, p, grad: Optional[torch.Tensor] = None) -> torch.Tensor:
        """grad[l] += sum_k <left[k, :], M_l[rows[k], :] @ p>  -- the per-length reduction.

        left [n, t], p [n_cols, t]; returns float32 [L]."""
        dev = self.device
        left = self._rhs(left, dev)
        p = self._rhs(p, dev)
        rows = self._ids(rows, dev)
        n = self.n_rows if rows is None else rows.numel()
        if left.shape[0] != n or p.shape[0] != self.n_cols or left.shape[1] != p.shape[1]:
            raise ValueError("fgrad_half: shape mismatch")
        if grad is None:
            grad = torch.zeros(self.n_steps, dtype=torch.float32, device=dev)
        phi = self.c_struct()
        check(_lib.lib().grf_phi_fgrad(ctypes.byref(phi), _ptr(rows), n, _ptr(left), left.stride(0), _ptr(p),
                                       p.stride(0), left.shape[1], _ptr(grad), _stream(dev)))
        return grad

    def fgrad(self, f, left, right, x1=None, x2=None) -> torch.Tensor:
        """d/df of sum(left * (Phi[x1] Phi[x2]^T right)): left [n1, t], right [n2, t] -> [L]."""
        left = torch.as_tensor(left, device=self.device)
        right = torch.as_tensor(right, device=self.device)
        if left.dim() == 1:
            left, right = left[:, None], right[:, None]
        p = self.apply_t(f, right, rows=x2)   # Phi[x2]^T right
        q = self.apply_t(f, left, rows=x1)    # Phi[x1]^T left
        grad = self.fgrad_half(x1, left, p)
        return self.fgrad_half(x2, right, q, grad=grad)

    # ---- construction ----------------------------------------------------
    @staticmethod
    def from_step_matrices(sm: StepMatrices, transpose: bool = True) -> "PhiBlocks":
        """float32 Phi blocks from the reference layout (values rounded like
        torch ``.float()``, graph_preprocessor.py:131-139)."""
        L = _lib.lib()
        dev = sm.device
        row_cnt = torch.empty(max(1, sm.n_rows * sm.n_steps), dtype=torch.int32, device=dev)
        check(L.grf_count_from_steps(_ptr(sm.offsets), sm.n_rows, sm.n_steps, _ptr(row_cnt), _stream(dev)))
        blk_ptr = scan_counts(row_cnt, sm.n_rows, sm.n_steps, _lib.ORDER_ROW_MAJOR, i64=True)
        total = int(blk_ptr[-1].item())
        if total >= 2 ** 31:
            raise ValueError("Phi shard exceeds 2^31 entries; shard the start nodes over more GPUs")
        blk_ptr = blk_ptr.to(torch.int32)
        entries = torch.empty((max(1, total), 2), dtype=torch.int32, device=dev)[:total]
        check(L.grf_blocks_from_steps(_ptr(sm.offsets), _ptr(sm.col), _ptr(sm.val), _ptr(blk_ptr), sm.n_rows,
                                      sm.n_steps, _ptr(entries), _stream(dev)))
        phi = PhiBlocks(blk_ptr, entries, sm.n_rows, sm.n_cols, sm.n_steps, sm.row_lo, sm.visits)
        return phi.build_transpose() if transpose else phi

    @staticmethod
    def concat_rows(parts: Sequence["PhiBlocks"]) -> "PhiBlocks":
        """Row chunks of one shard -> one PhiBlocks.  Parts that already carry their Phi^T keep it: the
        result's Phi^T is the list of those row blocks (nothing is re-sorted)."""
        if len(parts) == 1:
            return parts[0]
        ptrs, base = [], 0
        for p in parts:
            ptrs.append(p.blk_ptr[:-1].to(torch.int64) + base)
            base += p.nnz
        if base >= 2 ** 31:
            raise ValueError("Phi shard exceeds 2^31 entries; shard the start nodes over more GPUs")
        ptrs.append(torch.tensor([base], dtype=torch.int64, device=parts[0].device))
        out = PhiBlocks(torch.cat(ptrs).to(torch.int32), torch.cat([p.entries for p in parts]),
                        sum(p.n_rows for p in parts), parts[0].n_cols, parts[0].n_steps, parts[0].row_lo,
                        sum(p.visits for p in parts))
        if all(p.tblocks is not None for p in parts):
            out.tblocks, r0 = [], 0
            for p in parts:
                for tb in p.tblocks:
                    nb = TBlock(r0 + tb.r0, tb.n_rows, tb.nnz, tb.tblk_ptr, tb.tentries)
                    nb.census = tb.census
                    out.tblocks.append(nb)
                r0 += p.n_rows
        return out

    def to_scipy_steps(self):
        """float32 step matrices back on the host (tests / interchange)."""
        import scipy.sparse as sp

        ptr = self.blk_ptr.cpu().numpy().astype(np.int64)
        ent = self.entries.cpu().numpy()
        cols = (ent[:, 0] & ((1 << _lib.ENTRY_STEP_SHIFT) - 1)) if self.nnz else np.zeros(0, np.int32)
        vals = ent[:, 1].copy().view(np.float32) if self.nnz else np.zeros(0, np.float32)
        L, n = self.n_steps, self.n_rows
        mats = []
        for s in range(L):
            b = ptr[s:n * L:L] if n else np.zeros(0, np.int64)
            e = ptr[s + 1:n * L + 1:L] if n else np.zeros(0, np.int64)
            cnt = e - b
            ip = np.zeros(n + 1, dtype=np.int64)
            np.cumsum(cnt, out=ip[1:])
            idx = np.concatenate([np.arange(bb, ee) for bb, ee in zip(b, e)]) if n and ip[-1] else np.zeros(0, np.int64)
            mats.append(sp.csr_matrix((vals[idx], cols[idx], ip), shape=(n, self.n_cols)))
        return mats


def _blocks_from_staging(st: Staging, cfg: WalkConfig, n_cols: int, scale_mode: int) -> PhiBlocks:
    L = cfg.max_walk_length
    dev = st.row_cnt.device
    blk_ptr, total = scan_counts(st.row_cnt, st.n_rows, L, _lib.ORDER_ROW_MAJOR, i64=False, with_total=True)
    capacity = st.n_rows * st.stride            # one entry per staging slot at most
    pending = None
    if 0 < capacity * 8 <= _LAZY_ENTRY_BYTES:
        # small shard: allocate the bound, launch the compaction, and let the count arrive on the side
        base = _small_pinned()
        host = base[:2].view(torch.int64)
        host.copy_(total, non_blocking=True)
        arrived = torch.cuda.Event()
        arrived.record(torch.cuda.current_stream(dev))
        _keep_until_done(base, arrived)
        pending = (host, arrived, base)
        entries = torch.empty((capacity, 2), dtype=torch.int32, device=dev)
    else:
        total = int(total.item())
        if total >= 2 ** 31:
            raise ValueError("Phi shard exceeds 2^31 entries; shard the start nodes over more GPUs")
        entries = torch.empty((max(1, total), 2), dtype=torch.int32, device=dev)[:total]
    if st.stage_ent is not None:    # the walker already scaled and packed the entries
        check(_lib.lib().grf_compact_entries(_ptr(st.stage_ent), _ptr(blk_ptr), st.n_rows, L, st.stride,
                                             _ptr(entries), _stream(dev)))
    else:
        check(_lib.lib().grf_compact_blocks(_ptr(st.stage_col), _ptr(st.stage_sum), _ptr(st.row_cnt), _ptr(blk_ptr),
                                            st.n_rows, L, st.stride, cfg.walks_per_node, scale_mode, _ptr(entries),
                                            _stream(dev)))
    phi = PhiBlocks(blk_ptr, entries, st.n_rows, n_cols, L, st.row_lo)
    phi._nnz_pending = pending
    phi._col_counts = st.col_counts
    return phi


def build_phi_blocks(graph: DeviceGraph, cfg: WalkConfig, start_lo: int = 0, start_hi: Optional[int] = None,
                     scale_mode: int = _lib.SCALE_MUL_RECIP, transpose: bool = True,
                     max_stage_bytes: int = _MAX_STAGE_BYTES, block_rows: Optional[int] = None,
                     phase_hook=None) -> PhiBlocks:
    """Walker + compaction straight into the matvec layout (no float64 CSR, no host round trip).  A shard
    beyond ~T_BLOCK_ROWS rows is walked, compacted and transposed one row block at a time: the walker counts
    the Phi^T segment sizes of the block while it emits the entries, and the staging of one block is
    recycled for the next."""
    cfg.validate()
    start_hi = graph.n_nodes if start_hi is None else start_hi
    stride = _lib.lib().grf_walk_stage_stride(cfg.walks_per_node, cfg.max_walk_length)
    visits = torch.zeros(1, dtype=torch.int64, device=graph.device)
    block_rows = T_BLOCK_ROWS if block_rows is None else int(block_rows)
    n_rows = start_hi - start_lo
    n_blocks = 1 if n_rows <= block_rows + block_rows // 2 else -(-n_rows // block_rows)
    bounds = [start_lo + n_rows * b // n_blocks for b in range(n_blocks + 1)]
    parts = []
    for b in range(n_blocks):
        col_counts = None
        if transpose:   # the walker counts the Phi^T segment sizes while it emits the entries
            col_counts = torch.zeros(max(1, graph.n_nodes * cfg.max_walk_length), dtype=torch.int32,
                                     device=graph.device)
        chunks = []
        for lo, hi in _row_chunks(bounds[b], bounds[b + 1], stride, max_stage_bytes, slot_bytes=8):
            if phase_hook is not None:
                phase_hook("walk")
            st = run_walker(graph, cfg, lo, hi, visits=visits, col_counts=col_counts, entries_scale_mode=scale_mode)
            if phase_hook is not None:
                phase_hook("compact")
            chunks.append(_blocks_from_staging(st, cfg, graph.n_nodes, scale_mode))
            del st
        if phase_hook is not None:
            phase_hook("transpose")
        part = PhiBlocks.concat_rows(chunks)
        part._col_counts = col_counts
        if transpose:
            part.build_transpose(block_rows=1 << 40)      # this row block is one Phi^T block
        parts.append(part)
    phi = PhiBlocks.concat_rows(parts)
    phi.row_lo = start_lo
    phi.visits = visits  # device counter; int(phi.visits) syncs
    if phase_hook is not None:
        phase_hook("end")
    return phi


def phi_blocks_from_scipy(mats, device=None, row_lo: int = 0, transpose: bool = True) -> PhiBlocks:
    """Phi blocks from a list of scipy CSR step matrices (e.g. one of the
    reference's pickle caches, graph_preprocessor.py:141-165)."""
    dev = _device(device)
    n_rows, n_cols = mats[0].shape
    L = len(mats)
    offs, cols, vals, base = [], [], [], 0
    for m in mats:
        m = m.tocsr()
        if not m.has_sorted_indices:
            m = m.sorted_indices()
        offs.append(m.indptr[:-1].astype(np.int64) + base)
        base += m.nnz
        cols.append(m.indices.astype(np.int32))
        vals.append(m.data.astype(np.float64))
    offs.append(np.array([base], dtype=np.int64))
    # step-major offsets need one terminator per step boundary == next step's first offset: already contiguous
    sm = StepMatrices(torch.from_numpy(np.concatenate(offs)).to(dev), torch.from_numpy(np.concatenate(cols)).to(dev),
                      torch.from_numpy(np.concatenate(vals)).to(dev), n_rows, n_cols, L, row_lo)
    return PhiBlocks.from_step_matrices(sm, transpose=transpose)


def _canonical_csr(t: torch.Tensor) -> torch.Tensor:
    """``t`` with strictly increasing column indices in every row.  The union pattern, the Phi^T segments and the
    binary searches assume that; torch accepts CSR tensors with unsorted or repeated columns (its SpMM adds
    repeats), so such a tensor is coalesced -- sorted, repeats summed -- instead of multiplying wrongly.  One
    comparison pass + one sync per tensor, once per Phi."""
    col, crow = t.col_indices(), t.crow_indices()
    if col.numel() < 2:
        return t
    bad = col[1:] <= col[:-1]
    starts = crow[1:-1]                      # first entry of rows 1 .. n-1: no order across a row boundary
    starts = starts[(starts > 0) & (starts < col.numel())]
    bad[starts - 1] = False
    if not bool(bad.any()):
        return t
    # (t.to_sparse_coo() would mark the result as already coalesced: rebuild the triplets by hand)
    n_rows = t.shape[0]
    rows = torch.repeat_interleave(torch.arange(n_rows, device=col.device), crow[1:] - crow[:-1],
                                   output_size=col.numel())
    coo = torch.sparse_coo_tensor(torch.stack([rows, col.long()]), t.values(), tuple(t.shape)).coalesce()
    return coo.to_sparse_csr()


def phi_blocks_from_torch_csr(tensors, row_lo: int = 0, transpose: bool = True) -> PhiBlocks:
    """Phi blocks from one torch sparse-CSR tensor or a list of them (one per
    walk length) already on the GPU -- the layout ``from_scipy_csr`` produces
    (graph_preprocessor.py:117-139: int64 indices, float32 values)."""
    if isinstance(tensors, torch.Tensor):
        tensors = [tensors]
    dev = _device(tensors[0].device)
    n_rows, n_cols = tensors[0].shape
    offs, cols, vals, base = [], [], [], 0
    for t in tensors:
        if not t.is_sparse_csr:
            raise ValueError("Input tensor must be a sparse CSR tensor")
        t = _canonical_csr(t)
        crow = t.crow_indices().to(torch.int64)
        offs.append(crow[:-1] + base)
        base += int(t.values().numel())
        cols.append(t.col_indices().to(torch.int32))
        vals.append(t.values().to(torch.float64))
    offs.append(torch.tensor([base], dtype=torch.int64, device=dev))
    sm = StepMatrices(torch.cat(offs).contiguous(), torch.cat(cols).contiguous(), torch.cat(vals).contiguous(),
                      n_rows, n_cols, len(tensors), row_lo)
    return PhiBlocks.from_step_matrices(sm, transpose=transpose)


class MatvecPlan:
    """``out = Phi[x1] (Phi[x2]^T v)`` with everything but ``v`` / ``out`` fixed.

    A CG solve calls the kernel matvec hundreds of times with the same Phi, f,
    index sets and shapes (SURVEY.md 3.3); the plan keeps the argument block,
    the U workspace and the scatter buffer alive so that a product is a single
    ``grf_phi_matvec`` call -- or, for a row-sharded Phi (``group``), the first
    half, one all-reduce of U over NCCL, and the second half.

    ``merged=True`` (default): the products run on Phi_f materialised on the union
    pattern of the per-length matrices (``PhiBlocks.merged``), re-materialised by
    ``set_modulator``; ``merged=False`` applies f per entry on the per-length blocks."""

    def __init__(self, phi: PhiBlocks, f, t: int, x1=None, x2=None, group=None, merged: bool = True, exchange=None):
        dev = phi.device
        self.base, self.merged = phi, bool(merged)
        self.t, self.group = int(t), group
        self.exchange = exchange if group is not None else None
        if self.merged:
            phi.build_transpose()
            if len(phi.tblocks) != 1:
                self.merged = False     # a multi-block Phi^T multiplies the per-length blocks
        if self.merged:
            self.phi = phi.merged(f)
            self.f = torch.ones(1, dtype=torch.float32, device=dev)
        else:
            self.phi = phi
            self.f = phi._f(f).clone()
        self.phi.use_tiles = phi.use_tiles
        self.phi.dynamic_rows = phi.dynamic_rows
        self.phi.build_windows()
        self.phi.build_long_rows()
        phi.check_ids(x1)
        phi.check_ids(x2)
        self.x1, self.x2 = phi._ids(x1, dev), phi._ids(x2, dev)
        self.n1 = phi.n_rows if self.x1 is None else self.x1.numel()
        self.n2 = phi.n_rows if self.x2 is None else self.x2.numel()
        self.ldu = (self.t + 3) // 4 * 4
        if self.exchange is not None:
            if tuple(self.exchange.u.shape) != (max(1, phi.n_cols), self.ldu):
                raise ValueError("exchange buffer must be [n_cols, (t + 3) // 4 * 4] float32")
            self.u = self.exchange.u
        else:
            self.u = torch.empty((max(1, phi.n_cols), self.ldu), dtype=torch.float32, device=dev)
        self.vfull = (torch.zeros((max(1, phi.n_rows), self.ldu), dtype=torch.float32, device=dev)
                      if (self.x2 is not None or self.t % 4 != 0) else None)
        # no repeated ids in x2 (the usual case: a training set) -> scatter without memset / atomics
        self._flags = 8 if (self.x2 is not None and self.x2.numel() > 0
                            and int(torch.unique(self.x2).numel()) == self.x2.numel()) else 0
        self._fn = _lib.lib().grf_phi_matvec
        self._dev = dev
        # line-pair path (csrc/grf_pairs.cu): the merged product over all rows with t = 16, when no row needs the
        # long-row split and at least a fifth of the union entries find their line partner
        self._pair = None
        if (self.merged and PAIR_LAYOUT and self.t == 16 and self.x2 is None and self.phi._long_fwd is None
                and all(tb.long is None for tb in self.phi.tblocks) and phi.nnz > 0
                and phi.pair_ratio <= PAIR_MAX_RATIO):
            phi.merged(f, into=self.phi, pairs=True)
            if self.u.stride(0) == 16 and self.u.data_ptr() % 128 == 0:
                fwd, tr = phi._pairs
                pent, tpent = self.phi._pent
                self._pair = phi._pairs
                self._pair_fn = _lib.lib().grf_pairs_matvec
                self._pair_u = self.u.data_ptr()
                self._pair_args = (tr["pptr"].data_ptr(), tpent.data_ptr(), fwd["pptr"].data_ptr(), pent.data_ptr(),
                                   None if self.x1 is None else self.x1.data_ptr(), self.n1, self.phi.row_lo,
                                   self.phi.n_rows, self.phi.n_cols)
        self._single = len(self.phi.tblocks) == 1
        self._c = self.phi.c_struct(self.ldu)                                   # all rows (+ the only Phi^T block)
        self._cb = [self.phi.c_struct(self.ldu, block=b) for b in range(len(self.phi.tblocks))]
        self._gt, self._gf = self.phi._gather_flags()
        self._shared = self._shared_buf = None
        if group is not None and self.exchange is None:
            # exchange only the columns that more than one row shard touches (sharding.shared_columns)
            from . import sharding

            if phi.shared_hint is not None:
                self._shared = None if isinstance(phi.shared_hint, str) else phi.shared_hint
            else:
                touched = self.phi._touched
                if touched is None:     # most columns touched: a plain all-reduce follows
                    touched = torch.ones(phi.n_cols, dtype=torch.int32, device=dev)
                self._shared = sharding.shared_columns(touched, None if group is True else group)
            if self._shared is not None and self._shared.numel():
                self._shared_buf = torch.empty((self._shared.numel(), self.ldu), dtype=torch.float32, device=dev)

    def set_modulator(self, f) -> None:
        if self.merged:
            self.base.merged(f, into=self.phi, pairs=self._pair is not None)
        else:
            self.f.copy_(torch.as_tensor(f, device=self._dev).detach().to(torch.float32).reshape(-1))

    def _tune_gathers(self):
        """(Phi^T V, Phi U): does gathering with L1::no_allocate loads beat the cached loads on this Phi?
        Measured once per Phi with CUDA events on a random right-hand side (3 products each way)."""
        dev = self._dev
        v = torch.randn((max(1, self.n2), self.t), dtype=torch.float32, device=dev)
        out = torch.empty((max(1, self.n1), self.t), dtype=torch.float32, device=dev)
        best = []
        for half in (1, 2):
            ms = []
            for flag in (0, 32):
                self._gt = self._gf = flag
                self._call(v, out, half)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(torch.cuda.current_stream(dev))
                for _ in range(3):
                    self._call(v, out, half)
                b.record(torch.cuda.current_stream(dev))
                b.synchronize()
                ms.append(a.elapsed_time(b))
            best.append(ms[1] < 0.97 * ms[0])
        return tuple(best)

    def _call_pairs(self, v, out, which) -> bool:
        """The halves of the product on the line-pair entries (one C call); False when an operand is not laid out
        for it (a misaligned view of V, an output with an odd leading dimension)."""
        if which & 1 and (v.stride(0) != 16 or v.data_ptr() % 128):
            return False
        if which & 2 and (out.stride(0) % 4 or out.data_ptr() % 16):
            return False
        rc = self._pair_fn(*self._pair_args, None if v is None else v.data_ptr(), self._pair_u,
                           None if out is None else out.data_ptr(), 0 if out is None else out.stride(0), which,
                           _stream(self._dev))
        if rc:
            check(rc)
        return True

    def _call(self, v, out, which):
        if self._pair is not None and self._call_pairs(v, out, which):
            return
        st = _stream(self._dev)
        if which == 3 and self._single and self._gt == self._gf:
            rc = self._fn(ctypes.byref(self._c), _ptr(self.f), _ptr(self.x1), self.n1, _ptr(self.x2), self.n2,
                          ctypes.c_void_p(v.data_ptr()), v.stride(0), ctypes.c_void_p(out.data_ptr()), out.stride(0),
                          _ptr(self.u), self.ldu, _ptr(self.vfull), self.t, 3 | self._flags | self._gt, st)
            if rc:
                check(rc)
            return
        if which & 1:
            self.phi._first_half(self.f, self.x2, self.n2, v.data_ptr(), v.stride(0), self.u.data_ptr(), self.ldu,
                                 None if self.vfull is None else self.vfull.data_ptr(), self.t,
                                 self._flags | self._gt, structs=self._cb)
        if which & 2:
            rc = self._fn(ctypes.byref(self._c), _ptr(self.f), _ptr(self.x1), self.n1, None, self.phi.n_rows, None, 0,
                          ctypes.c_void_p(out.data_ptr()), out.stride(0), _ptr(self.u), self.ldu, None, self.t,
                          2 | self._gf, st)
            if rc:
                check(rc)

    def __call__(self, v: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """v: float32 [n2, t] with unit column stride; out: float32 [n1, t] (allocated if None)."""
        if v.dtype != torch.float32 or v.dim() != 2 or v.shape[0] != self.n2 or v.shape[1] != self.t \
                or (v.stride(1) != 1 and v.shape[1] != 1) or (v.shape[0] > 1 and v.stride(0) < self.t):
            raise ValueError("plan: v must be float32 [n2, t] with unit column stride")
        if out is None:
            out = torch.zeros((self.n1, self.t), dtype=torch.float32, device=self._dev)
        if self.group is None:
            self._call(v, out, 3)
        else:
            from . import sharding

            self._call(v, None, 1)
            if self.exchange is not None:
                self.exchange.reduce(_stream(self._dev))
            else:
                sharding.reduce_shared(self.u, self._shared, self._shared_buf,
                                       None if self.group is True else self.group)
            self._call(None, out, 2)
        return out
