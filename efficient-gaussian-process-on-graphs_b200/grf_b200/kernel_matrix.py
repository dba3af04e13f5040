"""The sparse kernel matrix K = Phi_f Phi_f^T on the device (csrc/grf_kernel_matrix.cu).

Replaces the host half of the reference's sparse ``fast_general_grf_kernel``
(graph_kernels_sparse/fast_grf_kernel_general.py:48-55): ``Phi += f_p * M_p`` by scipy additions and
``Phi @ Phi.T`` by scipy's single-threaded SpGEMM.  The device result equals scipy's in all three CSR
arrays, element for element (the rules are in include/grf_b200.h and the header of the .cu file).
"""

from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from ._lib import check
from .engine import _free_bytes, _ptr, _stream, scan_counts

_INT32_MAX = np.iinfo(np.int32).max
MAX_STEPS = 128        # modulator values merged per row of Phi_f (min(len(f), L))
GLOBAL_CTAS = 2 * 148  # CTAs of the hub-row bin (each owns one hash table in global memory)


def modulator_f64(f, n_steps: int) -> np.ndarray:
    """The f_p the reference's loop uses (p < min(len(f), L)), widened to float64 as numpy promotes
    ``f_p * M_p.data``.  The whole iterable is consumed, as the reference's ``enumerate`` does."""
    out = []
    for p, f_p in enumerate(f):
        if p >= n_steps:
            continue
        a = np.asarray(f_p)
        if a.ndim != 0 or a.dtype.kind not in "biuf" or np.result_type(np.float64, a.dtype) != np.float64:
            raise TypeError(f"modulator value {p} ({f_p!r}) does not widen to float64")
        out.append(np.float64(a))
    return np.asarray(out, dtype=np.float64)


def kernel_index_dtype(n: int, touched: int, stored: int):
    """Index dtype of scipy's ``Phi @ Phi.T`` (csr_matrix).  ``_matmul_sparse`` computes in int64 when the
    touched count (csr_matmat_maxnnz) or an input index array needs it, but the csr_matrix it returns is built
    with ``check_contents=True``: the arrays are narrowed back to int32 whenever N and the stored count fit.
    With nothing touched it returns ``csr_matrix((N, N))``, whose dtype depends on N alone."""
    if touched == 0:
        return np.int64 if n > _INT32_MAX else np.int32
    return np.int64 if max(n, stored) > _INT32_MAX else np.int32


@dataclass
class KernelMatrix:
    """K = Phi_f Phi_f^T in HBM: indptr int64 [n + 1], indices int32, data float64, rows in scipy's order."""

    indptr: torch.Tensor
    indices: torch.Tensor
    data: torch.Tensor
    n: int
    touched: int        # sum over rows of the distinct j touched (scipy's csr_matmat_maxnnz)
    nnz_phi: int        # stored entries of Phi_f

    @property
    def nnz(self) -> int:
        return int(self.data.numel())

    def to_scipy(self):
        """The scipy csr_matrix ``Phi @ Phi.T`` returns: same arrays and dtypes.  One device-to-host copy per
        array into pinned memory."""
        import scipy.sparse as sp

        if self.touched == 0:
            return sp.csr_matrix((self.n, self.n))
        idx = kernel_index_dtype(self.n, self.touched, self.nnz)
        ip = self.indptr.to(torch.int32) if idx == np.int32 else self.indptr

        def fetch(t):
            host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            host.copy_(t, non_blocking=True)
            return host

        ip_h, col_h, val_h = fetch(ip), fetch(self.indices), fetch(self.data)
        torch.cuda.current_stream(self.data.device).synchronize()
        col = col_h.numpy() if idx == np.int32 else col_h.numpy().astype(np.int64)
        return sp.csr_matrix((val_h.numpy(), col, ip_h.numpy()), shape=(self.n, self.n))


def _bins(size: torch.Tensor, n: int, dev) -> tuple:
    rows = torch.empty(max(1, 3 * n), dtype=torch.int32, device=dev)
    stats = torch.empty(4, dtype=torch.int64, device=dev)
    check(_lib.lib().grf_kmat_bin(_ptr(size), n, _ptr(rows), _ptr(stats), _stream(dev)))
    return rows, [int(x) for x in stats.cpu().tolist()]


def _workspace(stats, dev, budget: int, what: str):
    n_global, max_size = stats[2], int(stats[3])
    if n_global == 0:
        return None, 0, 0
    L = _lib.lib()
    ctas = min(GLOBAL_CTAS, n_global)
    per = L.grf_kmat_workspace_bytes(max_size, 1)
    if per > budget:
        raise MemoryError(f"kernel matrix {what}: a hash table for a row touching up to {max_size} columns needs "
                          f"{per} bytes, {budget} bytes of device memory are free")
    ctas = max(1, min(ctas, budget // (4 * per)))
    nbytes = L.grf_kmat_workspace_bytes(max_size, ctas)
    return torch.empty(nbytes, dtype=torch.uint8, device=dev), ctas, nbytes


def kernel_matrix(steps, f, events: Optional[Dict[str, torch.cuda.Event]] = None,
                  mem_limit: Optional[int] = None) -> KernelMatrix:
    """K = Phi_f Phi_f^T of ``steps`` (a StepMatrices), Phi_f = sum_p f_p M_p over p < min(len(f), L).

    ``events``: CUDA events recorded at the stage boundaries (keys "start", "phi", "transpose", "count",
    "fill").  ``mem_limit``: bytes K may take instead of the free device memory.  Raises MemoryError, naming
    nnz(K), before allocating K when it does not fit."""
    L = _lib.lib()
    dev = steps.device
    n, n_cols, n_steps = int(steps.n_rows), int(steps.n_cols), int(steps.n_steps)
    fv = modulator_f64(f, n_steps)
    n_f = int(fv.size)
    if n_f > MAX_STEPS:
        raise ValueError(f"kernel_matrix merges at most {MAX_STEPS} modulator values, got {n_f}")

    def mark(name):
        if events is not None:
            events[name] = torch.cuda.Event(enable_timing=True)
            events[name].record(torch.cuda.current_stream(dev))

    with torch.cuda.device(dev):
        st = _stream(dev)
        mark("start")
        fd = torch.from_numpy(fv).to(dev) if n_f else None
        # Phi_f
        cnt = torch.empty(max(1, n), dtype=torch.int32, device=dev)
        args = (_ptr(steps.offsets), _ptr(steps.col), _ptr(steps.val), n, n_steps, _ptr(fd), n_f, 0)
        check(L.grf_kmat_phi_count(*args, _ptr(cnt), st))
        phi_ptr = scan_counts(cnt, n, 1, _lib.ORDER_ROW_MAJOR, i64=True)
        nnz_phi = int(phi_ptr[-1].item()) if n else 0
        phi_col = torch.empty(max(1, nnz_phi), dtype=torch.int32, device=dev)
        phi_val = torch.empty(max(1, nnz_phi), dtype=torch.float64, device=dev)
        check(L.grf_kmat_phi_fill(*args, _ptr(phi_ptr), _ptr(phi_col), _ptr(phi_val), st))
        mark("phi")
        # Phi_f^T
        tcnt = torch.empty(max(1, n_cols), dtype=torch.int32, device=dev)
        check(L.grf_kmat_transpose_count(_ptr(phi_ptr), _ptr(phi_col), n, n_cols, _ptr(tcnt), st))
        tptr = scan_counts(tcnt, n_cols, 1, _lib.ORDER_ROW_MAJOR, i64=True)
        cursor = torch.empty(max(1, n_cols), dtype=torch.int64, device=dev)
        trow = torch.empty(max(1, nnz_phi), dtype=torch.int32, device=dev)
        tval = torch.empty(max(1, nnz_phi), dtype=torch.float64, device=dev)
        check(L.grf_kmat_transpose_fill(_ptr(phi_ptr), _ptr(phi_col), _ptr(phi_val), n, n_cols, _ptr(tptr),
                                        _ptr(cursor), _ptr(trow), _ptr(tval), st))
        del cursor, tcnt
        mark("transpose")
        ops = (_ptr(phi_ptr), _ptr(phi_col), _ptr(phi_val), _ptr(tptr), _ptr(trow), _ptr(tval), n)
        overflow = torch.empty(1, dtype=torch.int32, device=dev)
        budget = _free_bytes(dev) if mem_limit is None else int(mem_limit)
        # count: sizes = products per row (capped at n)
        size = torch.empty(max(1, n), dtype=torch.int32, device=dev)
        check(L.grf_kmat_row_sizes(_ptr(phi_ptr), _ptr(phi_col), _ptr(tptr), n, _ptr(size), st))
        rows, stats = _bins(size, n, dev)
        ws, ctas, wsb = _workspace(stats, dev, budget, "count")
        touched = torch.empty(max(1, n), dtype=torch.int32, device=dev)
        stored = torch.empty(max(1, n), dtype=torch.int32, device=dev)
        bin_rows = (ctypes.c_int64 * 3)(*stats[:3])
        check(L.grf_kmat_count(*ops, _ptr(size), _ptr(rows), bin_rows, stats[3], ctas, _ptr(ws), wsb, _ptr(touched),
                               _ptr(stored), _ptr(overflow), st))
        del ws
        kptr = scan_counts(stored, n, 1, _lib.ORDER_ROW_MAJOR, i64=True)
        n_touched = int(touched[:n].sum(dtype=torch.int64).item()) if n else 0
        nnz_k = int(kptr[-1].item()) if n else 0
        if int(overflow.item()):
            raise RuntimeError("grf_kmat_count: a row touched more columns than its size bound")
        mark("count")
        need = nnz_k * 12
        if need > budget:
            raise MemoryError(f"K = Phi_f Phi_f^T has nnz(K) = {nnz_k} stored entries ({need} bytes of indices and "
                              f"values); {budget} bytes of device memory are free")
        # fill: sizes = touched (exact), re-binned
        rows, stats = _bins(touched, n, dev)
        ws, ctas, wsb = _workspace(stats, dev, budget - need, "fill")
        kcol = torch.empty(max(1, nnz_k), dtype=torch.int32, device=dev)
        kval = torch.empty(max(1, nnz_k), dtype=torch.float64, device=dev)
        bin_rows = (ctypes.c_int64 * 3)(*stats[:3])
        check(L.grf_kmat_fill(*ops, _ptr(touched), _ptr(rows), bin_rows, stats[3], ctas, _ptr(ws), wsb, _ptr(kptr),
                              _ptr(kcol), _ptr(kval), _ptr(overflow), st))
        mark("fill")
        if int(overflow.item()):
            raise RuntimeError("grf_kmat_fill: a row outgrew its table or disagrees with the counted row pointers")
    if n == 0:
        kptr = torch.zeros(1, dtype=torch.int64, device=dev)
    return KernelMatrix(kptr, kcol[:nnz_k], kval[:nnz_k], n, n_touched, nnz_phi)
