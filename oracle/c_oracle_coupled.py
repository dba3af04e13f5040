"""ctypes front-end of ``oracle/grf_oracle_coupled.c``: step matrices of coupled walk draws
(TEST INFRASTRUCTURE ONLY).  Independent draws stay with :mod:`oracle.c_oracle`."""

from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import scipy.sparse as sp

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libgrf_oracle_coupled.so")
_lib = None

COUPLE_HALT, COUPLE_NEIGHBOURS = 2, 4   # GRF_DRAW_COUPLE_* of include/grf_b200.h


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("grf_oracle_coupled.c", "grf_oracle.c")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call(
            ["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", _SO, srcs[0], "-lm"]
        )
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_SO)
        _lib.grf_oracle_build_coupled.restype = ctypes.c_void_p
        _lib.grf_oracle_build_coupled.argtypes = [
            ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
            ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_double,
            ctypes.c_int32, ctypes.c_uint64, ctypes.c_int32, ctypes.c_int32,
        ]
        _lib.grf_oracle_nnz.restype = ctypes.c_int64
        _lib.grf_oracle_nnz.argtypes = [ctypes.c_void_p, ctypes.c_int32]
        _lib.grf_oracle_visits.restype = ctypes.c_int64
        _lib.grf_oracle_visits.argtypes = [ctypes.c_void_p]
        _lib.grf_oracle_copy.restype = None
        _lib.grf_oracle_copy.argtypes = [ctypes.c_void_p, ctypes.c_int32] + [ctypes.c_void_p] * 3
        _lib.grf_oracle_free.restype = None
        _lib.grf_oracle_free.argtypes = [ctypes.c_void_p]
    return _lib


def step_matrices(adj_csr, num_walks, p_halt, max_walk_length, coupling, seed=42, load_mode=0, scale_mode=0,
                  start_lo=0, start_hi=None, return_visits=False):
    """Step matrices M_l[start_lo:start_hi, :] of coupled Philox draws as scipy CSR (float64, int32, sorted
    columns), same conventions as ``c_oracle.step_matrices``.  ``coupling``: COUPLE_HALT | COUPLE_NEIGHBOURS
    bits, at least one."""
    if not coupling or coupling & ~(COUPLE_HALT | COUPLE_NEIGHBOURS):
        raise ValueError("coupling must be a non-empty combination of COUPLE_HALT and COUPLE_NEIGHBOURS")
    a = adj_csr.tocsr()
    n = a.shape[0]
    start_hi = n if start_hi is None else start_hi
    indptr = np.ascontiguousarray(a.indptr, dtype=np.int32)
    indices = np.ascontiguousarray(a.indices, dtype=np.int32)
    data = np.ascontiguousarray(a.data, dtype=np.float64)
    L = max_walk_length
    h = lib().grf_oracle_build_coupled(
        n, indptr.ctypes.data, indices.ctypes.data, data.ctypes.data, start_lo, start_hi, num_walks, L,
        float(p_halt), int(coupling), int(seed), load_mode, scale_mode,
    )
    try:
        mats = []
        n_local = start_hi - start_lo
        for s in range(L):
            nnz = lib().grf_oracle_nnz(h, s)
            ip = np.zeros(n_local + 1, dtype=np.int64)
            ix = np.zeros(nnz, dtype=np.int32)
            dv = np.zeros(nnz, dtype=np.float64)
            lib().grf_oracle_copy(h, s, ip.ctypes.data, ix.ctypes.data, dv.ctypes.data)
            mats.append(sp.csr_matrix((dv, ix, ip), shape=(n_local, n)))
        visits = lib().grf_oracle_visits(h)
    finally:
        lib().grf_oracle_free(h)
    return (mats, visits) if return_visits else mats
