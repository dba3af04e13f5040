"""ctypes front-end of ``oracle/grf_oracle_weighted.c``: alias tables and step matrices of weight-proportional
neighbour draws (TEST INFRASTRUCTURE ONLY).  Uniform draws stay with :mod:`oracle.c_oracle`."""

from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import scipy.sparse as sp

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libgrf_oracle_weighted.so")
_lib = None

# GrfAliasEdge of include/grf_b200.h as a numpy record
ALIAS_DTYPE = np.dtype([("scaled", "<f8"), ("scaled_alias", "<f8"), ("col", "<i4"), ("col_alias", "<i4"),
                        ("thr", "<u4"), ("pad", "<i4")])


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("grf_oracle_weighted.c", "grf_oracle.c")]
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
        vp = ctypes.c_void_p
        _lib.grf_oracle_build_weighted.restype = vp
        _lib.grf_oracle_build_weighted.argtypes = [
            ctypes.c_int64, vp, vp, vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
            ctypes.c_double, ctypes.c_int32, ctypes.c_uint64, ctypes.c_int32,
        ]
        _lib.grf_oracle_alias_records.restype = None
        _lib.grf_oracle_alias_records.argtypes = [ctypes.c_int64, vp, vp, vp, ctypes.c_double, vp]
        _lib.grf_oracle_alias_masses.restype = ctypes.c_double
        _lib.grf_oracle_alias_masses.argtypes = [ctypes.c_int32, vp, vp]
        _lib.grf_oracle_alias_edge_bytes.restype = ctypes.c_int32
        _lib.grf_oracle_alias_edge_bytes.argtypes = []
        _lib.grf_oracle_nnz.restype = ctypes.c_int64
        _lib.grf_oracle_nnz.argtypes = [vp, ctypes.c_int32]
        _lib.grf_oracle_visits.restype = ctypes.c_int64
        _lib.grf_oracle_visits.argtypes = [vp]
        _lib.grf_oracle_copy.restype = None
        _lib.grf_oracle_copy.argtypes = [vp, ctypes.c_int32] + [vp] * 3
        _lib.grf_oracle_free.restype = None
        _lib.grf_oracle_free.argtypes = [vp]
    return _lib


def _csr(adj_csr):
    a = adj_csr.tocsr()
    return (a.shape[0], np.ascontiguousarray(a.indptr, dtype=np.int32),
            np.ascontiguousarray(a.indices, dtype=np.int32), np.ascontiguousarray(a.data, dtype=np.float64))


def masses(weights):
    """(S, m) of one row: the float64 sum of |w| and the uint64 masses with the deficit applied."""
    w = np.ascontiguousarray(weights, dtype=np.float64)
    m = np.zeros(max(1, w.size), dtype=np.uint64)
    s = lib().grf_oracle_alias_masses(w.size, w.ctypes.data, m.ctypes.data)
    return s, m[: w.size]


def alias_records(adj_csr, p_halt):
    """GrfAliasEdge records of every row (numpy structured array [nnz], ALIAS_DTYPE)."""
    n, indptr, indices, data = _csr(adj_csr)
    out = np.zeros(max(1, data.size), dtype=ALIAS_DTYPE)
    lib().grf_oracle_alias_records(n, indptr.ctypes.data, indices.ctypes.data, data.ctypes.data, float(p_halt),
                                   out.ctypes.data)
    return out[: data.size]


def step_matrices(adj_csr, num_walks, p_halt, max_walk_length, antithetic=False, seed=42, scale_mode=0,
                  start_lo=0, start_hi=None, return_visits=False):
    """Step matrices M_l[start_lo:start_hi, :] of weight-proportional Philox draws as scipy CSR (float64, int32,
    sorted columns), same conventions as ``c_oracle.step_matrices`` (cumulative load rule)."""
    n, indptr, indices, data = _csr(adj_csr)
    start_hi = n if start_hi is None else start_hi
    L = max_walk_length
    h = lib().grf_oracle_build_weighted(
        n, indptr.ctypes.data, indices.ctypes.data, data.ctypes.data, start_lo, start_hi, num_walks, L,
        float(p_halt), int(bool(antithetic)), int(seed), scale_mode,
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
