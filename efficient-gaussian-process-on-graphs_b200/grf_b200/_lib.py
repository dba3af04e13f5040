"""ctypes binding of ``libgrf_b200.so`` (the C ABI declared in include/grf_b200.h)."""

from __future__ import annotations

import ctypes
import os
import subprocess
import sys
from ctypes import POINTER, Structure, c_double, c_float, c_int32, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
PKG_ROOT = os.path.dirname(_HERE)
REPO_ROOT = os.path.dirname(PKG_ROOT)
CSRC = os.path.join(PKG_ROOT, "csrc")
INCLUDE = os.path.join(REPO_ROOT, "include")
SO_PATH = os.environ.get("GRF_B200_SO") or os.path.join(_HERE, "libgrf_b200.so")   # override: tuning experiments

GRF_OK, GRF_ERR_INVALID, GRF_ERR_CUDA, GRF_ERR_UNSUPPORTED = 0, -1, -2, -3
DRAW_PHILOX, DRAW_REPLAY = 0, 1
DRAW_COUPLE_HALT, DRAW_COUPLE_NEIGHBOURS = 2, 4   # OR-ed into draw_mode with DRAW_PHILOX
LOAD_CUMULATIVE, LOAD_LAST_STEP, LOAD_ABLATION = 0, 1, 2
SCALE_MUL_RECIP, SCALE_DIV = 0, 1
ORDER_ROW_MAJOR, ORDER_STEP_MAJOR = 0, 1
ENTRY_STEP_SHIFT = 27  # GRF_ENTRY_STEP_SHIFT
ABI_VERSION = 8        # GRF_B200_ABI_VERSION

# every symbol include/grf_b200.h declares (tests/test_abi.py checks the header against this)
EXPORTS = (
    "grf_abi_version", "grf_last_error", "grf_walk_stage_stride", "grf_walk", "grf_scan_workspace_bytes",
    "grf_scan_counts", "grf_compact_steps", "grf_compact_blocks", "grf_blocks_from_steps", "grf_count_from_steps",
    "grf_row_census", "grf_long_rows_build", "grf_nonempty_rows", "grf_transpose_workspace_bytes", "grf_transpose_offsets", "grf_transpose_fill",
    "grf_phi_matvec", "grf_phi_fgrad", "grf_phi_row_dots", "grf_block_windows", "grf_edge_records", "grf_compact_entries", "grf_union_rank", "grf_union_fill",
    "grf_union_materialize", "grf_pairs_count", "grf_pairs_index", "grf_pairs_fill", "grf_pairs_spmm", "grf_pairs_matvec", "grf_cg_num_partials", "grf_cg_dot", "grf_cg_update", "grf_cg_direction",
    "grf_laplacian_count", "grf_laplacian_fill", "grf_shard_reach", "grf_exchange_flag_bytes", "grf_exchange_sum", "grf_exchange_sum_nvls",
    "grf_kmat_phi_count", "grf_kmat_phi_fill", "grf_kmat_transpose_count", "grf_kmat_transpose_fill", "grf_kmat_row_sizes",
    "grf_kmat_bin", "grf_kmat_workspace_bytes", "grf_kmat_count", "grf_kmat_fill",
)


class GrfGraph(Structure):
    _fields_ = [("n_nodes", c_int64), ("nnz", c_int64), ("row_ptr", c_void_p), ("col_idx", c_void_p),
                ("val", c_void_p)]


class GrfWalkCfg(Structure):
    _fields_ = [("start_lo", c_int64), ("start_hi", c_int64), ("walks_per_node", c_int32),
                ("max_walk_length", c_int32), ("p_halt", c_double), ("draw_mode", c_int32), ("load_mode", c_int32),
                ("seed", c_uint64), ("trace_u", c_void_p), ("trace_k", c_void_p), ("edges", c_void_p),
                ("col_counts", c_void_p), ("trace_walk_base", c_int64), ("stage_entries", c_void_p),
                ("scale_mode", c_int32)]


class GrfLongRows(Structure):
    _fields_ = [("threshold", c_int32), ("n_long", c_int32), ("n_chunks", c_int32), ("rows", c_void_p),
                ("chunk_ptr", c_void_p), ("chunk_bounds", c_void_p), ("partial", c_void_p), ("ld", c_int64),
                ("chunk_order", c_void_p)]


class GrfPhi(Structure):
    _fields_ = [("n_rows", c_int64), ("n_cols", c_int64), ("row_lo", c_int64), ("n_steps", c_int32),
                ("blk_ptr", c_void_p), ("entries", c_void_p), ("tblk_ptr", c_void_p), ("tentries", c_void_p),
                ("win", c_void_p), ("twin", c_void_p), ("win_max_width", c_int32), ("twin_max_width", c_int32),
                ("long_fwd", POINTER(GrfLongRows)), ("long_t", POINTER(GrfLongRows)),
                ("tcols", c_void_p), ("n_tcols", c_int64), ("nnz", c_int64), ("sched", c_void_p)]


def nvcc_command(out_path: str = SO_PATH):
    srcs = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))
    return ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
            "-Xcompiler", "-fPIC", "-shared", "-I", INCLUDE, "-I", CSRC, "-o", out_path] + srcs


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into libgrf_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "grf_b200.h")]
    newest = max(os.path.getmtime(s) for s in srcs)
    if force or not os.path.exists(SO_PATH) or os.path.getmtime(SO_PATH) < newest:
        cmd = nvcc_command()
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.check_call(cmd)
    return SO_PATH


_lib = None


def lib():
    """The loaded library.  Missing library => loud failure (no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"grf_b200: {SO_PATH} is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    L = ctypes.CDLL(SO_PATH)
    vp, i32, i64 = c_void_p, c_int32, c_int64
    L.grf_abi_version.restype = c_int32
    L.grf_abi_version.argtypes = []
    L.grf_last_error.restype = ctypes.c_char_p
    L.grf_last_error.argtypes = []
    L.grf_walk_stage_stride.restype = i64
    L.grf_walk_stage_stride.argtypes = [i32, i32]
    L.grf_walk.restype = i32
    L.grf_walk.argtypes = [POINTER(GrfGraph), POINTER(GrfWalkCfg), i64, vp, vp, vp, vp, vp]
    L.grf_scan_workspace_bytes.restype = i64
    L.grf_scan_workspace_bytes.argtypes = [i64]
    L.grf_scan_counts.restype = i32
    L.grf_scan_counts.argtypes = [vp, i64, i32, i32, vp, i32, vp, vp]
    L.grf_compact_steps.restype = i32
    L.grf_compact_steps.argtypes = [vp, vp, vp, vp, i64, i32, i64, i32, i32, vp, vp, vp]
    L.grf_compact_blocks.restype = i32
    L.grf_compact_blocks.argtypes = [vp, vp, vp, vp, i64, i32, i64, i32, i32, vp, vp]
    L.grf_blocks_from_steps.restype = i32
    L.grf_blocks_from_steps.argtypes = [vp, vp, vp, vp, i64, i32, vp, vp]
    L.grf_count_from_steps.restype = i32
    L.grf_count_from_steps.argtypes = [vp, i64, i32, vp, vp]
    L.grf_row_census.restype = i32
    L.grf_row_census.argtypes = [vp, i64, i32, i32, vp, vp]
    L.grf_shard_reach.restype = i32
    L.grf_shard_reach.argtypes = [POINTER(GrfGraph), vp, i32, i32, vp, vp, vp]
    L.grf_nonempty_rows.restype = i32
    L.grf_nonempty_rows.argtypes = [vp, i64, i32, vp, vp, vp, vp, vp]
    L.grf_transpose_workspace_bytes.restype = i64
    L.grf_transpose_workspace_bytes.argtypes = [i64, i32, i64]
    L.grf_transpose_offsets.restype = i32
    L.grf_transpose_offsets.argtypes = [vp, vp, i64, i64, i32, vp, vp, vp, i32, vp, vp]
    L.grf_transpose_fill.restype = i32
    L.grf_transpose_fill.argtypes = [vp, vp, i64, i64, i32, i64, i64, vp, vp, vp]
    L.grf_phi_matvec.restype = i32
    L.grf_phi_matvec.argtypes = [POINTER(GrfPhi), vp, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp, i32, i32, vp]
    L.grf_union_rank.restype = i32
    L.grf_union_rank.argtypes = [vp, vp, i32, vp, vp, vp, i64, vp, vp, vp, vp]
    L.grf_union_fill.restype = i32
    L.grf_union_fill.argtypes = [vp, vp, i32, vp, vp, vp, i64, vp, vp, vp, vp]
    L.grf_long_rows_build.restype = i32
    L.grf_long_rows_build.argtypes = [vp, vp, i64, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    L.grf_pairs_count.restype = i32
    L.grf_pairs_count.argtypes = [vp, vp, i64, vp, vp]
    L.grf_pairs_index.restype = i32
    L.grf_pairs_index.argtypes = [vp, vp, i64, vp, vp, vp]
    L.grf_pairs_fill.restype = i32
    L.grf_pairs_fill.argtypes = [vp, vp, i64, i64, vp, vp]
    L.grf_pairs_spmm.restype = i32
    L.grf_pairs_spmm.argtypes = [vp, vp, vp, i64, i64, i64, vp, i64, vp, i64, vp]
    L.grf_pairs_matvec.restype = i32
    L.grf_pairs_matvec.argtypes = [vp, vp, vp, vp, vp, i64, i64, i64, i64, vp, vp, vp, i64, i32, vp]
    L.grf_union_materialize.restype = i32
    L.grf_union_materialize.argtypes = [vp, vp, i64, vp, vp, vp, i32, vp, vp]
    L.grf_cg_num_partials.restype = i32
    L.grf_cg_num_partials.argtypes = [i64, i32]
    L.grf_cg_dot.restype = i32
    L.grf_cg_dot.argtypes = [vp, i64, vp, i64, c_float, i64, i32, vp, vp]
    L.grf_cg_update.restype = i32
    L.grf_cg_update.argtypes = [vp, i64, vp, i64, vp, i64, vp, i64, vp, vp, i64, i32, c_float, vp, vp]
    L.grf_cg_direction.restype = i32
    L.grf_cg_direction.argtypes = [vp, i64, vp, i64, vp, vp, i64, i32, c_float, vp, vp]
    L.grf_laplacian_count.restype = i32
    L.grf_laplacian_count.argtypes = [POINTER(GrfGraph), vp, vp, vp, vp]
    L.grf_laplacian_fill.restype = i32
    L.grf_laplacian_fill.argtypes = [POINTER(GrfGraph), vp, vp, vp, vp, vp, vp]
    L.grf_edge_records.restype = i32
    L.grf_edge_records.argtypes = [POINTER(GrfGraph), c_double, vp, vp]
    L.grf_compact_entries.restype = i32
    L.grf_compact_entries.argtypes = [vp, vp, i64, i32, i64, vp, vp]
    L.grf_exchange_flag_bytes.restype = i64
    L.grf_exchange_flag_bytes.argtypes = [i32]
    L.grf_exchange_sum.restype = i32
    L.grf_exchange_sum.argtypes = [POINTER(vp), POINTER(vp), i32, i32, i64, ctypes.c_uint32, vp]
    L.grf_exchange_sum_nvls.restype = i32
    L.grf_exchange_sum_nvls.argtypes = [vp, POINTER(vp), i32, i32, i64, ctypes.c_uint32, vp]
    L.grf_block_windows.restype = i32
    L.grf_block_windows.argtypes = [vp, vp, i64, i32, vp, vp, vp]
    L.grf_phi_fgrad.restype = i32
    L.grf_phi_fgrad.argtypes = [POINTER(GrfPhi), vp, i64, vp, i64, vp, i64, i32, vp, vp]
    L.grf_phi_row_dots.restype = i32
    L.grf_phi_row_dots.argtypes = [POINTER(GrfPhi), vp, vp, vp, i64, vp, vp]
    L.grf_kmat_phi_count.restype = i32
    L.grf_kmat_phi_count.argtypes = [vp, vp, vp, i64, i32, vp, i32, i32, vp, vp]
    L.grf_kmat_phi_fill.restype = i32
    L.grf_kmat_phi_fill.argtypes = [vp, vp, vp, i64, i32, vp, i32, i32, vp, vp, vp, vp]
    L.grf_kmat_transpose_count.restype = i32
    L.grf_kmat_transpose_count.argtypes = [vp, vp, i64, i64, vp, vp]
    L.grf_kmat_transpose_fill.restype = i32
    L.grf_kmat_transpose_fill.argtypes = [vp, vp, vp, i64, i64, vp, vp, vp, vp, vp]
    L.grf_kmat_row_sizes.restype = i32
    L.grf_kmat_row_sizes.argtypes = [vp, vp, vp, i64, vp, vp]
    L.grf_kmat_bin.restype = i32
    L.grf_kmat_bin.argtypes = [vp, i64, vp, vp, vp]
    L.grf_kmat_workspace_bytes.restype = i64
    L.grf_kmat_workspace_bytes.argtypes = [i32, i32]
    L.grf_kmat_count.restype = i32
    L.grf_kmat_count.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp, vp, POINTER(c_int64), i32, i32, vp, i64, vp, vp, vp,
                                 vp]
    L.grf_kmat_fill.restype = i32
    L.grf_kmat_fill.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp, vp, POINTER(c_int64), i32, i32, vp, i64, vp, vp, vp,
                                vp, vp]
    if L.grf_abi_version() != ABI_VERSION:
        raise RuntimeError("grf_b200: ABI version mismatch between _lib.py and libgrf_b200.so")
    _lib = L
    return _lib


def check(rc: int) -> None:
    """0 -> ok; invalid argument -> ValueError (as the reference raises); else RuntimeError."""
    if rc == GRF_OK:
        return
    msg = lib().grf_last_error().decode("utf-8", "replace")
    if rc == GRF_ERR_INVALID:
        raise ValueError(msg)
    raise RuntimeError(f"grf_b200 error {rc}: {msg}")
