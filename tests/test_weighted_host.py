"""Weight-proportional neighbour draws without a GPU: argument checks of the C ABI and the Python layer, the cache
name of GraphPreprocessor, and the weighted C oracle (the definitions at GrfAliasEdge in include/grf_b200.h) --
exact alias tables, bit-identity with uniform draws on +-1 weights, and unbiasedness of every M_l."""

import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

from grf_b200 import _lib
from grf_b200.engine import NEIGHBOUR_SAMPLINGS, WalkConfig
from gpu_util import csr_bits_equal, powerlaw_graph, random_graph, ring_graph
from oracle import c_oracle, c_oracle_coupled, c_oracle_weighted

T = 1 << 32
FAKE = 0x1000   # a non-NULL pointer the argument checks never dereference


@pytest.fixture(scope="module")
def lib():
    _lib.build()
    return _lib.lib()


def _walk_weighted(lib, draw_mode=_lib.DRAW_PHILOX, load_mode=_lib.LOAD_CUMULATIVE, edges=None, alias=FAKE, L=3,
                   p=0.1, nnz=8):
    g = _lib.GrfGraph(4, nnz, FAKE, FAKE, FAKE)
    c = _lib.GrfWalkCfg(0, 4, 5, L, p, draw_mode, load_mode, 42, None, None, edges)
    c.scale_mode = _lib.SCALE_MUL_RECIP
    return lib.grf_walk_weighted(ctypes.byref(g), ctypes.byref(c), alias, 401, FAKE, FAKE, FAKE, None, None)


@pytest.mark.parametrize("kw, match", [
    ({"draw_mode": _lib.DRAW_REPLAY}, "draw_mode"),
    ({"draw_mode": _lib.DRAW_COUPLE_NEIGHBOURS}, "draw_mode"),
    ({"draw_mode": _lib.DRAW_COUPLE_HALT | _lib.DRAW_COUPLE_NEIGHBOURS}, "draw_mode"),
    ({"load_mode": _lib.LOAD_LAST_STEP}, "load_mode"),
    ({"load_mode": _lib.LOAD_ABLATION}, "load_mode"),
    ({"edges": FAKE}, "edges"),
    ({"alias": None}, "null alias"),
], ids=["replay", "repelling", "antithetic+repelling", "last-step", "ablation", "edges", "no-alias"])
def test_weighted_walk_argument_errors(lib, kw, match):
    rc = _walk_weighted(lib, **kw)
    assert rc == _lib.GRF_ERR_INVALID
    with pytest.raises(ValueError, match=match):
        _lib.check(rc)


def test_shared_validation_names_the_weighted_entry_point(lib):
    g = _lib.GrfGraph(4, 8, FAKE, FAKE, FAKE)
    c = _lib.GrfWalkCfg(0, 4, 5, 3, 0.1, _lib.DRAW_PHILOX, _lib.LOAD_CUMULATIVE, 42, None, None, None)
    rc = lib.grf_walk_weighted(ctypes.byref(g), ctypes.byref(c), FAKE, 3, FAKE, FAKE, FAKE, None, None)
    with pytest.raises(ValueError, match=r"^grf_walk_weighted: stage_stride too small"):
        _lib.check(rc)
    rc = lib.grf_walk(ctypes.byref(g), ctypes.byref(c), 3, FAKE, FAKE, FAKE, None, None)
    with pytest.raises(ValueError, match=r"^grf_walk: stage_stride too small"):
        _lib.check(rc)


def test_alias_records_argument_errors(lib):
    g = _lib.GrfGraph(4, 8, FAKE, FAKE, FAKE)
    for p in (-0.1, 1.5):
        with pytest.raises(ValueError, match="p_halt"):
            _lib.check(lib.grf_alias_records(ctypes.byref(g), p, FAKE, None))
    with pytest.raises(ValueError, match="null"):
        _lib.check(lib.grf_alias_records(ctypes.byref(g), 0.1, None, None))
    assert lib.grf_alias_records(ctypes.byref(_lib.GrfGraph(4, 0, FAKE, None, None)), 0.1, None, None) == 0


def test_walk_config_validation():
    assert NEIGHBOUR_SAMPLINGS == ("uniform", "weighted")
    assert WalkConfig(8, 0.1, 3).neighbour_sampling == "uniform"
    for coupling in ("iid", "antithetic"):
        WalkConfig(8, 0.1, 3, coupling=coupling, neighbour_sampling="weighted").validate()
    with pytest.raises(ValueError, match="neighbour_sampling must be one of"):
        WalkConfig(8, 0.1, 3, neighbour_sampling="importance").validate()
    for coupling in ("repelling", "antithetic+repelling"):
        with pytest.raises(ValueError, match="repelling"):
            WalkConfig(8, 0.1, 3, coupling=coupling, neighbour_sampling="weighted").validate()
    trace = (np.zeros(1), np.zeros(1, dtype=np.int32))
    with pytest.raises(ValueError, match="native Philox"):
        WalkConfig(8, 0.1, 3, draw_mode=_lib.DRAW_REPLAY, trace=trace, neighbour_sampling="weighted").validate()
    for load_mode in (_lib.LOAD_LAST_STEP, _lib.LOAD_ABLATION):
        with pytest.raises(ValueError, match="cumulative"):
            WalkConfig(8, 0.1, 3, load_mode=load_mode, neighbour_sampling="weighted").validate()


def test_cache_filename_is_the_reference_one_for_uniform_and_suffixed_for_weighted():
    import hashlib

    from efficient_graph_gp_sparse.preprocessor.graph_preprocessor import GraphPreprocessor

    adj = random_graph(30, 60, 2)
    h = hashlib.md5(adj.data.tobytes() + adj.indices.tobytes() + adj.indptr.tobytes()).hexdigest()[:8]
    reference = f"experiments_sparse/step_matrices/step_matrices_{h}_30_10_0.5_10_42.pkl"
    assert GraphPreprocessor(adj, neighbour_sampling="uniform").cache_filename == reference
    assert GraphPreprocessor(adj, neighbour_sampling="weighted").cache_filename == reference[:-4] + "_weighted.pkl"
    both = GraphPreprocessor(adj, coupling="antithetic", neighbour_sampling="weighted").cache_filename
    assert both == reference[:-4] + "_antithetic_weighted.pkl"


def test_alias_edge_is_one_sector_by_gcc(tmp_path):
    src = tmp_path / "size.c"
    src.write_text('#include "grf_b200.h"\n#include <stddef.h>\n'
                   "_Static_assert(sizeof(GrfAliasEdge) == 32, \"size\");\n"
                   "_Static_assert(offsetof(GrfAliasEdge, scaled_alias) == 8, \"scaled_alias\");\n"
                   "_Static_assert(offsetof(GrfAliasEdge, col) == 16, \"col\");\n"
                   "_Static_assert(offsetof(GrfAliasEdge, thr) == 24, \"thr\");\n"
                   "int main(void) { return 0; }\n")
    subprocess.check_call(["gcc", "-fsyntax-only", "-I", _lib.INCLUDE, str(src)])
    assert c_oracle_weighted.lib().grf_oracle_alias_edge_bytes() == 32
    assert c_oracle_weighted.ALIAS_DTYPE.itemsize == 32


# ------------------------------------------------------------------ alias tables: exact
def _reconstructed_masses(rec, start, d):
    """Probability mass (in units of 1 / (d 2^32)) of every entry of one row, read back from its buckets."""
    got = np.zeros(d, dtype=object)
    idx = {}
    for k in range(d):
        idx.setdefault(int(rec["col"][start + k]), k)
    for k in range(d):
        r = rec[start + k]
        if int(r["thr"]) == 0xFFFFFFFF:
            assert int(r["col_alias"]) == int(r["col"]) and r["scaled_alias"] == r["scaled"]   # full: itself
            got[k] += T
        else:
            got[k] += int(r["thr"])
            got[idx[int(r["col_alias"])]] += T - int(r["thr"])
    return got


def _row_graph(weights):
    d = len(weights)
    return sp.csr_matrix((np.asarray(weights, dtype=np.float64), np.arange(d), np.array([0, d])), shape=(1, d))


ROWS = {
    "negative": [0.5, -2.0, 0.25, 1.0, -0.125],
    "explicit-zeros": [0.0, 3.0, 0.0, 0.0, 1.0, 0.0, 2.0],
    "single": [-1.5],
    "laplacian-hub": [1.0] + [-1.0 / np.sqrt(1000.0 * (2 + i % 7)) for i in range(999)],
    "1e5": list(np.random.default_rng(5).standard_normal(100_000) * np.exp(np.random.default_rng(6).standard_normal(100_000) * 3)),
}


@pytest.mark.parametrize("name", list(ROWS))
def test_alias_table_reproduces_the_masses_exactly(name):
    w = np.asarray(ROWS[name])
    d = w.size
    s, m = c_oracle_weighted.masses(w)
    assert sum(int(x) for x in m) == d * T
    assert s == pytest.approx(np.abs(w).sum(), rel=1e-12)
    assert all(int(m[k]) == 0 for k in range(d) if w[k] == 0.0)        # w = 0 is never taken
    rec = c_oracle_weighted.alias_records(_row_graph(w), 0.2)
    got = _reconstructed_masses(rec, 0, d)
    assert all(int(got[k]) == int(m[k]) for k in range(d))
    q = s / (1.0 - 0.2)
    assert np.array_equal(rec["scaled"], np.where(w < 0, -q, q))
    # the probabilities are |w| / S to within d / 2^32 per entry
    assert np.abs(m.astype(np.float64) / (d * float(T)) - np.abs(w) / np.abs(w).sum()).max() <= 2.0 / T


def test_equal_weights_give_full_buckets_and_a_zero_row_is_a_dead_end():
    rec = c_oracle_weighted.alias_records(_row_graph([-0.3] * 7), 0.1)
    assert (rec["thr"] == 0xFFFFFFFF).all() and np.array_equal(rec["col_alias"], rec["col"])
    rec = c_oracle_weighted.alias_records(_row_graph([0.0, -0.0, 0.0]), 0.1)
    assert (rec["thr"] == 0xFFFFFFFF).all() and (rec["scaled"] == 0.0).all() and (rec["scaled_alias"] == 0.0).all()


# ------------------------------------------------------------------ oracle: exact consequences
def _pm1(adj, seed):
    a = adj.tocsr().astype(np.float64)
    a.data = np.where(np.random.default_rng(seed).random(a.nnz) < 0.5, -1.0, 1.0)
    return a


@pytest.mark.parametrize("graph", ["ring", "random", "powerlaw"])
def test_weighted_oracle_equals_uniform_oracle_on_pm1_weights(graph):
    adj = {"ring": lambda: ring_graph(37), "random": lambda: random_graph(60, 200, 3),
           "powerlaw": lambda: powerlaw_graph(200, 800, 4)}[graph]()
    a = _pm1(adj, 9)
    for W, p, L, seed in ((16, 0.2, 5, 7), (5, 0.5, 4, 11)):
        want = c_oracle.step_matrices(a, W, p, L, seed=seed)
        got = c_oracle_weighted.step_matrices(a, W, p, L, seed=seed)
        assert all(csr_bits_equal(x, y) for x, y in zip(want, got))
        want = c_oracle_coupled.step_matrices(a, W, p, L, c_oracle_coupled.COUPLE_HALT, seed=seed)
        got = c_oracle_weighted.step_matrices(a, W, p, L, antithetic=True, seed=seed)
        assert all(csr_bits_equal(x, y) for x, y in zip(want, got))


def test_weighted_loads_are_bounded_by_the_row_sums():
    """|load factor| = S / (1 - p) <= (1 + sqrt(deg)) / (1 - p) on the normalized Laplacian."""
    from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian

    lap = get_normalized_laplacian(powerlaw_graph(300, 1500, 2))
    rec = c_oracle_weighted.alias_records(lap, 0.1)
    deg = np.repeat(np.diff(lap.indptr), np.diff(lap.indptr))
    assert (np.abs(rec["scaled"]) <= (1 + np.sqrt(deg)) / 0.9 * (1 + 1e-12)).all()


# ------------------------------------------------------------------ oracle: unbiasedness
def _hub_laplacian():
    """Normalized Laplacian of a 12-node graph with two hubs, an isolated node and a row of explicit zeros."""
    from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian

    n = 12
    e = [(0, j) for j in range(1, 9)] + [(1, j) for j in range(5, 10)] + [(3, 4), (6, 7), (9, 10)]
    i, j = np.array(e).T
    adj = sp.csr_matrix((np.ones(2 * len(e)), (np.r_[i, j], np.r_[j, i])), shape=(n, n))
    c = get_normalized_laplacian(adj).tocoo()
    keep = (c.data != 0) & (c.row != 11)
    # node 11 is isolated: its row holds two explicit zeros; row 3 holds one beside its weights
    i = np.r_[c.row[keep], 11, 11, 3]
    j = np.r_[c.col[keep], 2, 11, 8]
    v = np.r_[c.data[keep], 0.0, -0.0, 0.0]
    lap = sp.csr_matrix((v, (i, j)), shape=(n, n))
    lap.sort_indices()
    return lap


@pytest.mark.parametrize("antithetic", [False, True], ids=["weighted", "weighted+antithetic"])
def test_weighted_draws_are_unbiased(antithetic):
    """Mean of M_l over 400 seeds == L^l within 5 standard errors per entry (L: the hub Laplacian, negative
    off-diagonals, a zero row); W = 15 leaves one walk unpaired.  (At length 3 some entries of this graph are
    reached with probability ~5e-4 per walk: too rare to estimate their standard error from 400 seeds.)"""
    a = _hub_laplacian()
    assert a.nnz > np.count_nonzero(a.toarray())          # explicit zeros are stored
    W, p, L, seeds = 15, 0.3, 3, 400
    runs = np.stack([np.stack([m.toarray() for m in c_oracle_weighted.step_matrices(a, W, p, L, antithetic, seed=s)])
                     for s in range(seeds)])
    mean, se = runs.mean(0), runs.std(0, ddof=1) / np.sqrt(seeds)
    ad = a.toarray()
    for l in range(L):
        exact = np.linalg.matrix_power(ad, l)
        z = np.abs(mean[l] - exact)
        assert (z <= 5 * se[l] + 1e-12).all(), (l, float((z / np.maximum(se[l], 1e-300)).max()))
        assert (se[l][exact != 0] > 0).all() or l == 0
