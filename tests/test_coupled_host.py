"""Coupled walk draws without a GPU: argument checks of the C ABI and the Python layer, the cache name of
GraphPreprocessor, and the coupled modes of the C oracle (the definitions at GrfWalkCfg.seed in
include/grf_b200.h) -- exact consequences on rings and complete graphs, and unbiasedness of every M_l."""

import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

from grf_b200 import _lib
from grf_b200.engine import COUPLINGS, WalkConfig
from gpu_util import random_graph, ring_graph
from oracle import c_oracle, c_oracle_coupled

HALT, NEIGH = c_oracle_coupled.COUPLE_HALT, c_oracle_coupled.COUPLE_NEIGHBOURS


def oracle_steps(adj, W, p, L, coupling=0, **kw):
    """Step matrices from the C oracle: independent draws (c_oracle) or coupled ones (c_oracle_coupled)."""
    if coupling:
        return c_oracle_coupled.step_matrices(adj, W, p, L, coupling, **kw)
    return c_oracle.step_matrices(adj, W, p, L, **kw)


MODES = [0, HALT, NEIGH, HALT | NEIGH]


@pytest.fixture(scope="module")
def lib():
    _lib.build()
    return _lib.lib()


def _walk(lib, draw_mode):
    g = _lib.GrfGraph(4, 8, None, None, None)
    c = _lib.GrfWalkCfg(0, 4, 5, 3, 0.1, draw_mode, 0, 42, None, None)
    return lib.grf_walk(ctypes.byref(g), ctypes.byref(c), 401, None, None, None, None, None)


def test_flag_values_agree_between_header_binding_and_oracle():
    assert (_lib.DRAW_COUPLE_HALT, _lib.DRAW_COUPLE_NEIGHBOURS) == (HALT, NEIGH) == (2, 4)
    assert COUPLINGS == {"iid": 0, "antithetic": 2, "repelling": 4, "antithetic+repelling": 6}


@pytest.mark.parametrize("flags", [HALT, NEIGH, HALT | NEIGH])
def test_replay_with_coupling_is_an_argument_error(lib, flags):
    rc = _walk(lib, _lib.DRAW_REPLAY | flags)
    assert rc == _lib.GRF_ERR_INVALID
    with pytest.raises(ValueError, match="coupled draws need native Philox draws"):
        _lib.check(rc)


@pytest.mark.parametrize("draw_mode", [8, 16 | HALT, 1 << 30, -1])
def test_unknown_draw_bits_are_an_argument_error(lib, draw_mode):
    rc = _walk(lib, draw_mode)
    assert rc == _lib.GRF_ERR_INVALID
    with pytest.raises(ValueError, match="bad draw_mode"):
        _lib.check(rc)


def test_walk_config_validation():
    for name, bits in COUPLINGS.items():
        cfg = WalkConfig(8, 0.1, 3, coupling=name)
        cfg.validate()
        assert cfg.draw_flags() == bits
    assert WalkConfig(8, 0.1, 3).coupling == "iid" and WalkConfig(8, 0.1, 3).draw_flags() == _lib.DRAW_PHILOX
    with pytest.raises(ValueError, match="coupling must be one of"):
        WalkConfig(8, 0.1, 3, coupling="quasi").validate()
    with pytest.raises(ValueError, match="coupling must be one of"):
        WalkConfig(8, 0.1, 3, coupling="repelling+antithetic").validate()
    trace = (np.zeros(1), np.zeros(1, dtype=np.int32))
    for name in ("antithetic", "repelling", "antithetic+repelling"):
        with pytest.raises(ValueError, match="native Philox"):
            WalkConfig(8, 0.1, 3, draw_mode=_lib.DRAW_REPLAY, trace=trace, coupling=name).validate()
        with pytest.raises(ValueError, match="native Philox"):
            WalkConfig(8, 0.1, 3, trace=trace, coupling=name).validate()
    WalkConfig(8, 0.1, 3, draw_mode=_lib.DRAW_REPLAY, trace=trace).validate()   # iid replay stays valid


def test_cache_filename_is_the_reference_one_for_iid_and_distinct_otherwise():
    import hashlib

    from efficient_graph_gp_sparse.preprocessor.graph_preprocessor import GraphPreprocessor

    adj = random_graph(30, 60, 2)
    h = hashlib.md5(adj.data.tobytes() + adj.indices.tobytes() + adj.indptr.tobytes()).hexdigest()[:8]
    reference = f"experiments_sparse/step_matrices/step_matrices_{h}_30_10_0.5_10_42.pkl"
    assert GraphPreprocessor(adj).cache_filename == reference
    assert GraphPreprocessor(adj, coupling="iid").cache_filename == reference
    names = {GraphPreprocessor(adj, coupling=c).cache_filename for c in COUPLINGS}
    assert len(names) == len(COUPLINGS)
    for c in COUPLINGS:
        if c != "iid":
            assert GraphPreprocessor(adj, coupling=c).cache_filename.endswith(f"_{c}.pkl")


# ------------------------------------------------------------------ oracle: exact consequences
@pytest.mark.parametrize("flags", [HALT, HALT | NEIGH])
def test_antithetic_halting_at_one_half_halts_exactly_one_walk_of_each_pair(flags):
    """p = 1/2, even W, L = 2, ring (no dead ends): of every pair exactly one walk takes the single step, so
    the walk-steps are n*W (length 0) + n*W/2 (length 1) for every seed."""
    n, W = 40, 10
    ring = ring_graph(n)
    for seed in range(5):
        _, visits = oracle_steps(ring, W, 0.5, 2, seed=seed, coupling=flags, return_visits=True)
        assert visits == n * W + n * W // 2
    _, visits = oracle_steps(ring, W, 0.5, 2, seed=0, return_visits=True)
    assert visits != n * W + n * W // 2        # independent halting draws do not have this property


@pytest.mark.parametrize("flags", [NEIGH, HALT | NEIGH])
def test_repelling_walks_fewer_than_the_degree_take_distinct_neighbours(flags):
    """K_12 (deg 11), W = 8, p = 0: the 8 walks of each start node take 8 distinct first steps."""
    n = 12
    k12 = sp.csr_matrix(np.ones((n, n)) - np.eye(n))
    for seed in range(4):
        m1 = oracle_steps(k12, 8, 0.0, 2, seed=seed, coupling=flags)[1]
        assert np.array_equal(np.diff(m1.indptr), np.full(n, 8))
    m1 = oracle_steps(k12, 8, 0.0, 2, seed=0)[1]
    assert (np.diff(m1.indptr) < 8).any()       # independent draws collide


def test_repelling_walks_more_than_the_degree_spread_evenly():
    """Ring (deg 2, load factor 2 at p = 0), W = 7: each row of M_1 holds 3 and 4 walks' worth, 6/7 and 8/7."""
    n, W = 33, 7
    for seed in range(4):
        m1 = oracle_steps(ring_graph(n), W, 0.0, 2, seed=seed, coupling=NEIGH)[1]
        assert np.array_equal(np.diff(m1.indptr), np.full(n, 2))
        vals = np.sort(m1.data.reshape(n, 2), axis=1)
        assert np.array_equal(vals[:, 0], np.full(n, 6.0 * (1.0 / W)))
        assert np.array_equal(vals[:, 1], np.full(n, 8.0 * (1.0 / W)))


def test_coupled_oracle_needs_coupling_bits():
    g = random_graph(20, 40, 4)
    for bad in (0, 8, HALT | 16):
        with pytest.raises(ValueError, match="coupling"):
            c_oracle_coupled.step_matrices(g, 4, 0.2, 3, bad)


# ------------------------------------------------------------------ oracle: unbiasedness
@pytest.mark.parametrize("flags", MODES, ids=["iid", "antithetic", "repelling", "antithetic+repelling"])
def test_every_coupled_mode_is_unbiased(flags):
    """Mean of M_l over 400 seeds == A^l (A: the weighted walk graph) within 5 standard errors per entry,
    the standard errors estimated from the same seeds; W = 5 leaves one walk unpaired."""
    a = random_graph(12, 30, 6, weighted=True)
    W, p, L, seeds = 5, 0.3, 4, 400
    runs = np.stack([np.stack([m.toarray() for m in oracle_steps(a, W, p, L, seed=s, coupling=flags)])
                     for s in range(seeds)])
    mean, se = runs.mean(0), runs.std(0, ddof=1) / np.sqrt(seeds)
    ad = a.toarray()
    for l in range(L):
        exact = np.linalg.matrix_power(ad, l)
        z = np.abs(mean[l] - exact)
        assert (z <= 5 * se[l] + 1e-12).all(), (l, float((z / np.maximum(se[l], 1e-300)).max()))
        assert (se[l][exact > 0] > 0).all() or l == 0     # every reachable entry was sampled
