"""-m gpu tests of weight-proportional neighbour draws (WalkConfig.neighbour_sampling = "weighted";
grf_alias_records / grf_walk_weighted, definitions at GrfAliasEdge in include/grf_b200.h): alias tables and walks
bit-exact against the C oracle in every launch shape, bit-identity with uniform draws on +-1 weights, row shards,
the error they remove on a power-law Laplacian, and the GP layer on a weighted Phi."""

import numpy as np
import pytest
import scipy.sparse as sp

from gpu_util import csr_bits_equal, grid_graph, random_graph, ring_graph

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import torch

    assert torch.cuda.is_available(), "these tests need a B200"
    from grf_b200 import _lib, engine
    from oracle import c_oracle, c_oracle_weighted, grf_oracle

    return dict(torch=torch, lib=_lib, eng=engine, cu=c_oracle, cw=c_oracle_weighted, o=grf_oracle)


def _signed(adj, seed, zeros=0.0):
    """Random magnitudes over three decades, random signs, a fraction `zeros` of explicit zeros."""
    a = adj.tocsr().astype(np.float64)
    rng = np.random.default_rng(seed)
    a.data = np.exp(rng.uniform(-3.5, 3.5, a.nnz)) * np.where(rng.random(a.nnz) < 0.3, -1.0, 1.0)
    a.data[rng.random(a.nnz) < zeros] = 0.0
    a.sort_indices()
    return a


def _records_equal(got, want):
    got = got.cpu().numpy().view(np.uint64).reshape(-1, 4)[: want.size]
    return np.array_equal(got, want.view(np.uint64).reshape(-1, 4))


def _case(env, graph, W, p, L, seed, antithetic=False, scale_mode=0, start_lo=0, start_hi=None):
    eng, cw = env["eng"], env["cw"]
    g = eng.DeviceGraph.from_scipy(graph)
    cfg = eng.WalkConfig(W, p, L, seed=seed, coupling="antithetic" if antithetic else "iid",
                         neighbour_sampling="weighted")
    got = eng.build_step_matrices(g, cfg, start_lo, start_hi, scale_mode=scale_mode)
    want, visits = cw.step_matrices(graph, W, p, L, antithetic, seed=seed, scale_mode=scale_mode,
                                    start_lo=start_lo, start_hi=start_hi, return_visits=True)
    mats = got.to_scipy()
    for s in range(L):
        assert csr_bits_equal(mats[s], want[s]), (W, L, s)
    assert got.visits == visits
    return g, cfg, want


def _phi_bits_equal(phi, want):
    got = phi.to_scipy_steps()
    for s, w in enumerate(want):
        w32 = w.astype(np.float32)
        assert np.array_equal(got[s].indptr, w32.indptr) and np.array_equal(got[s].indices, w32.indices), s
        assert np.array_equal(got[s].data.view(np.int32), w32.data.view(np.int32)), s


# ------------------------------------------------------------------ alias tables
def _star(leaves):
    i = np.zeros(leaves, dtype=np.int64)
    j = np.arange(1, leaves + 1)
    return sp.csr_matrix((np.ones(2 * leaves), (np.r_[i, j], np.r_[j, i])), shape=(leaves + 1, leaves + 1))


def test_alias_records_bit_exact_star_with_1e5_leaves(env):
    """The hub row (120 001 entries) takes the CTA path, the leaves the warp path; Laplacian and signed weights."""
    from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian

    eng, cw = env["eng"], env["cw"]
    for a in (get_normalized_laplacian(_star(120_000)), _signed(_star(120_000), 4, zeros=0.01)):
        g = eng.DeviceGraph.from_scipy(a)
        for p in (0.1, 0.5):
            assert _records_equal(g.alias_records(p), cw.alias_records(a, p))


def test_alias_records_bit_exact_rmat_and_edge_cases(env):
    from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian

    eng, cw = env["eng"], env["cw"]
    graphs = [get_normalized_laplacian(_rmat(16, 1_100_000)), _signed(random_graph(3000, 40_000, 2), 5, zeros=0.1)]
    # rows of one entry, all-zero rows, equal weights, a single huge weight among tiny ones, lengths around 2048
    rows = [[-2.0], [0.0, 0.0], [0.5] * 3000, [1e-9] * 2500 + [1e6], list(np.linspace(-1, 1, 2048)),
            list(np.linspace(-1, 2, 2049)), [0.0] * 5000]
    n = len(rows)
    ip = np.r_[0, np.cumsum([len(r) for r in rows])]
    cols = np.concatenate([np.arange(len(r)) % n for r in rows])
    graphs.append(sp.csr_matrix((np.concatenate(rows), cols, ip), shape=(n, n)))
    for a in graphs:
        g = eng.DeviceGraph.from_scipy(a)
        assert _records_equal(g.alias_records(0.2), cw.alias_records(a, 0.2))


def test_non_finite_weights_are_rejected(env):
    eng = env["eng"]
    for bad in (np.nan, np.inf, -np.inf):
        a = _signed(random_graph(50, 120, 1), 2)
        a.data[7] = bad
        g = eng.DeviceGraph.from_scipy(a)
        with pytest.raises(ValueError, match="finite"):
            g.alias_records(0.1)
        with pytest.raises(ValueError, match="finite"):
            eng.build_step_matrices(g, eng.WalkConfig(4, 0.1, 3, neighbour_sampling="weighted"))


def test_finite_weights_whose_graph_total_overflows_are_accepted(env):
    """Each row sum of |w| is finite; only the sum over the whole graph overflows."""
    eng, cw = env["eng"], env["cw"]
    a = sp.csr_matrix((np.array([1e308, -1e308, 1e308, 0.5]), np.array([1, 0, 3, 2]), np.array([0, 1, 2, 3, 4])),
                      shape=(4, 4))
    g = eng.DeviceGraph.from_scipy(a)
    assert _records_equal(g.alias_records(0.1), cw.alias_records(a, 0.1))


def test_edge_and_alias_records_are_cached_side_by_side(env):
    eng = env["eng"]
    g = eng.DeviceGraph.from_scipy(_signed(random_graph(200, 800, 3), 1))
    alias, edges = g.alias_records(0.1), g.edge_records(0.1)
    assert g.alias_records(0.1) is alias and g.edge_records(0.1) is edges
    for s in ("uniform", "weighted", "uniform"):
        eng.build_step_matrices(g, eng.WalkConfig(8, 0.1, 3, neighbour_sampling=s))
    assert g.alias_records(0.1) is alias and g.edge_records(0.1) is edges


# ------------------------------------------------------------------ walks: bit-exact in every launch shape
# W <= 32 / 64 / 128 / 256: warp per start node (1 / 2 / 4 / 8 keys per lane, 4 / 2 / 1 start nodes per CTA as
# the visit records allow: W = 200, L = 30 holds 68 KB); W = 300: CTA per start node with every length;
# W = 2100, L = 10 and W = 8192, L = 5: one length at a time.
SHAPES = [(1, 4), (5, 6), (31, 5), (33, 4), (100, 5), (130, 10), (200, 30), (256, 5), (300, 4), (2100, 10),
          (8192, 5)]


@pytest.mark.parametrize("antithetic", [False, True], ids=["weighted", "weighted+antithetic"])
@pytest.mark.parametrize("W,L", SHAPES)
@pytest.mark.parametrize("wide", ["0", "1"])
def test_bit_exact_every_launch_shape(env, monkeypatch, antithetic, W, L, wide):
    monkeypatch.setenv("GRF_B200_WALK_WIDE", wide)      # forces the wide / narrow warp forms
    lap = env["o"].normalized_laplacian_sparse(random_graph(60, 150, 11, weighted=True))
    a = _signed(lap, 3, zeros=0.05)
    g, cfg, want = _case(env, a, W, 0.2, L, 5, antithetic)
    _phi_bits_equal(env["eng"].build_phi_blocks(g, cfg), want)


@pytest.mark.parametrize("antithetic", [False, True], ids=["weighted", "weighted+antithetic"])
@pytest.mark.parametrize("W", [100, 300])
def test_bit_exact_64bit_keys_on_a_row_slice_of_a_huge_ring(env, antithetic, W):
    """2^25-node ring with random weights (node bits + walk bits > 31: 64-bit sort keys), a slice of start nodes."""
    n = 1 << 25
    ring = _signed(ring_graph(n), 6)
    lo, hi = n - 300, n - 44
    g, cfg, want = _case(env, ring, W, 0.1, 4, 1, antithetic, start_lo=lo, start_hi=hi)
    _phi_bits_equal(env["eng"].build_phi_blocks(g, cfg, lo, hi), want)


@pytest.mark.parametrize("antithetic", [False, True], ids=["weighted", "weighted+antithetic"])
def test_finished_entries_both_scale_modes_and_the_matvec(env, antithetic):
    eng, cw, o, torch = env["eng"], env["cw"], env["o"], env["torch"]
    lap = o.normalized_laplacian_sparse(grid_graph(30, 20))
    g = eng.DeviceGraph.from_scipy(lap)
    cfg = eng.WalkConfig(50, 0.1, 4, seed=42, coupling="antithetic" if antithetic else "iid",
                         neighbour_sampling="weighted")
    for scale_mode in (0, 1):
        want = cw.step_matrices(lap, 50, 0.1, 4, antithetic, seed=42, scale_mode=scale_mode)
        _case(env, lap, 50, 0.1, 4, 42, antithetic, scale_mode=scale_mode)
        phi = eng.build_phi_blocks(g, cfg, scale_mode=scale_mode)
        _phi_bits_equal(phi, want)
    rng = np.random.default_rng(0)
    f = rng.standard_normal(4).astype(np.float32)
    v = rng.standard_normal((600, 16)).astype(np.float32)
    out = phi.matvec(torch.tensor(f), torch.tensor(v).cuda()).cpu().numpy()
    ref = o.phi_matvec_f64(phi.to_scipy_steps(), f, v)
    assert np.max(np.abs(out - ref)) / np.max(np.abs(ref)) < 2e-5


def test_no_step_needs_no_alias_records(env):
    """L = 1, p = 1 and an edgeless graph: the walker takes no step and is called without records."""
    a = _signed(random_graph(40, 100, 7), 1)
    _case(env, a, 16, 0.2, 1, 3)
    _case(env, a, 16, 1.0, 4, 3)
    _case(env, sp.csr_matrix((40, 40)), 16, 0.2, 4, 3)


@pytest.mark.parametrize("W,L", [(5, 6), (100, 5), (200, 30), (300, 4), (2100, 10)])
def test_weighted_phi_equals_uniform_phi_on_pm1_weights(env, W, L):
    eng = env["eng"]
    a = random_graph(300, 1200, 12).astype(np.float64)
    a.data = np.where(np.random.default_rng(2).random(a.nnz) < 0.4, -1.0, 1.0)
    g = eng.DeviceGraph.from_scipy(a)
    for coupling in ("iid", "antithetic"):
        uni = eng.build_phi_blocks(g, eng.WalkConfig(W, 0.15, L, seed=8, coupling=coupling)).to_scipy_steps()
        wgt = eng.build_phi_blocks(g, eng.WalkConfig(W, 0.15, L, seed=8, coupling=coupling,
                                                     neighbour_sampling="weighted")).to_scipy_steps()
        for x, y in zip(uni, wgt):
            assert np.array_equal(x.indptr, y.indptr) and np.array_equal(x.indices, y.indices)
            assert np.array_equal(x.data.view(np.int32), y.data.view(np.int32))


def _rmat(scale, m, seed=0, a=0.57, b=0.19, c=0.19):
    """R-MAT (0.57, 0.19, 0.19, 0.05), symmetrised, de-duplicated, no self-loops, unit weights."""
    rng = np.random.default_rng(seed)
    n = 1 << scale
    src = np.zeros(m, dtype=np.int64)
    dst = np.zeros(m, dtype=np.int64)
    for bit in range(scale):
        r = rng.random(m)
        src |= (r >= a + b).astype(np.int64) << bit
        dst |= (((r >= a) & (r < a + b)) | (r >= a + b + c)).astype(np.int64) << bit
    keep = src != dst
    lo, hi = np.minimum(src[keep], dst[keep]), np.maximum(src[keep], dst[keep])
    key = np.unique(lo * n + hi)
    lo, hi = key // n, key % n
    return sp.csr_matrix((np.ones(2 * key.size), (np.r_[lo, hi], np.r_[hi, lo])), shape=(n, n))


def test_rmat_in_miniature_hubs_and_isolated_nodes(env):
    """Config 4 in miniature (65 k nodes, ~1 M edges, hubs, isolated nodes), W = 100, L = 5."""
    from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian

    lap = get_normalized_laplacian(_rmat(16, 1_100_000))
    for antithetic in (False, True):
        _case(env, lap, 100, 0.1, 5, 42, antithetic)


def test_row_shard_built_alone_equals_its_rows_of_the_whole_phi(env):
    eng = env["eng"]
    g = eng.DeviceGraph.laplacian_of(random_graph(500, 1500, 8))
    for coupling in ("iid", "antithetic"):
        cfg = eng.WalkConfig(100, 0.1, 5, seed=21, coupling=coupling, neighbour_sampling="weighted")
        full = eng.build_phi_blocks(g, cfg).to_scipy_steps()
        for lo, hi in ((0, 123), (123, 388), (388, 500)):
            part = eng.build_phi_blocks(g, cfg, lo, hi).to_scipy_steps()
            for s in range(5):
                a, b = part[s], full[s][lo:hi]
                assert np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
                assert np.array_equal(a.data.view(np.int32), b.data.view(np.int32))


def test_pilot_row_cost_follows_the_sampling(env):
    from grf_b200 import sharding

    eng = env["eng"]
    g = eng.DeviceGraph.laplacian_of(_rmat(12, 40_000))
    uni = sharding.pilot_row_cost(g, eng.WalkConfig(100, 0.1, 5))
    wgt = sharding.pilot_row_cost(g, eng.WalkConfig(100, 0.1, 5, neighbour_sampling="weighted"))
    assert not env["torch"].equal(uni, wgt)
    assert abs(float(wgt.sum()) - 1.0) < 1e-9


def test_weighted_draws_lower_the_kernel_error_on_a_power_law_laplacian(env):
    """Relative Frobenius error of K = Phi Phi^T against the exact series (L = 5, f_l = 2^-l, p = 0.1, W = 100) on
    the normalized Laplacian of a 4096-node R-MAT graph, mean of 3 seeds: the CPU simulation of the walk gives
    24.5 (uniform) against 0.31 (weighted); assert a factor of 10."""
    torch, eng = env["torch"], env["eng"]
    from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian

    lap = get_normalized_laplacian(_rmat(12, 40_000))
    n, L = lap.shape[0], 5
    f = [0.5 ** l for l in range(L)]
    a = torch.tensor(lap.toarray(), dtype=torch.float64, device="cuda")
    power = torch.eye(n, dtype=torch.float64, device="cuda")
    phi = torch.zeros_like(power)
    for l in range(L):
        if l:
            power = power @ a
        phi += f[l] * power
    k = phi @ phi.T
    nk = torch.linalg.norm(k)
    g = eng.DeviceGraph.from_scipy(lap)
    errs = {}
    for sampling in ("uniform", "weighted"):
        e = []
        for s in range(3):
            mats = eng.build_step_matrices(g, eng.WalkConfig(100, 0.1, L, seed=1000 + s,
                                                             neighbour_sampling=sampling)).to_scipy()
            est = torch.tensor(sum(fl * m for fl, m in zip(f, mats)).toarray(), device="cuda")
            e.append(float(torch.linalg.norm(est @ est.T - k) / nk))
        errs[sampling] = float(np.mean(e))
        print(f"rmat4096 laplacian W=100 p=0.1 {sampling}: {errs[sampling]:.4g} {e}")
    assert errs["weighted"] * 10 < errs["uniform"], errs
    assert errs["weighted"] < 1.0, errs


def test_posterior_mean_on_a_weighted_phi_matches_a_direct_solve(env):
    torch = env["torch"]
    from efficient_graph_gp_sparse.models import SparseGraphGP
    from efficient_graph_gp_sparse.preprocessor import GraphPreprocessor
    from grf_b200.gp_compat import GaussianLikelihood

    adj = random_graph(400, 1300, 21)
    pp = GraphPreprocessor(adj, walks_per_node=30, p_halt=0.1, max_walk_length=4, random_walk_seed=7,
                           use_tqdm=False, neighbour_sampling="weighted")
    ops = pp.preprocess_graph()
    assert pp.cache_filename.endswith("_weighted.pkl")
    uni = GraphPreprocessor(adj, walks_per_node=30, p_halt=0.1, max_walk_length=4, random_walk_seed=7,
                            use_tqdm=False)
    uni.preprocess_graph()
    assert not all(csr_bits_equal(a, b) for a, b in zip(pp.step_matrices_scipy, uni.step_matrices_scipy))
    torch.manual_seed(0)
    rng = np.random.default_rng(3)
    train = rng.permutation(400)[:240]
    test = np.setdiff1d(np.arange(400), train)
    y = np.sin(np.arange(400) / 20.0)[train] + 0.1 * rng.standard_normal(240)
    lik = GaussianLikelihood()
    lik.noise = 0.1
    model = SparseGraphGP(torch.tensor(train, dtype=torch.float32)[:, None].cuda(),
                          torch.tensor(y, dtype=torch.float32).cuda(), lik, ops, 4).cuda()
    f = model.covar_module.modulator_vector.detach().cpu().numpy()
    phi = sum(float(fl) * m.astype(np.float32).astype(np.float64) for fl, m in zip(f, pp.step_matrices_scipy))
    phi = phi.toarray()
    Ktt = phi[train] @ phi[train].T + float(lik.noise) * np.eye(240)
    want = phi[test] @ phi[train].T @ np.linalg.solve(Ktt, y.astype(np.float32).astype(np.float64))
    got, info = model.posterior_mean(torch.tensor(test).cuda(), cg_tolerance=1e-7, return_info=True)
    rel = np.linalg.norm(got.cpu().numpy() - want) / np.linalg.norm(want)
    assert rel <= 1e-4, (rel, info)


def test_public_drop_ins_take_the_neighbour_sampling_keyword(env):
    from efficient_graph_gp.graph_kernels.fast_grf_kernel_general import fast_general_grf_kernel as k_dense
    from efficient_graph_gp.graph_kernels.utils import get_normalized_laplacian as lap_dense
    from efficient_graph_gp.random_walk_samplers.sampler import Graph, RandomWalk
    from efficient_graph_gp_sparse.graph_kernels_sparse.fast_grf_kernel_general import fast_general_grf_kernel as k_sp
    from efficient_graph_gp_sparse.random_walk_samplers_sparse.sparse_sampler import SparseRandomWalk

    cw, o = env["cw"], env["o"]
    adj = random_graph(80, 240, 5)
    lap = o.normalized_laplacian_sparse(adj).tocsr()
    f = np.array([1.0, 0.5, 0.25])
    for coupling, anti in (("iid", False), ("antithetic", True)):
        rw = SparseRandomWalk(lap, seed=3)
        want = cw.step_matrices(lap, 12, 0.2, 3, anti, seed=3)
        got = rw.get_random_walk_matrices(12, 0.2, 3, coupling=coupling, neighbour_sampling="weighted")
        assert all(csr_bits_equal(a, b) for a, b in zip(got, want))
        _phi_bits_equal(rw.get_phi_blocks(12, 0.2, 3, coupling=coupling, neighbour_sampling="weighted"), want)
        dense = RandomWalk(Graph(lap.toarray()), seed=3).get_random_walk_matrices(
            12, 0.2, 3, coupling=coupling, neighbour_sampling="weighted")
        want_d = cw.step_matrices(lap, 12, 0.2, 3, anti, seed=3, scale_mode=1)
        for l in range(3):
            assert np.array_equal(dense[:, :, l], want_d[l].toarray())
        ks = k_sp(adj, f, walks_per_node=12, p_halt=0.2, max_walk_length=3, coupling=coupling,
                  neighbour_sampling="weighted")
        mats = cw.step_matrices(lap, 12, 0.2, 3, anti, seed=42)
        phi = sum(fl * m for fl, m in zip(f, mats))
        assert abs(ks - phi @ phi.T).max() <= 1e-10 * abs(ks).max()
        kd = k_dense(adj.toarray(), f, walks_per_node=12, p_halt=0.2, max_walk_length=3, coupling=coupling,
                     neighbour_sampling="weighted")
        mats = cw.step_matrices(sp.csr_matrix(lap_dense(adj.toarray())), 12, 0.2, 3, anti, seed=42, scale_mode=1)
        phi = sum(fl * m for fl, m in zip(f, mats)).toarray()
        assert np.abs(kd - phi @ phi.T).max() <= 1e-10 * np.abs(kd).max()
    # the default stays the reference's uniform draws
    rw = SparseRandomWalk(lap, seed=3)
    assert all(csr_bits_equal(a, b) for a, b in zip(rw.get_random_walk_matrices(12, 0.2, 3),
                                                     env["cu"].step_matrices(lap, 12, 0.2, 3, seed=3)))
