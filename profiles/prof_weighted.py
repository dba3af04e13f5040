"""Weight-proportional neighbour draws (WalkConfig.neighbour_sampling = "weighted"): what they cost and how much
kernel error they remove.

    python profiles/prof_weighted.py --out DIR      (one GPU; writes DIR/weighted_walks.json)

Cost, uniform against weighted, alternated within every repetition (median of --reps after two warm-up rounds;
CUDA events, L2 not flushed):
  config 4 -- the bench.py graph (R-MAT 2^22 nodes, >= 70 M edges, normalized Laplacian), W = 100, L = 5, p = 0.1
  config 2 -- 316 x 316 grid Laplacian, same W, L, p
  alias build ms (grf_alias_records; the uniform column: grf_edge_records) and its split over the two kernels
  (torch.profiler: warp per row of <= 2048 entries, CTA per longer row), walker ms (finished entries + column
  counts, as build_phi_blocks runs it), Phi build ms (build_phi_blocks: walk + compact + Phi^T, records cached),
  walk-steps/s of the walker, nnz(Phi).
Accuracy: relative Frobenius error of K = Phi Phi^T against the exact series sum_l f_l A^l (f_l = 2^-l, L = 5),
mean and sd over --seeds seeds, p in {0.1, 0.5}, on a 64 x 64 grid and a 4096-node R-MAT graph, walk graphs A =
the normalized Laplacian and the normalized adjacency; uniform draws at W in {16, 32, 64, 100, 200, 400},
weighted and weighted + antithetic termination at W in {16, 100}.  From the uniform curve (log-log interpolation,
extrapolated with the slope of its last two points while it falls): the uniform W that matches each weighted error.
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "efficient-gaussian-process-on-graphs_b200")]

import numpy as np  # noqa: E402
import scipy.sparse as sp  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from grf_b200 import _lib, engine, synth  # noqa: E402

MODES = {"uniform": ("iid", "uniform"), "weighted": ("iid", "weighted"),
         "weighted+antithetic": ("antithetic", "weighted")}
WS_UNIFORM = [16, 32, 64, 100, 200, 400]
WS_WEIGHTED = [16, 100]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed_alternating(fns, reps):
    """{name: (median ms, all ms)}: one run of every fn per round, two warm-up rounds."""
    out = {k: [] for k in fns}
    for i in range(reps + 2):
        for name, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            r = fn()
            b.record()
            torch.cuda.synchronize()
            if i >= 2:
                out[name].append(a.elapsed_time(b))
            del r
    return {k: (float(np.median(v)), v) for k, v in out.items()}


def alias_kernel_split(build, reps):
    """Mean device ms per call of each grf_alias_records kernel over `reps` calls."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            build()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for name in ("alias_rows_warp", "alias_rows_cta"):
            if name in ev.key:
                out[name] = getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1e3 / reps
    return out


def row_sizes(g):
    deg = (g.row_ptr[1:] - g.row_ptr[:-1]).to(torch.int64)
    return {"rows_le_32": int(((deg > 0) & (deg <= 32)).sum()),
            "rows_33_2048": int(((deg > 32) & (deg <= 2048)).sum()), "rows_gt_2048": int((deg > 2048).sum()),
            "entries_gt_2048": int(deg[deg > 2048].sum())}


def cost(g, reps):
    cfgs = {s: engine.WalkConfig(bench.W, bench.P_HALT, bench.L, seed=bench.SEED, neighbour_sampling=s)
            for s in ("uniform", "weighted")}
    visits = {s: torch.zeros(1, dtype=torch.int64, device="cuda") for s in cfgs}

    bufs = {"uniform": torch.empty((max(1, g.nnz), 2), dtype=torch.float64, device="cuda"),
            "weighted": torch.empty((max(1, g.nnz), 4), dtype=torch.float64, device="cuda")}

    def records(s):                     # the build itself, through the C ABI (the graph caches its own copy)
        fn = _lib.lib().grf_alias_records if s == "weighted" else _lib.lib().grf_edge_records
        gs = g.c_struct()
        _lib.check(fn(ctypes.byref(gs), float(bench.P_HALT), ctypes.c_void_p(bufs[s].data_ptr()), None))

    def walk(s):
        visits[s].zero_()
        return engine.run_walker(g, cfgs[s], visits=visits[s], count_columns=True,
                                 entries_scale_mode=_lib.SCALE_MUL_RECIP)

    rec = timed_alternating({s: (lambda s=s: records(s)) for s in cfgs}, reps)
    split = alias_kernel_split(lambda: records("weighted"), reps)
    g.edge_records(bench.P_HALT)
    g.alias_records(bench.P_HALT)           # both cached from here on
    wk = timed_alternating({s: (lambda s=s: walk(s)) for s in cfgs}, reps)
    bd = timed_alternating({s: (lambda s=s: engine.build_phi_blocks(g, cfgs[s])) for s in cfgs}, reps)
    rows = {}
    for s in cfgs:
        visits[s].zero_()
        walk(s)
        steps = int(visits[s].item())
        phi = engine.build_phi_blocks(g, cfgs[s])
        nnz = int(phi.blk_ptr.view(-1)[-1].item())
        del phi
        rows[s] = {"records_ms": rec[s][0], "records_ms_runs": rec[s][1], "walker_ms": wk[s][0],
                   "walker_ms_runs": wk[s][1], "phi_build_ms": bd[s][0], "phi_build_ms_runs": bd[s][1],
                   "walk_steps": steps, "walk_steps_per_s": steps / (wk[s][0] * 1e-3), "nnz_phi": nnz,
                   "records_plus_phi_build_ms": rec[s][0] + bd[s][0]}
        if s == "weighted":
            rows[s]["alias_kernel_ms"] = split
        print(s, {k: v for k, v in rows[s].items() if not k.endswith("runs")}, flush=True)
    torch.cuda.empty_cache()
    return rows


def normalized_adjacency(adj):
    d = np.asarray(adj.sum(1)).ravel()
    dis = sp.diags(np.where(d > 0, 1.0 / np.sqrt(np.where(d > 0, d, 1.0)), 0.0))
    a = (dis @ adj @ dis).tocsr()
    a.sort_indices()
    return a


def rmat_host(scale, m, seed=0, a=0.57, b=0.19, c=0.19):
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


def uniform_w_equivalent(ws, means, target):
    """Uniform W whose (log-log interpolated) error equals `target`; None when the curve does not reach it."""
    le, lw = np.log(means), np.log(ws)
    if target >= le[0]:
        return float(np.exp(lw[0] + (target - le[0]) * (lw[1] - lw[0]) / (le[1] - le[0]))) if le[1] < le[0] else None
    for i in range(1, len(ws)):
        if le[i] <= target:
            return float(np.exp(lw[i - 1] + (target - le[i - 1]) * (lw[i] - lw[i - 1]) / (le[i] - le[i - 1])))
    if le[-1] >= le[-2]:
        return None
    return float(np.exp(lw[-1] + (target - le[-1]) * (lw[-1] - lw[-2]) / (le[-1] - le[-2])))


def accuracy(walk_graph, seeds, L=5):
    f = [0.5 ** l for l in range(L)]
    a = torch.tensor(walk_graph.toarray(), dtype=torch.float64, device="cuda")
    power = torch.eye(a.shape[0], dtype=torch.float64, device="cuda")
    phi_x = torch.zeros_like(a)
    for l, fl in enumerate(f):
        if l:
            power = power @ a
        phi_x += fl * power
    k_x = phi_x @ phi_x.T
    norm_x = float(torch.linalg.norm(k_x))
    g = engine.DeviceGraph.from_scipy(walk_graph)
    n = walk_graph.shape[0]
    res = {}
    for p in (0.1, 0.5):
        for mode, (coupling, sampling) in MODES.items():
            for W in (WS_UNIFORM if mode == "uniform" else WS_WEIGHTED):
                errs = []
                for s in range(seeds):
                    st = engine.build_step_matrices(g, engine.WalkConfig(W, p, L, seed=1000 + s, coupling=coupling,
                                                                         neighbour_sampling=sampling))
                    phi = torch.zeros((n, n), dtype=torch.float64, device="cuda")
                    off = st.offsets
                    for l in range(L):
                        ip = off[l * n:(l + 1) * n + 1]
                        b, e = int(ip[0]), int(ip[-1])
                        rows = torch.repeat_interleave(torch.arange(n, device="cuda"), ip[1:] - ip[:-1])
                        phi[rows, st.col[b:e].long()] += f[l] * st.val[b:e]
                    errs.append(float(torch.linalg.norm(phi @ phi.T - k_x)) / norm_x)
                res[f"p={p} {mode} W={W}"] = {"mean": float(np.mean(errs)), "sd": float(np.std(errs, ddof=1)),
                                              "errors": errs}
            ws = WS_UNIFORM if mode == "uniform" else WS_WEIGHTED
            print(p, mode, {W: round(res[f"p={p} {mode} W={W}"]["mean"], 4) for W in ws}, flush=True)
        means = [res[f"p={p} uniform W={W}"]["mean"] for W in WS_UNIFORM]
        for mode in ("weighted", "weighted+antithetic"):
            for W0 in WS_WEIGHTED:
                res[f"p={p} {mode} uniform_W_equivalent_at_W={W0}"] = uniform_w_equivalent(
                    WS_UNIFORM, means, np.log(res[f"p={p} {mode} W={W0}"]["mean"]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for weighted_walks.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seeds", type=int, default=8)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "prof_weighted measures on the GPU"
    os.makedirs(args.out, exist_ok=True)
    t0 = time.time()
    result = {"card": card(), "torch": torch.__version__,
              "settings": {"W": bench.W, "L": bench.L, "p_halt": bench.P_HALT, "reps": args.reps,
                           "accuracy_seeds": args.seeds, "accuracy_L": 5, "accuracy_f": "2^-l"}}
    g4, stats = synth.rmat_walk_graph(bench.RMAT_SCALE, bench.RMAT_EDGES, seed=bench.RMAT_SEED)
    result["config4_graph"] = stats
    result["config4_row_sizes"] = row_sizes(g4)
    result["config4"] = cost(g4, args.reps)
    del g4
    torch.cuda.empty_cache()
    g2 = engine.DeviceGraph.from_scipy(bench.grid_laplacian(316, 316))
    result["config2"] = cost(g2, args.reps)
    del g2
    from efficient_graph_gp_sparse.utils_sparse.graph_utils import get_normalized_laplacian
    path = sp.diags([np.ones(63), np.ones(63)], [-1, 1], format="csr")
    grid = (sp.kron(sp.eye(64), path) + sp.kron(path, sp.eye(64))).tocsr()
    graphs = {"grid64x64": grid, "rmat4096": rmat_host(12, 40_000)}
    acc = {}
    for name, adj in graphs.items():
        for kind, wg in (("laplacian", get_normalized_laplacian(adj)), ("normalized_adjacency",
                                                                       normalized_adjacency(adj))):
            print(name, kind, flush=True)
            acc[f"{name} {kind}"] = accuracy(wg.tocsr(), args.seeds)
    result["accuracy"] = acc
    result["card_after"] = card()
    result["seconds"] = time.time() - t0
    with open(os.path.join(args.out, "weighted_walks.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print("wrote", os.path.join(args.out, "weighted_walks.json"))


if __name__ == "__main__":
    main()
