"""Coupled walk draws (WalkConfig.coupling): what they cost and how much kernel error they remove.

    python profiles/prof_coupled.py --out DIR      (one GPU; writes DIR/prof_coupled.json)

Cost, per coupling, median of --reps runs after two warm-up runs (CUDA events, L2 not flushed: both graphs'
working sets stream far beyond 126 MB on config 4; config 2 is L2-resident as in bench.py's config-2 section
without the flush):
  config 4 -- the bench.py graph (R-MAT 2^22 nodes, >= 70 M edges, normalized Laplacian), W = 100, L = 5, p = 0.1
  config 2 -- 316 x 316 grid Laplacian, same W, L, p
  walker ms (grf_walk with finished entries + column counts, as build_phi_blocks runs it), Phi build ms
  (build_phi_blocks: walk + compact + Phi^T), walk-steps/s of the walker, nnz(Phi).
Accuracy: relative Frobenius error of K = Phi Phi^T against the exact series sum_l f_l A^l (f_l = 2^-l, L = 5),
mean and sd over 8 seeds, W in {4, 8, 16, 32, 64, 100}, p in {0.1, 0.5}, on a 64 x 64 grid and a 4096-node
R-MAT graph, for two walk graphs A: the normalized Laplacian (what the project builds Phi on) and the
normalized adjacency D^-1/2 A D^-1/2.  From the iid curve (log-log interpolation, extrapolated with the slope of
its last two points): the iid W that matches each coupled mode's error at W = 16 and W = 100.
"""

import argparse
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

MODES = ["iid", "antithetic", "repelling", "antithetic+repelling"]
WS = [4, 8, 16, 32, 64, 100]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, reps):
    out = []
    for i in range(reps + 2):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        torch.cuda.synchronize()
        if i >= 2:
            out.append(a.elapsed_time(b))
        del r
    return float(np.median(out)), out


def cost(g, reps):
    rows = {}
    for mode in MODES:
        cfg = engine.WalkConfig(bench.W, bench.P_HALT, bench.L, seed=bench.SEED, coupling=mode)
        visits = torch.zeros(1, dtype=torch.int64, device="cuda")

        def walk():
            visits.zero_()
            return engine.run_walker(g, cfg, visits=visits, count_columns=True,
                                     entries_scale_mode=_lib.SCALE_MUL_RECIP)

        walk_ms, walk_all = timed(walk, reps)
        steps = int(visits.item())
        build_ms, build_all = timed(lambda: engine.build_phi_blocks(g, cfg), reps)
        phi = engine.build_phi_blocks(g, cfg)
        nnz = int(phi.blk_ptr.view(-1)[-1].item())
        del phi
        rows[mode] = {"walker_ms": walk_ms, "walker_ms_runs": walk_all, "phi_build_ms": build_ms,
                      "phi_build_ms_runs": build_all, "walk_steps": steps,
                      "walk_steps_per_s": steps / (walk_ms * 1e-3), "nnz_phi": nnz}
        print(mode, {k: v for k, v in rows[mode].items() if not k.endswith("runs")}, flush=True)
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
        for mode in MODES:
            for W in WS:
                errs = []
                for s in range(seeds):
                    st = engine.build_step_matrices(g, engine.WalkConfig(W, p, L, seed=1000 + s, coupling=mode))
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
            print(p, mode, [round(res[f"p={p} {mode} W={W}"]["mean"], 4) for W in WS], flush=True)
    # iid W with the same error as each coupled mode at W = 16 and W = 100
    for p in (0.1, 0.5):
        le = np.log([res[f"p={p} iid W={W}"]["mean"] for W in WS])
        lw = np.log(WS)
        for mode in MODES[1:]:
            for W0 in (16, 100):
                target = np.log(res[f"p={p} {mode} W={W0}"]["mean"])
                if target >= le[0]:
                    weq = float(np.exp(lw[0] + (target - le[0]) * (lw[1] - lw[0]) / (le[1] - le[0])))
                elif target <= le[-1]:
                    weq = float(np.exp(lw[-1] + (target - le[-1]) * (lw[-1] - lw[-2]) / (le[-1] - le[-2])))
                else:
                    i = int(np.nonzero(le <= target)[0][0])
                    weq = float(np.exp(lw[i - 1] + (target - le[i - 1]) * (lw[i] - lw[i - 1]) / (le[i] - le[i - 1])))
                res[f"p={p} {mode} iid_W_equivalent_at_W={W0}"] = weq
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for prof_coupled.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seeds", type=int, default=8)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "prof_coupled measures on the GPU"
    os.makedirs(args.out, exist_ok=True)
    t0 = time.time()
    result = {"card": card(), "torch": torch.__version__,
              "settings": {"W": bench.W, "L": bench.L, "p_halt": bench.P_HALT, "reps": args.reps,
                           "accuracy_seeds": args.seeds, "accuracy_L": 5, "accuracy_f": "2^-l"}}
    g4, stats = synth.rmat_walk_graph(bench.RMAT_SCALE, bench.RMAT_EDGES, seed=bench.RMAT_SEED)
    result["config4_graph"] = stats
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
    result["seconds"] = time.time() - t0
    with open(os.path.join(args.out, "prof_coupled.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print("wrote", os.path.join(args.out, "prof_coupled.json"))


if __name__ == "__main__":
    main()
