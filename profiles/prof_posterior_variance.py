"""Cost of the exact posterior variance (grf_b200/posterior.py): the float64 factor on the columns the training rows
touch, and one grf_phi_row_quadform pass over every node of the graph.

    python profiles/prof_posterior_variance.py --out DIR [--reps 3] [--configs 2,4]

Cases: config 2 (the 316^2 grid, W = 100, L = 5) and config 4 (R-MAT 2^22 nodes, 7e7 edges, W = 100, L = 5), each
with n in {100, 600, 4096} random training nodes and every node as a test node.  Per case: CUDA-event times of the
stages (merge, slots, G, G^T G, Cholesky, triangular solve, quadform; medians over --reps after one warm-up), m (the
touched columns), the touched entries sum_i |{e in row i : slot >= 0}|, and the quadform's algorithmic bytes: 8 B
per entry and 4 B per slot lookup of every test row, plus 4 n B per touched entry gathered from C.  Card name and
power limit are read in the same run and written with the results (DIR/posterior_variance.json)."""

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "efficient-gaussian-process-on-graphs_b200")]

STAGES = ("merge", "slots", "G", "gram", "cholesky", "solve")


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                                       "--format=csv,noheader"], text=True).splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers are still worth writing; say why the card is unknown
        return {"error": repr(e)}


def phi_of(config, dev):
    from grf_b200 import engine, synth

    cfg = engine.WalkConfig(100, 0.1, 5, seed=42)
    if config == 2:
        import scipy.sparse as sp

        path = sp.diags([np.ones(315), np.ones(315)], [-1, 1], format="csr")
        grid = (sp.kron(sp.eye(316), path) + sp.kron(path, sp.eye(316))).tocsr()
        g = engine.DeviceGraph.laplacian_of(grid, dev)
    else:
        g, _ = synth.rmat_walk_graph(22, int(70e6), seed=0, device=dev)
    return engine.build_phi_blocks(g, cfg, transpose=True)


def run_case(name, phi, n, reps):
    import torch

    from grf_b200.posterior import ExactPosterior

    dev = phi.device
    rng = np.random.default_rng(n)
    x = torch.tensor(rng.choice(phi.n_rows, n, replace=False), device=dev)
    f = torch.tensor([1.0 / (1 + p) ** 2 for p in range(phi.n_steps)])
    xt = torch.arange(phi.n_rows, device=dev)
    ExactPosterior(phi, f, x, 0.1).variance(xt)            # warm-up: union pattern, libraries, kernel
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        ev = {}
        post = ExactPosterior(phi, f, x, 0.1, events=ev)
        var = post.variance(xt)
        torch.cuda.synchronize()
        t = {}
        prev = "start"
        for s in STAGES:
            t[s + "_ms"] = ev[prev].elapsed_time(ev[s])
            prev = s
        t["quadform_ms"] = ev["quadform_start"].elapsed_time(ev["quadform"])
        times.append(t)
    ent = post.phi_f.entries
    nnz = int(ent.shape[0])
    touched = int((post.slot[ent[:, 0].long()] >= 0).sum().item())
    qf_bytes = 12 * nnz + 4 * n * touched
    med = {k: float(np.median([t[k] for t in times])) for k in times[0]}
    res = {"case": name, "n_train": n, "n_test": phi.n_rows, "m": post.m, "nnz_phi_f": nnz,
           "touched_entries": touched, "quadform_bytes": qf_bytes, "stages_ms": times, "median_stages_ms": med,
           "quadform_GB_per_s": qf_bytes / (med["quadform_ms"] * 1e6),
           "variance_min": float(var.min()), "variance_max": float(var.max())}
    print(json.dumps({k: v for k, v in res.items() if k != "stages_ms"}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--configs", default="2,4")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("prof_posterior_variance needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {"card": card(), "torch": torch.__version__, "cases": []}
    for config in (int(c) for c in a.configs.split(",")):
        phi = phi_of(config, dev)
        for n in (100, 600, 4096):
            out["cases"].append(run_case(f"config{config}_W100_L5", phi, n, a.reps))
        del phi
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "posterior_variance.json"), "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
