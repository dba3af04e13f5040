"""Cost of the sparse fast_general_grf_kernel: K = Phi_f Phi_f^T on the device against the host path.

    python profiles/prof_kernel_matrix.py --out DIR

Three shapes (config 1: G(2708, 5429), W = 50, L = 3; config 2: the 316^2 grid, W = 100, L = 5; the 316^2 grid
with the function's defaults W = 50, L = 10).  For each: wall time of the old path (walks, StepMatrices.to_scipy,
scipy sum and SpGEMM) and of the new one (walks, kernel_matrix, to_scipy), CUDA-event times of the device stages,
the host-clock time of the copy of K (to_scipy, which ends in a synchronise), nnz(Phi_f), nnz(K), the touched
count and the bytes copied.  Both results are compared array for array.  Card name and power limit are read in
the same run and written with the results (DIR/kernel_matrix.json)."""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "efficient-gaussian-process-on-graphs_b200")]


def grid(nx, ny):
    def path(n):
        return sp.diags([np.ones(n - 1), np.ones(n - 1)], [-1, 1], format="csr")

    return (sp.kron(sp.eye(ny), path(nx)) + sp.kron(path(ny), sp.eye(nx))).tocsr()


def gnm(n, m, seed):
    rng = np.random.default_rng(seed)
    i, j = rng.integers(0, n, m), rng.integers(0, n, m)
    keep = i != j
    a = sp.coo_matrix((np.ones(keep.sum()), (i[keep], j[keep])), shape=(n, n)).tocsr()
    a.data[:] = 1.0
    a = a.maximum(a.T).tocsr()
    a.sort_indices()
    return a


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                                       "--format=csv,noheader"], text=True).splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers are still worth writing; say why the card is unknown
        return {"error": repr(e)}


def same(a, b):
    return (a.indptr.dtype == b.indptr.dtype and a.indices.dtype == b.indices.dtype and np.array_equal(a.indptr, b.indptr)
            and np.array_equal(a.indices, b.indices) and np.array_equal(a.data.view(np.int64), b.data.view(np.int64)))


def run_shape(name, adj, W, L, p_halt=0.1, reps=3):
    import torch

    from efficient_graph_gp_sparse.random_walk_samplers_sparse import SparseRandomWalk

    f = [1.0 / (1 + p) ** 2 for p in range(L)]
    rw = SparseRandomWalk.on_normalized_laplacian(adj)
    steps = rw.get_step_matrices_device(W, p_halt, L)       # warm-up of the walker and of every kernel
    steps.kernel_matrix(f).to_scipy()
    torch.cuda.synchronize()
    res = {"shape": name, "n": adj.shape[0], "W": W, "L": L, "p_halt": p_halt}
    old, new, stage = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        steps = rw.get_step_matrices_device(W, p_halt, L)
        mats = steps.to_scipy()
        phi = sp.csr_matrix(mats[0].shape)
        for s, f_p in enumerate(f):
            phi += f_p * mats[s]
        k_old = phi @ phi.T
        old.append(time.perf_counter() - t0)

        torch.cuda.synchronize()
        t0 = time.perf_counter()
        steps = rw.get_step_matrices_device(W, p_halt, L)
        ev = {}
        km = steps.kernel_matrix(f, events=ev)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        k_new = km.to_scipy()
        t2 = time.perf_counter()
        new.append(t2 - t0)
        stage.append({"assembly_ms": ev["start"].elapsed_time(ev["phi"]),
                      "transpose_ms": ev["phi"].elapsed_time(ev["transpose"]),
                      "count_ms": ev["transpose"].elapsed_time(ev["count"]),
                      "fill_ms": ev["count"].elapsed_time(ev["fill"]),
                      "copy_to_host_ms": 1e3 * (t2 - t1)})
        assert same(k_new, k_old), name
    res["old_path_s"] = old
    res["new_path_s"] = new
    res["stages"] = stage
    res["median_old_s"] = float(np.median(old))
    res["median_new_s"] = float(np.median(new))
    res["median_stages_ms"] = {k: float(np.median([s[k] for s in stage])) for k in stage[0]}
    res["nnz_phi_f"] = km.nnz_phi
    res["nnz_k"] = km.nnz
    res["touched"] = km.touched
    idx_bytes = 4 if k_new.indices.dtype == np.int32 else 8
    res["copy_bytes"] = km.nnz * (8 + idx_bytes) + (adj.shape[0] + 1) * idx_bytes
    res["results_equal"] = True
    print(json.dumps({k: v for k, v in res.items() if k not in ("stages",)}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("prof_kernel_matrix needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    out = {"card": card(), "torch": torch.__version__, "shapes": []}
    g316 = grid(316, 316)
    for name, adj, W, L in [("config1_gnm2708", gnm(2708, 5429, 0), 50, 3), ("config2_grid316_W100_L5", g316, 100, 5),
                            ("grid316_defaults_W50_L10", g316, 50, 10)]:
        out["shapes"].append(run_shape(name, adj, W, L, reps=a.reps))
    with open(os.path.join(a.out, "kernel_matrix.json"), "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
