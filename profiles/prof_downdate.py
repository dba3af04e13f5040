"""Cost of removing observations from the exact posterior (grf_b200/posterior.py): ExactPosterior.forget of b rows
plus a PosteriorMarginals refresh at every node, against rebuilding the posterior on the kept rows (constructor +
variance + mean), and of ExactPosterior.set_targets plus the refresh of the mean.

    python profiles/prof_downdate.py --out DIR [--reps 2] [--configs 2,4]

Cases: config 2 (the 316^2 grid, W = 100, L = 5) and config 4 (R-MAT 2^22 nodes, 7e7 edges, W = 100, L = 5), each
with n in {100, 600, 4096} random training nodes, b in {1, 16, 50, 100} removed rows taken from the front (a sliding
window: j0 = 0, the largest C' product), the middle and the end (a truncation).  Per case, medians over --reps after
one warm-up of CUDA-event times of:
  - the stages of forget ("factor": T T^T and its Cholesky; "columns": the right factors, C' and U in float64 row
    chunks, the retired rows; "weights": a);
  - the refresh pass over every node (b + 1 <= 64: row_downdate; b = 100: row_quadform + row_project);
  - the rebuild on the kept rows: constructor (merge .. solve), variance and mean;
the refresh's algorithmic bytes (as profiles/prof_condition.py) over its time, and the largest difference of the
refreshed variance and mean from the rebuild's.  For the front removals, the C'[:, j0:] = C[:, j0:] M product alone
both ways, alternated: float64 row chunks (what forget does) and one float32 GEMM, with the largest difference of
the float32 result from the float64 one.  Card name and power limit are read in the same run and written with the
results (DIR/downdate.json)."""

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "efficient-gaussian-process-on-graphs_b200"), os.path.dirname(__file__)]

from prof_condition import _clone, _ms, refresh_bytes  # noqa: E402
from prof_posterior_variance import card, phi_of  # noqa: E402


def _events():
    import torch

    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def product_both_ways(post, b, reps):
    """C[:, :n] M for the front removal of b rows: float64 row chunks against one float32 GEMM."""
    import torch

    from grf_b200.posterior import _condition_chunk

    n, m = post.n, post.m
    T = post.L[b:, :]                                   # j0 = 0: the kept rows after j0 are b .. n - 1
    l22 = torch.linalg.cholesky(T @ T.T)
    M = torch.linalg.solve_triangular(l22, T, upper=False).T.contiguous()      # [n, n - b]
    M32 = M.to(torch.float32)
    out64 = torch.empty((m, n - b), dtype=torch.float32, device=post.device)
    chunk = _condition_chunk(n, m)

    def f64():
        for r0 in range(0, m, chunk):
            r1 = min(m, r0 + chunk)
            out64[r0:r1] = (post.C[r0:r1, :n].to(torch.float64) @ M).to(torch.float32)

    def f32():
        return post.C[:, :n] @ M32

    t = {"float64_chunks_ms": [], "float32_gemm_ms": []}
    for rep in range(reps + 1):
        for key, fn in (("float64_chunks_ms", f64), ("float32_gemm_ms", f32)):
            a, e = _events()
            a.record()
            res = fn()
            e.record()
            torch.cuda.synchronize()
            if rep:
                t[key].append(a.elapsed_time(e))
            if key == "float32_gemm_ms":
                out32 = res
    diff = float((out32 - out64).abs().max())
    flop = 2.0 * m * n * (n - b)
    med = {k: float(np.median(v)) for k, v in t.items()}
    return {"m": m, "flop": flop, **med, "times_ms": t, "max_abs_diff_f32_vs_f64": diff,
            "max_abs_c_new": float(out64.abs().max()),
            "float64_TFLOP_per_s": flop / (med["float64_chunks_ms"] * 1e9),
            "float32_TFLOP_per_s": flop / (med["float32_gemm_ms"] * 1e9)}


def run_case(name, phi, n, reps):
    import torch

    from grf_b200.posterior import ExactPosterior

    dev = phi.device
    rng = np.random.default_rng(n + 1)
    nodes = torch.tensor(rng.choice(phi.n_rows, n, replace=False), device=dev)
    yall = torch.sin(nodes.double() / 1000.0)
    f = torch.tensor([1.0 / (1 + p) ** 2 for p in range(phi.n_steps)])
    xt = torch.arange(phi.n_rows, device=dev, dtype=torch.int32)
    base = ExactPosterior(phi, f, nodes, 0.1, y_train=yall)
    bmarg = base.marginals(xt)
    out, products = [], []
    for b in (1, 16, 50, 100):
        bb = min(b, n)
        wheres = {"front": np.arange(bb), "middle": np.arange((n - bb) // 2, (n - bb) // 2 + bb),
                  "end": np.arange(n - bb, n)}
        for where, pos in wheres.items():
            if bb == n and where != "front":
                continue
            kept = torch.tensor(np.setdiff1d(np.arange(n), pos), device=dev)
            times = []
            for rep in range(reps + 1):
                post, marg = _clone(base, bmarg)
                ev = {}
                post.events = ev
                torch.cuda.synchronize()
                post.forget(pos)
                marg.refresh()
                torch.cuda.synchronize()
                rb = {}
                fresh = ExactPosterior(phi, f, nodes[kept], 0.1, events=rb, y_train=yall[kept])
                var_f = fresh.variance(xt)
                mean_f = fresh.mean(xt)
                torch.cuda.synchronize()
                t = {"factor_ms": _ms(ev, "downdate_start", "downdate_factor"),
                     "columns_ms": _ms(ev, "downdate_factor", "downdate_columns"),
                     "weights_ms": _ms(ev, "downdate_columns", "downdate_weights"),
                     "forget_ms": _ms(ev, "downdate_start", "downdate_weights"),
                     "refresh_ms": _ms(ev, "refresh_start", "refresh"),
                     "rebuild_constructor_ms": _ms(rb, "start", "solve"),
                     "rebuild_variance_ms": _ms(rb, "quadform_start", "quadform"),
                     "rebuild_mean_ms": _ms(rb, "project_start", "project")}
                t["update_ms"] = t["forget_ms"] + t["refresh_ms"]
                t["rebuild_ms"] = t["rebuild_constructor_ms"] + t["rebuild_variance_ms"] + t["rebuild_mean_ms"]
                if rep:
                    times.append(t)
                if rep == reps:
                    dv = (marg.variance() - var_f).abs()
                    dp = (post.variance(xt) - var_f).abs()
                    dm = (marg.mean - mean_f).abs()
                    diff = {"max_abs_var_diff": float(dv.max()), "max_abs_posterior_var_diff": float(dp.max()),
                            "max_var": float(var_f.max()), "max_abs_mean_diff": float(dm.max()),
                            "max_abs_mean": float(mean_f.abs().max())}
                del fresh, var_f, mean_f, post, marg
                torch.cuda.empty_cache()
            med = {k: float(np.median([t[k] for t in times])) for k in times[0]}
            entry = {"case": name, "n_train": n, "b": bb, "where": where, "j0": int(pos[0]),
                     "refresh_path": "row_downdate" if bb + 1 <= 64 else "row_quadform + row_project",
                     "m": base.m, "median_ms": med, "times_ms": times, **diff,
                     "speedup": med["rebuild_ms"] / med["update_ms"]}
            if bb + 1 <= 64:
                nbytes, streamed, touched = refresh_bytes(base, bb, 1)
                entry.update(refresh_bytes=nbytes, streamed_entries=streamed, touched_entries=touched,
                             refresh_GB_per_s=nbytes / (med["refresh_ms"] * 1e6))
            print(json.dumps({k: v for k, v in entry.items() if k != "times_ms"}), flush=True)
            out.append(entry)
        if bb < n:
            pr = {"case": name, "n_train": n, "b": bb, **product_both_ways(base, bb, reps)}
            print(json.dumps({k: v for k, v in pr.items() if k != "times_ms"}), flush=True)
            products.append(pr)
            torch.cuda.empty_cache()
    # set_targets: all targets, plus the refresh of the mean
    times = []
    for rep in range(reps + 1):
        post, marg = _clone(base, bmarg)
        a, e = _events()
        a.record()
        post.set_targets(torch.cos(nodes.double() / 1000.0))
        e.record()
        c, d = _events()
        c.record()
        marg.refresh()
        d.record()
        torch.cuda.synchronize()
        if rep:
            times.append({"set_targets_ms": a.elapsed_time(e), "refresh_ms": c.elapsed_time(d)})
        del post, marg
    st = {"case": name, "n_train": n, **{k: float(np.median([t[k] for t in times])) for k in times[0]},
          "times_ms": times}
    print(json.dumps({k: v for k, v in st.items() if k != "times_ms"}), flush=True)
    del base, bmarg
    torch.cuda.empty_cache()
    return out, products, st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--configs", default="2,4")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("prof_downdate needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {"card": card(), "torch": torch.__version__, "cases": [], "products": [], "set_targets": []}
    for config in (int(c) for c in a.configs.split(",")):
        phi = phi_of(config, dev)
        for n in (100, 600, 4096):
            cases, products, st = run_case(f"config{config}_W100_L5", phi, n, a.reps)
            out["cases"] += cases
            out["products"] += products
            out["set_targets"].append(st)
        del phi
        torch.cuda.empty_cache()
        with open(os.path.join(a.out, "downdate.json"), "w") as fh:      # after each config
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
