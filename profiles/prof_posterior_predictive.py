"""Cost of the exact posterior mean, samples and joint covariance (grf_b200/posterior.py) once the factor is built:
one grf_phi_row_project pass each, plus the prior SpMM, the float64 triangular solve and the float32 GEMM of the
samples, and the K** pair dots and float64 P P^T of the covariance.

    python profiles/prof_posterior_predictive.py --out DIR [--reps 3] [--configs 2,4]

Cases: config 2 (the 316^2 grid, W = 100, L = 5) and config 4 (R-MAT 2^22 nodes, 7e7 edges, W = 100, L = 5), each
with n in {100, 600, 4096} random training nodes.  Per case, medians over --reps after one warm-up of CUDA-event
times of:
  - the mean at every node (r = 1);
  - samples with s = 1, 16 and 64 at every node, split into prior apply, triangular solve, GEMM and projection;
  - the covariance between q = 50, 500 and 2000 random nodes (projection with r = n, and the whole call).
For every projection: its algorithmic bytes, 12 B per streamed entry of the projected rows of Phi_f (8 B entry, 4 B
slot lookup), 4 r B of B per touched entry and 4 r B of out per row, and that over the projection's time.  Card name
and power limit are read in the same run and written with the results (DIR/posterior_predictive.json)."""

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "efficient-gaussian-process-on-graphs_b200"), os.path.dirname(__file__)]

from prof_posterior_variance import card, phi_of  # noqa: E402


def _ms(ev, a, b):
    return ev[a].elapsed_time(ev[b])


def _median(times):
    return {k: float(np.median([t[k] for t in times])) for k in times[0]}


def project_bytes(post, xt, r):
    """12 B per streamed entry of the rows xt, 4 r B per touched entry, 4 r B per output row."""
    ptr = post.phi_f.blk_ptr.long()
    xl = xt.long()
    streamed = int((ptr[xl + 1] - ptr[xl]).sum().item())
    ent = post.phi_f.entries
    touched_row = post.slot[ent[:, 0].long()] >= 0
    if xt.numel() == post.phi_f.n_rows:
        touched = int(touched_row.sum().item())
    else:
        import torch

        cum = torch.cat([torch.zeros(1, dtype=torch.int64, device=ptr.device), torch.cumsum(touched_row.long(), 0)])
        touched = int((cum[ptr[xl + 1]] - cum[ptr[xl]]).sum().item())
    return 12 * streamed + 4 * r * touched + 4 * r * int(xt.numel()), streamed, touched


def timed(fn, reps, stages):
    import torch

    fn(None)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        ev = {}
        fn(ev)
        torch.cuda.synchronize()
        times.append({k: _ms(ev, a, b) for k, (a, b) in stages.items()})
    return _median(times), times


def run_case(name, phi, n, reps):
    import torch

    from grf_b200.posterior import ExactPosterior

    dev = phi.device
    rng = np.random.default_rng(n)
    x = torch.tensor(rng.choice(phi.n_rows, n, replace=False), device=dev)
    y = torch.sin(x.double() / 1000.0)
    f = torch.tensor([1.0 / (1 + p) ** 2 for p in range(phi.n_steps)])
    post = ExactPosterior(phi, f, x, 0.1, y_train=y)
    xt = torch.arange(phi.n_rows, device=dev, dtype=torch.int32)
    res = {"case": name, "n_train": n, "n_test": phi.n_rows, "m": post.m}

    def with_events(ev, call):
        post.events = ev
        call()
        post.events = None

    def add_rate(entry, r, rows):
        b, streamed, touched = project_bytes(post, rows, r)
        entry.update(project_bytes=b, streamed_entries=streamed, touched_entries=touched,
                     project_GB_per_s=b / (entry["median_ms"]["project_ms"] * 1e6))

    med, times = timed(lambda ev: with_events(ev, lambda: post.mean(xt)), reps,
                       {"project_ms": ("project_start", "project")})
    res["mean"] = {"r": 1, "median_ms": med, "times_ms": times}
    add_rate(res["mean"], 1, xt)

    res["samples"] = []
    for s in (1, 16, 64):
        gen = torch.Generator(device=dev).manual_seed(s)
        stages = {"prior_ms": ("sample_start", "prior"), "solve_ms": ("prior", "triangular"),
                  "gemm_ms": ("triangular", "gemm"), "project_ms": ("project_start", "project"),
                  "total_ms": ("sample_start", "project")}
        med, times = timed(lambda ev: with_events(ev, lambda: post.sample(xt, s, generator=gen)), reps, stages)
        entry = {"s": s, "median_ms": med, "times_ms": times}
        add_rate(entry, s, xt)
        res["samples"].append(entry)

    res["covariance"] = []
    for q in (50, 500, 2000):
        xq = torch.tensor(rng.choice(phi.n_rows, q, replace=False), device=dev, dtype=torch.int32)

        def cov(ev):
            post.events = ev
            post._mark("cov_start")
            post.covariance(xq)
            post._mark("cov_end")
            post.events = None

        med, times = timed(cov, reps, {"project_ms": ("project_start", "project"),
                                       "total_ms": ("cov_start", "cov_end")})
        entry = {"q": q, "median_ms": med, "times_ms": times}
        add_rate(entry, n, xq)
        res["covariance"].append(entry)
    print(json.dumps({k: v for k, v in res.items()}, default=str)[:2000], flush=True)
    del post
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--configs", default="2,4")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("prof_posterior_predictive needs a CUDA device")
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
    with open(os.path.join(a.out, "posterior_predictive.json"), "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
