"""Cost of one BO iteration's update of the exact posterior (grf_b200/posterior.py): ExactPosterior.condition_on
with b new rows plus a PosteriorMarginals refresh at every node, against rebuilding the posterior on the n + b rows
(constructor + variance + mean at every node).

    python profiles/prof_condition.py --out DIR [--reps 3] [--configs 2,4]

Cases: config 2 (the 316^2 grid, W = 100, L = 5) and config 4 (R-MAT 2^22 nodes, 7e7 edges, W = 100, L = 5), each
with n in {100, 600, 4096} random training nodes and b in {1, 16, 50, 100} new ones.  b + 1 <= 64 columns take the
row_condition pass; b = 100 takes row_quadform on the new columns plus a row_project onto a.  Per case, medians over
--reps after one warm-up of CUDA-event times of:
  - the stages of condition_on ("cross", "factor", "append", "weights");
  - the refresh pass over every node;
  - the rebuild: constructor (merge .. solve), variance and mean;
  - allocating the grown C and copying the old columns into it alone (part of "append": what spare capacity in C
    would save);
the refresh's algorithmic bytes (12 B per streamed entry of Phi_f, 4 k B of B per touched entry, and per row
the 8 B read and 8 B write of q, 4 B of d, 4 B of var and 4 B of mean) over its time, and the largest difference of
the refreshed variance and mean from the rebuild's; and, for the selection between the two refresh paths, both
on the same k = 8 .. 63 new columns (alternated, CUDA events around each whole path).  Card name and power limit
are read in the same run and written with the results (DIR/condition.json)."""

import argparse
import copy
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "efficient-gaussian-process-on-graphs_b200"), os.path.dirname(__file__)]

from prof_posterior_variance import card, phi_of  # noqa: E402


def _ms(ev, a, b):
    return ev[a].elapsed_time(ev[b])


def _clone(post, marg):
    """A copy of the posterior and its marginals: condition_on replaces the posterior's tensors it changes, a
    refresh updates q, var and mean in place."""
    p = copy.copy(post)
    m = copy.copy(marg)
    m.post = p
    for k in ("q", "d", "_var", "_mean"):
        if getattr(m, k) is not None:
            setattr(m, k, getattr(m, k).clone())
    return p, m


def refresh_bytes(post, k, wm):
    ptr = post.phi_f.blk_ptr.long()
    ent = post.phi_f.entries
    streamed = int(ent.shape[0])
    touched = int((post.slot[ent[:, 0].long()] >= 0).sum().item())
    rows = int(ptr.numel() - 1)
    return 12 * streamed + 4 * (k + wm) * touched + (24 + 4 * wm) * rows, streamed, touched


def run_case(name, phi, n, reps):
    import torch

    from grf_b200.posterior import ExactPosterior

    dev = phi.device
    rng = np.random.default_rng(n)
    nodes = torch.tensor(rng.choice(phi.n_rows, n + 100, replace=False), device=dev)
    yall = torch.sin(nodes.double() / 1000.0)
    f = torch.tensor([1.0 / (1 + p) ** 2 for p in range(phi.n_steps)])
    xt = torch.arange(phi.n_rows, device=dev, dtype=torch.int32)
    base = ExactPosterior(phi, f, nodes[:n], 0.1, y_train=yall[:n])
    bmarg = base.marginals(xt)
    out = []
    for b in (1, 16, 50, 100):
        xb, yb = nodes[n:n + b], yall[n:n + b]
        times = []
        for rep in range(reps + 1):
            post, marg = _clone(base, bmarg)
            ev = {}
            post.events = ev
            torch.cuda.synchronize()
            post.condition_on(xb, yb)
            marg.refresh()
            torch.cuda.synchronize()
            rb = {}
            fresh = ExactPosterior(phi, f, nodes[:n + b], 0.1, events=rb, y_train=yall[:n + b])
            var_f = fresh.variance(xt)
            mean_f = fresh.mean(xt)
            torch.cuda.synchronize()
            t = {"cross_ms": _ms(ev, "condition_start", "cross"), "factor_ms": _ms(ev, "cross", "factor"),
                 "append_ms": _ms(ev, "factor", "append"), "weights_ms": _ms(ev, "append", "weights"),
                 "condition_ms": _ms(ev, "condition_start", "weights"), "refresh_ms": _ms(ev, "refresh_start", "refresh"),
                 "rebuild_constructor_ms": _ms(rb, "start", "solve"),
                 "rebuild_variance_ms": _ms(rb, "quadform_start", "quadform"),
                 "rebuild_mean_ms": _ms(rb, "project_start", "project")}
            t["update_ms"] = t["condition_ms"] + t["refresh_ms"]
            t["rebuild_ms"] = t["rebuild_constructor_ms"] + t["rebuild_variance_ms"] + t["rebuild_mean_ms"]
            if rep:
                times.append(t)
            if rep == reps:
                dv = (marg.variance() - var_f).abs()
                dm = (marg.mean - mean_f).abs()
                diff = {"max_abs_var_diff": float(dv.max()), "max_var": float(var_f.max()),
                        "max_abs_mean_diff": float(dm.max()), "max_abs_mean": float(mean_f.abs().max())}
            del fresh, var_f, mean_f, post, marg
            torch.cuda.empty_cache()
        # what spare capacity in C would save: the new C and the copy of the old columns into it, alone
        for rep in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            C = torch.zeros((base.m, (n + b + 3) // 4 * 4), dtype=torch.float32, device=dev)
            C[:, :n] = base.C[:, :n]
            e1.record()
            torch.cuda.synchronize()
            del C
            if rep:
                times[rep - 1]["realloc_copy_ms"] = e0.elapsed_time(e1)
        med = {k: float(np.median([t[k] for t in times])) for k in times[0]}
        entry = {"case": name, "n_train": n, "b": b, "refresh_path": "row_condition" if b + 1 <= 64 else
                 "row_quadform + row_project", "m": base.m, "median_ms": med, "times_ms": times, **diff,
                 "speedup": med["rebuild_ms"] / med["update_ms"]}
        if b + 1 <= 64:
            nb, streamed, touched = refresh_bytes(_m_after(base, xb), b, 1)
            entry.update(refresh_bytes=nb, streamed_entries=streamed, touched_entries=touched,
                         refresh_GB_per_s=nb / (med["refresh_ms"] * 1e6))
        print(json.dumps({k: v for k, v in entry.items() if k != "times_ms"}), flush=True)
        out.append(entry)
    sel = selection(name, base, bmarg, nodes, yall, n, reps)
    del base, bmarg
    torch.cuda.empty_cache()
    return out, sel


def selection(name, base, bmarg, nodes, yall, n, reps):
    """The two refresh paths on the same k new columns of C (after conditioning on 63 rows), alternated:
    row_condition over [C_new[:, :k] | a] against row_quadform on C_new[:, :k] plus row_project onto a."""
    import torch

    post, marg = _clone(base, bmarg)
    post.condition_on(nodes[n:n + 63], yall[n:n + 63])
    one = torch.ones(1, device=post.device)
    res = {"case": name, "n_train": n, "selection": []}
    for k in (8, 16, 17, 32, 48, 63):
        cols = post.C[:, n:n + k]

        def fused():
            B = torch.empty((post.m, k + 1), dtype=torch.float32, device=post.device)
            B[:, :k] = cols
            B[:, k] = post.a[:, 0]
            post.phi_f.row_condition(one, marg.x, post.slot, B, k, True, marg.q.clone(), marg.d, marg._var,
                                     marg._mean)

        def split():
            dq, _ = post.phi_f.row_quadform(one, marg.x, post.slot, cols)
            q = marg.q + dq.to(torch.float64)
            torch.clamp_min((marg.d.to(torch.float64) - q).to(torch.float32), 0.0)
            post.phi_f.row_project(one, marg.x, post.slot, post.a)

        t = {"row_condition_ms": [], "quadform_project_ms": []}
        for rep in range(reps + 1):
            for key, fn in (("row_condition_ms", fused), ("quadform_project_ms", split)):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                torch.cuda.synchronize()
                if rep:
                    t[key].append(a.elapsed_time(b))
        entry = {"k": k, **{key: float(np.median(v)) for key, v in t.items()}, "times_ms": t}
        print(json.dumps({"case": name, "n_train": n, **{kk: v for kk, v in entry.items() if kk != "times_ms"}}),
              flush=True)
        res["selection"].append(entry)
    del post, marg
    return res


def _m_after(base, xb):
    """The slot map after conditioning (touched entries are counted against it)."""
    p = copy.copy(base)          # condition_on replaces the tensors it changes, so base stays as it was
    p.events = None
    return p.condition_on(xb, base.y.new_zeros(xb.numel()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--configs", default="2,4")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("prof_condition needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {"card": card(), "torch": torch.__version__, "cases": [], "selection": []}
    for config in (int(c) for c in a.configs.split(",")):
        phi = phi_of(config, dev)
        for n in (100, 600, 4096):
            cases, sel = run_case(f"config{config}_W100_L5", phi, n, a.reps)
            out["cases"] += cases
            out["selection"].append(sel)
        del phi
        torch.cuda.empty_cache()
        with open(os.path.join(a.out, "condition.json"), "w") as fh:     # after each config
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
