"""Cost of the exact marginal likelihood (grf_b200/mll.py): the per-length training Gram E built once
(PhiBlocks.training_gram: gather, light kernel, hub columns' H H^T, symmetrise), then one loss + backward per
evaluation, against one neg_mll_backward call at the reference setting (16 probes, cg_tolerance = 1e-2).

    python profiles/prof_exact_mll.py --out DIR [--reps 3] [--configs 2,4]

Cases: config 2 (the 316^2 grid) and config 4 (R-MAT 2^22 nodes, 7e7 edges), W = 100, L = 5, each with n in
{100, 600, 4096} random training nodes (the seeds of prof_posterior_variance.py).  Per case:
  - CUDA-event times of the Gram stages at the default hub threshold T (medians over --reps after a warm-up), with
    nnz_train, m (touched columns), h (hub columns), P_light = sum over light slots of t_s^2 and the light kernel's
    algorithmic bytes: per product of the upper triangle (sum_s t_s (t_s + 1) / 2 of them) the float64 E element
    read and written and the 8-byte slot-list entry, plus 8 B per row entry and its slot bounds;
  - the whole Gram at other thresholds, alternated in one loop (T = 0 is the dense alternative, the stacked G_l
    float64 GEMM over every touched column; it is run where its H fits, n <= 600);
  - loss + backward per evaluation, and one neg_mll_backward call.
Card name and power limit are read in the same run and written with the results (DIR/exact_mll.json)."""

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "efficient-gaussian-process-on-graphs_b200"), os.path.dirname(__file__)]

from prof_posterior_variance import card, phi_of  # noqa: E402

STAGES = ("gather", "light", "heavy", "symmetrise")
SWEEP = (0, 64, 256, 1024, 4096, 1 << 30)


def _gram_ms(phi, x, T):
    import torch

    from grf_b200 import engine

    engine.GRAM_HEAVY_THRESHOLD = T
    ev = {"start": torch.cuda.Event(enable_timing=True)}
    ev["start"].record()
    E, st = phi._training_gram(x, events=ev)
    torch.cuda.synchronize()
    t = {}
    prev = "start"
    for s in STAGES:
        t[s + "_ms"] = ev[prev].elapsed_time(ev[s])
        prev = s
    t["total_ms"] = ev["start"].elapsed_time(ev["symmetrise"])
    return E, st, t


def run_case(name, phi, n, reps):
    import torch

    from efficient_graph_gp_sparse.gptorch_kernels_sparse import SparseGRFKernel
    from grf_b200 import engine
    from grf_b200.gp_compat import GaussianLikelihood
    from grf_b200.mll import ExactMLL, neg_mll_backward

    dev = phi.device
    default_T = engine.GRAM_HEAVY_THRESHOLD
    rng = np.random.default_rng(n)
    x = torch.tensor(rng.choice(phi.n_rows, n, replace=False), device=dev)
    y = torch.sin(x.double() / 1000.0) + 0.1 * torch.randn(n, dtype=torch.float64, device=dev,
                                                           generator=torch.Generator(device=dev).manual_seed(n))
    res = {"case": name, "n_train": n, "default_threshold": default_T}

    # the Gram at the default threshold: stages and sizes
    E, st, _ = _gram_ms(phi, x, default_T)                   # warm-up
    E_default = E
    times = [_gram_ms(phi, x, default_T)[2] for _ in range(reps)]
    res.update(st)
    res["median_stages_ms"] = {k: float(np.median([t[k] for t in times])) for k in times[0]}

    # light kernel bytes: the products of the upper triangle, from the per-slot counts
    xl = x.long()
    ptr = phi.blk_ptr.long()
    L = phi.n_steps
    start, lens = ptr[xl * L], ptr[(xl + 1) * L] - ptr[xl * L]
    i = torch.repeat_interleave(torch.arange(n, device=dev), lens)
    idx = start[i] + torch.arange(int(lens.sum()), device=dev) - (torch.cumsum(lens, 0) - lens)[i]
    cols = phi.entries[idx, 0].long() & ((1 << 27) - 1)
    t_s = torch.unique(cols, return_counts=True)[1]
    lt = t_s[t_s <= default_T]
    upper = int((lt * (lt + 1) // 2).sum())
    light_entries = int(lt.sum())
    res["light_upper_products"] = upper
    res["light_bytes"] = 24 * upper + 16 * light_entries
    res["light_GB_per_s"] = res["light_bytes"] / (res["median_stages_ms"]["light_ms"] * 1e6)

    # other thresholds, alternated (they differ from the default only in how the sums round)
    sweep = [T for T in SWEEP if T != 0 or engine.training_gram_bytes(n, L, st["m"]) < 40 << 30]
    per_T = {T: [] for T in sweep}
    scale = float(E_default.abs().max())
    worst = 0.0
    for _ in range(reps):
        for T in sweep:
            E2, st2, t = _gram_ms(phi, x, T)
            per_T[T].append(t["total_ms"])
            worst = max(worst, float((E2 - E_default).abs().max()) / scale)
            del E2
    res["threshold_sweep_ms"] = {str(T): float(np.median(v)) for T, v in per_T.items()}
    res["threshold_sweep_h"] = {str(T): int((t_s > T).sum()) for T in sweep}
    res["threshold_sweep_max_rel_diff"] = worst
    engine.GRAM_HEAVY_THRESHOLD = default_T
    del E

    # per evaluation
    mll = ExactMLL(phi, x, y)
    f = torch.tensor([1.0 / (1 + p) ** 2 for p in range(L)], dtype=torch.float64, requires_grad=True)
    noise = torch.tensor(0.1, dtype=torch.float64, requires_grad=True)
    for _ in range(2):
        mll.loss(f, noise).backward()
    torch.cuda.synchronize()
    ev_times = []
    for _ in range(max(reps, 5)):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        loss = mll.loss(f, noise)
        loss.backward()
        b.record()
        torch.cuda.synchronize()
        ev_times.append(a.elapsed_time(b))
    res["eval_ms"] = float(np.median(ev_times))
    res["loss"] = loss.item()
    del mll

    # one neg_mll_backward call at the reference setting
    kern = SparseGRFKernel(L, None).to(dev)
    kern._blocks = phi
    with torch.no_grad():
        kern.raw_modulator_vector.copy_(f.detach().float())
    lik = GaussianLikelihood().to(dev)
    lik.noise = 0.1
    gen = torch.Generator(device=dev).manual_seed(0)
    neg_mll_backward(kern, lik, x, y.float(), num_probes=16, cg_tolerance=1e-2, generator=gen)
    torch.cuda.synchronize()
    cg_times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = neg_mll_backward(kern, lik, x, y.float(), num_probes=16, cg_tolerance=1e-2, generator=gen)
        b.record()
        torch.cuda.synchronize()
        cg_times.append(a.elapsed_time(b))
    res["neg_mll_backward_ms"] = float(np.median(cg_times))
    res["neg_mll_backward_loss"] = out["loss"]
    res["neg_mll_backward_cg_iterations"] = out["cg_iterations"]
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--configs", default="2,4")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("prof_exact_mll needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {"card": card(), "torch": torch.__version__, "cases": []}
    for config in (int(c) for c in a.configs.split(",")):
        phi = phi_of(config, dev)
        for n in (100, 600, 4096):
            out["cases"].append(run_case(f"config{config}_W100_L5", phi, n, a.reps))
            torch.cuda.empty_cache()
        del phi
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "exact_mll.json"), "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
