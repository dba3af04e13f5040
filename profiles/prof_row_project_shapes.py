"""grf_phi_row_project: the warp shape chosen for r against the 128-column panels forced for every r.

    python profiles/prof_row_project_shapes.py --out DIR [--reps 7] [--configs 2,4]

The panel form (row_project_kernel) serves every r > 64.  For r <= 4 the library takes row_project_narrow_kernel
(lanes own entries) and for 4 < r <= 64 row_project_mid_kernel (entry groups x column quads).  This script builds,
in a temporary directory, a second library from csrc/grf_api.cu and csrc/grf_posterior.cu with those two branches
of the dispatch removed, so the same call runs the panels at every r.  On config 2 (the 316^2 grid) and config 4
(R-MAT 2^22 nodes), W = 100, L = 5, with the slot map of n = 100, 600 and 4096 random training nodes and every node
as a projected row, it times both libraries at r = 1, 4, 16 and 64 (CUDA events, one call each in alternation,
median of --reps after a warm-up) and reports the largest difference of the two results next to the largest
magnitude.  Card name and power limit are read in the same run (DIR/row_project_shapes.json)."""

import argparse
import ctypes
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "efficient-gaussian-process-on-graphs_b200")
sys.path[:0] = [ROOT, PKG, os.path.dirname(os.path.abspath(__file__))]

from prof_posterior_variance import card, phi_of  # noqa: E402

NARROW = "    if (r <= 4) {"
MID = "    if (r <= 64) {"


def panels_library(tmp):
    """The library with the narrow and mid branches of grf_phi_row_project's dispatch turned off."""
    csrc = os.path.join(PKG, "csrc")
    for name in ("grf_api.cu", "grf_common.cuh"):
        shutil.copy(os.path.join(csrc, name), tmp)
    src = open(os.path.join(csrc, "grf_posterior.cu")).read()
    assert src.count(NARROW) == 1 and src.count(MID) == 1, "the dispatch of grf_phi_row_project has changed"
    with open(os.path.join(tmp, "grf_posterior.cu"), "w") as fh:
        fh.write(src.replace(NARROW, "    if (false) {").replace(MID, "    if (false) {"))
    so = os.path.join(tmp, "libpanels.so")
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler",
                           "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-I", tmp, "-o", so,
                           os.path.join(tmp, "grf_api.cu"), os.path.join(tmp, "grf_posterior.cu")])
    return so


def project(lib, st, one, slot, B, out, n, r):
    import torch

    rc = lib.grf_phi_row_project(ctypes.byref(st), one.data_ptr(), None, n, slot.data_ptr(), B.data_ptr(), r, r,
                                 out.data_ptr(), r, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--configs", default="2,4")
    a = ap.parse_args()
    import torch

    from grf_b200 import _lib
    from grf_b200.posterior import ExactPosterior

    if not torch.cuda.is_available():
        raise SystemExit("prof_row_project_shapes needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    tmp = tempfile.mkdtemp(prefix="grf_row_project_")
    try:
        libs = {"chosen": _lib.lib(), "panels": ctypes.CDLL(panels_library(tmp))}
        libs["panels"].grf_phi_row_project.restype = ctypes.c_int32
        libs["panels"].grf_phi_row_project.argtypes = libs["chosen"].grf_phi_row_project.argtypes
        out = {"card": card(), "torch": torch.__version__, "cases": []}
        for config in (int(c) for c in a.configs.split(",")):
            phi = phi_of(config, dev)
            for n in (100, 600, 4096):
                rng = np.random.default_rng(n)
                x = torch.tensor(rng.choice(phi.n_rows, n, replace=False), device=dev)
                f = torch.tensor([1.0 / (1 + p) ** 2 for p in range(phi.n_steps)])
                post = ExactPosterior(phi, f, x, 0.1)
                st = post.phi_f.c_struct()
                one = torch.ones(1, device=dev)
                N = post.phi_f.n_rows
                for r in (1, 4, 16, 64):
                    B = torch.randn((post.m, r), device=dev)
                    res = {k: torch.empty((N, r), device=dev) for k in libs}
                    for k, lib in libs.items():       # warm-up
                        project(lib, st, one, post.slot, B, res[k], N, r)
                    torch.cuda.synchronize()
                    ms = {k: [] for k in libs}
                    for _ in range(a.reps):
                        for k, lib in libs.items():
                            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            t0.record()
                            project(lib, st, one, post.slot, B, res[k], N, r)
                            t1.record()
                            torch.cuda.synchronize()
                            ms[k].append(t0.elapsed_time(t1))
                    case = {"config": config, "n_train": n, "m": post.m, "r": r,
                            "chosen_ms": float(np.median(ms["chosen"])), "panels_ms": float(np.median(ms["panels"])),
                            "times_ms": ms, "max_abs_diff": float((res["chosen"] - res["panels"]).abs().max()),
                            "max_abs": float(res["panels"].abs().max())}
                    print(json.dumps({k: v for k, v in case.items() if k != "times_ms"}), flush=True)
                    out["cases"].append(case)
                del post
                torch.cuda.empty_cache()
            del phi
            torch.cuda.empty_cache()
        with open(os.path.join(a.out, "row_project_shapes.json"), "w") as fh:
            json.dump(out, fh, indent=1)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
