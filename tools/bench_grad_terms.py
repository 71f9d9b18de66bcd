#!/usr/bin/env python
"""Value + gradient of the OILMM logpdf at the C3 shape (p = 64, m = 16, N = 8192, D = 1) for four latent families:
(a) SE latents through lmm_oilmm_logpdf_grad, (b) the same through lmm_oilmm_logpdf_grad_terms, (c) SE + Periodic sums,
(d) Matern52 * Periodic products -- what the per-term kernel-gradient contraction (kgrad_terms_kernel) adds to a call.

Default: after one warm-up call per variant, `--reps` rounds that call the variants in turn; each call is timed by the
library's CUDA events (lmm_ctx_last_timings()[0]) and by the host clock; the medians are printed as one JSON line with the
card's name and power limit.  `--profile DIR`: a separate run, one call per variant under torch.profiler (CUDA activities),
kernel times summed by name into DIR/grad_terms_kernels.json (the new kernel next to the potri GEMMs)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lmm_b200 as lmm  # noqa: E402

N, P, M = 8192, 64, 16


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True).stdout.strip()
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


def problem():
    rng = np.random.default_rng(0)
    x = np.sort(rng.uniform(0, N / 100.0, N))
    U, S, _ = np.linalg.svd(np.random.default_rng(1).uniform(0, 1, (P, M)), full_matrices=False)
    s = np.random.default_rng(2).uniform(0.5, 2.0, M)
    y = rng.standard_normal(P * N)
    sc = lambda k, i: k.compose(lmm.ScaleTransform(float(s[i])))  # noqa: E731
    fams = {
        "a_se_single_entry": [sc(lmm.SEKernel(), i) for i in range(M)],
        "c_se_plus_periodic": [sc(lmm.SEKernel(), i) + 0.5 * sc(lmm.PeriodicKernel(1.3), i) for i in range(M)],
        "d_matern52_times_periodic": [sc(lmm.Matern52Kernel(), i) * sc(lmm.PeriodicKernel(1.3), i) for i in range(M)],
    }
    fxs = {k: lmm.ILMM(lmm.independent_mogp([lmm.GP(kk) for kk in ks]), lmm.Orthogonal(U, S))(lmm.MOInputIsotopicByOutputs(x, P), 0.1)
           for k, ks in fams.items()}
    calls = {
        "a_se_single_entry": lambda: lmm.logpdf_and_gradient(fxs["a_se_single_entry"], y, with_grad_y=True),
        "b_se_terms_entry": lambda: lmm.logpdf_and_gradient(fxs["a_se_single_entry"], y, with_grad_y=True, kernel_terms=True),
        "c_se_plus_periodic": lambda: lmm.logpdf_and_gradient(fxs["c_se_plus_periodic"], y, with_grad_y=True, kernel_terms=True),
        "d_matern52_times_periodic": lambda: lmm.logpdf_and_gradient(fxs["d_matern52_times_periodic"], y, with_grad_y=True, kernel_terms=True),
    }
    return calls


def timing(reps):
    ctx = lmm.default_context()
    calls = problem()
    out = {k: f() for k, f in calls.items()}  # warm-up of every shape
    # the _terms entry point leaves the single-kernel outputs bit-identical
    ga, gb = out["a_se_single_entry"][1], out["b_se_terms_entry"][1]
    same = all(np.array_equal(ga[k], gb[k]) for k in ("variance", "inv_lengthscale", "mean_const", "y", "U", "S"))
    dev = {k: [] for k in calls}
    wall = {k: [] for k in calls}
    for _ in range(reps):
        for k, f in calls.items():  # variants alternate
            t0 = time.perf_counter()
            f()
            wall[k].append((time.perf_counter() - t0) * 1e3)
            dev[k].append(float(ctx.last_timings()[0]))
    res = {"shape": f"C3 OILMM p={P} m={M} N={N} D=1", "reps": reps, **card(), "single_outputs_identical_a_vs_b": bool(same)}
    for k in calls:
        res[k] = {"device_ms_median": statistics.median(dev[k]), "wall_ms_median": statistics.median(wall[k]),
                  "device_ms_min": min(dev[k]), "device_ms_max": max(dev[k])}
    print(json.dumps(res), flush=True)


def profile(outdir):
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile

    calls = problem()
    for f in calls.values():
        f()
    torch.cuda.synchronize()
    res = {"shape": f"C3 OILMM p={P} m={M} N={N} D=1", **card()}
    for k, f in calls.items():
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            f()
            torch.cuda.synchronize()
        by = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                by[ev.name] = by.get(ev.name, 0.0) + ev.device_time_total / 1e3
        total = sum(by.values())
        groups = {"kgrad_terms": 0.0, "kgrad_single": 0.0, "gemm (potrf updates, potri TRSM / SYRK)": 0.0}
        for name, ms in by.items():
            if "kgrad_terms" in name:
                groups["kgrad_terms"] += ms
            elif "kgrad" in name:
                groups["kgrad_single"] += ms
            elif "gemm" in name.lower():
                groups["gemm (potrf updates, potri TRSM / SYRK)"] += ms
        top = sorted(by.items(), key=lambda kv: -kv[1])[:12]
        res[k] = {"kernel_ms_total": total, "groups_ms": groups, "kgrad_terms_share": groups["kgrad_terms"] / total if total else 0.0,
                  "top_kernels_ms": dict(top)}
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, "grad_terms_kernels.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--profile", metavar="DIR", help="torch.profiler run instead of the timing run; summary written to DIR")
    a = ap.parse_args()
    if a.reps < 5:
        ap.error("--reps must be at least 5")
    if a.profile:
        profile(a.profile)
    else:
        timing(a.reps)


if __name__ == "__main__":
    main()
