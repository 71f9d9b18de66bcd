#!/usr/bin/env python
"""Missing-data logpdf of the dense model against its value + gradient (lmm_ilmm_masked_logpdf_grad): p = 8, m = 4, N = 2048
with 20 % of the entries missing at random (nobs ≈ 13 100), SE + Periodic sum latents, D = 1.

Default: after one warm-up call of each, `--reps` rounds that call the two in turn; each call is timed by the library's CUDA
events (lmm_ctx_last_timings()[0]) and by the host clock.  The medians, the card's name and power limit go to one JSON line
and to OUT/r04_missing_grad_timing.json.  `--profile`: a separate run, one call of each under torch.profiler (CUDA
activities), kernel times summed by name; the share of the new contraction kernels (kgrad_masked_*, the per-term finish and
the diagonal sum) in the value + gradient call's kernel time goes to OUT/r04_missing_grad_kernels.json."""
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

N, P, M, MISSING = 2048, 8, 4, 0.2
CONTRACTION = ("kgrad_masked", "kgrad_terms_finish", "sym_diag_sum")


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True).stdout.strip()
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


def problem():
    rng = np.random.default_rng(0)
    x = np.sort(rng.uniform(0, N / 100.0, N))
    H = rng.uniform(0.2, 1.2, (P, M))
    s = np.random.default_rng(2).uniform(0.5, 2.0, M)
    ks = [lmm.SEKernel().compose(lmm.ScaleTransform(float(s[i]))) + 0.5 * lmm.PeriodicKernel(1.3).compose(lmm.ScaleTransform(float(s[i])))
          for i in range(M)]
    y = rng.standard_normal(P * N)
    y[rng.uniform(size=P * N) < MISSING] = np.nan
    fx = lmm.ILMM(lmm.independent_mogp([lmm.GP(k) for k in ks]), H)(lmm.MOInputIsotopicByOutputs(x, P), 0.1)
    calls = {"logpdf_only": lambda: lmm.logpdf_missing(fx, y),
             "value_and_gradient": lambda: lmm.logpdf_missing_and_gradient(fx, y, with_grad_y=True, kernel_terms=True)}
    return calls, int(np.sum(~np.isnan(y)))


def shape(nobs):
    return f"dense missing-data ILMM p={P} m={M} N={N} D=1, {int(MISSING * 100)}% missing at random, nobs={nobs}, SE + Periodic sums"


def timing(reps, out):
    ctx = lmm.default_context()
    calls, nobs = problem()
    vals = {k: f() for k, f in calls.items()}  # warm-up of both shapes
    lp0, lp1 = vals["logpdf_only"], vals["value_and_gradient"][0]
    dev = {k: [] for k in calls}
    wall = {k: [] for k in calls}
    for _ in range(reps):
        for k, f in calls.items():  # alternate
            t0 = time.perf_counter()
            f()
            wall[k].append((time.perf_counter() - t0) * 1e3)
            dev[k].append(float(ctx.last_timings()[0]))
    res = {"shape": shape(nobs), "reps": reps, **card(), "logpdf_rel_diff": abs(lp0 - lp1) / abs(lp0)}
    for k in calls:
        res[k] = {"device_ms_median": statistics.median(dev[k]), "wall_ms_median": statistics.median(wall[k]),
                  "device_ms_min": min(dev[k]), "device_ms_max": max(dev[k])}
    res["ratio_value_and_gradient_over_logpdf"] = res["value_and_gradient"]["device_ms_median"] / res["logpdf_only"]["device_ms_median"]
    with open(os.path.join(out, "r04_missing_grad_timing.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res), flush=True)


def profile(out):
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile

    calls, nobs = problem()
    for f in calls.values():
        f()
    torch.cuda.synchronize()
    res = {"shape": shape(nobs), **card()}
    for k, f in calls.items():
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            f()
            torch.cuda.synchronize()
        by = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                by[ev.name] = by.get(ev.name, 0.0) + ev.device_time_total / 1e3
        total = sum(by.values())
        contraction = sum(ms for name, ms in by.items() if any(c in name for c in CONTRACTION))
        top = sorted(by.items(), key=lambda kv: -kv[1])[:12]
        res[k] = {"kernel_ms_total": total, "contraction_ms": contraction, "contraction_share": contraction / total if total else 0.0,
                  "top_kernels_ms": dict(top)}
    with open(os.path.join(out, "r04_missing_grad_kernels.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--profile", action="store_true", help="torch.profiler run instead of the timing run")
    ap.add_argument("--out", default="profiles", help="directory of the JSON output (default: profiles)")
    a = ap.parse_args()
    if a.reps < 5:
        ap.error("--reps must be at least 5")
    os.makedirs(a.out, exist_ok=True)
    if a.profile:
        profile(a.out)
    else:
        timing(a.reps, a.out)


if __name__ == "__main__":
    main()
