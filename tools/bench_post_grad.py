#!/usr/bin/env python
"""Posterior-predictive logpdf gradient through the conditioning at the C3 shape: an OILMM posterior (p = 64, m = 16,
N = 8192, D = 1) scored at N* = 1024 test points, with SE latents and with SE + Periodic sums.  Four calls per family:
lmm_post_logpdf (value), lmm_post_logpdf_grad (σ*², y*), lmm_post_logpdf_grad_full (the new call) and
lmm_oilmm_logpdf_grad_terms on the training data (the training gradient at the same N).

Default: after one warm-up call of each, `--reps` rounds that call the four in turn; each call ends in a device
synchronise, so the host clock around it is the call's time.  Medians are written with the card's name and power limit and
the achieved FP64 rate of the new call against its flop model (`flops_full` below).  `--profile`: a separate run, one call
of each under torch.profiler (CUDA activities), kernel times summed by name, with the share of the three gradient
contractions (kgrad_terms_kernel twice, kgrad_cross_terms_kernel) in the new call's kernel time.
Output: one JSON line on stdout and profiles/r05_post_grad_{timing,kernels}.json (or --out DIR)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lmm_b200 as lmm  # noqa: E402

N, NS, P, M = 8192, 1024, 64, 16


def flops_full(n, ns):
    """FP64 flops per latent of lmm_post_logpdf_grad_full: the predictive factor of lmm_post_logpdf_grad (V = K(x*,x) L⁻ᵀ,
    K** - VV', chol, L*⁻ᵀ) plus X = L⁻ᵀ, V again, W = X V' (X triangular), Φ = W L*⁻ᵀ, X* = L*⁻ᵀ, -X*X*', Φ X*' and ΦΦ'."""
    pred = n * ns * n + ns * ns * n + ns ** 3 / 3 + ns ** 3 / 3
    grad = n ** 3 / 3 + n * ns * n + n * ns * n + n * ns * ns + ns ** 3 / 3 + ns ** 3 / 3 + 2 * n * ns * ns + n * n * ns
    return pred + grad


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True).stdout.strip()
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


def problem():
    rng = np.random.default_rng(0)
    xa = np.sort(rng.uniform(0, (N + NS) / 100.0, N + NS))
    x, xs = xa[:N], xa[N:]  # forecast: the test points follow the training points
    U, S, _ = np.linalg.svd(np.random.default_rng(1).uniform(0, 1, (P, M)), full_matrices=False)
    s = np.random.default_rng(2).uniform(0.5, 2.0, M)
    y, ys = rng.standard_normal(P * N), rng.standard_normal(P * NS)
    sc = lambda k, i: k.compose(lmm.ScaleTransform(float(s[i])))  # noqa: E731
    fams = {
        "se": [sc(lmm.SEKernel(), i) for i in range(M)],
        "se_plus_periodic": [sc(lmm.SEKernel(), i) + 0.5 * sc(lmm.PeriodicKernel(1.3), i) for i in range(M)],
    }
    O = lmm.MOInputIsotopicByOutputs
    calls = {}
    for name, ks in fams.items():
        f = lmm.ILMM(lmm.independent_mogp([lmm.GP(k) for k in ks]), lmm.Orthogonal(U, S))
        fx = f(O(x, P), 0.1)
        fxp = lmm.posterior(fx, y)(O(xs, P), 0.1)
        calls[name] = {
            "post_logpdf": lambda fxp=fxp: lmm.logpdf(fxp, ys),
            "post_logpdf_grad": lambda fxp=fxp: lmm.logpdf_and_gradient(fxp, ys, with_grad_y=True),
            "post_logpdf_grad_full": lambda fxp=fxp: lmm.predictive_logpdf_and_gradient(fxp, ys, y, with_grad_y=True),
            "train_logpdf_grad_terms": lambda fx=fx: lmm.logpdf_and_gradient(fx, y, with_grad_y=True, kernel_terms=True),
        }
    return calls


def timing(reps, out):
    import torch

    calls = problem()
    for fam in calls.values():
        for f in fam.values():  # warm-up of every shape
            f()
    torch.cuda.synchronize()
    res = {"shape": f"C3 OILMM posterior p={P} m={M} N={N} N*={NS} D=1", "reps": reps, **card(),
           "flops_full_per_latent": flops_full(N, NS), "flops_train_grad_per_latent": float(N) ** 3}
    for fam, fs in calls.items():
        wall = {k: [] for k in fs}
        for _ in range(reps):
            for k, f in fs.items():  # calls alternate
                t0 = time.perf_counter()
                f()
                wall[k].append((time.perf_counter() - t0) * 1e3)
        r = {k: {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v)} for k, v in wall.items()}
        full = r["post_logpdf_grad_full"]["ms_median"]
        r["full_over_train_grad"] = full / r["train_logpdf_grad_terms"]["ms_median"]
        r["full_tflops"] = M * flops_full(N, NS) / (full * 1e-3) / 1e12
        res[fam] = r
    with open(os.path.join(out, "r05_post_grad_timing.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res), flush=True)


def profile(out):
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile

    calls = problem()
    for fam in calls.values():
        for f in fam.values():
            f()
    torch.cuda.synchronize()
    res = {"shape": f"C3 OILMM posterior p={P} m={M} N={N} N*={NS} D=1", **card()}
    for fam, fs in calls.items():
        res[fam] = {}
        for k, f in fs.items():
            with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
                f()
                torch.cuda.synchronize()
            by = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA:
                    by[ev.name] = by.get(ev.name, 0.0) + ev.device_time_total / 1e3
            total = sum(by.values())
            contr = sum(ms for name, ms in by.items() if "kgrad_terms" in name or "kgrad_cross_terms" in name)
            res[fam][k] = {"kernel_ms_total": total, "contraction_ms": contr, "contraction_share": contr / total if total else 0.0,
                           "top_kernels_ms": dict(sorted(by.items(), key=lambda kv: -kv[1])[:14])}
    with open(os.path.join(out, "r05_post_grad_kernels.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--profile", action="store_true", help="torch.profiler run instead of the timing run")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory of the JSON output")
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
