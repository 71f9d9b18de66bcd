#!/usr/bin/env python
"""Leave-one-input-out cross-validation at the C3 shape: an OILMM (p = 64, m = 16, N = 8192, D = 1) with SE latents and
with SE + Periodic sums.  Four calls per family: lmm_oilmm_logpdf (value), lmm_oilmm_loo without gradient outputs (the
LOO value path), lmm_oilmm_logpdf_grad_terms (the training gradient) and lmm_oilmm_loo with every gradient output.

Default: after one warm-up call of each, `--reps` rounds that call the four in turn; each call ends in a device
synchronise, so the host clock around it is the call's time.  Medians are written with the card's name and power limit and
the achieved FP64 rate of the two LOO calls against the flop model below.  `--profile`: a separate run, one call of each
under torch.profiler (CUDA activities), kernel times summed by name, with the share of the kernels the LOO adds
(loo_terms, sym_expand_scale, loo_grad_vectors) in each call's kernel time.
Output: one JSON line on stdout and profiles/r09_loo_{timing,kernels}.json (or --out DIR)."""
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

N, P, M = 8192, 64, 16
LOO_KERNELS = ("loo_terms", "sym_expand_scale", "loo_grad_vectors")


def flops_loo_value(n):
    """FP64 flops per latent of the LOO value path: the factorisation (N³/3) and X = L⁻ᵀ (triangular TRSM, N³/3)."""
    return 2 * n ** 3 / 3


def flops_loo_grad(n):
    """FP64 flops per latent of the LOO value and gradient: the value path plus -A = -XX' (triangular SYRK, N³/3) and -2BB' with B = A R^{1/2} full (SYRK, N³): 2N³ in all."""
    return flops_loo_value(n) + n ** 3 / 3 + n ** 3


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
        "se": [sc(lmm.SEKernel(), i) for i in range(M)],
        "se_plus_periodic": [sc(lmm.SEKernel(), i) + 0.5 * sc(lmm.PeriodicKernel(1.3), i) for i in range(M)],
    }
    O = lmm.MOInputIsotopicByOutputs
    calls = {}
    for name, ks in fams.items():
        fx = lmm.ILMM(lmm.independent_mogp([lmm.GP(k) for k in ks]), lmm.Orthogonal(U, S))(O(x, P), 0.1)
        calls[name] = {
            "logpdf": lambda fx=fx: lmm.logpdf(fx, y),
            "loo_value": lambda fx=fx: lmm.loo_logpdf(fx, y),
            "train_logpdf_grad_terms": lambda fx=fx: lmm.logpdf_and_gradient(fx, y, with_grad_y=True, kernel_terms=True),
            "loo_value_grad": lambda fx=fx: lmm.loo_logpdf_and_gradient(fx, y, with_grad_y=True),
        }
    return calls


def timing(reps, out):
    import torch

    calls = problem()
    for fam in calls.values():
        for f in fam.values():  # warm-up of every shape
            f()
    torch.cuda.synchronize()
    res = {"shape": f"C3 OILMM p={P} m={M} N={N} D=1", "reps": reps, **card(), "flops_loo_value_per_latent": flops_loo_value(N),
           "flops_loo_grad_per_latent": flops_loo_grad(N), "flops_train_grad_per_latent": float(N) ** 3}
    for fam, fs in calls.items():
        wall = {k: [] for k in fs}
        for _ in range(reps):
            for k, f in fs.items():  # calls alternate
                t0 = time.perf_counter()
                f()
                wall[k].append((time.perf_counter() - t0) * 1e3)
        r = {k: {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v)} for k, v in wall.items()}
        val, grad = r["loo_value"]["ms_median"], r["loo_value_grad"]["ms_median"]
        r["loo_value_over_logpdf"] = val / r["logpdf"]["ms_median"]
        r["loo_grad_over_train_grad"] = grad / r["train_logpdf_grad_terms"]["ms_median"]
        r["loo_value_tflops"] = M * flops_loo_value(N) / (val * 1e-3) / 1e12
        r["loo_grad_tflops"] = M * flops_loo_grad(N) / (grad * 1e-3) / 1e12
        res[fam] = r
    with open(os.path.join(out, "r09_loo_timing.json"), "w") as fh:
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
    res = {"shape": f"C3 OILMM p={P} m={M} N={N} D=1", **card()}
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
            new = sum(ms for name, ms in by.items() if any(n in name for n in LOO_KERNELS))
            res[fam][k] = {"kernel_ms_total": total, "loo_kernels_ms": new, "loo_kernels_share": new / total if total else 0.0,
                           "top_kernels_ms": dict(sorted(by.items(), key=lambda kv: -kv[1])[:14])}
    with open(os.path.join(out, "r09_loo_kernels.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true", help="torch.profiler run instead of the timing run")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"), help="directory of the JSON output")
    a = ap.parse_args()
    if a.reps < 3:
        ap.error("--reps must be at least 3")
    os.makedirs(a.out, exist_ok=True)
    if a.profile:
        profile(a.out)
    else:
        timing(a.reps, a.out)


if __name__ == "__main__":
    main()
