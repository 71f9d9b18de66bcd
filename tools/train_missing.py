#!/usr/bin/env python
"""Hyper-parameter learning on partially observed data: Adam on log(variance), log(inv_lengthscale) per latent and log(σ²)
of an ILMM (dense mixing matrix H, held at its true value) whose data were sampled from known hyper-parameters, with
`--missing` of the entries of y removed (NaN) at random.  Every step is one `lmm_ilmm_masked_logpdf_grad` call on the GPU
(the dense model on the observed entries).

    python tools/train_missing.py --N 1024 --m 3 --p 6 --steps 40
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lmm_b200 as lmm  # noqa: E402


def build(H, var, ils, kinds):
    ks = [(float(v) * (lmm.Matern32Kernel() if k == 0 else lmm.Matern52Kernel())).compose(lmm.ScaleTransform(float(s))) for v, s, k in zip(var, ils, kinds)]
    return lmm.ILMM(lmm.independent_mogp([lmm.GP(k) for k in ks]), H)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=1024)
    ap.add_argument("--p", type=int, default=6)
    ap.add_argument("--m", type=int, default=3)
    ap.add_argument("--missing", type=float, default=0.3)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--lr", type=float, default=0.08)
    args = ap.parse_args()
    rng = np.random.default_rng(0)
    N, p, m = args.N, args.p, args.m
    x = np.sort(rng.uniform(0, N / 50.0, N))
    H = rng.uniform(0.2, 1.2, (p, m))
    kinds = [i % 2 for i in range(m)]
    true_var, true_ils, true_s2 = rng.uniform(0.5, 2.0, m), rng.uniform(0.6, 1.8, m), 0.05
    f_true = build(H, true_var, true_ils, kinds)
    # latent draws through the IndependentMOGP sampler (1e-4 jitter keeps the smooth prior covariance numerically PD), mixed
    # and corrupted on the host, then a random share of the entries removed
    lat = lmm.rand(np.random.default_rng(1), f_true.f(lmm.MOInputIsotopicByOutputs(x, m), 1e-4)).reshape(m, N)
    y = (H @ lat + np.sqrt(true_s2) * np.random.default_rng(2).standard_normal((p, N))).reshape(-1)
    y[np.random.default_rng(3).uniform(size=p * N) < args.missing] = np.nan
    xin = lmm.MOInputIsotopicByOutputs(x, p)
    theta = np.zeros(2 * m + 1)  # log var, log ils, log σ²  (start at 1, 1, 1)
    mom, vel = np.zeros_like(theta), np.zeros_like(theta)
    t0 = time.perf_counter()
    hist = []
    for it in range(1, args.steps + 1):
        var, ils, s2 = np.exp(theta[:m]), np.exp(theta[m:2 * m]), float(np.exp(theta[-1]))
        lp, g = lmm.logpdf_missing_and_gradient(build(H, var, ils, kinds)(xin, s2), y)
        grad = np.concatenate([g["variance"] * var, g["inv_lengthscale"] * ils, [g["sigma2"] * s2]])  # chain rule to log-space
        mom = 0.9 * mom + 0.1 * grad
        vel = 0.999 * vel + 0.001 * grad * grad
        theta += args.lr * (mom / (1 - 0.9 ** it)) / (np.sqrt(vel / (1 - 0.999 ** it)) + 1e-8)
        hist.append(lp)
    dt = time.perf_counter() - t0
    print(json.dumps({"N": N, "p": p, "m": m, "missing": args.missing, "n_observed": int(np.sum(~np.isnan(y))), "steps": args.steps,
                      "sec_per_step": dt / args.steps, "logpdf_first": hist[0], "logpdf_last": hist[-1],
                      "sigma2_true_vs_fit": [true_s2, float(np.exp(theta[-1]))],
                      "variance_true_vs_fit": [[round(float(a), 3), round(float(b), 3)] for a, b in zip(true_var, np.exp(theta[:m]))],
                      "inv_ls_true_vs_fit": [[round(float(a), 3), round(float(b), 3)] for a, b in zip(true_ils, np.exp(theta[m:2 * m]))]}))
    assert hist[-1] > hist[0]


if __name__ == "__main__":
    main()
