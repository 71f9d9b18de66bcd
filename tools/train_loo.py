#!/usr/bin/env python
"""Cross-validation training: Adam on log(variance), log(inv_lengthscale) per latent and log(σ²) of a seeded OILMM maximises
its leave-one-input-out log predictive density.  Every step is one `loo_logpdf_and_gradient` call (lmm_oilmm_loo with
gradient outputs): no data split, no refits.  U and S are held at their true values.

    python tools/train_loo.py --N 2000 --m 3 --p 6 --steps 40
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lmm_b200 as lmm  # noqa: E402


def build(U, S, var, ils):
    ks = [(float(v) * lmm.Matern52Kernel()).compose(lmm.ScaleTransform(float(s))) for v, s in zip(var, ils)]
    return lmm.ILMM(lmm.independent_mogp([lmm.GP(k) for k in ks]), lmm.Orthogonal(U, S))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=2000)
    ap.add_argument("--p", type=int, default=6)
    ap.add_argument("--m", type=int, default=3)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--lr", type=float, default=0.08)
    args = ap.parse_args()
    rng = np.random.default_rng(0)
    N, p, m = args.N, args.p, args.m
    x = np.linspace(0.0, N / 50.0, N)
    U, S, _ = np.linalg.svd(rng.uniform(0, 1, (p, m)), full_matrices=False)
    true_var, true_ils, true_s2 = rng.uniform(0.5, 2.0, m), rng.uniform(0.6, 1.8, m), 0.05
    f_true = build(U, S, true_var, true_ils)
    # latent draws through the IndependentMOGP sampler (1e-4 jitter keeps the smooth prior covariance numerically PD), mixed and
    # corrupted on the host
    lat = lmm.rand(np.random.default_rng(1), f_true.f(lmm.MOInputIsotopicByOutputs(x, m), 1e-4)).reshape(m, N)
    y = ((U * np.sqrt(S)) @ lat + np.sqrt(true_s2) * np.random.default_rng(2).standard_normal((p, N))).reshape(-1)
    O = lmm.MOInputIsotopicByOutputs
    theta = np.zeros(2 * m + 1)  # log var, log ils, log σ²  (start at 1, 1, 1)
    mom, vel = np.zeros_like(theta), np.zeros_like(theta)
    t0 = time.perf_counter()
    hist = []
    for it in range(1, args.steps + 1):
        var, ils, s2 = np.exp(theta[:m]), np.exp(theta[m:2 * m]), float(np.exp(theta[-1]))
        lp, g = lmm.loo_logpdf_and_gradient(build(U, S, var, ils)(O(x, p), s2), y)
        grad = np.concatenate([g["variance"] * var, g["inv_lengthscale"] * ils, [g["sigma2"] * s2]])  # chain rule to log-space
        mom = 0.9 * mom + 0.1 * grad
        vel = 0.999 * vel + 0.001 * grad * grad
        theta += args.lr * (mom / (1 - 0.9 ** it)) / (np.sqrt(vel / (1 - 0.999 ** it)) + 1e-8)
        hist.append(lp)
    dt = time.perf_counter() - t0
    print(json.dumps({"N": N, "p": p, "m": m, "steps": args.steps, "sec_per_step": dt / args.steps,
                      "loo_logpdf_first": hist[0], "loo_logpdf_last": hist[-1], "loo_logpdf_max": max(hist),
                      "sigma2_true_vs_fit": [true_s2, float(np.exp(theta[-1]))],
                      "variance_true_vs_fit": [[round(float(a), 3), round(float(b), 3)] for a, b in zip(true_var, np.exp(theta[:m]))],
                      "inv_ls_true_vs_fit": [[round(float(a), 3), round(float(b), 3)] for a, b in zip(true_ils, np.exp(theta[m:2 * m]))]}))
    assert hist[-1] > hist[0], "the LOO score did not rise"


if __name__ == "__main__":
    main()
