#!/usr/bin/env python
"""Sparse variational (VFE) bound of an OILMM: p = 64, m = 16, N = 2^18, M = 2048 inducing inputs, D = 1, one family of SE and
one of Matern52 latents.  The exact logpdf at N = 16384 is timed alongside for scale (the largest N the exact path's benchmark
runs).

Default: after one warm-up call of each, `--reps` rounds that call elbo and elbo_and_gradient (SE, Matern52) and the exact logpdf in turn; every
call ends in a device synchronise, so the host clock around it is the call's time.  Medians are written with the card's name,
power limit and SM clocks.  `--profile`: a separate run, one elbo call per family under torch.profiler (CUDA activities),
kernel times summed by name, and the Gram kernel's achieved FP64 rate against 37.2 TFLOP/s (the FP64 tensor pipe's peak).
`--parity`: the first latent's bound at full size against a chunked NumPy evaluation of the oracle formula.
Output: one JSON line on stdout and profiles/r11_vfe_{timing,kernels,parity}.json (or --out DIR)."""
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

N, P, M_LAT, M_IND, N_EXACT = 1 << 18, 64, 16, 2048, 16384
PEAK_FP64_TC = 37.2e12


def gram_flops(n, mi, m):
    """FP64 flops of vfe_gram_kernel for m latents: every stored 128 x 128 tile of the packed-lower Gram (diagonal tiles in
    full) over the padded training rows, 2 flop per multiply-add."""
    mt, npad = -(-mi // 128), -(-n // 128) * 128
    return 2.0 * (mt * (mt + 1) // 2) * 128 * 128 * npad * m


def card():
    import torch

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"device": torch.cuda.get_device_name(), "nvidia_smi name,power.limit,clocks.sm,clocks.max.sm": q}


def problem():
    rng = np.random.default_rng(0)
    x = np.sort(rng.uniform(0, N / 100.0, N))
    z = np.linspace(0.0, N / 100.0, M_IND)
    U, S, _ = np.linalg.svd(np.random.default_rng(1).uniform(0, 1, (P, M_LAT)), full_matrices=False)
    s = np.random.default_rng(2).uniform(0.5, 2.0, M_LAT) * 0.2  # lengthscales of a few inducing-point spacings
    y = rng.standard_normal(P * N)
    O = lmm.MOInputIsotopicByOutputs
    fams = {"se": lmm.SEKernel, "matern52": lmm.Matern52Kernel}
    calls = {}
    for name, K in fams.items():
        lat = lmm.independent_mogp([lmm.GP(K().compose(lmm.ScaleTransform(float(s[i])))) for i in range(M_LAT)])
        fx = lmm.ILMM(lat, lmm.Orthogonal(U, S))(O(x, P), 0.1)
        calls["elbo_" + name] = (lambda fx=fx: lmm.elbo(lmm.VFE(z, 1e-6), fx, y))
        calls["elbo_and_gradient_" + name] = (lambda fx=fx: lmm.elbo_and_gradient(lmm.VFE(z, 1e-6), fx, y))
    lat = lmm.independent_mogp([lmm.GP(lmm.SEKernel().compose(lmm.ScaleTransform(float(s[i])))) for i in range(M_LAT)])
    fxe = lmm.ILMM(lat, lmm.Orthogonal(U, S))(O(x[:N_EXACT], P), 0.1)
    ye = y.reshape(P, N)[:, :N_EXACT].reshape(-1)
    calls["exact_logpdf_N16384"] = lambda: lmm.logpdf(fxe, ye)
    return calls, (x, z, U, S, s, y)


def timed(fn):
    import torch

    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def parity(data):
    """Latent 0 of the SE family: ELBO_0 on the projected data, chunked NumPy (Cholesky of K(z, z), triangular solves)."""
    import scipy.linalg as sl

    x, z, U, S, s, y = data
    T = (U / np.sqrt(S)[None, :]).T
    ty = T[:1] @ y.reshape(P, N)
    nu = 0.1 / S[0]
    k = lambda a, b: np.exp(-0.5 * (s[0] * (a[:, None] - b[None, :])) ** 2)  # noqa: E731
    Lz = np.linalg.cholesky(k(z, z) + 1e-6 * np.eye(M_IND))
    Psi, b, dd = np.zeros((M_IND, M_IND)), np.zeros(M_IND), 0.0
    for r0 in range(0, N, 16384):
        Bt = sl.solve_triangular(Lz, k(z, x[r0:r0 + 16384]), lower=True).T
        d = ty[0, r0:r0 + 16384]
        Psi += Bt.T @ Bt
        b += Bt.T @ d
        dd += d @ d
    Ls = np.linalg.cholesky(np.eye(M_IND) + Psi / nu)
    c = sl.solve_triangular(Ls, b, lower=True)
    return -0.5 * (N * np.log(2 * np.pi) + N * np.log(nu) + 2 * np.sum(np.log(np.diag(Ls))) + dd / nu - c @ c / nu ** 2
                   + (N - np.trace(Psi)) / nu)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--parity", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    calls, data = problem()
    res = {"shape": {"p": P, "m": M_LAT, "N": N, "M": M_IND, "D": 1, "exact_N": N_EXACT}, **card()}
    if a.parity:
        # latent 0 alone: the same model with one latent and U's first column
        x, z, U, S, s, y = data
        lat = lmm.independent_mogp([lmm.GP(lmm.SEKernel().compose(lmm.ScaleTransform(float(s[0]))))])
        fx1 = lat(lmm.MOInputIsotopicByOutputs(x, 1), 0.1 / S[0])
        T = (U / np.sqrt(S)[None, :]).T
        got = lmm.elbo(lmm.VFE(z, 1e-6), fx1, (T[:1] @ y.reshape(P, N)).reshape(-1))
        ref = parity(data)
        res["parity_latent0"] = {"library": got, "numpy": ref, "rel": abs(got - ref) / abs(ref)}
        json.dump(res, open(os.path.join(a.out, "r11_vfe_parity.json"), "w"), indent=1)
    elif a.profile:
        import torch
        from torch.profiler import ProfilerActivity, profile

        for name, fn in calls.items():
            fn()
        per = {}
        for name in ("elbo_se", "elbo_matern52"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                calls[name]()
                torch.cuda.synchronize()
            k = {}
            for e in prof.events():
                if e.device_type.name == "CUDA":
                    k[e.name] = k.get(e.name, 0.0) + e.device_time_total / 1e3  # ms
            gram = sum(v for n, v in k.items() if "vfe_gram_kernel" in n)
            per[name] = {"kernels_ms": dict(sorted(k.items(), key=lambda t: -t[1])[:20]), "total_kernel_ms": sum(k.values()),
                         "gram_ms": gram, "gram_tflops": gram_flops(N, M_IND, M_LAT) / (gram * 1e-3) / 1e12,
                         "gram_share_of_37.2_tflops": gram_flops(N, M_IND, M_LAT) / (gram * 1e-3) / PEAK_FP64_TC}
        res.update(per)
        res.update({"after": card()})
        json.dump(res, open(os.path.join(a.out, "r11_vfe_kernels.json"), "w"), indent=1)
    else:
        for fn in calls.values():
            fn()
        t = {k: [] for k in calls}
        for _ in range(a.reps):
            for k, fn in calls.items():
                t[k].append(timed(fn))
        res["median_s"] = {k: statistics.median(v) for k, v in t.items()}
        res["all_s"] = t
        res["after"] = card()
        json.dump(res, open(os.path.join(a.out, "r11_vfe_timing.json"), "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
