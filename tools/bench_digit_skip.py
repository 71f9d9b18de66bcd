#!/usr/bin/env python
"""The int8 wide update with the digit-plane filter, measured honestly: bench.py's workload at N = 16384 with m = 8 latents (small
enough to recount every latent on the host), one OILMM logpdf on one stream with CUDA events around every int8 update launch
(library option "ozaki_time").  The host recount (tools/ozaki_digits.py, the slice kernel's rule applied to the returned factors)
gives the tile products the kernel actually multiplied -- pass A members x the MMAs of d = 0..3, pass B members x the rest -- and with
them the kernel's real int8 rate, beside the nominal one bench.py reports (envelope tile products x all S(S+1)/2 MMAs).

    python tools/bench_digit_skip.py --out profiles/r07_digit_skip.json"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import int8_peak_tops, workload  # noqa: E402
from tools.ozaki_digits import T, first_planes, update_products  # noqa: E402

_FACTORS = []


def _count(args):
    i, env, S, bits = args
    return update_products(first_planes(_FACTORS[i], S, bits), env, S, bits)


def envelope(x, inv_ls, nt):
    """First tile column with an entry the library's exp does not flush to 0 (0.5 d^2 <= 708), for sorted x."""
    r = np.sqrt(2 * 708.0) / inv_ls
    j0 = np.searchsorted(x, x[np.arange(nt) * T] - r, side="left")
    return np.minimum(j0 // T, np.arange(nt))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--p", type=int, default=64)
    ap.add_argument("--m", type=int, default=8)
    ap.add_argument("--N", type=int, default=16384)
    ap.add_argument("--ozaki", type=int, default=7)
    ap.add_argument("--ozaki-bits", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import lmm_b200 as lmm

    S, bits = a.ozaki, a.ozaki_bits
    x, U, Sv, inv_ls, y, s2 = workload(a.p, a.m, a.N)
    ctx = lmm.default_context()
    ctx.set_option("ozaki", S)
    ctx.set_option("ozaki_bits", bits)
    ctx.set_option("streams", 1)
    fs = [lmm.GP(lmm.SEKernel().compose(lmm.ScaleTransform(float(il)))) for il in inv_ls]  # as bench.py builds it
    f = lmm.ILMM(lmm.independent_mogp(fs), lmm.Orthogonal(U, Sv))
    fx = f(lmm.MOInputIsotopicByOutputs(x, a.p), s2)
    lmm.logpdf(fx, y)  # warm-up (module load, workspace)
    ctx.set_option("ozaki_time", 1)
    runs = []
    for _ in range(a.reps):
        ctx.last_timings()
        lmm.logpdf(fx, y)
        tm = ctx.last_timings()
        runs.append({"int8_kernel_ms": float(tm[7]), "envelope_tile_products": float(tm[5])})
    ctx.set_option("ozaki_time", 0)
    post = lmm.posterior(fx, y)
    nt = a.N // T
    _FACTORS.extend(np.array(g.C) for g in post.f.fs)
    t0 = time.time()
    with mp.get_context("fork").Pool(min(a.m, os.cpu_count() or 1)) as pool:
        cnt = pool.map(_count, [(i, envelope(x, inv_ls[i], nt), S, bits) for i in range(a.m)])
    recount_s = time.time() - t0
    tot = {k: int(sum(int(c[k]) for c in cnt)) for k in cnt[0]}
    nmma = S * (S + 1) // 2
    nA = sum(1 for t in range(min(S, 4)) for u in range(min(S, 4)) if t + u <= min(S, 4) - 1)  # MMAs of pass A (d = 0..3)
    ms = float(np.median([r["int8_kernel_ms"] for r in runs]))
    nominal_ops = tot["envelope"] * nmma * 2.0 * T ** 3
    real_ops = (tot["pass_a"] * nA + tot["pass_b"] * (nmma - nA)) * 2.0 * T ** 3
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:  # noqa: BLE001
        gpu = f"unavailable: {exc}"
    peak, peak_src = int8_peak_tops()
    res = {"workload": f"bench.py workload(p={a.p}, m={a.m}, N={a.N}), OILMM logpdf, one stream", "ozaki": S, "ozaki_bits": bits,
           "gpu": gpu, "runs": runs, "int8_kernel_ms_median": ms,
           "tile_products": {"envelope": tot["envelope"], "pass_b_members": tot["pass_b"], "pass_a_members": tot["pass_a"],
                             "ctas_run": tot["ctas"], "ctas_with_empty_pass_a": tot["ctas_pass_a_empty"]},
           "counter_matches_envelope": all(r["envelope_tile_products"] == tot["envelope"] for r in runs),
           "nominal_int8_tops": nominal_ops / (ms * 1e-3) / 1e12, "real_int8_tops": real_ops / (ms * 1e-3) / 1e12,
           "int8_peak_tops": peak, "int8_peak_source": peak_src, "real_frac_of_peak": real_ops / (ms * 1e-3) / 1e12 / peak,
           "per_latent": [{k: int(v) for k, v in c.items()} for c in cnt], "host_recount_s": recount_s,
           "note": "real = MMAs the kernel issued (pass A members x the pairs of d = 0..3, pass B members x the pairs of d = 4..S-1); "
                   "nominal = envelope tile products x S(S+1)/2, what bench.py's roofline reports; row scales of the recount from the "
                   "returned factor's row norms"}
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
