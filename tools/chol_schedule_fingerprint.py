#!/usr/bin/env python
"""Fingerprint of the Cholesky schedules (csrc/host_chol.cu): for each configuration below one JSON record with the launch count
(Context.counters()), last_timings()[6] (in-block updates) and [5] (int8 tile products, with "ozaki_time"), the sorted multiset of
(kernel, grid, block) from a torch.profiler trace (as [kernel, grid, block, count]), and the sha256 of every output array.  Two
builds that give identical files enqueue the same kernels with the same grids and compute the same bits; a refactor of the host
schedules is checked that way.

    python tools/chol_schedule_fingerprint.py --out FILE.json

Covers: the left-looking schedule on 4 stream groups (DMMA, int8 with the panel TRSM or separate launches writing the digit
planes, ozaki_time accounting), the one-stream fused chain of small grids, the right-looking schedule (lookahead, chain_fused,
the ozaki_single_nt crossover), info of non-PD inputs, the tile envelope at widths 1 and 2, the jstart > 0 block update of a
conditioned posterior, the prediction sweep incl. its int8 path, the potri sweep of the gradient, and the chunked int8 workspace."""
import argparse
import hashlib
import json
import os
import sys
import tempfile
from collections import Counter

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def spd(batch, N, seed):
    """SE kernel matrices of sorted points plus noise: dense and positive definite."""
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(0, N / 40.0, N))
    d2 = (x[:, None] - x[None, :]) ** 2
    return np.stack([np.exp(-0.5 * d2 * (0.5 + 0.3 * b) ** 2) + 0.1 * np.eye(N) for b in range(batch)])


def oilmm(lmm, p, m, N, span, seed):
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(0, span, N))
    U = np.linalg.qr(rng.standard_normal((p, m)))[0]
    S = rng.uniform(0.5, 2.0, m)
    fs = [lmm.GP(lmm.SEKernel().compose(lmm.ScaleTransform(0.9 + 0.2 * a / m))) for a in range(m)]
    return lmm.ILMM(lmm.independent_mogp(fs), lmm.Orthogonal(U, S)), x, rng


def run(lmm, name, opts, call):
    """call() -> dict of output arrays, run once under torch.profiler in a fresh Context with the options `opts`."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    ctx = lmm.Context()
    lmm.set_default_context(ctx)
    for k, v in opts.items():
        ctx.set_option(k, v)
    c0 = ctx.counters()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        outs = call(ctx)
        torch.cuda.synchronize()
    c1 = ctx.counters()
    tm = ctx.last_timings()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            trace = json.load(fh)
    launched = Counter((ev["name"], tuple(ev["args"].get("grid", ())), tuple(ev["args"].get("block", ())))
                       for ev in trace["traceEvents"] if ev.get("cat") == "kernel")
    kernels = sorted([name, list(grid), list(block), n] for (name, grid, block), n in launched.items())
    rec = {"name": name, "options": opts, "launches": c1[0] - c0[0], "counters_delta": [b - a for a, b in zip(c0, c1)],
           "timings6": float(tm[6]), "kernels": kernels, "sha256": {k: sha(v) for k, v in outs.items()}}
    if opts.get("ozaki_time"):
        rec["timings5"] = float(tm[5])
    lmm.set_default_context(None)
    del ctx
    return rec


def configs(lmm):
    import torch

    def potrf(A):
        def call(ctx):
            L, logdet, info = lmm.potrf_batched(A, ctx)
            return {"L": L, "logdet": logdet, "info": info}
        return call

    A8 = spd(8, 4096, 1)
    yield "potrf 8x4096", {}, potrf(A8)
    yield "potrf 8x4096 int8", {"ozaki": 7, "ozaki_bits": 8}, potrf(A8)
    yield "potrf 8x4096 int8 trsm_slice 0", {"ozaki": 7, "ozaki_bits": 8, "trsm_slice": 0}, potrf(A8)
    yield "potrf 8x4096 int8 timed", {"ozaki": 7, "ozaki_bits": 8, "streams": 1, "ozaki_time": 1}, potrf(A8)
    del A8
    yield "potrf 20x640", {}, potrf(spd(20, 640, 2))
    for batch, N in ((1, 2300), (2, 2300), (1, 4500), (2, 4500), (1, 12288)):
        A = spd(batch, N, 3)
        for oz in ((0, 7) if N == 12288 else (0,)):
            for la in (0, 1):
                for cf in (0, 1, 2):
                    yield f"potrf {batch}x{N}", {"ozaki": oz, "ozaki_bits": 8, "lookahead": la, "chain_fused": cf}, potrf(A)
    A = spd(3, 200, 4)
    A[1, 150, 150] = -1.0
    A[2, 10, 10] = -1.0
    for cf in (0, 1):
        yield "potrf 3x200 non-PD", {"chain_fused": cf}, potrf(A)

    def logpdf(N):
        def call(ctx):
            f, x, rng = oilmm(lmm, 16, 16, N, 100.0, 5)
            y = rng.standard_normal(16 * N)
            return {"logpdf": lmm.logpdf(f(lmm.MOInputIsotopicByOutputs(x, 16), 0.1), y)}
        return call

    for N in (8192, 4096):
        for oz in (0, 7):
            yield f"oilmm logpdf N={N}", {"ozaki": oz, "ozaki_bits": 8}, logpdf(N)

    def conditioned(ctx):
        f, x1, rng = oilmm(lmm, 8, 8, 4096, 200.0, 6)
        mo = lambda x: lmm.MOInputIsotopicByOutputs(x, 8)  # noqa: E731
        x2, xt = rng.uniform(0, 200.0, 1000), rng.uniform(0, 200.0, 1024)
        post1 = lmm.posterior(f(mo(x1), 0.1), rng.standard_normal(8 * 4096))
        post2 = lmm.posterior(post1(mo(x2), 0.2), rng.standard_normal(8 * 1000))
        M, V = lmm.mean_and_var(post2(mo(xt), 0.1))
        return {"mean": M, "var": V}

    for oz in (0, 7):
        for streams in (1, 4):
            yield "oilmm posterior 4096+1000, mean_and_var 1024", {"ozaki": oz, "ozaki_bits": 8, "streams": streams}, conditioned

    def gradient(ctx):
        f, x, rng = oilmm(lmm, 8, 8, 4096, 200.0, 7)
        lp, g = lmm.logpdf_and_gradient(f(lmm.MOInputIsotopicByOutputs(x, 8), 0.1), rng.standard_normal(8 * 4096))
        return {"logpdf": lp, **{k: v for k, v in g.items() if k != "terms"}}

    yield "oilmm logpdf_and_gradient 4096", {}, gradient

    A4 = spd(4, 8192, 8)
    per_latent = 2080 * 7 * 16384  # sym_tiles(64) tiles x 7 planes x 16 KB

    yield "potrf 4x8192 int8", {"ozaki": 7, "ozaki_bits": 8}, potrf(A4)

    def chunked(ctx):
        # leave free: 6 GiB reserve + 1.5 latents' planes + what lmm_potrf_batched allocates before the factorisation (A, L, W)
        own = A4.nbytes + 4 * 2080 * 16384 * 8 + 4 * 64 * 16384 * 8
        free = torch.cuda.mem_get_info()[0]
        fill = torch.empty(max(free - (6 << 30) - int(1.5 * per_latent) - own, 0), dtype=torch.uint8, device="cuda")
        out = potrf(A4)(ctx)
        del fill
        return out

    yield "potrf 4x8192 int8, chunked workspace", {"ozaki": 7, "ozaki_bits": 8}, chunked


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    import torch

    import lmm_b200 as lmm

    if not torch.cuda.is_available():
        raise SystemExit("chol_schedule_fingerprint.py needs a CUDA device")
    recs = [run(lmm, name, opts, call) for name, opts, call in configs(lmm)]
    with open(a.out, "w") as fh:
        json.dump(recs, fh, indent=1)
    print(json.dumps([{"name": r["name"], "options": r["options"], "launches": r["launches"]} for r in recs]))


if __name__ == "__main__":
    main()
