#!/usr/bin/env python
"""Where the time of the int8 Cholesky goes: one eval of bench.py's headline workload (C4: OILMM p = 64, m = 64, N = 16384, SE
latents, 7 digit planes of 8 bits, the library's default streams) under torch.profiler with CUDA activities, kernel time summed
by kernel and, for the tile GEMM, by mode (UPDATE / TRSM).  Beside it the work model of the batched left-looking schedule
(csrc/host_chol.cu: chol_factor_stream) computed on the host from the tile envelope of the workload's inputs: tiles of the
panel TRSMs, DMMA tile products of the narrow in-block updates and of the short wide updates (k < ozaki_min_k), int8 tile
products of the wide updates, tiles the digit-plane slicing reads, diagonal tiles -- with the FP64 floors at the DMMA peak.

    python tools/bench_chol_phases.py [--outer-block B] [--trsm-slice 0|1] [--tag NAME] [--out DIR]

--outer-block 0 (default) leaves the library's block width; --trsm-slice leaves the library's default when not given.  A few
unprofiled evals first give the stage times (last_timings) of the same build; the profiled eval is a run of its own.
Output: one JSON line on stdout and DIR/r10_chol_phases_<tag>.json (DIR defaults to profiles/)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import workload  # noqa: E402

T = 128
DMMA_PEAK_TFLOPS = 37.2  # FP64 tensor pipe of the B200 (tools/microbench/fp64_peak.cu)
TRSM_FLOP = 2.0 * T ** 3 * 136 / 256  # the TRSM kernel skips 120 of the 256 8x8 block products of the triangular W
KERNELS = ("ozaki_update_kernel", "gemm_tile_kernel_v2", "gemm_direct2_kernel", "potrf_tile_kernel2", "ozaki_slice_kernel",
           "chain_column_kernel")


def envelope(x, inv_ls, nt):
    """First tile column of each tile row with an SE entry the library's exp does not flush to 0 (d^2 <= 1416), for sorted x."""
    r = np.sqrt(2 * 708.0) / inv_ls
    j0 = np.searchsorted(x, x[np.arange(nt) * T] - r, side="left")
    return np.minimum(j0 // T, np.arange(nt))


def work_model(envs, nt, ob, min_k):
    """Tile counts of chol_factor_stream at block width ob for the envelopes `envs` (one int array of nt per latent)."""
    w = {"envelope_tiles": 0, "trsm_tiles": 0, "narrow_dmma_products": 0, "wide_dmma_products": 0, "wide_int8_products": 0,
         "slice_tiles": 0, "diagonal_tiles": 0}
    for env in envs:
        env = np.asarray(env, dtype=np.int64)
        I = np.arange(nt)
        w["envelope_tiles"] += int((I - env + 1).sum())
        w["diagonal_tiles"] += nt
        for s0 in range(0, nt, ob):
            s1 = min(s0 + ob, nt)
            for J in range(s0, s1):
                rows = I[J:]
                kb = np.maximum(env[rows], env[J])
                if s0 > 0:  # wide update of column J by k < s0
                    n = int(np.clip(s0 - kb, 0, None).sum())
                    w["wide_int8_products" if s0 >= min_k else "wide_dmma_products"] += n
                # narrow update of column J by k in [s0, J)
                w["narrow_dmma_products"] += int(np.clip(J - np.maximum(kb, s0), 0, None).sum())
                w["trsm_tiles"] += int((env[J + 1:] <= J).sum())
            if s1 < nt:  # tiles (I >= s1, k in [s0, s1)) inside the envelope, sliced for the later wide updates
                rows = I[s1:]
                w["slice_tiles"] += int(sum((env[rows] <= k).sum() for k in range(s0, s1)))
    fl = 2.0 * T ** 3
    w["floors_ms_at_dmma_peak"] = {
        "trsm": w["trsm_tiles"] * TRSM_FLOP / (DMMA_PEAK_TFLOPS * 1e9),
        "narrow_dmma": w["narrow_dmma_products"] * fl / (DMMA_PEAK_TFLOPS * 1e9),
        "wide_dmma": w["wide_dmma_products"] * fl / (DMMA_PEAK_TFLOPS * 1e9),
    }
    w["slice_first_read_gb"] = w["slice_tiles"] * T * T * 8 / 1e9
    return w


def classify(name):
    for k in KERNELS:
        if k in name:
            if k in ("gemm_tile_kernel_v2", "gemm_direct2_kernel"):
                mode = name.split(k + "<", 1)[1][0] if k + "<" in name else "?"
                tag = "UPDATE" if mode == "0" else "TRSM" if mode == "1" else mode
                return f"{k}_{tag}{'_SLICE' if 'true>' in name else ''}"
            return k
    return "other"


def card():
    import torch

    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        q = f"unavailable: {exc}"
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--p", type=int, default=64)
    ap.add_argument("--m", type=int, default=64)
    ap.add_argument("--N", type=int, default=16384)
    ap.add_argument("--outer-block", type=int, default=0, help="library option outer_block (0: the library's choice)")
    ap.add_argument("--trsm-slice", type=int, choices=(0, 1), default=None,
                    help="library option trsm_slice: digit planes written by the panel TRSM (1) or by separate slice launches (0)")
    ap.add_argument("--model-only", action="store_true", help="print the work model and stop (no GPU needed)")
    ap.add_argument("--tag", default="run")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    x, U, S, inv_ls, y, s2 = workload(a.p, a.m, a.N)
    nt = (a.N + T - 1) // T
    envs = [envelope(x, il, nt) for il in inv_ls]
    min_k = 4
    # the block width the library takes on this path when outer_block is not set: 1 from 64 tile rows on, 2 below
    model = {f"ob{ob}": work_model(envs, nt, ob, min_k) for ob in sorted({1, 2, a.outer_block or 1})}
    res = {"workload": f"bench.py workload(p={a.p}, m={a.m}, N={a.N}), OILMM logpdf + posterior, ozaki 7 x 8 bits", "model": model}
    if a.model_only:
        print(json.dumps(res))
        return

    import torch
    from torch.profiler import ProfilerActivity, profile

    import lmm_b200 as lmm

    if not torch.cuda.is_available():
        raise SystemExit("bench_chol_phases.py needs a CUDA device")
    ctx = lmm.default_context()
    ctx.set_option("ozaki", 7)
    ctx.set_option("ozaki_bits", 8)
    if a.outer_block:
        ctx.set_option("outer_block", a.outer_block)
    if a.trsm_slice is not None:
        ctx.set_option("trsm_slice", a.trsm_slice)
    fs = [lmm.GP(lmm.SEKernel().compose(lmm.ScaleTransform(float(s)))) for s in inv_ls]  # as bench.py builds it
    f = lmm.ILMM(lmm.independent_mogp(fs), lmm.Orthogonal(U, S))
    fx = f(lmm.MOInputIsotopicByOutputs(torch.from_numpy(x.reshape(-1, 1)).cuda(), a.p), s2)
    yd = torch.from_numpy(y).cuda()

    def step():
        post, lp = lmm.posterior(fx, yd, with_logpdf=True)
        tm = ctx.last_timings().copy()
        post.f.fs[0]._owner.free()
        return lp, tm

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    stages = [step()[1] for _ in range(3)]
    res["stage_ms_median"] = {k: statistics.median(float(t[i]) for t in stages)
                              for i, k in enumerate(("eval", "kmat", "cholesky", "solves", "proj"))}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        lp, _ = step()
        torch.cuda.synchronize()
    by, cnt = {}, {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            k = classify(ev.name)
            by[k] = by.get(k, 0.0) + ev.device_time_total / 1e3
            cnt[k] = cnt.get(k, 0) + 1
    res.update(card())
    res["options"] = {"outer_block": a.outer_block, "trsm_slice": a.trsm_slice}
    res["logpdf"] = float(lp)
    res["kernel_ms"] = dict(sorted(by.items(), key=lambda kv: -kv[1]))
    res["kernel_launches"] = cnt
    res["kernel_ms_total"] = sum(by.values())
    res["note"] = ("kernel_ms: device time summed over all launches of one eval under torch.profiler (4 streams overlap, so the sum "
                   "exceeds the eval's wall time); model: counts from the SE envelope of the inputs, floors at the FP64 DMMA peak")
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, f"r10_chol_phases_{a.tag}.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
