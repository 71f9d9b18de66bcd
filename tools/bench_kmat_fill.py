"""Cost of the deferred zero fill of a kept posterior (library option "kmat_skip"): the headline eval (BASELINE config 4, as
bench.py builds it) leaves the kernel-matrix tiles that are provably exact zeros unwritten, and the first call that reads the
posterior's factors writes them.  Times a prediction at 256 points as the first read (fill + prediction) and again as the
second read of the same posterior (prediction only), over `--reps` fresh posteriors; prints one JSON line."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ozaki", type=int, default=7)
    ap.add_argument("--ozaki-bits", type=int, default=8)
    args = ap.parse_args()
    import torch

    import lmm_b200 as lmm
    from bench import workload

    p, m, N = 64, 64, 16384
    ctx = lmm.Context(0)
    lmm.set_default_context(ctx)
    ctx.set_option("ozaki", args.ozaki)
    ctx.set_option("ozaki_bits", args.ozaki_bits)
    x, U, S, inv_ls, y, s2 = workload(p, m, N)
    fs = [lmm.GP(lmm.SEKernel().compose(lmm.ScaleTransform(float(s)))) for s in inv_ls]
    f = lmm.ILMM(lmm.independent_mogp(fs), lmm.Orthogonal(U, S))
    fx = f(lmm.MOInputIsotopicByOutputs(torch.from_numpy(x.reshape(-1, 1)).cuda(), p), s2)
    yd = torch.from_numpy(y).cuda()
    xs = lmm.MOInputIsotopicByOutputs(np.linspace(x[0], x[-1], 256), p)
    first, second = [], []
    for r in range(args.reps + 1):
        post, _ = lmm.posterior(fx, yd, with_logpdf=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        lmm.mean_and_var(post(xs, s2))
        t1 = time.perf_counter()
        lmm.mean_and_var(post(xs, s2))
        t2 = time.perf_counter()
        if r > 0:  # the first posterior warms up the prediction's kernels
            first.append((t1 - t0) * 1e3)
            second.append((t2 - t1) * 1e3)
        del post
    fill = float(np.median(first) - np.median(second))
    nt = N // 128
    print(json.dumps({"what": "deferred zero fill of a C4 posterior (first read minus second read of the same posterior)",
                      "gpu": torch.cuda.get_device_name(0), "first_read_ms": first, "second_read_ms": second, "fill_ms": fill,
                      "dense_lower_tile_bytes": 8.0 * 128 * 128 * m * nt * (nt + 1) / 2}))


if __name__ == "__main__":
    main()
