#!/usr/bin/env python
"""Leave-one-input-out value, marginals and gradient with latents sharded over the ranks (run under torchrun, one rank per
GPU): the LOO terms, gradients and marginals are summed over the ranks by the library's NCCL all-reduces.  Rank 0 then
repeats the calls on a context of its own (one rank, every latent local) and prints one JSON line comparing the two; exit
code 1 if they differ by more than 1e-12."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lmm_b200 as lmm  # noqa: E402


def problem():
    rng = np.random.default_rng(0)
    N, p = 900, 8
    x = np.sort(rng.uniform(0, 9, N))
    s = lambda k, v: k.compose(lmm.ScaleTransform(v))  # noqa: E731
    ks = [s(lmm.SEKernel(), 0.4) + 0.5 * s(lmm.PeriodicKernel(0.8), 0.7),
          s(0.9 * lmm.Matern52Kernel(), 0.3) * lmm.PeriodicKernel(1.3),
          s(0.7 * lmm.Matern32Kernel(), 1.1),
          s(lmm.RationalQuadraticKernel(1.4), 0.9),
          s(0.6 * lmm.SEKernel(), 1.5) + s(0.3 * lmm.ExponentialKernel(), 0.8) + s(0.4 * lmm.RationalQuadraticKernel(1.7), 0.6)]
    m = len(ks)
    Q, _ = np.linalg.qr(np.random.default_rng(1).standard_normal((p, m)))
    S = np.random.default_rng(2).uniform(0.5, 2.0, m)
    y = rng.standard_normal(p * N)
    f = lmm.ILMM(lmm.independent_mogp([lmm.GP(0.1 * i, k) for i, k in enumerate(ks)]), lmm.Orthogonal(Q, S))
    return f(lmm.MOInputIsotopicByOutputs(x, p), 0.1), y


def flat(g):
    t = [np.array([q["variance"], q["inv_lengthscale"], q["param"], *q["ard"]]) for lat in g["terms"] for q in lat]
    return np.concatenate(t + [g["variance"], g["inv_lengthscale"], g["mean_const"], [g["sigma2"]], g["y"], g["U"].ravel(), g["S"], g["ard"].ravel()])


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    ctx = lmm.Context(local)
    lmm.set_default_context(ctx)
    lmm.dist.init_context_distributed(ctx)
    fx, y = problem()
    lp_d, g_d = lmm.loo_logpdf_and_gradient(fx, y, with_grad_y=True)
    v_d = lmm.loo_logpdf(fx, y)
    M_d, V_d = lmm.loo_mean_and_var(fx, y)
    dist.barrier()
    ok = True
    if rank == 0:
        lmm.set_default_context(lmm.Context(local))
        fx1, y1 = problem()
        lp_1, g_1 = lmm.loo_logpdf_and_gradient(fx1, y1, with_grad_y=True)
        v_1 = lmm.loo_logpdf(fx1, y1)
        M_1, V_1 = lmm.loo_mean_and_var(fx1, y1)
        a, b = np.concatenate([flat(g_d), M_d, V_d]), np.concatenate([flat(g_1), M_1, V_1])
        terms_d = np.concatenate([[q["variance"], q["inv_lengthscale"], q["param"]] for lat in g_d["terms"] for q in lat])
        terms_1 = np.concatenate([[q["variance"], q["inv_lengthscale"], q["param"]] for lat in g_1["terms"] for q in lat])
        rel = float(np.max(np.abs(a - b)) / np.max(np.abs(b)))
        ok = rel <= 1e-12 and abs(lp_d - lp_1) <= 1e-12 * abs(lp_1) and abs(v_d - v_1) <= 1e-12 * abs(v_1)
        print(json.dumps({"ranks": world, "device": torch.cuda.get_device_name(local), "loo_ranks": lp_d, "loo_one_rank": lp_1,
                          "loo_value_path_ranks": v_d, "loo_value_path_one_rank": v_1,
                          "grad_terms_identical": bool(np.array_equal(terms_d, terms_1)), "max_rel_diff_all_outputs": rel, "ok": bool(ok)}),
              flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
