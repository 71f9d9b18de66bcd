#!/usr/bin/env python
"""Bit-identity check of the logpdf gradient outputs between two builds.

    python tools/grad_bitidentity.py dump ROOT OUT.npz     # seeded lmm_*_logpdf_grad[_terms] outputs of the package in ROOT
    python tools/grad_bitidentity.py compare A.npz B.npz   # np.array_equal on every array

Inputs: seeded x (N = 300 and 1300), y, U, S (p = 5, m = 3); single-kernel latents through the plain and the _terms entry
points, composite / periodic / rational-quadratic latents through the _terms entry points; OILMM and IndependentMOGP; every
output (value, variance, inv_lengthscale, mean_const, ard, sigma2, y, U, S, terms).  Run each dump in its own process."""
import sys

import numpy as np


def dump(root, path):
    sys.path.insert(0, root)
    import lmm_b200 as lmm
    from oracle import lmm_oracle as o

    out = {}
    O = lmm.MOInputIsotopicByOutputs
    for N in (300, 1300):
        rng = np.random.default_rng(N)
        x = np.sort(rng.uniform(0, N / 50.0, N))
        p, m = 5, 3
        U, S = o.orthogonal_from_seed(p, m, seed=3)
        y = rng.standard_normal(p * N)
        single = [lmm.GP(0.2, lmm.SEKernel().compose(lmm.ScaleTransform(1.3))), lmm.GP(-0.1, lmm.Matern52Kernel()), lmm.GP(lmm.Matern32Kernel())]
        comp = [lmm.GP(0.3, lmm.SEKernel() + 0.5 * lmm.PeriodicKernel(1.1)), lmm.GP(lmm.RationalQuadraticKernel(1.5)),
                lmm.GP(0.1, lmm.Matern52Kernel() * lmm.PeriodicKernel(0.8))]
        for fam, ks in (("single", single), ("comp", comp)):
            for terms in ((False, True) if fam == "single" else (True,)):
                fo = lmm.ILMM(lmm.independent_mogp(ks), lmm.Orthogonal(U, S))(O(x, p), 0.1)
                fi = lmm.independent_mogp(ks)(O(x, m), 0.15)
                res = {"oilmm": lmm.logpdf_and_gradient(fo, y, with_grad_y=True, kernel_terms=terms),
                       "imogp": lmm.logpdf_and_gradient(fi, y[: m * N], with_grad_y=True, kernel_terms=terms)}
                for tag, (v, g) in res.items():
                    key = f"{tag}_{fam}_{int(terms)}_{N}"
                    out[key + "_value"] = np.array([v])
                    for k, a in g.items():
                        if k == "terms":
                            out[key + "_terms"] = np.concatenate([[t["variance"], t["inv_lengthscale"], t["param"], *t["ard"]] for lat in a for t in lat])
                        else:
                            out[key + "_" + k] = np.atleast_1d(np.asarray(a, dtype=np.float64))
    np.savez(path, **out)
    print(len(out), "arrays")


def compare(pa, pb):
    a, b = np.load(pa), np.load(pb)
    assert sorted(a.files) == sorted(b.files), set(a.files) ^ set(b.files)
    bad = [k for k in a.files if not np.array_equal(a[k], b[k])]
    print(f"{len(a.files)} arrays compared with np.array_equal; differing: {bad}")
    return not bad


if __name__ == "__main__":
    if sys.argv[1] == "dump":
        dump(sys.argv[2], sys.argv[3])
    else:
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
