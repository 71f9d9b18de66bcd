"""Kernel-matrix build inside the provable tile envelope (library option "kmat_skip", csrc/kmat.cu: kmat_bound_kernel).  The
OILMM / IndependentMOGP eval builds only the tiles that are not provably exact zeros and leaves the others unwritten; a kept
posterior writes those zeros on its first read.  Every result must be the same bits as with every tile built: logpdf, the
exported factors, marginals, seeded samples, conditioning, the posterior-predictive logpdf and a save / load
round trip -- for sorted and tile-shuffled inputs, every stationary kernel kind, a composite latent, 1 and 4 streams, and the
DMMA and int8 updates.  A logpdf-only eval first leaves its unwritten tiles' garbage in the pool memory the posterior reuses."""
import os

import numpy as np
import pytest

from oracle import lmm_oracle as o

T = 128


def latents():
    comp = o.Kernel(o.SE, 1.2, 0.9, op=o.COMPOSE_SUM, terms=(o.Kernel(o.PERIODIC, 0.5, 0.7, param=0.8),))
    return [o.GP(o.Kernel(o.SE, 1.0, 12.0), 0.1), o.GP(o.Kernel(o.EXPONENTIAL, 0.8, 0.4), 0.0), o.GP(o.Kernel(o.MATERN32, 1.1, 2.0), -0.2),
            o.GP(o.Kernel(o.MATERN52, 0.9, 20.0), 0.0), o.GP(o.Kernel(o.SE, 0.7, 0.05), 0.0), o.GP(comp, 0.3)]


def problem(N, order):
    rng = np.random.default_rng(N + (order == "shuffled"))
    x = np.sort(rng.uniform(0, N / 20.0, N))
    if order == "shuffled":
        x = np.concatenate([x[i * T:(i + 1) * T] for i in rng.permutation(-(-N // T))])
    xs = rng.uniform(0, N / 20.0, 40)
    return x, xs, rng.standard_normal(8 * N)


@pytest.fixture()
def lmm():
    import lmm_b200

    yield lmm_b200
    ctx = lmm_b200.default_context()
    ctx.set_option("kmat_skip", 1)
    ctx.set_option("ozaki", int(os.environ.get("LMM_OZAKI", "0")))
    ctx.set_option("ozaki_bits", int(os.environ.get("LMM_OZAKI_BITS", "7")))
    ctx.set_option("streams", 4)


def run(lmm, kind, N, order, skip, tmp_path):
    from test_composite_kernels import to_lmm

    lmm.default_context().set_option("kmat_skip", skip)
    x, xs, y = problem(N, order)
    gs = latents()
    m = len(gs)
    O = lmm.MOInputIsotopicByOutputs
    fs = lmm.independent_mogp([to_lmm(lmm, g) for g in gs])
    if kind == "oilmm":
        U, S = o.orthogonal_from_seed(8, m, seed=2)
        f, p = lmm.ILMM(fs, lmm.Orthogonal(U, S)), 8
    else:
        f, p = fs, m
    fx = f(O(x, p), 0.1)
    y = y[:p * N]
    out = {"lp_only": lmm.logpdf(fx, y)}  # streamed arena: its unwritten tiles are left in the pool memory
    post, lp = lmm.posterior(fx, y, with_logpdf=True)
    out["lp"] = lp
    lat = post.f.fs if kind == "oilmm" else post.fs
    out["L"] = [lat[i].C for i in range(m)]  # export: the first read writes the zeros
    M, V = lmm.mean_and_var(post(O(xs, p), 0.1))
    out["M"], out["V"] = M, V
    out["rand"] = lmm.rand(np.random.default_rng(3), post(O(xs[:9], p), 0.1))
    ys = np.random.default_rng(4).standard_normal(p * len(xs))
    out["plp"] = lmm.logpdf(post(O(xs, p), 0.1), ys)  # posterior-predictive logpdf
    post2 = lmm.posterior(post(O(xs[:20], p), 0.1), ys[:p * 20])
    out["cond"] = lmm.mean_and_var(post2(O(xs, p), 0.1))
    path = str(tmp_path / f"post_{skip}.bin")
    lmm.save_posterior(post, path)
    loaded = lmm.load_posterior(path, f)
    out["loaded"] = lmm.mean_and_var(loaded(O(xs, p), 0.1))
    return out


def same(a, b):
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(same(u, v) for u, v in zip(a, b))
    return np.array_equal(np.asarray(a), np.asarray(b))


@pytest.mark.gpu
@pytest.mark.parametrize("int8", [False, True])
@pytest.mark.parametrize("streams", [1, 4])
@pytest.mark.parametrize("order", ["sorted", "shuffled"])
@pytest.mark.parametrize("kind", ["oilmm", "imogp"])
def test_skipped_build_is_bit_identical(lmm, kind, order, streams, int8, tmp_path):
    ctx = lmm.default_context()
    ctx.set_option("streams", streams)
    ctx.set_option("ozaki", 7 if int8 else 0)
    ctx.set_option("ozaki_bits", 8)
    N = 4096
    ref = run(lmm, kind, N, order, 0, tmp_path)
    new = run(lmm, kind, N, order, 1, tmp_path)
    for k in ref:
        assert same(ref[k], new[k]), k
    # the skip is not vacuous: the narrow SE / Matern latents have exact-zero tiles
    L0 = ref["L"][0]
    assert not np.any(L0[N - T:, :T])
