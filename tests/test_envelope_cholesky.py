"""Tile envelope of the batched Cholesky: far-apart points give kernel entries that are exactly 0.0, and a Cholesky factor keeps
each row's envelope -- if the first nonzero tile of tile row I of K + noise I is F_I, then L(I, k) = 0 for k < F_I, bit for bit.
The OILMM / IndependentMOGP eval path records F_I while it builds the kernel matrices and skips every tile product, TRSM,
digit-plane slice and solve term with an all-zero operand.  CPU: the invariant on LAPACK factors of oracle kernel matrices.  GPU:
logpdf / posterior marginals against the oracle at 1e-9 with bands narrower than a tile, medium bands, dense latents, Matern52 and
SE + Periodic in one batch; the kept factors are exactly 0 outside the envelope; and the int8 update runs exactly the tile products
whose k range is inside the envelope."""
import os

import numpy as np
import pytest
import scipy.linalg as sla

from _tol import assert_isapprox
from oracle import lmm_oracle as o

T = 128


def dense_envelope(nonzero):
    """env[I] = first tile column J <= I of tile row I with a nonzero entry (the diagonal tile always counts)."""
    N = nonzero.shape[0]
    nt = -(-N // T)
    env = np.empty(nt, dtype=np.int64)
    for I in range(nt):
        rows = nonzero[I * T:(I + 1) * T, :(I + 1) * T]
        cols = np.flatnonzero(rows.any(axis=0))
        env[I] = min(cols[0] // T if cols.size else I, I)
    return env


def zero_outside(L, env):
    return all(not np.any(L[I * T:(I + 1) * T, :env[I] * T]) for I in range(len(env)))


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("order", ["sorted", "shuffled"])
def test_lapack_factor_is_zero_outside_the_tile_envelope(order):
    rng = np.random.default_rng(11)
    N = 1000
    x = np.sort(rng.uniform(0, 50, N))
    if order == "shuffled":
        x = rng.permutation(x)
    for inv_ls in (12.0, 1.5, 40.0):
        C = o.kernelmatrix(o.Kernel(o.SE, 1.0, inv_ls), x)
        C[np.diag_indices_from(C)] += 0.1
        env = dense_envelope(C != 0.0)
        assert env.min() < np.arange(len(env)).max()  # some tile row has zero tiles: the check below is not vacuous
        L = sla.cholesky(C, lower=True)
        assert zero_outside(L, env), inv_ls


# ------------------------------------------------------------------------------------------------ GPU
def latents():
    """A band narrower than a tile, a medium band, no zero tile, Matern52, SE + Periodic (dense)."""
    per = o.Kernel(o.SE, 1.2, 0.9, op=o.COMPOSE_SUM, terms=(o.Kernel(o.PERIODIC, 0.5, 0.7, param=0.8),))
    return [o.GP(o.Kernel(o.SE, 1.0, 12.0), 0.1), o.GP(o.Kernel(o.SE, 0.8, 1.5), 0.0), o.GP(o.Kernel(o.SE, 1.1, 0.05), -0.2),
            o.GP(o.Kernel(o.MATERN52, 0.9, 20.0), 0.0), o.GP(per, 0.3)]


def gpu_nonzero(g, x):
    """Where the library's kernel entries are not exactly 0: its exp flushes below e^-708 (csrc/common.cuh: exp_nonpos)."""
    d = np.abs(x[:, None] - x[None, :]) * g.kernel.inv_lengthscale
    if g.kernel.terms:  # a periodic term never vanishes
        return np.ones_like(d, dtype=bool)
    if g.kernel.kind == o.SE:
        return 0.5 * d * d <= 708.0
    assert g.kernel.kind == o.MATERN52
    return np.sqrt(5.0) * d <= 708.0


def problem(N, order):
    rng = np.random.default_rng(N + (order == "shuffled"))
    x = np.sort(rng.uniform(0, N / 20.0, N))
    if order == "shuffled":  # 128-point runs in random order: bands stay, the envelope is no longer monotone
        x = np.concatenate([x[i * T:(i + 1) * T] for i in rng.permutation(-(-N // T))])
    xs = rng.uniform(0, N / 20.0, 40)
    return x, xs


_REF = {}


def reference(kind, N, order):
    key = (kind, N, order)
    if key not in _REF:
        x, xs = problem(N, order)
        gs = latents()
        m = len(gs)
        rng = np.random.default_rng(5)
        if kind == "oilmm":
            p = 7
            U, S = o.orthogonal_from_seed(p, m, seed=2)
            y = rng.standard_normal(p * N)
            om = o.OILMMModel(gs, U, S)
            lp = o.oilmm_logpdf(om, x, 0.1, y)
            M, V = o.oilmm_mean_and_var(o.oilmm_posterior(om, x, 0.1, y), xs, 0.1)
            extra = (U, S)
        else:
            y = rng.standard_normal(m * N)
            lp = o.imogp_logpdf(gs, x, 0.1, y)
            M, V = o.imogp_mean_and_var(o.imogp_posterior(gs, x, 0.1, y), xs, 0.1)
            extra = None
        envs = []
        for g in gs:
            nz = gpu_nonzero(g, x)
            np.fill_diagonal(nz, True)
            envs.append(dense_envelope(nz))
        _REF[key] = (x, xs, y, lp, M, V, extra, np.array(envs))
    return _REF[key]


@pytest.fixture()
def lmm():
    import lmm_b200

    ctx = lmm_b200.default_context()
    yield lmm_b200
    ctx.set_option("ozaki", int(os.environ.get("LMM_OZAKI", "0")))
    ctx.set_option("ozaki_bits", int(os.environ.get("LMM_OZAKI_BITS", "7")))
    ctx.set_option("ozaki_time", 0)
    ctx.set_option("streams", 4)


def build(lmm, kind, N, order):
    from test_composite_kernels import to_lmm

    x, xs, y, lp, M, V, extra, envs = reference(kind, N, order)
    O = lmm.MOInputIsotopicByOutputs
    fs = lmm.independent_mogp([to_lmm(lmm, g) for g in latents()])
    if kind == "oilmm":
        U, S = extra
        f, p = lmm.ILMM(fs, lmm.Orthogonal(U, S)), U.shape[0]
    else:
        f, p = fs, len(latents())
    return f(O(x, p), 0.1), O(xs, p), y


@pytest.mark.gpu
@pytest.mark.parametrize("int8", [False, True])
@pytest.mark.parametrize("streams", [1, 4])
@pytest.mark.parametrize("order", ["sorted", "shuffled"])
@pytest.mark.parametrize("N", [1000, 4096])
@pytest.mark.parametrize("kind", ["oilmm", "imogp"])
def test_envelope_eval_matches_oracle(lmm, kind, N, order, streams, int8):
    ctx = lmm.default_context()
    ctx.set_option("streams", streams)
    ctx.set_option("ozaki", 7 if int8 else 0)
    ctx.set_option("ozaki_bits", 8)
    x, xs, y, lp_ref, M_ref, V_ref, _, envs = reference(kind, N, order)
    fx, Oxs, y = build(lmm, kind, N, order)
    post, lp = lmm.posterior(fx, y, with_logpdf=True)
    assert abs(lp - lp_ref) <= 1e-9 * abs(lp_ref), (lp, lp_ref)
    M, V = lmm.mean_and_var(post(Oxs, 0.1))
    assert_isapprox(M, M_ref, 1e-9, "posterior mean")
    np.testing.assert_allclose(V, V_ref, rtol=1e-9)
    lat = post.f.fs if kind == "oilmm" else post.fs
    for i in range(len(envs)):
        assert zero_outside(lat[i].C, envs[i]), i


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["oilmm", "imogp"])
@pytest.mark.parametrize("order", ["sorted", "shuffled"])
def test_int8_update_runs_only_the_envelope_tile_products(lmm, kind, order):
    """With "ozaki_time" the library reports the 128^3 tile products its int8 launches ran: per tile (I, J) of the wide update of
    block column [s0, s1) (2 tile columns under int8), max(0, s0 - max(env[I], env[J])) -- not s0."""
    ctx = lmm.default_context()
    N, S, bits, ob, min_k = 4096, 7, 8, 2, 4
    ctx.set_option("streams", 1)
    ctx.set_option("ozaki", S)
    ctx.set_option("ozaki_bits", bits)
    ctx.set_option("ozaki_time", 1)
    x, xs, y, lp_ref, _, _, _, envs = reference(kind, N, order)
    fx, _, y = build(lmm, kind, N, order)
    ctx.last_timings()  # drop what earlier calls recorded
    lp = lmm.logpdf(fx, y)
    tm = ctx.last_timings()
    assert abs(lp - lp_ref) <= 1e-9 * abs(lp_ref)
    nt = envs.shape[1]
    want, dense = 0, 0
    for s0 in range(ob, nt, ob):
        if s0 < min_k or s0 * T * S * 16384 >= 2 ** 31:
            continue
        for J in range(s0, min(s0 + ob, nt)):
            for I in range(J, nt):
                kb = np.maximum(envs[:, I], envs[:, J])
                want += int(np.maximum(s0 - kb, 0).sum())
                dense += s0 * len(envs)
    assert want < dense
    assert tm[5] == want, (tm[5], want, dense)
