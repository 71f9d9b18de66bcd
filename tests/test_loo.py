"""Leave-one-input-out (LOO) cross-validation of OILMM / IndependentMOGP: value, LOO predictive marginals and gradient.

The closed-form oracle lives here, on top of the unchanged oracle: per latent (C = K + νI, A = C⁻¹, α = Aδ, d = diag A,
q = α/d, r = (1 + αq)/(2d), w = Aq) LOO = Σ_i (-½ log 2π + ½ log d_i - ½ α_i q_i), dLOO/dC = ½(αw' + wα') - A diag(r) A,
dLOO/dδ = -w; the OILMM adds the regulariser of `o.oilmm_logpdf`.  CPU: it is checked against the brute-force
Σ_i [logpdf(all) - logpdf(without input i)] (value, every gradient block by central differences) and against the oracle
posterior on y_{-i} at x_i (marginals).  GPU: `loo_logpdf` / `loo_mean_and_var` / `loo_logpdf_and_gradient` against it."""
import dataclasses
import os

import numpy as np
import pytest

from _tol import assert_isapprox, relnorm
from oracle import lmm_oracle as o
from test_composite_gradient import _contract, _inputs, _params, _shift, _xin, to_lmm
from test_missing_gradient import KERNEL_CASES, kernel_case


# ------------------------------------------------------------------------------------------------ closed-form oracle
def _latent_loo(f, x, noise, ty):
    K = o.kernelmatrix(f.kernel, x)
    C = K + noise * np.eye(K.shape[0])
    L = o._chol_lower(C)
    A = o._bwd(L, o._fwd(L, np.eye(K.shape[0])))
    alpha = A @ (ty - f.mean_const)
    d = np.diag(A).copy()
    q = alpha / d
    r = (1.0 + alpha * q) / (2.0 * d)
    w = A @ q
    G = 0.5 * (np.outer(alpha, w) + np.outer(w, alpha)) - (A * r[None, :]) @ A
    val = float(np.sum(-0.5 * o.LOG2PI + 0.5 * np.log(d) - 0.5 * alpha * q))
    return val, G, w, ty - q, 1.0 / d - noise


def loo_oracle(fs, x, s2, y, U=None, S=None):
    """(value, (M, V), grads) of the LOO of an OILMM (U, S given) or an IndependentMOGP.  grads: "terms" (per latent,
    (nterms, 3 + D)), "mean_const", "sigma2", "y" (p*N,), and "U" / "S" for an OILMM."""
    N = o._as2d(x).shape[0]
    Y = o.reshape_y(y, N)
    m = len(fs)
    if U is not None:
        T, nu = o.project_orthogonal(U, S, s2)
        H = U * np.sqrt(S)[None, :]
    else:
        T, nu, H = np.eye(m), np.full(m, s2), np.eye(m)
    Ty = T @ Y
    parts = [_latent_loo(f, x, nu[i], Ty[i]) for i, f in enumerate(fs)]
    val = sum(q[0] for q in parts)
    W = np.stack([q[2] for q in parts])
    trG = np.array([np.trace(q[1]) for q in parts])
    M = H @ np.stack([q[3] for q in parts])
    V = (H * H) @ np.stack([q[4] for q in parts]) + s2
    g = {"terms": [_contract(q[1], f, x) for q, f in zip(parts, fs)], "mean_const": W.sum(axis=1)}
    if U is None:
        g["sigma2"] = float(np.sum(trG))
        g["y"] = (-W).reshape(-1)
        return val, (M.reshape(-1), V.reshape(-1)), g
    p = U.shape[0]
    val += o.regulariser_orthogonal(U, S, s2, Y)
    R = (np.eye(p) - U @ U.T) @ Y
    resid = float(np.sum(R * R))
    g["sigma2"] = float(np.sum(trG / S)) - 0.5 * (N * (p - m) / s2 - resid / s2 ** 2)
    g["y"] = (-T.T @ W - R / s2).reshape(-1)
    g["S"] = np.array([(W[i] @ Ty[i]) / (2 * S[i]) - trG[i] * s2 / S[i] ** 2 - N / (2 * S[i]) for i in range(m)])
    Z = U.T @ Y
    g["U"] = -(Y @ W.T) / np.sqrt(S)[None, :] + (R @ Z.T + Y @ (R.T @ U)) / s2
    return val, (M.reshape(-1), V.reshape(-1)), g


def _drop(x, y, p, i):
    N = o._as2d(x).shape[0]
    return np.delete(x, i, axis=0), np.delete(o.reshape_y(y, N), i, axis=1).reshape(-1)


def brute_loo(fs, x, s2, y, U=None, S=None):
    """Σ_i [logpdf(all) - logpdf(without input i)] by N + 1 oracle logpdfs."""
    N = o._as2d(x).shape[0]
    if U is not None:
        model = o.OILMMModel(fs, U, S)
        lp = lambda xx, yy: o.oilmm_logpdf(model, xx, s2, yy)  # noqa: E731
        p = U.shape[0]
    else:
        lp = lambda xx, yy: o.imogp_logpdf(fs, xx, s2, yy)  # noqa: E731
        p = len(fs)
    full = lp(x, y)
    return sum(full - lp(*_drop(x, y, p, i)) for i in range(N))


def _case(case, model, N, seed):
    rng = np.random.default_rng(seed)
    fs, D = kernel_case(case)
    x = _inputs(rng, N, D, hi=max(6.0, N / 40.0))
    if model == "oilmm":
        p = 5
        U, S = o.orthogonal_from_seed(p, len(fs), seed=seed % 7 + 1)
    else:
        p, U, S = len(fs), None, None
    y = rng.standard_normal(p * N)
    return fs, D, x, p, U, S, y


MODELS = ["oilmm", "imogp"]


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oracle_loo_value_and_marginals_equal_the_brute_force(case, model):
    fs, D, x, p, U, S, y = _case(case, model, 25, 3 + KERNEL_CASES.index(case))
    val, (M, V), _ = loo_oracle(fs, x, 0.2, y, U, S)
    ref = brute_loo(fs, x, 0.2, y, U, S)
    assert abs(val - ref) <= 1e-12 * abs(ref), (val, ref)
    N = len(x)
    for i in range(N):
        xm, ym = _drop(x, y, p, i)
        if U is not None:
            Mr, Vr = o.oilmm_mean_and_var(o.oilmm_posterior(o.OILMMModel(fs, U, S), xm, 0.2, ym), x[i:i + 1], 0.2)
        else:
            Mr, Vr = o.imogp_mean_and_var(o.imogp_posterior(fs, xm, 0.2, ym), x[i:i + 1], 0.2)
        assert relnorm(M.reshape(p, N)[:, i], Mr) <= 1e-10
        assert relnorm(V.reshape(p, N)[:, i], Vr) <= 1e-10


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oracle_loo_gradient_matches_finite_differences_of_the_brute_force(case, model):
    s2, h, rtol = 0.2, 1e-6, 5e-6
    fs, D, x, p, U, S, y = _case(case, model, 14, 30 + KERNEL_CASES.index(case))
    _, _, g = loo_oracle(fs, x, s2, y, U, S)

    def lp(fs2=fs, s=s2, y2=y, U2=U, S2=S):
        return brute_loo(fs2, x, s, y2, U2, S2)

    def close(fd, an, scale, what):
        assert abs(fd - an) <= rtol * max(abs(an), 1e-2 * scale), (what, fd, an)

    for i, f in enumerate(fs):
        scale = max(1e-3, float(np.max(np.abs(g["terms"][i]))))
        for t, j, v in _params(f, D):
            hh = h * max(1.0, abs(v))
            close((lp(fs2=_shift(fs, i, t, j, hh)) - lp(fs2=_shift(fs, i, t, j, -hh))) / (2 * hh), g["terms"][i][t, j], scale, (i, t, j))

        def mshift(dm, i=i):
            return [dataclasses.replace(q, mean_const=q.mean_const + dm) if n == i else q for n, q in enumerate(fs)]

        close((lp(fs2=mshift(h)) - lp(fs2=mshift(-h))) / (2 * h), g["mean_const"][i], max(1e-3, float(np.max(np.abs(g["mean_const"])))),
              "mean")
    close((lp(s=s2 * (1 + h)) - lp(s=s2 * (1 - h))) / (2 * h * s2), g["sigma2"], abs(g["sigma2"]), "sigma2")
    scale = max(1e-3, float(np.max(np.abs(g["y"]))))
    for a in range(0, len(y), max(1, len(y) // 10)):
        yp, ym = y.copy(), y.copy()
        yp[a] += h
        ym[a] -= h
        close((lp(y2=yp) - lp(y2=ym)) / (2 * h), g["y"][a], scale, ("y", a))
    if U is None:
        return
    for i in range(len(fs)):
        Sp, Sm = S.copy(), S.copy()
        Sp[i] += h
        Sm[i] -= h
        close((lp(S2=Sp) - lp(S2=Sm)) / (2 * h), g["S"][i], max(1e-3, float(np.max(np.abs(g["S"])))), ("S", i))
    scale = max(1e-3, float(np.max(np.abs(g["U"]))))
    for j in range(U.shape[0]):
        for i in range(U.shape[1]):
            Up, Um = U.copy(), U.copy()
            Up[j, i] += h
            Um[j, i] -= h
            close((lp(U2=Up) - lp(U2=Um)) / (2 * h), g["U"][j, i], scale, ("U", j, i))


def test_oracle_loo_at_n1_is_the_prior_logpdf():
    """N = 1: nothing is left to condition on, so LOO is the prior logpdf."""
    fs, _, x, p, U, S, y = _case("se_matern52", "oilmm", 1, 5)
    val, _, _ = loo_oracle(fs, x, 0.2, y, U, S)
    assert abs(val - o.oilmm_logpdf(o.OILMMModel(fs, U, S), x, 0.2, y)) <= 1e-13 * abs(val)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def lmm():
    import lmm_b200

    lmm_b200.default_context()
    return lmm_b200


def _fx(lmm, fs, x, p, s2, U=None, S=None):
    lat = lmm.independent_mogp([to_lmm(lmm, g) for g in fs])
    f = lmm.ILMM(lat, lmm.Orthogonal(U, S)) if U is not None else lat
    return f(lmm.MOInputIsotopicByOutputs(_xin(lmm, x), p), s2)


def _terms_array(got):
    return [np.array([[t["variance"], t["inv_lengthscale"], t["param"]] + list(t["ard"]) for t in lat]) for lat in got]


def _assert_grads(g, ref, orth, rtol=1e-9):
    got = _terms_array(g["terms"])
    assert_isapprox(np.concatenate([a.ravel() for a in got]), np.concatenate([r.ravel() for r in ref["terms"]]), rtol, what="terms")
    assert_isapprox(g["variance"], [r[0, 0] for r in ref["terms"]], rtol, what="variance")
    assert_isapprox(g["inv_lengthscale"], [r[0, 1] for r in ref["terms"]], rtol, what="inv_lengthscale")
    # term 0's ARD slots (zeros for a term without an ARDTransform), as grad_ard returns them
    assert_isapprox(g["ard"], np.stack([r[0, 3:] for r in ref["terms"]]), rtol, what="ard")
    assert_isapprox(g["mean_const"], ref["mean_const"], rtol, what="mean_const")
    assert_isapprox([g["sigma2"]], [ref["sigma2"]], rtol, what="sigma2")
    assert_isapprox(g["y"], ref["y"], rtol, what="y")
    if orth:
        assert_isapprox(g["U"], ref["U"], rtol, what="U")
        assert_isapprox(g["S"], ref["S"], rtol, what="S")


def _check_against_oracle(lmm, fs, x, p, s2, y, U, S, rtol=1e-9):
    fx = _fx(lmm, fs, x, p, s2, U, S)
    val, (Mr, Vr), ref = loo_oracle(fs, x, s2, y, U, S)
    v, g = lmm.loo_logpdf_and_gradient(fx, y, with_grad_y=True)
    assert abs(v - val) <= rtol * abs(val), (v, val)
    _assert_grads(g, ref, U is not None, rtol)
    M, V = lmm.loo_mean_and_var(fx, y)
    assert_isapprox(M, Mr, rtol, what="LOO mean")
    assert_isapprox(V, Vr, rtol, what="LOO var")
    vv = lmm.loo_logpdf(fx, y)
    assert abs(vv - v) <= 1e-12 * abs(v), (vv, v)  # the value path against the gradient path's value
    return fx


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 50, 129, 300, 700, 2300])
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oilmm_loo_matches_oracle(lmm, case, N):
    """Ragged N (50, 129, 300, 700, 2300) leaves identity padding rows in the last tile: they must contribute nothing."""
    fs, D, x, p, U, S, y = _case(case, "oilmm", N, 100 + N + KERNEL_CASES.index(case))
    _check_against_oracle(lmm, fs, x, p, 0.15, y, U, S)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 129, 700])
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_imogp_loo_matches_oracle(lmm, case, N):
    fs, D, x, p, U, S, y = _case(case, "imogp", N, 200 + N + KERNEL_CASES.index(case))
    _check_against_oracle(lmm, fs, x, p, 0.15, y, None, None)


@pytest.mark.gpu
def test_loo_at_n1_is_the_prior_logpdf(lmm):
    fs, _, x, p, U, S, y = _case("periodic_sum", "oilmm", 1, 9)
    fx = _fx(lmm, fs, x, p, 0.2, U, S)
    assert abs(lmm.loo_logpdf(fx, y) - lmm.logpdf(fx, y)) <= 1e-12 * abs(lmm.logpdf(fx, y))


@pytest.mark.gpu
def test_loo_agrees_with_the_library_posterior_and_logpdf(lmm):
    """LOO marginals are what the library's own posterior on y_{-i} predicts at x_i; at N = 300 the LOO value is the sum
    over every input of logpdf(all) - logpdf(without i)."""
    fs, D, x, p, U, S, y = _case("se_matern52", "oilmm", 300, 11)
    s2 = 0.15
    fx = _fx(lmm, fs, x, p, s2, U, S)
    M, V = lmm.loo_mean_and_var(fx, y)
    N = len(x)
    for i in (0, 1, 127, 128, 200, N - 1):
        xm, ym = _drop(x, y, p, i)
        post = lmm.posterior(_fx(lmm, fs, xm, p, s2, U, S), ym)
        Mi, Vi = lmm.mean_and_var(post(lmm.MOInputIsotopicByOutputs(_xin(lmm, x[i:i + 1]), p), s2))
        assert_isapprox(M.reshape(p, N)[:, i], Mi, what=f"mean {i}")
        assert_isapprox(V.reshape(p, N)[:, i], Vi, what=f"var {i}")
    full = lmm.logpdf(fx, y)
    brute = 0.0
    for i in range(N):
        xm, ym = _drop(x, y, p, i)
        brute += full - lmm.logpdf(_fx(lmm, fs, xm, p, s2, U, S), ym)
    v = lmm.loo_logpdf(fx, y)
    assert abs(v - brute) <= 1e-9 * abs(v), (v, brute)


@pytest.mark.gpu
def test_loo_is_deterministic(lmm):
    fs, D, x, p, U, S, y = _case("ard_D2", "oilmm", 400, 12)
    fx = _fx(lmm, fs, x, p, 0.2, U, S)
    va, a = lmm.loo_logpdf_and_gradient(fx, y, with_grad_y=True)
    vb, b = lmm.loo_logpdf_and_gradient(fx, y, with_grad_y=True)
    assert va == vb
    for k in ("variance", "inv_lengthscale", "mean_const", "ard", "y", "U", "S"):
        assert np.array_equal(a[k], b[k]), k
    assert a["sigma2"] == b["sigma2"]
    for ta, tb in zip(_terms_array(a["terms"]), _terms_array(b["terms"])):
        assert np.array_equal(ta, tb)
    assert lmm.loo_logpdf(fx, y) == lmm.loo_logpdf(fx, y)
    Ma, Va = lmm.loo_mean_and_var(fx, y)
    Mb, Vb = lmm.loo_mean_and_var(fx, y)
    assert np.array_equal(Ma, Mb) and np.array_equal(Va, Vb)


@pytest.mark.gpu
def test_loo_reports_a_failed_factorisation(lmm):
    """Duplicate inputs and a vanishing noise: singular latent covariance, reported as the logpdf reports it, on the value
    path and on the gradient path."""
    fs = [o.GP(o.Kernel(o.SE), 0.0)]
    x = np.array([0.0, 0.0, 1.0])
    fx = _fx(lmm, fs, x, 1, 1e-300)
    with pytest.raises(lmm.PosDefException) as e:
        lmm.loo_logpdf(fx, np.zeros(3))
    assert e.value.info > 0 and e.value.latent == 0
    with pytest.raises(lmm.PosDefException):
        lmm.loo_logpdf_and_gradient(fx, np.zeros(3))


@pytest.mark.gpu
def test_loo_refusals(lmm):
    fs, D, x, p, U, S, y = _case("se_matern52", "oilmm", 30, 13)
    lat = lmm.independent_mogp([to_lmm(lmm, g) for g in fs])
    O = lmm.MOInputIsotopicByOutputs
    fx = _fx(lmm, fs, x, p, 0.2, U, S)
    with pytest.raises(TypeError):  # general ILMM
        lmm.loo_logpdf(lmm.ILMM(lat, U * np.sqrt(S)[None, :])(O(_xin(lmm, x), p), 0.2), y)
    post = lmm.posterior(fx, y)
    with pytest.raises(TypeError):  # posterior FiniteGP
        lmm.loo_logpdf(post(O(_xin(lmm, x), p), 0.2), y)
    with pytest.raises(TypeError):  # by-features inputs
        lmm.loo_mean_and_var(lmm.ILMM(lat, lmm.Orthogonal(U, S))(lmm.MOInputIsotopicByFeatures(_xin(lmm, x), p), 0.2), y)
    with pytest.raises(TypeError):  # non-scalar noise
        lmm.loo_logpdf_and_gradient(lat(O(_xin(lmm, x), len(fs)), np.full(len(fs) * len(x), 0.2)), y[: len(fs) * len(x)])
    y2 = y.copy()
    y2[7] = np.nan
    with pytest.raises(ValueError):
        lmm.loo_logpdf(fx, y2)
    with pytest.raises(ValueError):
        lmm.loo_logpdf_and_gradient(fx, y2)
    # the C entry points refuse a NaN in y and m > p themselves
    import ctypes as C

    lib = lmm._lib
    ctx = lmm.default_context()
    descs = lmm.api._descs([to_lmm(lmm, g) for g in fs])
    pts = np.ascontiguousarray(np.asarray(x, dtype=np.float64).reshape(len(x), 1))
    out = C.c_double()
    Uf, Sv = np.asfortranarray(U), np.ascontiguousarray(S)
    rc = ctx.lib.lmm_oilmm_loo(ctx.handle, descs, 2, lib.ptr(pts), len(x), 1, lib.ptr(Uf), lib.ptr(Sv), p, 0.2, lib.ptr(y2), p,
                               C.byref(out), None, None, None, None, None, None, None, None, None, None)
    assert rc == lib.LMM_E_ARG
    U1 = np.asfortranarray(U[:1, :])
    rc = ctx.lib.lmm_oilmm_loo(ctx.handle, descs, 2, lib.ptr(pts), len(x), 1, lib.ptr(U1), lib.ptr(Sv), 1, 0.2, lib.ptr(y[: len(x)]), 1,
                               C.byref(out), None, None, None, None, None, None, None, None, None, None)
    assert rc == lib.LMM_E_ARG


@pytest.mark.gpu
def test_loo_with_the_int8_factorisation(lmm):
    """"ozaki" = 7 planes of 8 bits (the setting bench.py times): three latents put the factorisation on the batched schedule,
    whose wide updates then run on the int8 tensor cores ("ozaki_time" counts their tile products); the potri and the SYRKs
    stay FP64."""
    fs, D, x, p, U, S, y = _case("se_matern52", "oilmm", 2300, 14)
    fs = fs + [o.GP(o.Kernel(o.MATERN32, 0.8, 0.7), 0.05)]
    U, S = o.orthogonal_from_seed(p, len(fs), seed=3)
    ctx = lmm.default_context()
    ctx.set_option("ozaki", 7)
    ctx.set_option("ozaki_bits", 8)
    ctx.set_option("ozaki_time", 1)
    try:
        ctx.last_timings()  # drop what earlier calls recorded
        _check_against_oracle(lmm, fs, x, p, 0.15, y, U, S)
        assert ctx.last_timings()[5] > 0  # int8 tile products ran
    finally:
        ctx.set_option("ozaki_time", 0)
        ctx.set_option("ozaki", int(os.environ.get("LMM_OZAKI", "0")))  # the library default, or what the whole run was started with
        ctx.set_option("ozaki_bits", int(os.environ.get("LMM_OZAKI_BITS", "7")))
