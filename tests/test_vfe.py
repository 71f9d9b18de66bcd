"""Sparse variational (VFE) bound and posterior of OILMM / IndependentMOGP priors.

The closed-form oracle lives here, on top of the unchanged oracle, in the whitened form the library uses: per latent
(Kz = K(z, z) + jitter I = Lz Lz', B' = K(x, z) Lz^{-T}, Ψ = B B', b = B δ, Σ = I + Ψ/ν = L_Σ L_Σ')
    ELBO_l = -½ [N log 2π + N log ν + log|Σ| + δ'δ/ν - b'Σ⁻¹b/ν² + (Σ_i k_ii - tr Ψ)/ν]
plus the regulariser of `o.oilmm_logpdf` for an OILMM.  CPU: it is checked against Titsias' bound of the dense pN model, against
the exact logpdf (a lower bound, equal for z = x and jitter 0) and against the unwhitened predictive formulas.  GPU: `elbo` and
`posterior(VFE(z), fx, y)` against it."""
import ctypes as C
import dataclasses
import os

import numpy as np
import pytest

from _tol import assert_isapprox
from oracle import lmm_oracle as o
from test_composite_gradient import _inputs, _params, _shift, _xin, to_lmm
from test_missing_gradient import KERNEL_CASES, kernel_case


# ------------------------------------------------------------------------------------------------ closed-form oracle
def _latent_vfe(f, x, z, jitter, nu, ty, xs=None):
    M = o._as2d(z).shape[0]
    Lz = o._chol_lower(o.kernelmatrix(f.kernel, z) + jitter * np.eye(M))
    Bt = o._fwd(Lz, o.kernelmatrix(f.kernel, z, x)).T  # K(x, z) Lz^{-T}
    d = ty - f.mean_const
    Psi = Bt.T @ Bt
    b = Bt.T @ d
    Ls = o._chol_lower(np.eye(M) + Psi / nu)
    c = o._fwd(Ls, b)
    N = len(d)
    val = -0.5 * (N * o.LOG2PI + N * np.log(nu) + 2 * np.sum(np.log(np.diag(Ls))) + d @ d / nu - c @ c / nu ** 2
                  + (np.sum(o.kernelmatrix_diag(f.kernel, x)) - np.trace(Psi)) / nu)
    if xs is None:
        return val, None, None
    V = o._fwd(Lz, o.kernelmatrix(f.kernel, z, xs)).T
    W = o._fwd(Ls, V.T).T  # V L_Σ^{-T}
    mean = f.mean_const + W @ c / nu
    var = o.kernelmatrix_diag(f.kernel, xs) - np.sum(V * V, axis=1) + np.sum(W * W, axis=1)
    return val, mean, var


def vfe_oracle(fs, x, z, jitter, s2, y, U=None, S=None, xs=None):
    """(ELBO, (mean, var) at xs by outputs or None) of an OILMM (U, S given) or an IndependentMOGP."""
    N = o._as2d(x).shape[0]
    Y = o.reshape_y(y, N)
    m = len(fs)
    if U is not None:
        T, nu = o.project_orthogonal(U, S, s2)
        H = U * np.sqrt(S)[None, :]
    else:
        T, nu, H = np.eye(m), np.full(m, s2), np.eye(m)
    Ty = T @ Y
    parts = [_latent_vfe(f, x, z, jitter, nu[i], Ty[i], xs) for i, f in enumerate(fs)]
    val = sum(q[0] for q in parts)
    if U is not None:
        val += o.regulariser_orthogonal(U, S, s2, Y)
    if xs is None:
        return val, None
    ML, VL = np.stack([q[1] for q in parts]), np.stack([q[2] for q in parts])
    if U is not None:
        return val, ((H @ ML).reshape(-1), ((H * H) @ (VL + 1e-18) + s2).reshape(-1))
    return val, (ML.reshape(-1), (VL + s2).reshape(-1))


def dense_titsias(fs, x, z, jitter, s2, y, U=None, S=None):
    """Titsias' bound of the dense pN model: log N(y; Hμ, Σ_l h_l h_l' ⊗ Q_l + σ²I) - Σ_l |h_l|² tr(K_l - Q_l) / (2σ²)."""
    N = o._as2d(x).shape[0]
    m = len(fs)
    H = U * np.sqrt(S)[None, :] if U is not None else np.eye(m)
    p = H.shape[0]
    Cov = s2 * np.eye(p * N)
    mean = np.zeros(p * N)
    trace = 0.0
    for i, f in enumerate(fs):
        Kz = o.kernelmatrix(f.kernel, z) + jitter * np.eye(o._as2d(z).shape[0])
        Kzx = o.kernelmatrix(f.kernel, z, x)
        Q = Kzx.T @ np.linalg.solve(Kz, Kzx)
        h = H[:, i]
        Cov += np.kron(np.outer(h, h), Q)
        mean += np.kron(h, np.full(N, f.mean_const))
        trace += (h @ h) * (np.sum(o.kernelmatrix_diag(f.kernel, x)) - np.trace(Q))
    Lc = o._chol_lower(Cov)
    r = o._fwd(Lc, y - mean)
    return -0.5 * (p * N * o.LOG2PI + 2 * np.sum(np.log(np.diag(Lc))) + r @ r) - trace / (2 * s2)


def _case(case, model, N, M, seed, spread=False):
    rng = np.random.default_rng(seed)
    fs, D = kernel_case(case)
    hi = max(6.0, N / 40.0)
    x = _inputs(rng, N, D, hi=hi)
    z = _inputs(rng, M, D, hi=hi)
    if model == "oilmm":
        p = 5
        U, S = o.orthogonal_from_seed(p, len(fs), seed=seed % 7 + 1)
    else:
        p, U, S = len(fs), None, None
    y = rng.standard_normal(p * N)
    return fs, D, x, z, p, U, S, y


MODELS = ["oilmm", "imogp"]
JIT = 1e-4  # keeps K(z, z) well conditioned for every kernel case (periodic latents repeat inducing inputs modulo the period)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oracle_elbo_is_the_titsias_bound_of_the_dense_model(case, model):
    fs, D, x, z, p, U, S, y = _case(case, model, 30, 7, 3 + KERNEL_CASES.index(case))
    val, _ = vfe_oracle(fs, x, z, JIT, 0.2, y, U, S)
    ref = dense_titsias(fs, x, z, JIT, 0.2, y, U, S)
    assert abs(val - ref) <= 1e-12 * abs(ref), (val, ref)


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oracle_elbo_bounds_the_logpdf_and_is_exact_at_z_equal_x(case, model):
    fs, D, x, z, p, U, S, y = _case(case, model, 12, 5, 20 + KERNEL_CASES.index(case))
    x = np.arange(12.0) * 1.7 if D == 1 else np.stack([np.arange(12.0) * 1.7, np.arange(12.0)[::-1] * 1.3], axis=1)
    exact = o.oilmm_logpdf(o.OILMMModel(fs, U, S), x, 0.2, y) if U is not None else o.imogp_logpdf(fs, x, 0.2, y)
    val, _ = vfe_oracle(fs, x, z[:5], JIT, 0.2, y, U, S)
    assert val <= exact
    val_x, _ = vfe_oracle(fs, x, x, 0.0, 0.2, y, U, S)
    assert abs(val_x - exact) <= 1e-10 * abs(exact), (val_x, exact)


@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oracle_marginals_match_the_unwhitened_formulas(case):
    fs, D, x, z, p, U, S, y = _case(case, "imogp", 40, 9, 40 + KERNEL_CASES.index(case))
    xs = _inputs(np.random.default_rng(1), 11, D)
    nu = 0.2
    for i, f in enumerate(fs):
        d = y[i * 40:(i + 1) * 40] - f.mean_const
        _, mean, var = _latent_vfe(f, x, z, JIT, nu, y[i * 40:(i + 1) * 40], xs)
        Kz = o.kernelmatrix(f.kernel, z) + JIT * np.eye(9)
        Kzx, Ksz = o.kernelmatrix(f.kernel, z, x), o.kernelmatrix(f.kernel, xs, z)
        Sig = Kz + Kzx @ Kzx.T / nu
        m_ref = f.mean_const + Ksz @ np.linalg.solve(Sig, Kzx @ d) / nu
        v_ref = (o.kernelmatrix_diag(f.kernel, xs) - np.sum(Ksz * np.linalg.solve(Kz, Ksz.T).T, axis=1)
                 + np.sum(Ksz * np.linalg.solve(Sig, Ksz.T).T, axis=1))
        assert_isapprox(mean, m_ref, 1e-10, what="mean")
        assert_isapprox(var, v_ref, 1e-10, what="var")


def _latent_vfe_grad(f, x, z, jitter, nu, ty):
    """The whitened cotangents of ELBO_l: (Ḡxz, Ḡz, dELBO/dδ, dELBO/dν)."""
    M = o._as2d(z).shape[0]
    Lz = o._chol_lower(o.kernelmatrix(f.kernel, z) + jitter * np.eye(M))
    Lzi = o._fwd(Lz, np.eye(M))
    Bt = o.kernelmatrix(f.kernel, x, z) @ Lzi.T
    d = ty - f.mean_const
    Psi, b = Bt.T @ Bt, Bt.T @ d
    Sig = np.eye(M) + Psi / nu
    Si = np.linalg.inv(Sig)
    bw = Si @ b
    beta = Lzi.T @ bw
    Gxz = Bt @ ((np.eye(M) - Si) / nu - np.outer(bw, bw) / nu ** 3) @ Lzi + np.outer(d, beta) / nu ** 2
    Gz = 0.5 * Lzi.T @ (2 * np.eye(M) - Si - Sig - np.outer(bw, bw) / nu ** 2) @ Lzi
    N = len(d)
    kd = np.sum(o.kernelmatrix_diag(f.kernel, x))
    dnu = -0.5 * (N / nu - np.trace(Si @ Psi) / nu ** 2 - d @ d / nu ** 2 + 2 * b @ bw / nu ** 3 - bw @ Psi @ bw / nu ** 4
                  - (kd - np.trace(Psi)) / nu ** 2)
    return Gxz, Gz, -(d - Bt @ bw / nu) / nu, dnu


@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oracle_gradient_formulas_match_finite_differences(case):
    """Every kernel hyper-parameter (through K(x, z), K(z, z) and k(x, x)), δ and ν against central differences of ELBO_l."""
    fs, D, x, z, p, U, S, y = _case(case, "imogp", 20, 6, 60 + KERNEL_CASES.index(case))
    nu, h, rtol = 0.2, 1e-6, 5e-6
    for i, f in enumerate(fs):
        ty = y[i * 20:(i + 1) * 20]
        Gxz, Gz, gd, dnu = _latent_vfe_grad(f, x, z, JIT, nu, ty)
        val = lambda g=f, n=nu, t=ty: _latent_vfe(g, x, z, JIT, n, t)[0]  # noqa: E731
        for t, j, v in _params(f, D):
            hh = h * max(1.0, abs(v))
            fp, fm = _shift([f], 0, t, j, hh)[0], _shift([f], 0, t, j, -hh)[0]
            dKxz = (o.kernelmatrix(fp.kernel, x, z) - o.kernelmatrix(fm.kernel, x, z)) / (2 * hh)
            dKz = (o.kernelmatrix(fp.kernel, z) - o.kernelmatrix(fm.kernel, z)) / (2 * hh)
            dkd = (np.sum(o.kernelmatrix_diag(fp.kernel, x)) - np.sum(o.kernelmatrix_diag(fm.kernel, x))) / (2 * hh)
            an = np.sum(Gxz * dKxz) + np.sum(Gz * dKz) - dkd / (2 * nu)
            fd = (val(g=fp) - val(g=fm)) / (2 * hh)
            assert abs(fd - an) <= rtol * max(abs(an), 1e-2), (i, t, j, fd, an)
        fd = (val(n=nu * (1 + h)) - val(n=nu * (1 - h))) / (2 * h * nu)
        assert abs(fd - dnu) <= rtol * abs(dnu), ("nu", fd, dnu)
        for a in range(0, 20, 4):
            tp, tm = ty.copy(), ty.copy()
            tp[a] += h
            tm[a] -= h
            fd = (val(t=tp) - val(t=tm)) / (2 * h)
            assert abs(fd - gd[a]) <= rtol * max(abs(gd[a]), 1e-2), ("delta", a, fd, gd[a])


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


def _check(lmm, fs, D, x, z, p, U, S, y, s2=0.15, jitter=JIT, rtol=1e-9):
    xs = _inputs(np.random.default_rng(5), 77, D, hi=float(np.max(x)) + 0.5)
    val, (Mr, Vr) = vfe_oracle(fs, x, z, jitter, s2, y, U, S, xs)
    fx = _fx(lmm, fs, x, p, s2, U, S)
    approx = lmm.VFE(_xin(lmm, z), jitter)
    v = lmm.elbo(approx, fx, y)
    assert abs(v - val) <= rtol * abs(val), (v, val)
    post = lmm.posterior(approx, fx, y)
    Mg, Vg = lmm.mean_and_var(post(lmm.MOInputIsotopicByOutputs(_xin(lmm, xs), p), s2))
    assert_isapprox(Mg, Mr, rtol, what="mean")
    assert_isapprox(Vg, Vr, rtol, what="var")
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 50, 129, 300])
@pytest.mark.parametrize("N", [1, 129, 700, 2300])
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oilmm_vfe_matches_oracle(lmm, case, N, M):
    """Ragged N and M leave padding rows in the last tiles of K(x, z) and K(z, z): they must contribute nothing."""
    _check(lmm, *_case(case, "oilmm", N, M, 100 + N + M + KERNEL_CASES.index(case)))


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 50, 129, 300])
@pytest.mark.parametrize("N", [1, 129, 700, 2300])
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_imogp_vfe_matches_oracle(lmm, case, N, M):
    _check(lmm, *_case(case, "imogp", N, M, 200 + N + M + KERNEL_CASES.index(case)))


@pytest.mark.gpu
def test_vfe_chunks_agree_with_one_chunk(lmm):
    """"vfe_chunk" = 2 tile rows splits N = 700 (6 tile rows) into 3 chunks whose Gram sums are added in chunk order."""
    fs, D, x, z, p, U, S, y = _case("se_matern52", "oilmm", 700, 129, 7)
    fx = _fx(lmm, fs, x, p, 0.15, U, S)
    approx = lmm.VFE(_xin(lmm, z), JIT)
    ctx = lmm.default_context()
    one = lmm.elbo(approx, fx, y)
    ctx.set_option("vfe_chunk", 2)
    try:
        three = lmm.elbo(approx, fx, y)
        xs = _xin(lmm, x[:50])
        M3, V3 = lmm.mean_and_var(lmm.posterior(approx, fx, y)(lmm.MOInputIsotopicByOutputs(xs, p), 0.15))
    finally:
        ctx.set_option("vfe_chunk", 0)
    M1, V1 = lmm.mean_and_var(lmm.posterior(approx, fx, y)(lmm.MOInputIsotopicByOutputs(xs, p), 0.15))
    assert abs(one - three) <= 1e-12 * abs(one), (one, three)
    assert_isapprox(M3, M1, 1e-12, what="mean")
    assert_isapprox(V3, V1, 1e-12, what="var")


@pytest.mark.gpu
@pytest.mark.parametrize("model", MODELS)
def test_vfe_at_z_equal_x_is_the_logpdf(lmm, model):
    fs, D, _, _, p, U, S, y = _case("se_matern52", model, 40, 1, 8)
    x = np.arange(40.0) * 2.5
    fx = _fx(lmm, fs, x, p, 0.2, U, S)
    lp = lmm.logpdf(fx, y)
    v = lmm.elbo(lmm.VFE(_xin(lmm, x), 0.0), fx, y)
    assert abs(v - lp) <= 1e-9 * abs(lp), (v, lp)


@pytest.mark.gpu
def test_vfe_is_deterministic(lmm):
    fs, D, x, z, p, U, S, y = _case("ard_D2", "oilmm", 2300, 300, 12)
    fx = _fx(lmm, fs, x, p, 0.2, U, S)
    approx = lmm.VFE(_xin(lmm, z), JIT)
    assert lmm.elbo(approx, fx, y) == lmm.elbo(approx, fx, y)
    xs = lmm.MOInputIsotopicByOutputs(_xin(lmm, x[:300]), p)
    Ma, Va = lmm.mean_and_var(lmm.posterior(approx, fx, y)(xs, 0.2))
    Mb, Vb = lmm.mean_and_var(lmm.posterior(approx, fx, y)(xs, 0.2))
    assert np.array_equal(Ma, Mb) and np.array_equal(Va, Vb)


@pytest.mark.gpu
def test_vfe_reports_a_failed_factorisation(lmm):
    """Duplicate inducing inputs with jitter 0: K(z, z) is singular, reported with the latent as the logpdf reports it."""
    fs, D, x, _, p, U, S, y = _case("se_matern52", "oilmm", 50, 3, 9)
    fx = _fx(lmm, fs, x, p, 0.2, U, S)
    approx = lmm.VFE(np.array([1.0, 2.0, 2.0]), 0.0)
    with pytest.raises(lmm.PosDefException) as e:
        lmm.elbo(approx, fx, y)
    assert e.value.info > 0 and e.value.latent == 0
    with pytest.raises(lmm.PosDefException):
        lmm.posterior(approx, fx, y)


@pytest.mark.gpu
def test_vfe_refusals(lmm):
    fs, D, x, z, p, U, S, y = _case("se_matern52", "oilmm", 30, 5, 13)
    lat = lmm.independent_mogp([to_lmm(lmm, g) for g in fs])
    O = lmm.MOInputIsotopicByOutputs
    fx = _fx(lmm, fs, x, p, 0.2, U, S)
    approx = lmm.VFE(_xin(lmm, z))
    with pytest.raises(TypeError):  # general ILMM
        lmm.elbo(approx, lmm.ILMM(lat, U * np.sqrt(S)[None, :])(O(_xin(lmm, x), p), 0.2), y)
    post = lmm.posterior(fx, y)
    with pytest.raises(TypeError):  # posterior FiniteGP
        lmm.elbo(approx, post(O(_xin(lmm, x), p), 0.2), y)
    with pytest.raises(TypeError):  # by-features inputs
        lmm.posterior(approx, lmm.ILMM(lat, lmm.Orthogonal(U, S))(lmm.MOInputIsotopicByFeatures(_xin(lmm, x), p), 0.2), y)
    with pytest.raises(TypeError):  # non-scalar noise
        lmm.elbo(approx, lat(O(_xin(lmm, x), len(fs)), np.full(len(fs) * len(x), 0.2)), y[: len(fs) * len(x)])
    y2 = y.copy()
    y2[7] = np.nan
    with pytest.raises(ValueError):
        lmm.elbo(approx, fx, y2)
    # the C entry points refuse a NaN in y, M < 1, a negative jitter and m > p themselves
    lib = lmm._lib
    ctx = lmm.default_context()
    descs = lmm.api._descs([to_lmm(lmm, g) for g in fs])
    pts = np.ascontiguousarray(np.asarray(x, dtype=np.float64).reshape(len(x), 1))
    zp = np.ascontiguousarray(np.asarray(z, dtype=np.float64))
    out = C.c_double()
    Uf, Sv = np.asfortranarray(U), np.ascontiguousarray(S)

    def call(yv, M=len(z), jitter=JIT, Um=Uf, pp=p):
        return ctx.lib.lmm_oilmm_vfe(ctx.handle, descs, 2, lib.ptr(pts), len(x), 1, lib.ptr(zp), M, jitter, lib.ptr(Um), lib.ptr(Sv), pp,
                                     0.2, lib.ptr(yv), pp, C.byref(out), None, None, None, None, None, None, None, None)

    assert call(y) == lib.LMM_OK
    assert call(y2) == lib.LMM_E_ARG
    assert call(y, M=0) == lib.LMM_E_ARG
    assert call(y, jitter=-1.0) == lib.LMM_E_ARG
    assert call(np.ascontiguousarray(y[: len(x)]), Um=np.asfortranarray(U[:1, :]), pp=1) == lib.LMM_E_ARG
    rc = ctx.lib.lmm_imogp_vfe(ctx.handle, descs, 2, lib.ptr(pts), len(x), 1, lib.ptr(zp), len(z), JIT, 0.0, lib.ptr(y[: 2 * len(x)]), 2,
                               C.byref(out), None, None, None, None, None, None)
    assert rc == lib.LMM_E_ARG  # σ² must be positive


@pytest.mark.gpu
def test_vfe_posterior_refuses_everything_but_the_marginals(lmm):
    fs, D, x, z, p, U, S, y = _case("se_matern52", "oilmm", 200, 20, 14)
    s2 = 0.2
    fx = _fx(lmm, fs, x, p, s2, U, S)
    approx = lmm.VFE(_xin(lmm, z), JIT)
    post = lmm.posterior(approx, fx, y)
    owner = lmm.api._post_owner(post(lmm.MOInputIsotopicByOutputs(_xin(lmm, x[:3]), p), s2))
    lib, ctx, h = lmm._lib, owner.ctx, owner.handle
    xs = np.ascontiguousarray(x[:9].reshape(9, 1))
    ys = np.zeros(p * 9)
    buf = np.zeros(p * 9 * p * 9)
    P = lib.ptr
    out, il, h2 = C.c_double(), C.c_int(), C.c_void_p()
    kind = C.c_int()
    assert ctx.lib.lmm_post_info(h, C.byref(kind), None, None, None, None, None) == lib.LMM_OK
    calls = {
        "mean_and_cov": lambda: ctx.lib.lmm_post_mean_and_cov(h, P(xs), 9, s2, None, P(buf)),
        "condition": lambda: ctx.lib.lmm_post_condition(h, P(xs), 9, s2, P(ys), C.byref(h2), C.byref(il)),
        "logpdf": lambda: ctx.lib.lmm_post_logpdf(h, P(xs), 9, s2, P(ys), C.byref(out), C.byref(il)),
        "logpdf_grad": lambda: ctx.lib.lmm_post_logpdf_grad(h, P(xs), 9, s2, P(ys), C.byref(out), None, None, C.byref(il)),
        "logpdf_grad_full": lambda: ctx.lib.lmm_post_logpdf_grad_full(h, P(xs), 9, s2, P(ys), P(y), C.byref(out), None, None, None, None,
                                                                      None, None, None, None, None, C.byref(il)),
        "rand": lambda: ctx.lib.lmm_post_rand(h, P(xs), 9, s2, P(np.zeros(2 * 9)), P(np.zeros(p * 9)), P(ys), C.byref(il)),
        "export": lambda: ctx.lib.lmm_post_export(h, 0, None, P(np.zeros(20)), None),
        "save": lambda: ctx.lib.lmm_post_save(h, os.devnull.encode()),
    }
    Mx, Vx = lmm.mean_and_var(post(lmm.MOInputIsotopicByOutputs(_xin(lmm, x[:9]), p), s2))
    for name, fn in calls.items():
        assert fn() == lib.LMM_E_UNSUPPORTED, name
        assert "VFE" in ctx.error(), name
    M2, V2 = lmm.mean_and_var(post(lmm.MOInputIsotopicByOutputs(_xin(lmm, x[:9]), p), s2))  # still usable
    assert np.array_equal(Mx, M2) and np.array_equal(Vx, V2)
    with pytest.raises(ValueError):
        lmm.rand(post(lmm.MOInputIsotopicByOutputs(_xin(lmm, x[:9]), p), s2))


@pytest.mark.gpu
@pytest.mark.parametrize("bits", [7, 8])
def test_vfe_with_the_int8_path(lmm, bits):
    """"ozaki" = 7 planes: with M > 1024 inducing inputs the factorisation of K(z, z) and the sweep K(x, z) Lz^{-T} take their
    wide updates on the int8 tensor cores; the Gram stays FP64."""
    fs, D, x, z, p, U, S, y = _case("se_matern52", "oilmm", 1300, 1100, 15)
    z = np.linspace(0.0, float(np.max(x)), 1100)
    fs = fs + [o.GP(o.Kernel(o.MATERN32, 0.8, 0.7), 0.05)]
    U, S = o.orthogonal_from_seed(p, len(fs), seed=3)
    ctx = lmm.default_context()
    ctx.set_option("ozaki", 7)
    ctx.set_option("ozaki_bits", bits)
    try:
        _check(lmm, fs, D, x, z, p, U, S, y, jitter=1e-3)
    finally:
        ctx.set_option("ozaki", int(os.environ.get("LMM_OZAKI", "0")))  # the library default, or what the whole run was started with
        ctx.set_option("ozaki_bits", int(os.environ.get("LMM_OZAKI_BITS", "7")))


def _check_gradient_fd(lmm, fs, D, x, z, p, U, S, y, s2=0.15, h=1e-6, rtol=5e-6):
    """The library's gradient against central differences of the oracle ELBO, every block.  The step h trades the difference's
    truncation error against the oracle's rounding: at N = 300, M = 129 the ELBO (~1e3) carries ~1e-10 of rounding through
    K(z, z), which h = 1e-6 would turn into 1e-5 relative noise, so that case takes h = 2e-5."""
    fx = _fx(lmm, fs, x, p, s2, U, S)
    approx = lmm.VFE(_xin(lmm, z), JIT)
    v, g = lmm.elbo_and_gradient(approx, fx, y, with_grad_y=True)
    val = vfe_oracle(fs, x, z, JIT, s2, y, U, S)[0]
    assert abs(v - val) <= 1e-9 * abs(val), (v, val)

    def lp(fs2=fs, s=s2, y2=y, U2=U, S2=S):
        return vfe_oracle(fs2, x, z, JIT, s, y2, U2, S2)[0]

    def close(fd, an, scale, what):
        assert abs(fd - an) <= rtol * max(abs(an), 1e-2 * scale), (what, fd, an)

    terms = [np.array([[t["variance"], t["inv_lengthscale"], t["param"]] + list(t["ard"]) for t in lat]) for lat in g["terms"]]
    for i, f in enumerate(fs):
        scale = max(1e-3, float(np.max(np.abs(terms[i]))))
        for t, j, vv in _params(f, D):
            hh = h * max(1.0, abs(vv))
            close((lp(fs2=_shift(fs, i, t, j, hh)) - lp(fs2=_shift(fs, i, t, j, -hh))) / (2 * hh), terms[i][t, j], scale, (i, t, j))
        assert g["variance"][i] == terms[i][0, 0] and g["inv_lengthscale"][i] == terms[i][0, 1]

        def mshift(dm, i=i):
            return [dataclasses.replace(q, mean_const=q.mean_const + dm) if n == i else q for n, q in enumerate(fs)]

        close((lp(fs2=mshift(h)) - lp(fs2=mshift(-h))) / (2 * h), g["mean_const"][i], max(1e-3, float(np.max(np.abs(g["mean_const"])))),
              "mean")
    close((lp(s=s2 * (1 + h)) - lp(s=s2 * (1 - h))) / (2 * h * s2), g["sigma2"], abs(g["sigma2"]), "sigma2")
    scale = max(1e-3, float(np.max(np.abs(g["y"]))))
    for a in range(0, len(y), max(1, len(y) // 12)):
        yp, ym = y.copy(), y.copy()
        yp[a] += h
        ym[a] -= h
        close((lp(y2=yp) - lp(y2=ym)) / (2 * h), g["y"][a], scale, ("y", a))
    if U is None:
        return g
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
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,h", [(60, 7, 1e-6), (300, 129, 2e-5), (1, 3, 1e-6)])
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_vfe_gradient_matches_finite_differences_of_the_oracle(lmm, case, model, N, M, h):
    _check_gradient_fd(lmm, *_case(case, model, N, M, 300 + N + M + KERNEL_CASES.index(case)), h=h)


@pytest.mark.gpu
def test_vfe_gradient_is_deterministic_chunked_and_reports_failures(lmm):
    fs, D, x, z, p, U, S, y = _case("ard_D2", "oilmm", 700, 129, 16)
    fx = _fx(lmm, fs, x, p, 0.2, U, S)
    approx = lmm.VFE(_xin(lmm, z), JIT)
    va, a = lmm.elbo_and_gradient(approx, fx, y, with_grad_y=True)
    vb, b = lmm.elbo_and_gradient(approx, fx, y, with_grad_y=True)
    assert va == vb and va == lmm.elbo(approx, fx, y)
    for k in ("variance", "inv_lengthscale", "mean_const", "ard", "y", "U", "S"):
        assert np.array_equal(a[k], b[k]), k
    ctx = lmm.default_context()
    ctx.set_option("vfe_chunk", 2)  # three row chunks in both passes
    try:
        vc, c = lmm.elbo_and_gradient(approx, fx, y, with_grad_y=True)
    finally:
        ctx.set_option("vfe_chunk", 0)
    assert abs(vc - va) <= 1e-12 * abs(va)
    for k in ("variance", "inv_lengthscale", "mean_const", "ard", "y", "U", "S"):
        assert_isapprox(c[k], a[k], 1e-11, what=k)
    with pytest.raises(lmm.PosDefException) as e:
        lmm.elbo_and_gradient(lmm.VFE(_xin(lmm, np.array([[1.0, 2.0], [1.0, 2.0]])), 0.0), fx, y)
    assert e.value.info > 0 and e.value.latent == 0


@pytest.mark.gpu
def test_vfe_latent_marginals(lmm):
    """lmm_post_latent_mean_and_var on a VFE handle: one latent's approximate posterior, noise added."""
    fs, D, x, z, p, U, S, y = _case("periodic_sum", "oilmm", 400, 40, 17)
    s2 = 0.15
    fx = _fx(lmm, fs, x, p, s2, U, S)
    post = lmm.posterior(lmm.VFE(_xin(lmm, z), JIT), fx, y)
    xs = _inputs(np.random.default_rng(3), 55, D, hi=float(np.max(x)))
    T, nu = o.project_orthogonal(U, S, s2)
    Ty = T @ o.reshape_y(y, len(x))
    for i, f in enumerate(fs):
        _, mr, vr = _latent_vfe(f, x, z, JIT, nu[i], Ty[i], xs)
        Mg, Vg = lmm.mean_and_var(lmm.get_latent_gp(post).fs[i](_xin(lmm, xs), 0.3))
        assert_isapprox(Mg, mr, what="latent mean")
        assert_isapprox(Vg, vr + 0.3, what="latent var")
