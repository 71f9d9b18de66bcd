"""Per-term logpdf gradient of composite latents: KernelSum / KernelProduct of up to 4 terms, PeriodicKernel(r) and
RationalQuadraticKernel(α) (the shape parameters included), through OILMM, IndependentMOGP and general ILMM.

The analytic per-term derivatives (`dkernel_dterms`, `*_logpdf_grad_terms`) live here, on top of the oracle's kernel
matrices and its G = (αα' - C⁻¹)/2 construction.  CPU: they are checked against central differences of the oracle logpdf
and against the oracle's single-kernel gradient.  GPU: `logpdf_and_gradient(..., kernel_terms=True)` against them."""
import dataclasses
import math

import numpy as np
import pytest

from oracle import lmm_oracle as o


# ------------------------------------------------------------------------------------------------ analytic per-term oracle
def _single_term_derivs(k: o.Kernel, x):
    """(K_t, [∂K_t/∂variance, ∂K_t/∂s, ∂K_t/∂param, ∂K_t/∂ard_0 ..]) of one single kernel, direct differences."""
    X = o._as2d(x)
    D = X.shape[1]
    a = np.ones(D) if k.ard is None else np.asarray(k.ard, dtype=np.float64)
    s = k.inv_lengthscale
    U = (X[:, None, :] - X[None, :, :]) * (s * a)  # u_k = s a_k (x_k - x'_k)
    zero = np.zeros(U.shape[:2])
    if k.kind == o.PERIODIC:
        r = k.param
        sn = o._sinpi(U) / r
        q = np.sum(sn * sn, axis=-1)
        kap = np.exp(-0.5 * q)
        w = -kap * math.pi / (2.0 * r * r)
        f = U * o._sinpi(2.0 * U)
        ds = w * np.sum(f, axis=-1) / s
        dp = kap * q / r
        dard = [w * f[..., j] / a[j] for j in range(D)]
    else:
        d2 = np.sum(U * U, axis=-1)
        d = np.sqrt(d2)
        kap = o.kappa(k.kind, d2, k.param)
        with np.errstate(divide="ignore", invalid="ignore"):  # g = 2 κ'(d²): ∂κ/∂s = g d²/s, ∂κ/∂a_j = g u_j²/a_j
            if k.kind == o.SE:
                g = -kap
            elif k.kind == o.MATERN32:
                g = -3.0 * np.exp(-math.sqrt(3.0) * d)
            elif k.kind == o.MATERN52:
                g = -(5.0 / 3.0) * (1.0 + math.sqrt(5.0) * d) * np.exp(-math.sqrt(5.0) * d)
            elif k.kind == o.EXPONENTIAL:
                g = np.where(d > 0, -kap / d, 0.0)
            else:
                g = -kap / (1.0 + d2 / (2.0 * k.param))
        ds = g * d2 / s
        dard = [g * U[..., j] ** 2 / a[j] for j in range(D)]
        dp = zero
        if k.kind == o.RATQUAD:
            base = 1.0 + d2 / (2.0 * k.param)
            dp = kap * (d2 / (2.0 * k.param * base) - np.log(base))
    if k.ard is None:
        dard = [zero] * D
    v = k.variance
    return v * kap, [kap, v * ds, v * dp] + [v * t for t in dard]


def terms_of(k: o.Kernel) -> list:
    return [dataclasses.replace(k, op=o.COMPOSE_NONE, terms=())] + list(k.terms)


def dkernel_dterms(k: o.Kernel, x) -> list:
    """Per term t, the list [∂K/∂variance_t, ∂K/∂s_t, ∂K/∂param_t, ∂K/∂ard_t[0..D)] of the whole kernel matrix K:
    ∂K/∂θ_t = ∂k_t/∂θ_t for a sum, (Π_{u≠t} k_u) ∂k_t/∂θ_t for a product."""
    parts = [_single_term_derivs(t, x) for t in terms_of(k)]
    out = []
    for t, (_, ds) in enumerate(parts):
        if k.op == o.COMPOSE_PRODUCT:
            others = np.ones_like(parts[0][0])
            for u, (Ku, _) in enumerate(parts):
                if u != t:
                    others = others * Ku
            ds = [others * m for m in ds]
        out.append(ds)
    return out


def _G(K, noise, delta):
    C = K.copy()
    C[np.diag_indices_from(C)] += noise
    L = o._chol_lower(C)
    alpha = o._bwd(L, o._fwd(L, delta))
    return 0.5 * (np.outer(alpha, alpha) - o._bwd(L, o._fwd(L, np.eye(C.shape[0]))))


def _contract(G, f: o.GP, x) -> np.ndarray:
    """(nterms, 3 + D): <G, ∂K/∂θ> per term and parameter."""
    return np.array([[float(np.sum(G * dK)) for dK in ds] for ds in dkernel_dterms(f.kernel, x)])


def gp_logpdf_grad_terms(f: o.GP, x, noise: float, y) -> np.ndarray:
    G = _G(o.kernelmatrix(f.kernel, x), noise, np.asarray(y, dtype=np.float64) - f.mean_const)
    return _contract(G, f, x)


def oilmm_logpdf_grad_terms(model: o.OILMMModel, x, sigma2: float, y) -> list:
    N = o._as2d(x).shape[0]
    T, ST = o.project_orthogonal(model.U, model.S, sigma2)
    Ty = T @ o.reshape_y(y, N)
    return [gp_logpdf_grad_terms(f, x, ST[i], Ty[i]) for i, f in enumerate(model.fs)]


def imogp_logpdf_grad_terms(fs, x, sigma2: float, y) -> list:
    Y = o.reshape_y(y, o._as2d(x).shape[0])
    return [gp_logpdf_grad_terms(f, x, sigma2, Y[i]) for i, f in enumerate(fs)]


def ilmm_logpdf_grad_terms(fs, H, x, sigma2: float, y) -> list:
    N = o._as2d(x).shape[0]
    T, ST = o.project_general(np.asarray(H, dtype=np.float64), sigma2)
    delta = (T @ o.reshape_y(y, N)).reshape(-1) - np.concatenate([np.full(N, f.mean_const) for f in fs])
    G = _G(o._latent_prior_cov(fs, x) + np.kron(ST, np.eye(N)), 0.0, delta)
    return [_contract(G[a * N:(a + 1) * N, a * N:(a + 1) * N], f, x) for a, f in enumerate(fs)]


# ------------------------------------------------------------------------------------------------ fixtures
def composite_latents(D: int = 1):
    """Trend + seasonal sum, locally periodic product, plain kernel, 3-term sum; with D = 2 the periodic term of the sum and
    the Matern52 term of the product carry an ARDTransform."""
    ard_p, ard_m = (None, None) if D == 1 else ((1.3, 0.6), (0.7, 1.6))
    k_sum = o.Kernel(o.SE, 1.2, 0.4, op=o.COMPOSE_SUM, terms=(o.Kernel(o.PERIODIC, 0.5, 0.7, ard=ard_p, param=0.8),))
    k_prod = o.Kernel(o.MATERN52, 0.9, 0.3, ard=ard_m, op=o.COMPOSE_PRODUCT, terms=(o.Kernel(o.PERIODIC, 1.0, 1.0, param=1.3),))
    k_plain = o.Kernel(o.MATERN32, 0.7, 1.1)
    k_three = o.Kernel(o.SE, 0.6, 1.5, op=o.COMPOSE_SUM, terms=(o.Kernel(o.EXPONENTIAL, 0.3, 0.8), o.Kernel(o.RATQUAD, 0.4, 0.6, param=1.7)))
    return [o.GP(k_sum, 0.3), o.GP(k_prod, 0.0), o.GP(k_plain, -0.2), o.GP(k_three, 0.1)]


def shape_latents():
    """Single RationalQuadratic (α) and single Periodic (r, s) latents."""
    return [o.GP(o.Kernel(o.RATQUAD, 0.8, 0.9, param=1.4), 0.1), o.GP(o.Kernel(o.PERIODIC, 1.1, 0.6, param=0.9), -0.3)]


def to_lmm(lmm, g):
    base = {o.SE: lmm.SEKernel, o.MATERN32: lmm.Matern32Kernel, o.MATERN52: lmm.Matern52Kernel, o.EXPONENTIAL: lmm.ExponentialKernel}

    def single(k):
        b = lmm.RationalQuadraticKernel(k.param) if k.kind == o.RATQUAD else lmm.PeriodicKernel(k.param) if k.kind == o.PERIODIC else base[k.kind]()
        b = (k.variance * b).compose(lmm.ScaleTransform(k.inv_lengthscale))
        return b.compose(lmm.ARDTransform(k.ard)) if k.ard is not None else b

    ts = terms_of(g.kernel)
    k = single(ts[0])
    for t in ts[1:]:
        k = k * single(t) if g.kernel.op == o.COMPOSE_PRODUCT else k + single(t)
    return lmm.GP(g.mean_const, k)


def _inputs(rng, N, D, hi=6.0):
    return np.sort(rng.uniform(0, hi, N)) if D == 1 else rng.uniform(0, hi, (N, D))


# parameter j of term t of latent i, shifted by h
def _shift(fs, i, t, j, h):
    g = fs[i]
    ts = terms_of(g.kernel)
    q = ts[t]
    if j == 0:
        q = dataclasses.replace(q, variance=q.variance + h)
    elif j == 1:
        q = dataclasses.replace(q, inv_lengthscale=q.inv_lengthscale + h)
    elif j == 2:
        q = dataclasses.replace(q, param=q.param + h)
    else:
        a = list(q.ard)
        a[j - 3] += h
        q = dataclasses.replace(q, ard=tuple(a))
    ts[t] = q
    k = dataclasses.replace(ts[0], op=g.kernel.op if len(ts) > 1 else o.COMPOSE_NONE, terms=tuple(ts[1:]))
    return [dataclasses.replace(g, kernel=k) if n == i else f for n, f in enumerate(fs)]


def _params(g, D):
    """(t, j, value) of every free hyper-parameter of a latent."""
    out = []
    for t, q in enumerate(terms_of(g.kernel)):
        out += [(t, 0, q.variance), (t, 1, q.inv_lengthscale)]
        if q.kind in (o.RATQUAD, o.PERIODIC):
            out.append((t, 2, q.param))
        if q.ard is not None:
            out += [(t, 3 + j, q.ard[j]) for j in range(D)]
    return out


def _check_fd(fs, grads, logpdf_of, D, h=1e-6, rtol=5e-6):
    for i, g in enumerate(fs):
        scale = max(1e-3, float(np.max(np.abs(grads[i]))))
        for t, j, v in _params(g, D):
            hh = h * max(1.0, abs(v))
            fd = (logpdf_of(_shift(fs, i, t, j, hh)) - logpdf_of(_shift(fs, i, t, j, -hh))) / (2 * hh)
            an = grads[i][t, j]
            assert abs(fd - an) <= rtol * max(abs(an), 1e-2 * scale), (i, t, j, fd, an)


MODELS = ["oilmm", "imogp", "ilmm"]


def _model_case(model, fs, x, rng):
    """(analytic per-term gradients, logpdf as a function of the latents) of one model."""
    N, m = o._as2d(x).shape[0], len(fs)
    if model == "oilmm":
        p = m + 2
        U, S = o.orthogonal_from_seed(p, m, seed=5)
        y = rng.standard_normal(p * N)
        return (oilmm_logpdf_grad_terms(o.OILMMModel(fs, U, S), x, 0.1, y),
                lambda f2: o.oilmm_logpdf(o.OILMMModel(f2, U, S), x, 0.1, y))
    if model == "imogp":
        y = rng.standard_normal(m * N)
        return imogp_logpdf_grad_terms(fs, x, 0.15, y), lambda f2: o.imogp_logpdf(f2, x, 0.15, y)
    p = m + 1
    H = rng.uniform(0, 1, (p, m))
    y = rng.standard_normal(p * N)
    return ilmm_logpdf_grad_terms(fs, H, x, 0.2, y), lambda f2: o.ilmm_logpdf(f2, H, x, 0.2, y)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("case", ["sum_product_three", "shape_params", "ard_product_D2"])
def test_oracle_term_gradients_match_finite_differences(model, case):
    rng = np.random.default_rng(7)
    D = 2 if case == "ard_product_D2" else 1
    if case == "sum_product_three":
        fs = [g for i, g in enumerate(composite_latents()) if i != 2]
    elif case == "shape_params":
        fs = shape_latents()
    else:
        fs = composite_latents(2)[:2]
    x = _inputs(rng, 24, D)
    grads, logpdf_of = _model_case(model, fs, x, rng)
    _check_fd(fs, grads, logpdf_of, D)


@pytest.mark.parametrize("D", [1, 2])
def test_oracle_term_gradients_reduce_to_the_single_kernel_gradient(D):
    rng = np.random.default_rng(11)
    x = _inputs(rng, 30, D)
    y = rng.standard_normal(30)
    kinds = [o.SE, o.MATERN32, o.MATERN52, o.EXPONENTIAL, o.RATQUAD]
    for kind in kinds:
        f = o.GP(o.Kernel(kind, 0.8, 0.7, ard=None if D == 1 else (1.2, 0.5), param=1.9), 0.2)
        g = gp_logpdf_grad_terms(f, x, 0.1, y)
        ref = o.gp_logpdf_grad(f, x, 0.1, y)
        np.testing.assert_allclose(g[0, 0], ref[1], rtol=1e-10)
        np.testing.assert_allclose(g[0, 1], ref[2], rtol=1e-10)
        if D == 2:
            np.testing.assert_allclose(g[0, 3:], o.gp_logpdf_grad_ard(f, x, 0.1, y), rtol=1e-10)


def test_shared_scale_transform_chain_rule():
    """(k1 + k2) ∘ ScaleTransform(s): every term's s_t = c_t s, so d logpdf / ds = Σ_t (s_t / s) g_t."""
    rng = np.random.default_rng(3)
    x = _inputs(rng, 26, 1)
    y = rng.standard_normal(26)
    c = (0.4, 0.7)

    def gp(s):
        return o.GP(o.Kernel(o.SE, 1.2, c[0] * s, op=o.COMPOSE_SUM, terms=(o.Kernel(o.PERIODIC, 0.5, c[1] * s, param=0.8),)), 0.3)

    s, h = 1.3, 1e-6
    g = gp_logpdf_grad_terms(gp(s), x, 0.1, y)
    chain = sum((c[t] * s / s) * g[t, 1] for t in range(2))
    fd = (o.gp_logpdf(gp(s + h), x, 0.1, y) - o.gp_logpdf(gp(s - h), x, 0.1, y)) / (2 * h)
    assert abs(chain - fd) <= 5e-6 * abs(chain)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def lmm():
    import lmm_b200

    lmm_b200.default_context()
    return lmm_b200


def _xin(lmm, x):
    return x if x.ndim == 1 else lmm.ColVecs(x.T)


def _assert_terms(got, ref, fs, D):
    assert len(got) == len(fs)
    for i, g in enumerate(fs):
        ts = terms_of(g.kernel)
        assert len(got[i]) == len(ts)
        for t, q in enumerate(ts):
            row = np.array([got[i][t]["variance"], got[i][t]["inv_lengthscale"], got[i][t]["param"]] + list(got[i][t]["ard"]))
            assert row.shape == (3 + D,)
            np.testing.assert_allclose(row, ref[i][t], rtol=1e-7, atol=1e-8, err_msg=f"latent {i} term {t}")
            if q.kind not in (o.RATQUAD, o.PERIODIC):
                assert got[i][t]["param"] == 0.0
            if q.ard is None:
                assert np.all(got[i][t]["ard"] == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [60, 700, 1300])
@pytest.mark.parametrize("D", [1, 2])
def test_oilmm_composite_gradient(lmm, N, D):
    rng = np.random.default_rng(N + D)
    fs = composite_latents(D) + shape_latents()
    m, p, s2 = len(fs), 8, 0.1
    x = _inputs(rng, N, D, hi=12.0)
    U, S = o.orthogonal_from_seed(p, m, seed=3)
    y = rng.standard_normal(p * N)
    om = o.OILMMModel(fs, U, S)
    f = lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), lmm.Orthogonal(U, S))
    lp, g = lmm.logpdf_and_gradient(f(lmm.MOInputIsotopicByOutputs(_xin(lmm, x), p), s2), y, with_grad_y=True, kernel_terms=True)
    lpr = o.oilmm_logpdf(om, x, s2, y)
    _, gr = o.oilmm_logpdf_grad(om, x, s2, y)  # σ², y, U, S and the mean need only the kernel matrices
    assert abs(lp - lpr) <= 1e-9 * abs(lpr)
    ref = oilmm_logpdf_grad_terms(om, x, s2, y)
    _assert_terms(g["terms"], ref, fs, D)
    np.testing.assert_allclose(g["variance"], [r[0, 0] for r in ref], rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(g["inv_lengthscale"], [r[0, 1] for r in ref], rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(g["mean_const"], gr["mean_const"], rtol=1e-7, atol=1e-8)
    assert abs(g["sigma2"] - gr["sigma2"]) <= 1e-7 * abs(gr["sigma2"])
    np.testing.assert_allclose(g["y"], gr["y"], rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose(g["S"], gr["S"], rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(g["U"], gr["U"], rtol=1e-7, atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("N,D", [(90, 1), (300, 2)])
def test_imogp_and_ilmm_composite_gradient(lmm, N, D):
    rng = np.random.default_rng(40 + N)
    fs = composite_latents(D)[:2] + shape_latents()[1:] + [composite_latents(D)[3]]
    m = len(fs)
    x = _inputs(rng, N, D, hi=9.0)
    O = lmm.MOInputIsotopicByOutputs
    # IndependentMOGP
    yi = rng.standard_normal(m * N)
    fi = lmm.independent_mogp([to_lmm(lmm, g) for g in fs])
    lpi, gi = lmm.logpdf_and_gradient(fi(O(_xin(lmm, x), m), 0.15), yi, with_grad_y=True, kernel_terms=True)
    assert abs(lpi - o.imogp_logpdf(fs, x, 0.15, yi)) <= 1e-9 * abs(lpi)
    _assert_terms(gi["terms"], imogp_logpdf_grad_terms(fs, x, 0.15, yi), fs, D)
    parts = [o.gp_logpdf_grad(fs[i], x, 0.15, yi.reshape(m, N)[i]) for i in range(m)]
    assert abs(gi["sigma2"] - sum(q[4] for q in parts)) <= 1e-7 * abs(gi["sigma2"])
    np.testing.assert_allclose(gi["mean_const"], [q[3] for q in parts], rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(gi["y"], np.concatenate([q[5] for q in parts]), rtol=1e-7, atol=1e-9)
    # general ILMM
    p = m + 2
    H = rng.uniform(0, 1, (p, m))
    y = rng.standard_normal(p * N)
    f = lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), H)
    lp, g = lmm.logpdf_and_gradient(f(O(_xin(lmm, x), p), 0.2), y, with_grad_y=True, kernel_terms=True)
    lpr, gr = o.ilmm_logpdf_grad(fs, H, x, 0.2, y)
    assert abs(lp - lpr) <= 1e-9 * abs(lpr)
    _assert_terms(g["terms"], ilmm_logpdf_grad_terms(fs, H, x, 0.2, y), fs, D)
    np.testing.assert_allclose(g["mean_const"], gr["mean_const"], rtol=1e-7, atol=1e-8)
    assert abs(g["sigma2"] - gr["sigma2"]) <= 1e-7 * abs(gr["sigma2"])
    np.testing.assert_allclose(g["y"], gr["y"], rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose(g["H"], gr["H"], rtol=1e-7, atol=1e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 2])
def test_single_kernel_latents_old_and_terms_entry_points_agree(lmm, D):
    """Single-kernel latents: the _terms entry points return exactly what the single-kernel ones do; the RQ α is the
    oracle's; two calls give bit-identical per-term gradients."""
    rng = np.random.default_rng(5 + D)
    ard = None if D == 1 else (1.2, 0.6)
    fs = [o.GP(o.Kernel(o.SE, 1.1, 0.8, ard=ard), 0.2), o.GP(o.Kernel(o.MATERN52, 0.7, 1.3), -0.1),
          o.GP(o.Kernel(o.RATQUAD, 0.9, 0.5, ard=ard, param=1.6), 0.0)]
    m, p, N = len(fs), 5, 500
    x = _inputs(rng, N, D, hi=10.0)
    U, S = o.orthogonal_from_seed(p, m, seed=9)
    y = rng.standard_normal(p * N)
    O = lmm.MOInputIsotopicByOutputs
    f = lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), lmm.Orthogonal(U, S))
    fx = f(O(_xin(lmm, x), p), 0.1)
    lp0, g0 = lmm.logpdf_and_gradient(fx, y, with_grad_y=True)
    lp1, g1 = lmm.logpdf_and_gradient(fx, y, with_grad_y=True, kernel_terms=True)
    _, g2 = lmm.logpdf_and_gradient(fx, y, with_grad_y=True, kernel_terms=True)
    assert lp0 == lp1
    for k in ("variance", "inv_lengthscale", "mean_const", "ard", "y", "U", "S"):
        assert np.array_equal(g0[k], g1[k]), k
    assert g0["sigma2"] == g1["sigma2"]
    ref = oilmm_logpdf_grad_terms(o.OILMMModel(fs, U, S), x, 0.1, y)
    _assert_terms(g1["terms"], ref, fs, D)
    for a, b in zip(g1["terms"], g2["terms"]):  # deterministic: fixed-order reductions, no atomics
        for ta, tb in zip(a, b):
            assert ta["variance"] == tb["variance"] and ta["inv_lengthscale"] == tb["inv_lengthscale"] and ta["param"] == tb["param"]
            assert np.array_equal(ta["ard"], tb["ard"])
    # the same through the general ILMM
    H = rng.uniform(0, 1, (p, m))
    fh = lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), H)(O(_xin(lmm, x[:200]), p), 0.2)
    yh = rng.standard_normal(p * 200)
    _, h0 = lmm.logpdf_and_gradient(fh, yh)
    _, h1 = lmm.logpdf_and_gradient(fh, yh, kernel_terms=True)
    for k in ("variance", "inv_lengthscale", "mean_const", "ard", "H"):
        assert np.array_equal(h0[k], h1[k]), k


@pytest.mark.gpu
def test_composite_gradient_is_deterministic_and_posterior_rejects_kernel_terms(lmm):
    rng = np.random.default_rng(2)
    fs = composite_latents(2)
    m, p, N = len(fs), 6, 700
    x = _inputs(rng, N, 2, hi=10.0)
    U, S = o.orthogonal_from_seed(p, m, seed=4)
    y = rng.standard_normal(p * N)
    O = lmm.MOInputIsotopicByOutputs
    f = lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), lmm.Orthogonal(U, S))
    fx = f(O(_xin(lmm, x), p), 0.1)
    _, a = lmm.logpdf_and_gradient(fx, y, kernel_terms=True)
    _, b = lmm.logpdf_and_gradient(fx, y, kernel_terms=True)
    for la, lb in zip(a["terms"], b["terms"]):
        for ta, tb in zip(la, lb):
            assert (ta["variance"], ta["inv_lengthscale"], ta["param"]) == (tb["variance"], tb["inv_lengthscale"], tb["param"])
            assert np.array_equal(ta["ard"], tb["ard"])
    with pytest.raises(ValueError, match="composite"):  # the single-kernel path still refuses composite latents
        lmm.logpdf_and_gradient(fx, y)
    post = lmm.posterior(fx, y)
    xs = rng.uniform(0, 10, (20, 2))
    with pytest.raises(ValueError, match="kernel_terms"):
        lmm.logpdf_and_gradient(post(O(lmm.ColVecs(xs.T), p), 0.1), rng.standard_normal(p * 20), kernel_terms=True)
