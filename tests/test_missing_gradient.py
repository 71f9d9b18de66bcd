"""Gradient of the missing-data (heterotopic) logpdf: the dense model y ~ N((H ⊗ I) m, Σ_l (h_l h_l') ⊗ K_l + σ² I) restricted
to the observed (non-NaN) entries of y, and the per-input-mask OILMM.

The analytic oracle lives here, on top of the unchanged oracle's `dense_mogp_cov` restricted to the observed entries and the
per-term derivatives of test_composite_gradient.py.  CPU: it is checked against central differences of
`o.missing_data_logpdf` for every hyper-parameter, H, the means, σ² and y.  GPU: `logpdf_missing_and_gradient` against it."""
import dataclasses

import numpy as np
import pytest

from _tol import assert_isapprox, relnorm
from oracle import lmm_oracle as o
from test_composite_gradient import _inputs, _params, _shift, _xin, dkernel_dterms, terms_of, to_lmm


# ------------------------------------------------------------------------------------------------ analytic oracle
def missing_data_logpdf_grad(fs, H, x, sigma2, y):
    """(logpdf, grads) of the dense model on the observed entries of y.  grads: "terms" (per latent, (nterms, 3 + D)),
    "H" (p, m), "mean_const" (m,), "sigma2", "y" (p*N,; 0 at NaN entries)."""
    H = np.asarray(H, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    N = o._as2d(x).shape[0]
    p, m = H.shape
    obs = np.flatnonzero(~np.isnan(y))
    jo, io = obs // N, obs % N
    Ks = [o.kernelmatrix(f.kernel, x)[np.ix_(io, io)] for f in fs]
    C = sum(np.outer(H[jo, l], H[jo, l]) * Ks[l] for l in range(m)) + sigma2 * np.eye(len(obs))
    L = o._chol_lower(C)
    delta = y[obs] - (H @ np.array([f.mean_const for f in fs]))[jo]
    z = o._fwd(L, delta)
    alpha = o._bwd(L, z)
    Cinv = o._bwd(L, o._fwd(L, np.eye(len(obs))))
    G = 0.5 * (np.outer(alpha, alpha) - Cinv)
    lp = -0.5 * (len(obs) * o.LOG2PI + 2.0 * float(np.sum(np.log(np.diag(L)))) + float(z @ z))
    terms, gH = [], np.zeros((p, m))
    for l, f in enumerate(fs):
        W = G * np.outer(H[jo, l], H[jo, l])
        terms.append(np.array([[float(np.sum(W * dK[np.ix_(io, io)])) for dK in ds] for ds in dkernel_dterms(f.kernel, x)]))
        v = (G * Ks[l]) @ H[jo, l]  # v_l(a) = Σ_b G_ab H[j_b,l] k_l(a,b)
        gH[:, l] = 2.0 * np.bincount(jo, weights=v, minlength=p) + f.mean_const * np.bincount(jo, weights=alpha, minlength=p)
    gy = np.zeros(p * N)
    gy[obs] = -alpha
    return lp, {"terms": terms, "H": gH, "mean_const": np.array([alpha @ H[jo, l] for l in range(m)]), "sigma2": float(np.trace(G)),
                "y": gy}


# ------------------------------------------------------------------------------------------------ fixtures
def kernel_case(case):
    """(latents, D) of one kernel case."""
    K = o.Kernel
    if case == "se_matern52":
        return [o.GP(K(o.SE, 1.1, 0.8), 0.3), o.GP(K(o.MATERN52, 0.7, 1.3), -0.2)], 1
    if case == "exponential_ratquad":
        return [o.GP(K(o.EXPONENTIAL, 0.9, 0.6), 0.1), o.GP(K(o.RATQUAD, 0.8, 0.9, param=1.4), 0.4)], 1
    if case == "periodic_sum":
        return [o.GP(K(o.PERIODIC, 1.1, 0.6, param=0.9), -0.3),
                o.GP(K(o.SE, 1.2, 0.4, op=o.COMPOSE_SUM, terms=(K(o.PERIODIC, 0.5, 0.7, param=0.8),)), 0.2)], 1
    if case == "product":
        return [o.GP(K(o.MATERN52, 0.9, 0.3, op=o.COMPOSE_PRODUCT, terms=(K(o.PERIODIC, 1.0, 1.0, param=1.3),)), 0.1),
                o.GP(K(o.SE, 0.6, 1.5), -0.1)], 1
    assert case == "ard_D2"
    return [o.GP(K(o.SE, 1.0, 0.7, ard=(1.3, 0.6)), 0.2),
            o.GP(K(o.MATERN52, 0.9, 0.5, ard=(0.7, 1.6), op=o.COMPOSE_PRODUCT, terms=(K(o.PERIODIC, 1.0, 0.8, param=1.2),)), -0.3)], 2


KERNEL_CASES = ["se_matern52", "exponential_ratquad", "periodic_sum", "product", "ard_D2"]
MASKS = ["none", "random30", "random70", "output_missing", "input_missing"]


def make_y(rng, p, N, mask):
    """A by-outputs y (p*N) with NaN at the missing entries of the named mask."""
    y = rng.standard_normal((p, N))
    if mask in ("random30", "random70"):
        miss = rng.uniform(size=(p, N)) < (0.3 if mask == "random30" else 0.7)
        miss[0, 0] = False  # something stays observed
        y[miss] = np.nan
    elif mask == "output_missing":
        y[1, :] = np.nan
        y[0, rng.uniform(size=N) < 0.2] = np.nan
    elif mask == "input_missing":
        y[:, N // 3] = np.nan
    return y.reshape(-1)


def _shift_H(H, j, l, h):
    H2 = H.copy()
    H2[j, l] += h
    return H2


def _check_fd(fs, H, x, s2, y, D, h=1e-6, rtol=5e-6):
    """Every block of the analytic gradient against central differences of o.missing_data_logpdf."""
    _, g = missing_data_logpdf_grad(fs, H, x, s2, y)

    def lp(fs2=fs, H2=H, s=s2, y2=y):
        return o.missing_data_logpdf(fs2, H2, x, s, y2)

    def close(fd, an, scale):
        assert abs(fd - an) <= rtol * max(abs(an), 1e-2 * scale), (fd, an)

    for i, f in enumerate(fs):
        scale = max(1e-3, float(np.max(np.abs(g["terms"][i]))))
        for t, j, v in _params(f, D):
            hh = h * max(1.0, abs(v))
            close((lp(fs2=_shift(fs, i, t, j, hh)) - lp(fs2=_shift(fs, i, t, j, -hh))) / (2 * hh), g["terms"][i][t, j], scale)
        def mshift(d, i=i):
            return [dataclasses.replace(q, mean_const=q.mean_const + d) if n == i else q for n, q in enumerate(fs)]

        close((lp(fs2=mshift(h)) - lp(fs2=mshift(-h))) / (2 * h), g["mean_const"][i], max(1e-3, float(np.max(np.abs(g["mean_const"])))))
    scale = max(1e-3, float(np.max(np.abs(g["H"]))))
    for j in range(H.shape[0]):
        for l in range(H.shape[1]):
            close((lp(H2=_shift_H(H, j, l, h)) - lp(H2=_shift_H(H, j, l, -h))) / (2 * h), g["H"][j, l], scale)
    close((lp(s=s2 + h * s2) - lp(s=s2 - h * s2)) / (2 * h * s2), g["sigma2"], abs(g["sigma2"]))
    obs = np.flatnonzero(~np.isnan(y))
    scale = max(1e-3, float(np.max(np.abs(g["y"]))))
    for a in obs[:: max(1, len(obs) // 12)]:
        yp, ym = y.copy(), y.copy()
        yp[a] += h
        ym[a] -= h
        close((lp(y2=yp) - lp(y2=ym)) / (2 * h), g["y"][a], scale)
    assert np.all(g["y"][np.isnan(y)] == 0.0)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oracle_missing_gradient_matches_finite_differences(case, mask):
    rng = np.random.default_rng(KERNEL_CASES.index(case) * 10 + MASKS.index(mask))
    fs, D = kernel_case(case)
    p, N = 3, 12
    x = _inputs(rng, N, D)
    H = rng.uniform(0.2, 1.2, (p, len(fs)))
    y = make_y(rng, p, N, mask)
    _check_fd(fs, H, x, 0.2, y, D)


def test_oracle_missing_gradient_without_missing_entries_is_the_dense_ilmm_gradient():
    """Nothing missing: the dense model is the general ILMM, so d/dH and the hyper-parameter gradients are the oracle's."""
    rng = np.random.default_rng(4)
    fs, _ = kernel_case("se_matern52")
    p, N = 3, 15
    x = _inputs(rng, N, 1)
    H = rng.uniform(0.2, 1.2, (p, 2))
    y = rng.standard_normal(p * N)
    lp, g = missing_data_logpdf_grad(fs, H, x, 0.2, y)
    lpr, gr = o.ilmm_logpdf_grad(fs, H, x, 0.2, y)
    assert abs(lp - lpr) <= 1e-10 * abs(lpr)
    np.testing.assert_allclose(g["H"], gr["H"], rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose([t[0, 0] for t in g["terms"]], gr["variance"], rtol=1e-6)
    np.testing.assert_allclose([t[0, 1] for t in g["terms"]], gr["inv_lengthscale"], rtol=1e-6)
    np.testing.assert_allclose(g["mean_const"], gr["mean_const"], rtol=1e-6, atol=1e-10)
    assert abs(g["sigma2"] - gr["sigma2"]) <= 1e-6 * abs(gr["sigma2"])


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def lmm():
    import lmm_b200

    lmm_b200.default_context()
    return lmm_b200


def _model(lmm, fs, H, x, p, s2):
    return lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), H)(lmm.MOInputIsotopicByOutputs(_xin(lmm, x), p), s2)


def _terms_array(got):
    return [np.array([[t["variance"], t["inv_lengthscale"], t["param"]] + list(t["ard"]) for t in lat]) for lat in got]


def _assert_matches_oracle(g, ref, fs):
    got = _terms_array(g["terms"])
    for i in range(len(fs)):
        assert got[i].shape == ref["terms"][i].shape
    assert_isapprox(np.concatenate([a.ravel() for a in got]), np.concatenate([r.ravel() for r in ref["terms"]]), what="terms")
    assert_isapprox(g["variance"], [r[0, 0] for r in ref["terms"]], what="variance")
    assert_isapprox(g["inv_lengthscale"], [r[0, 1] for r in ref["terms"]], what="inv_lengthscale")
    assert_isapprox(g["H"], ref["H"], what="H")
    assert_isapprox(g["mean_const"], ref["mean_const"], what="mean_const")
    assert_isapprox([g["sigma2"]], [ref["sigma2"]], what="sigma2")
    assert_isapprox(g["y"], ref["y"], what="y")


@pytest.mark.gpu
@pytest.mark.parametrize("N", [50, 300, 700])
@pytest.mark.parametrize("p,m", [(3, 2), (5, 3)])
def test_missing_gradient_matches_oracle(lmm, N, p, m):
    """N < 128 puts several outputs into one tile; the nobs values cross tile boundaries at random offsets."""
    rng = np.random.default_rng(N + 10 * p)
    K = o.Kernel
    fs = [o.GP(K(o.SE, 1.2, 0.4, op=o.COMPOSE_SUM, terms=(K(o.PERIODIC, 0.5, 0.7, param=0.8),)), 0.3), o.GP(K(o.MATERN52, 0.8, 0.9), -0.4),
          o.GP(K(o.RATQUAD, 0.7, 0.6, param=1.5), 0.2)][:m]
    x = _inputs(rng, N, 1, hi=12.0)
    H = rng.uniform(0.2, 1.2, (p, m))
    y = make_y(rng, p, N, "random30")
    lp, g = lmm.logpdf_missing_and_gradient(_model(lmm, fs, H, x, p, 0.15), y, with_grad_y=True, kernel_terms=True)
    lpr, ref = missing_data_logpdf_grad(fs, H, x, 0.15, y)
    assert abs(lp - lpr) <= 1e-9 * abs(lpr)
    _assert_matches_oracle(g, ref, fs)


@pytest.mark.gpu
@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_missing_gradient_kernel_and_mask_grid(lmm, case, mask):
    rng = np.random.default_rng(100 + KERNEL_CASES.index(case) * 10 + MASKS.index(mask))
    fs, D = kernel_case(case)
    p, N = 4, 90
    x = _inputs(rng, N, D, hi=8.0)
    H = rng.uniform(0.2, 1.2, (p, len(fs)))
    y = make_y(rng, p, N, mask)
    fx = _model(lmm, fs, H, x, p, 0.2)
    lp, g = lmm.logpdf_missing_and_gradient(fx, y, with_grad_y=True, kernel_terms=True)
    lpr, ref = missing_data_logpdf_grad(fs, H, x, 0.2, y)
    assert abs(lp - lpr) <= 1e-9 * abs(lpr)
    _assert_matches_oracle(g, ref, fs)
    # value: the logpdf of the value path; structure: exact zeros where nothing is observed
    assert abs(lp - lmm.logpdf_missing(fx, y)) <= 1e-14 * abs(lp)
    assert np.all(g["y"][np.isnan(y)] == 0.0)
    if mask == "output_missing":
        assert np.all(g["H"][1, :] == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("mask", ["none", "input_missing"])
def test_dense_path_agrees_with_oilmm_path(lmm, mask):
    """Orthogonal U: the dense model with H = U√S passed as an ndarray and the OILMM path are the same function of the
    hyper-parameters, σ², y and S; their U gradients agree in the tangent space of orthogonal U."""
    rng = np.random.default_rng(21 + MASKS.index(mask))
    fs, _ = kernel_case("periodic_sum")
    m, p, N, s2 = len(fs), 4, 150, 0.1
    x = _inputs(rng, N, 1, hi=10.0)
    U, S = o.orthogonal_from_seed(p, m, seed=6)
    y = make_y(rng, p, N, mask)
    O = lmm.MOInputIsotopicByOutputs
    lat = lmm.independent_mogp([to_lmm(lmm, g) for g in fs])
    lo, go = lmm.logpdf_missing_and_gradient(lmm.ILMM(lat, lmm.Orthogonal(U, S))(O(_xin(lmm, x), p), s2), y, with_grad_y=True, kernel_terms=True)
    ld, gd = lmm.logpdf_missing_and_gradient(lmm.ILMM(lat, U * np.sqrt(S)[None, :])(O(_xin(lmm, x), p), s2), y, with_grad_y=True,
                                             kernel_terms=True)
    assert "H" not in go and "H" in gd
    assert abs(lo - ld) <= 1e-9 * abs(lo)
    for k in ("variance", "inv_lengthscale", "mean_const", "y"):
        assert_isapprox(gd[k], go[k], what=k)
    assert_isapprox([gd["sigma2"]], [go["sigma2"]], what="sigma2")
    assert_isapprox(np.concatenate([a.ravel() for a in _terms_array(gd["terms"])]),
                    np.concatenate([a.ravel() for a in _terms_array(go["terms"])]), what="terms")
    rs = np.sqrt(S)
    gS = np.sum(gd["H"] * U, axis=0) / (2.0 * rs)
    assert_isapprox(gS, go["S"], what="S")

    def tangent(Gm):
        A = U.T @ Gm
        return Gm - U @ (0.5 * (A + A.T))

    assert_isapprox(tangent(gd["H"] * rs[None, :]), tangent(go["U"]), what="U (tangent space)")
    # the Orthogonal H through the dense path (a mask that is not per-input) returns the chain rule of H = U√S
    y2 = y.copy()
    y2[3] = np.nan
    _, gc = lmm.logpdf_missing_and_gradient(lmm.ILMM(lat, lmm.Orthogonal(U, S))(O(_xin(lmm, x), p), s2), y2, kernel_terms=True)
    _, gh = lmm.logpdf_missing_and_gradient(lmm.ILMM(lat, U * rs[None, :])(O(_xin(lmm, x), p), s2), y2, kernel_terms=True)
    assert np.array_equal(gc["H"], gh["H"])
    assert np.array_equal(gc["U"], gh["H"] * rs[None, :])
    assert relnorm(gc["S"], np.sum(gh["H"] * U, axis=0) / (2.0 * rs)) <= 1e-15


@pytest.mark.gpu
def test_missing_gradient_is_deterministic(lmm):
    rng = np.random.default_rng(8)
    fs, D = kernel_case("ard_D2")
    p, N = 5, 400
    x = _inputs(rng, N, D, hi=10.0)
    H = rng.uniform(0.2, 1.2, (p, len(fs)))
    y = make_y(rng, p, N, "random30")
    fx = _model(lmm, fs, H, x, p, 0.2)
    la, a = lmm.logpdf_missing_and_gradient(fx, y, with_grad_y=True, kernel_terms=True)
    lb, b = lmm.logpdf_missing_and_gradient(fx, y, with_grad_y=True, kernel_terms=True)
    assert la == lb
    for k in ("variance", "inv_lengthscale", "mean_const", "ard", "H", "y"):
        assert np.array_equal(a[k], b[k]), k
    assert a["sigma2"] == b["sigma2"]
    for ta, tb in zip(_terms_array(a["terms"]), _terms_array(b["terms"])):
        assert np.array_equal(ta, tb)


@pytest.mark.gpu
def test_missing_gradient_refusals(lmm):
    import ctypes as C

    rng = np.random.default_rng(9)
    fs, _ = kernel_case("periodic_sum")
    p, N = 3, 40
    x = _inputs(rng, N, 1)
    H = rng.uniform(0.2, 1.2, (p, 2))
    y = make_y(rng, p, N, "random30")
    fx = _model(lmm, fs, H, x, p, 0.2)
    with pytest.raises(ValueError, match="composite"):  # composite latents need kernel_terms, as in logpdf_and_gradient
        lmm.logpdf_missing_and_gradient(fx, y)
    with pytest.raises(ValueError, match="missing"):
        lmm.logpdf_missing_and_gradient(fx, np.full(p * N, np.nan), kernel_terms=True)
    yf = rng.standard_normal(p * N)
    post = lmm.posterior(fx, yf)
    with pytest.raises(TypeError):
        lmm.logpdf_missing_and_gradient(post(lmm.MOInputIsotopicByOutputs(x[:10], p), 0.2), yf[:p * 10], kernel_terms=True)
    # the OILMM entry refuses a mask that is not per-input
    U, S = o.orthogonal_from_seed(p, 2, seed=2)
    ctx = lmm.default_context()
    lib = lmm._lib
    descs = lmm.api._descs([to_lmm(lmm, g) for g in fs])
    pts = np.ascontiguousarray(x.reshape(N, 1))
    Uf, Sv = np.asfortranarray(U), np.ascontiguousarray(S)
    out, nobs, il = C.c_double(), C.c_int(0), C.c_int(-1)
    gt = np.zeros(2 * lib.LMM_MAX_TERMS * lib.LMM_GRAD_TERM_STRIDE)
    rc = ctx.lib.lmm_oilmm_masked_logpdf_grad(ctx.handle, descs, 2, lib.ptr(pts), N, 1, lib.ptr(Uf), lib.ptr(Sv), p, 0.2, lib.ptr(y), p,
                                              C.byref(out), None, None, None, None, None, None, lib.ptr(gt), C.byref(nobs), C.byref(il))
    assert rc == lib.LMM_E_UNSUPPORTED
