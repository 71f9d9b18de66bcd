"""Gradient of the posterior-predictive logpdf through the conditioning: logpdf(posterior(f(x, σ²), y)(x*, σ*²), y*)
w.r.t. every term's hyper-parameters, the means, σ², σ*², y, y*, U and S (OILMM and IndependentMOGP posteriors).

The analytic oracle here is built on the unchanged oracle (`o.oilmm_posterior`, `o.oilmm_post_logpdf_grad`) and the
per-term kernel derivatives of `test_composite_gradient.dkernel_dterms`, evaluated on the stacked points [x; x*] and sliced
into the K(x,x), K(x,x*) and K(x*,x*) blocks.  CPU: it is checked against central differences of the composed oracle value.
GPU: `predictive_logpdf_and_gradient` against it, and against the chain rule of the union logpdf
log p(y, y*) = log p(y) + log p(y* | y), which does not use the new oracle."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from _tol import assert_isapprox
from oracle import lmm_oracle as o
from test_composite_gradient import _inputs, _params, _shift, _xin, composite_latents, dkernel_dterms, terms_of, to_lmm
from test_missing_gradient import kernel_case


# ------------------------------------------------------------------------------------------------ analytic oracle
def post_value(fs, U, S, x, s2, y, xs, s2s, ys) -> float:
    """The composed oracle value logpdf(posterior(OILMM(fs, U, S)(x, σ²), y)(x*, σ*²), y*); U = I, S = 1 is an
    IndependentMOGP."""
    post = o.oilmm_posterior(o.OILMMModel(fs, U, S), x, s2, y)
    return o.oilmm_post_logpdf_grad(post, xs, s2s, ys)[0]


def post_full_grad(fs, U, S, x, s2, y, xs, s2s, ys):
    """(value, grads) of `post_value`: grads["terms"][i] is (nterms, 3 + D) as `_contract` of test_composite_gradient."""
    X, Xs = o._as2d(x), o._as2d(xs)
    N, Ns = X.shape[0], Xs.shape[0]
    p, m = U.shape
    Y, Ys = o.reshape_y(y, N), o.reshape_y(ys, Ns)
    T = U.T / np.sqrt(S)[:, None]
    Ty, Tys = T @ Y, T @ Ys
    Z = np.vstack([X, Xs])
    terms, gmean, tr_x, tr_s = [], np.zeros(m), np.zeros(m), np.zeros(m)
    g_ytr, bar_T = np.zeros((p, N)), np.zeros((m, p))
    for i, f in enumerate(fs):
        k = f.kernel
        Kxx, Kxs, Kss = o.kernelmatrix(k, X), o.kernelmatrix(k, X, Xs), o.kernelmatrix(k, Xs)
        Cx = Kxx + (s2 / S[i]) * np.eye(N)
        alpha = np.linalg.solve(Cx, Ty[i] - f.mean_const)
        W = np.linalg.solve(Cx, Kxs)
        Sig = Kss - Kxs.T @ W + (s2s / S[i]) * np.eye(Ns)
        P = np.linalg.inv(Sig)
        beta = P @ (Tys[i] - f.mean_const - Kxs.T @ alpha)
        gamma = W @ beta
        Gss = 0.5 * (np.outer(beta, beta) - P)
        Gc = np.outer(alpha - gamma, beta) + W @ P
        Gx = 0.5 * (np.outer(gamma - alpha, gamma - alpha) - np.outer(alpha, alpha) - W @ P @ W.T)
        terms.append(np.array([[float(np.sum(Gx * d[:N, :N]) + np.sum(Gc * d[:N, N:]) + np.sum(Gss * d[N:, N:])) for d in ds]
                               for ds in dkernel_dterms(k, Z)]))
        gmean[i] = beta.sum() - gamma.sum()
        tr_x[i], tr_s[i] = np.trace(Gx), np.trace(Gss)
        g_ytr += np.outer(T[i], gamma)
        bar_T[i] = gamma @ Y.T - beta @ Ys.T
    lp, gpost = o.oilmm_post_logpdf_grad(o.oilmm_posterior(o.OILMMModel(fs, U, S), x, s2, y), xs, s2s, ys)
    Rs = (np.eye(p) - U @ U.T) @ Ys
    gU = bar_T.T / np.sqrt(S)[None, :] + Rs @ (U.T @ Ys).T / s2s
    gS = -np.einsum("ij,ji->i", bar_T, U) / (2.0 * S ** 1.5) - tr_x * s2 / S ** 2 - tr_s * s2s / S ** 2 - Ns / (2.0 * S)
    return lp, {"terms": terms, "mean_const": gmean, "sigma2": gpost["sigma2"], "y": gpost["y"],
                "train": {"sigma2": float(np.sum(tr_x / S)), "y": g_ytr.reshape(-1)}, "U": gU, "S": gS}


# ------------------------------------------------------------------------------------------------ fixtures
def latents_case(case):
    """(latents, D): the kernel grid of test_missing_gradient plus Matern32 and a 3-term sum."""
    if case == "matern32_three":
        fs = composite_latents()
        return [fs[2], fs[3]], 1
    return kernel_case(case)


KERNEL_CASES = ["se_matern52", "exponential_ratquad", "periodic_sum", "product", "ard_D2", "matern32_three"]


def problem(rng, fs, model, N, Ns, D, hi=6.0):
    """(U, S, x, σ², y, x*, σ*², y*): OILMM with p = m + 2 (p > m), or IndependentMOGP (U = I, S = 1)."""
    m = len(fs)
    if model == "oilmm":
        p = m + 2
        U, S = o.orthogonal_from_seed(p, m, seed=4)
    else:
        p = m
        U, S = np.eye(m), np.ones(m)
    xa = _inputs(rng, N + Ns, D, hi)
    idx = rng.permutation(N + Ns)
    x, xs = xa[np.sort(idx[:N])], xa[np.sort(idx[N:])]
    return U, S, x, 0.12, rng.standard_normal(p * N), xs, 0.09, rng.standard_normal(p * Ns)


# ------------------------------------------------------------------------------------------------ CPU
def _fd(fun, v, h=1e-6):
    hh = h * max(1.0, abs(v))
    return (fun(v + hh) - fun(v - hh)) / (2 * hh)


def _close(fd, an, scale, rtol=5e-6):
    return abs(fd - an) <= rtol * max(abs(an), 1e-2 * scale)


@pytest.mark.parametrize("model", ["oilmm", "imogp"])
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_oracle_posterior_gradient_matches_finite_differences(model, case):
    rng = np.random.default_rng(17)
    fs, D = latents_case(case)
    U, S, x, s2, y, xs, s2s, ys = problem(rng, fs, model, 22, 9, D)
    lp, g = post_full_grad(fs, U, S, x, s2, y, xs, s2s, ys)
    assert abs(lp - post_value(fs, U, S, x, s2, y, xs, s2s, ys)) <= 1e-12 * abs(lp)
    # every term's hyper-parameters
    for i, gp_ in enumerate(fs):
        scale = max(1e-3, float(np.max(np.abs(g["terms"][i]))))
        for t, j, v in _params(gp_, D):
            fd = _fd(lambda w: post_value(_shift(fs, i, t, j, w - v), U, S, x, s2, y, xs, s2s, ys), v)
            assert _close(fd, g["terms"][i][t, j], scale), (i, t, j, fd, g["terms"][i][t, j])
        fd = _fd(lambda w: post_value([dataclasses.replace(f, mean_const=w) if n == i else f for n, f in enumerate(fs)],
                                      U, S, x, s2, y, xs, s2s, ys), gp_.mean_const)
        assert _close(fd, g["mean_const"][i], 1.0), (i, fd, g["mean_const"][i])
    # noise variances
    assert _close(_fd(lambda w: post_value(fs, U, S, x, w, y, xs, s2s, ys), s2), g["train"]["sigma2"], 1.0)
    assert _close(_fd(lambda w: post_value(fs, U, S, x, s2, y, xs, w, ys), s2s), g["sigma2"], 1.0)
    # observations (a sample of entries on each side)
    for k in rng.choice(len(y), 8, replace=False):
        def fy(w, k=k):
            yy = y.copy()
            yy[k] = w
            return post_value(fs, U, S, x, s2, yy, xs, s2s, ys)
        assert _close(_fd(fy, y[k]), g["train"]["y"][k], 1.0), k
    for k in rng.choice(len(ys), 8, replace=False):
        def fys(w, k=k):
            yy = ys.copy()
            yy[k] = w
            return post_value(fs, U, S, x, s2, y, xs, s2s, yy)
        assert _close(_fd(fys, ys[k]), g["y"][k], 1.0), k
    if model != "oilmm":
        return
    for (a, b) in [(0, 0), (U.shape[0] - 1, 1), (2, 0), (1, 1)]:
        def fu(w, a=a, b=b):
            UU = U.copy()
            UU[a, b] = w
            return post_value(fs, UU, S, x, s2, y, xs, s2s, ys)
        assert _close(_fd(fu, U[a, b]), g["U"][a, b], 1.0), (a, b)
    for b in range(len(S)):
        def fsv(w, b=b):
            SS = S.copy()
            SS[b] = w
            return post_value(fs, U, SS, x, s2, y, xs, s2s, ys)
        assert _close(_fd(fsv, S[b]), g["S"][b], 1.0), b


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def lmm():
    import lmm_b200

    lmm_b200.default_context()
    return lmm_b200


def _build(lmm, fs, model, U, S, x, s2, y, p):
    """The library's posterior handle of the problem."""
    O = lmm.MOInputIsotopicByOutputs
    lat = lmm.independent_mogp([to_lmm(lmm, g) for g in fs])
    f = lmm.ILMM(lat, lmm.Orthogonal(U, S)) if model == "oilmm" else lat
    return lmm.posterior(f(O(_xin(lmm, x), p), s2), y)


def _terms_array(got):
    return [np.array([[d["variance"], d["inv_lengthscale"], d["param"]] + list(d["ard"]) for d in lat]) for lat in got]


def _assert_matches_oracle(g, ref, model, rtol=1e-9):
    for i, (a, b) in enumerate(zip(_terms_array(g["terms"]), ref["terms"])):
        assert_isapprox(a, b, rtol, f"terms of latent {i}")
    assert_isapprox(g["mean_const"], ref["mean_const"], rtol, "mean_const")
    assert_isapprox([g["sigma2"]], [ref["sigma2"]], rtol, "sigma2*")
    assert_isapprox([g["train"]["sigma2"]], [ref["train"]["sigma2"]], rtol, "sigma2")
    assert_isapprox(g["y"], ref["y"], rtol, "y*")
    assert_isapprox(g["train"]["y"], ref["train"]["y"], rtol, "y")
    if model == "oilmm":
        assert_isapprox(g["U"], ref["U"], rtol, "U")
        assert_isapprox(g["S"], ref["S"], rtol, "S")
    else:
        assert "U" not in g and "S" not in g


def _run(lmm, fs, model, N, Ns, D, seed, hi=10.0):
    rng = np.random.default_rng(seed)
    U, S, x, s2, y, xs, s2s, ys = problem(rng, fs, model, N, Ns, D, hi)
    p = U.shape[0]
    post = _build(lmm, fs, model, U, S, x, s2, y, p)
    lp, g = lmm.predictive_logpdf_and_gradient(post(lmm.MOInputIsotopicByOutputs(_xin(lmm, xs), p), s2s), ys, y, with_grad_y=True)
    lpr, ref = post_full_grad(fs, U, S, x, s2, y, xs, s2s, ys)
    assert abs(lp - lpr) <= 1e-9 * abs(lpr)
    return g, ref


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["oilmm", "imogp"])
@pytest.mark.parametrize("N,Ns", [(50, 7), (300, 140), (700, 260)])
def test_posterior_gradient_matches_oracle(lmm, model, N, Ns):
    fs = composite_latents(1)
    g, ref = _run(lmm, fs, model, N, Ns, 1, seed=N + Ns)
    _assert_matches_oracle(g, ref, model)


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["oilmm", "imogp"])
@pytest.mark.parametrize("case", KERNEL_CASES)
def test_posterior_gradient_kernel_grid(lmm, model, case):
    fs, D = latents_case(case)
    g, ref = _run(lmm, fs, model, 230, 90, D, seed=3)
    _assert_matches_oracle(g, ref, model)
    D0 = len(g["ard"][0])
    for i, f in enumerate(fs):
        np.testing.assert_array_equal(g["variance"][i], g["terms"][i][0]["variance"])
        np.testing.assert_array_equal(g["inv_lengthscale"][i], g["terms"][i][0]["inv_lengthscale"])
        np.testing.assert_array_equal(g["ard"][i], g["terms"][i][0]["ard"] if f.kernel.ard is not None else np.zeros(D0))


@pytest.mark.gpu
@pytest.mark.parametrize("N,Ns", [(700, 300), (2300, 400)])
def test_union_identity(lmm, N, Ns):
    """log p(y, y*) = log p(y) + log p(y* | y) at σ*² = σ²: the union's gradient is the training gradient plus the new one."""
    rng = np.random.default_rng(N)
    fs = composite_latents(1)
    m, p, s2 = len(fs), len(fs) + 3, 0.1
    U, S = o.orthogonal_from_seed(p, m, seed=8)
    xa = _inputs(rng, N + Ns, 1, hi=40.0)
    idx = rng.permutation(N + Ns)
    x, xs = xa[np.sort(idx[:N])], xa[np.sort(idx[N:])]
    Y, Ys = rng.standard_normal((p, N)), rng.standard_normal((p, Ns))
    O = lmm.MOInputIsotopicByOutputs
    f = lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), lmm.Orthogonal(U, S))
    lp_tr, g_tr = lmm.logpdf_and_gradient(f(O(x, p), s2), Y.reshape(-1), with_grad_y=True, kernel_terms=True)
    xu, Yu = np.concatenate([x, xs]), np.hstack([Y, Ys])
    lp_u, g_u = lmm.logpdf_and_gradient(f(O(xu, p), s2), Yu.reshape(-1), with_grad_y=True, kernel_terms=True)
    post = lmm.posterior(f(O(x, p), s2), Y.reshape(-1))
    lp_c, g_c = lmm.predictive_logpdf_and_gradient(post(O(xs, p), s2), Ys.reshape(-1), Y.reshape(-1), with_grad_y=True)
    assert abs(lp_tr + lp_c - lp_u) <= 1e-9 * abs(lp_u)
    a, b, c = _terms_array(g_tr["terms"]), _terms_array(g_c["terms"]), _terms_array(g_u["terms"])
    assert_isapprox(np.concatenate([(s + t).ravel() for s, t in zip(a, b)]), np.concatenate([t.ravel() for t in c]), 1e-9, "terms")
    for k in ("mean_const", "U", "S"):
        assert_isapprox(g_tr[k] + g_c[k], g_u[k], 1e-9, k)
    assert_isapprox([g_tr["sigma2"] + g_c["train"]["sigma2"] + g_c["sigma2"]], [g_u["sigma2"]], 1e-9, "sigma2")
    gyu = g_u["y"].reshape(p, N + Ns)
    assert_isapprox((g_tr["y"] + g_c["train"]["y"]).reshape(p, N), gyu[:, :N], 1e-9, "y")
    assert_isapprox(g_c["y"].reshape(p, Ns), gyu[:, N:], 1e-9, "y*")


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["oilmm", "imogp"])
def test_value_and_test_side_are_bit_identical_and_calls_deterministic(lmm, model, tmp_path):
    rng = np.random.default_rng(21)
    fs = composite_latents(2)
    U, S, x, s2, y, xs, s2s, ys = problem(rng, fs, model, 500, 180, 2, hi=10.0)
    p = U.shape[0]
    post = _build(lmm, fs, model, U, S, x, s2, y, p)
    O = lmm.MOInputIsotopicByOutputs
    fxp = post(O(_xin(lmm, xs), p), s2s)
    mv0 = lmm.mean_and_var(fxp)
    lp0, g0 = lmm.logpdf_and_gradient(fxp, ys, with_grad_y=True)
    lp1, g1 = lmm.predictive_logpdf_and_gradient(fxp, ys, y, with_grad_y=True)
    lp2, g2 = lmm.predictive_logpdf_and_gradient(fxp, ys, y, with_grad_y=True)
    assert lp1 == lp0 == lmm.logpdf(fxp, ys)
    assert g1["sigma2"] == g0["sigma2"]
    assert np.array_equal(g1["y"], g0["y"])
    flat = lambda g: np.concatenate([np.concatenate([t.ravel() for t in _terms_array(g["terms"])]), g["mean_const"], [g["sigma2"]],
                                     [g["train"]["sigma2"]], g["y"], g["train"]["y"]] + ([g["U"].ravel(), g["S"]] if model == "oilmm" else []))
    assert lp2 == lp1 and np.array_equal(flat(g1), flat(g2))
    mv1 = lmm.mean_and_var(fxp)  # the handle is unchanged
    assert np.array_equal(mv0[0], mv1[0]) and np.array_equal(mv0[1], mv1[1])
    path = str(tmp_path / "post.bin")
    lmm.save_posterior(post, path)
    f = lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), lmm.Orthogonal(U, S)) if model == "oilmm" else \
        lmm.independent_mogp([to_lmm(lmm, g) for g in fs])
    loaded = lmm.load_posterior(path, f)
    lp3, g3 = lmm.predictive_logpdf_and_gradient(loaded(O(_xin(lmm, xs), p), s2s), ys, y, with_grad_y=True)
    assert lp3 == lp1 and np.array_equal(flat(g3), flat(g1))


@pytest.mark.gpu
def test_masked_oilmm_posterior_is_an_ordinary_oilmm_handle(lmm):
    """A per-input mask gives an OILMM posterior over the observed inputs: y_train is the observed block."""
    rng = np.random.default_rng(5)
    fs = composite_latents(1)[:2]
    m, p, N, Ns = 2, 4, 160, 50
    U, S = o.orthogonal_from_seed(p, m, seed=6)
    x, xs = _inputs(rng, N, 1, 10.0), _inputs(rng, Ns, 1, 10.0)
    Y = rng.standard_normal((p, N))
    keep = np.ones(N, bool)
    keep[rng.choice(N, 30, replace=False)] = False
    Ym = Y.copy()
    Ym[:, ~keep] = np.nan
    O = lmm.MOInputIsotopicByOutputs
    f = lmm.ILMM(lmm.independent_mogp([to_lmm(lmm, g) for g in fs]), lmm.Orthogonal(U, S))
    post = lmm.posterior_missing(f(O(x, p), 0.1), Ym.reshape(-1))
    ys = rng.standard_normal(p * Ns)
    lp, g = lmm.predictive_logpdf_and_gradient(post(O(xs, p), 0.1), ys, Y[:, keep].reshape(-1))
    lpr, ref = post_full_grad(fs, U, S, x[keep], 0.1, Y[:, keep].reshape(-1), xs, 0.1, ys)
    assert abs(lp - lpr) <= 1e-9 * abs(lpr)
    for i, (a, b) in enumerate(zip(_terms_array(g["terms"]), ref["terms"])):
        assert_isapprox(a, b, 1e-9, f"terms of latent {i}")
    assert_isapprox(g["S"], ref["S"], 1e-9, "S")


@pytest.mark.gpu
def test_refusals(lmm):
    rng = np.random.default_rng(12)
    fs = composite_latents(1)[:2]
    m, N, Ns = 2, 60, 20
    x, xs = _inputs(rng, N, 1), _inputs(rng, Ns, 1)
    O = lmm.MOInputIsotopicByOutputs
    lat = lmm.independent_mogp([to_lmm(lmm, g) for g in fs])
    # general ILMM (joint posterior)
    p = 3
    H = rng.uniform(0.2, 1.2, (p, m))
    y = rng.standard_normal(p * N)
    post = lmm.posterior(lmm.ILMM(lat, H)(O(x, p), 0.2), y)
    with pytest.raises(ValueError, match="per-latent"):
        lmm.predictive_logpdf_and_gradient(post(O(xs, p), 0.2), rng.standard_normal(p * Ns), y)
    # IndependentMOGP under a dense Σy (joint posterior)
    ym = rng.standard_normal(m * N)
    A = rng.standard_normal((m * N, m * N)) * 0.01
    post = lmm.posterior(lat(O(x, m), 0.1 * np.eye(m * N) + A @ A.T), ym)
    with pytest.raises(ValueError, match="per-latent"):
        lmm.predictive_logpdf_and_gradient(post(O(xs, m), 0.2), rng.standard_normal(m * Ns), ym)
    # dense missing-data posterior
    U, S = o.orthogonal_from_seed(p, m, seed=2)
    f = lmm.ILMM(lat, lmm.Orthogonal(U, S))
    yn = y.copy()
    yn[rng.choice(p * N, 20, replace=False)] = np.nan
    post = lmm.posterior_missing(f(O(x, p), 0.2), yn)
    with pytest.raises(ValueError, match="per-latent"):
        lmm.predictive_logpdf_and_gradient(post(O(xs, p), 0.2), rng.standard_normal(p * Ns), y)
    # sequentially conditioned OILMM posterior
    post = lmm.posterior(f(O(x, p), 0.2), y)
    y2 = rng.standard_normal(p * Ns)
    post2 = lmm.posterior(post(O(xs, p), 0.2), y2)
    with pytest.raises(ValueError, match="sequentially"):
        lmm.predictive_logpdf_and_gradient(post2(O(xs, p), 0.2), y2, np.concatenate([y.reshape(p, N), y2.reshape(p, Ns)], 1).reshape(-1))
    # y_train that is not the handle's data
    with pytest.raises(ValueError, match="y_train"):
        lmm.predictive_logpdf_and_gradient(post(O(xs, p), 0.2), y2, y + 1e-6)
    # NULL y_train, grad_U on an IndependentMOGP
    ctx = lmm.default_context()
    lib = lmm._lib
    pts = np.ascontiguousarray(xs.reshape(Ns, 1))
    out, il = C.c_double(), C.c_int(-1)
    h = lmm.api._post_owner(post(O(xs, p), 0.2)).handle
    rc = ctx.lib.lmm_post_logpdf_grad_full(h, lib.ptr(pts), Ns, 0.2, lib.ptr(y2), None, C.byref(out), None, None, None, None, None, None,
                                           None, None, None, C.byref(il))
    assert rc == lib.LMM_E_ARG
    post_i = lmm.posterior(lat(O(x, m), 0.2), ym)
    ys_i = rng.standard_normal(m * Ns)
    gU = np.zeros(m * m)
    h = lmm.api._post_owner(post_i(O(xs, m), 0.2)).handle
    rc = ctx.lib.lmm_post_logpdf_grad_full(h, lib.ptr(pts), Ns, 0.2, lib.ptr(ys_i), lib.ptr(ym), C.byref(out), None, None, None, None,
                                           None, None, None, lib.ptr(gU), None, C.byref(il))
    assert rc == lib.LMM_E_ARG
    # without grad_U the same call runs
    rc = ctx.lib.lmm_post_logpdf_grad_full(h, lib.ptr(pts), Ns, 0.2, lib.ptr(ys_i), lib.ptr(ym), C.byref(out), None, None, None, None,
                                           None, None, None, None, None, C.byref(il))
    assert rc == lib.LMM_OK
