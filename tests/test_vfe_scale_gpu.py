"""Sparse variational (VFE) bound, gradient and posterior at the shapes and options the small cases of test_vfe.py never reach:
inducing sets of 3 to 13 tiles, every factor schedule chol_factor picks for K(z, z) and Σ, short last row chunks, 16 latents, and
the int8 path at N = 12000.  The references are the closed-form oracle of test_vfe.py (`vfe_oracle`, `_latent_vfe`), computed
once per problem and shared by every option set that runs it.

Gradients past the size where per-parameter differences are affordable are checked along seeded random directions v (one
central difference of the oracle ELBO along v against g·v), see `directional_difference`; its error bound is checked against
the whitened cotangents of `_latent_vfe_grad` on the CPU before any GPU case relies on it.  A CPU test restates the rules that
select the schedules and asserts that every GPU case still reaches the branch it is there for."""
import contextlib
import dataclasses
import math
import os

import numpy as np
import pytest

from _tol import assert_isapprox
from oracle import lmm_oracle as o
from test_composite_gradient import _contract, _inputs, _params, _shift, _xin, terms_of
from test_missing_gradient import KERNEL_CASES, kernel_case
from test_vfe import JIT, _case, _fx, _latent_vfe, _latent_vfe_grad, vfe_oracle

T = 128


# ------------------------------------------------------------------------------------------------ problems
@dataclasses.dataclass
class Problem:
    fs: list
    D: int
    x: np.ndarray
    z: np.ndarray
    p: int
    U: object
    S: object
    y: np.ndarray
    xs: np.ndarray
    s2: float = 0.15
    jitter: float = JIT

    @property
    def oilmm(self):
        return self.U is not None


def _standard(case, model, N, M, seed, nxs):
    fs, D, x, z, p, U, S, y = _case(case, model, N, M, seed)
    xs = _inputs(np.random.default_rng(seed + 1), nxs, D, hi=float(np.max(x)) + 0.5)
    return Problem(fs, D, x, z, p, U, S, y, xs)


def latent_pool(m, seed):
    """m one-dimensional latents, each with its own kernel, hyper-parameters and mean: the latents of the 1-D KERNEL_CASES in turn,
    their leading term's variance and inverse lengthscale scaled by factors in [0.75, 1.35] and their means shifted, so that two
    latents built from the same case still differ.  The non-decaying periodic latents of "periodic_sum" are left out: over
    hundreds of inducing inputs their K(z, z) is numerically rank-deficient, and the oracle's central differences along their
    relative inverse lengthscale (a derivative that grows with the distance of the inputs) lose most of their digits."""
    base = [g for c in KERNEL_CASES if c != "periodic_sum" and kernel_case(c)[1] == 1 for g in kernel_case(c)[0]]
    rng = np.random.default_rng(seed)
    out = []
    for i in range(m):
        g = base[i % len(base)]
        a, b = rng.uniform(0.75, 1.35, 2)
        k = dataclasses.replace(g.kernel, variance=g.kernel.variance * a, inv_lengthscale=g.kernel.inv_lengthscale * b)
        out.append(o.GP(k, g.mean_const + rng.uniform(-0.3, 0.3)))
    return out


def _pooled(model, m, p, N, M, seed, nxs, linspace_z=False, jitter=JIT):
    rng = np.random.default_rng(seed)
    fs = latent_pool(m, seed)
    hi = max(6.0, N / 40.0)
    x = _inputs(rng, N, 1, hi=hi)
    z = np.linspace(0.0, hi, M) if linspace_z else _inputs(rng, M, 1, hi=hi)
    if model == "oilmm":
        U, S = o.orthogonal_from_seed(p, m, seed=seed % 7 + 1)
    else:
        p, U, S = m, None, None
    y = rng.standard_normal(p * N)
    xs = _inputs(rng, nxs, 1, hi=hi + 0.5)
    return Problem(fs, 1, x, z, p, U, S, y, xs, jitter=jitter)


def _scale_se(N, M, seed, nxs):
    pb = _standard("se_matern52", "imogp", N, M, seed, nxs)
    pb.z = np.linspace(0.0, float(np.max(pb.x)), M)  # evenly spread: no near-duplicate inducing inputs at M = 1600
    pb.jitter = 1e-3
    return pb


# key -> (builder, N, M, m): the shape is restated so the branch table below needs no problem build
PROBLEMS = {
    # 1. gradient past two inducing tiles (mt = 3, 5, 6); 333 test points = 3 tile rows, the last one ragged
    "oilmm_se_matern52_M300": (lambda: _standard("se_matern52", "oilmm", 2000, 300, 401, 333), 2000, 300, 2),
    "imogp_product_M520": (lambda: _standard("product", "imogp", 2500, 520, 402, 333), 2500, 520, 2),
    "oilmm_ard_D2_M700": (lambda: _standard("ard_D2", "oilmm", 1500, 700, 403, 333), 1500, 700, 2),
    # 2. factor schedules
    "oilmm_m2_M800": (lambda: _standard("se_matern52", "oilmm", 1200, 800, 411, 333), 1200, 800, 2),
    "imogp_m6_M800": (lambda: _pooled("imogp", 6, 6, 1200, 800, 412, 333), 1200, 800, 6),
    "oilmm_m14_M900": (lambda: _pooled("oilmm", 14, 16, 700, 900, 413, 333), 700, 900, 14),
    "imogp_m2_M1450": (lambda: _standard("exponential_ratquad", "imogp", 1500, 1450, 414, 333), 1500, 1450, 2),
    # 3. row chunks: N = 850 is 7 tile rows, the last one ragged
    "oilmm_product_N850": (lambda: _standard("product", "oilmm", 850, 300, 421, 200), 850, 300, 2),
    # 4. many latents
    "oilmm_m16": (lambda: _pooled("oilmm", 16, 24, 2000, 300, 431, 200), 2000, 300, 16),
    "imogp_m16": (lambda: _pooled("imogp", 16, 16, 2000, 300, 432, 200), 2000, 300, 16),
    # 5. production scale; 600 test points = 5 tile rows, the last one ragged
    "oilmm_m4_M1100": (lambda: _pooled("oilmm", 4, 5, 12000, 1100, 441, 600, linspace_z=True, jitter=1e-3), 12000, 1100, 4),
    "imogp_m2_M1600": (lambda: _scale_se(12000, 1600, 442, 600), 12000, 1600, 2),
}


# ------------------------------------------------------------------------------------------------ directional differences
# A direction moves every parameter at once.  Positive parameters (kernel hyper-parameters, σ², S) move relatively,
# θ -> θ (1 + t v_θ); means, y and U move absolutely.  Each block (hyper-parameters, means, σ², y, U, S) of v has unit 2-norm, so
# no block is drowned by the size of another (y has p N entries).
#
# Error of the central difference D(h) = (f(+h) - f(-h)) / 2h against the directional derivative f'(0):
#   truncation  h² |f'''| / 6, with |f'''| <= FD_C3 |f| along such a direction: the bound is a sum of p N terms that are at most
#               quadratic in y, U and the means, and depend on the relative hyper-parameters, σ² and S through smooth functions
#               whose derivatives are of the order of the terms themselves.  Measured with h = 1e-3 on the problems below: at most
#               5 |f| along the random directions, 130 |f| along a single coordinate (the inverse lengthscale of the periodic
#               factor of "ard_D2", whose derivative grows with the distance of the inputs); FD_C3 = 200 covers both;
#   rounding    ε |f| / h, with ε = FD_EPS bounding how much the oracle's relative rounding differs between the two ends.  It
#               grows with the conditioning of K(z, z); measured from the spread of the differences at h = 1e-6: up to 7e-12
#               (14 latents, 900 inducing inputs over 17.5 length units).  FD_EPS keeps a factor of 3 over that.
# h = 5e-5 about balances the two: bound = (FD_C3 h²/6 + FD_EPS/h) |f| = 4.8e-7 |f|, against directional derivatives of the
# order of |f|.  g·v carries the library's own error too, held to the 1e-9 relative of its values: GPU_RTOL times the sum of
# the absolute contributions |g_j s_j v_j|.
FD_H = 5e-5
FD_C3 = 200.0
FD_EPS = 2e-11
GPU_RTOL = 1e-9


def fd_bound(f):
    return (FD_C3 * FD_H ** 2 / 6.0 + FD_EPS / FD_H) * abs(f)


@dataclasses.dataclass
class Direction:
    terms: list  # per latent: (terms, 3 + D), the layout of the gradient's per-term rows
    mean: np.ndarray
    sigma2: float
    y: np.ndarray
    U: object
    S: object


BLOCKS = ("terms", "mean", "sigma2", "y", "U", "S")


def random_direction(pb, seed, blocks=BLOCKS):
    rng = np.random.default_rng(seed)

    def unit(n, on):
        if not on:
            return np.zeros(n)
        r = rng.standard_normal(n)
        return r / np.linalg.norm(r)

    idx = [(i, t, j) for i, f in enumerate(pb.fs) for t, j, _ in _params(f, pb.D)]
    r = unit(len(idx), "terms" in blocks)
    terms = [np.zeros((len(terms_of(f.kernel)), 3 + pb.D)) for f in pb.fs]
    for (i, t, j), ri in zip(idx, r):
        terms[i][t, j] = ri
    m = len(pb.fs)
    return Direction(terms, unit(m, "mean" in blocks), float(unit(1, "sigma2" in blocks)[0]), unit(len(pb.y), "y" in blocks),
                     unit(pb.U.size, "U" in blocks).reshape(pb.U.shape) if pb.oilmm else None,
                     unit(m, "S" in blocks) if pb.oilmm else None)


def moved(pb, v, t):
    """(fs, σ², y, U, S) at parameter + t v."""
    fs = pb.fs
    for i, f in enumerate(pb.fs):
        for tt, j, val in _params(f, pb.D):
            if v.terms[i][tt, j]:
                fs = _shift(fs, i, tt, j, t * v.terms[i][tt, j] * val)
    fs = [dataclasses.replace(f, mean_const=f.mean_const + t * v.mean[i]) for i, f in enumerate(fs)]
    U = pb.U + t * v.U if pb.oilmm else None
    S = pb.S * (1.0 + t * v.S) if pb.oilmm else None
    return fs, pb.s2 * (1.0 + t * v.sigma2), pb.y + t * v.y, U, S


def oracle_elbo(pb, fs, s2, y, U, S):
    return vfe_oracle(fs, pb.x, pb.z, pb.jitter, s2, y, U, S)[0]


def directional_difference(pb, v):
    """(D(h), the bound on |D(h) - f'(0)|) along v."""
    fp, fm = oracle_elbo(pb, *moved(pb, v, FD_H)), oracle_elbo(pb, *moved(pb, v, -FD_H))
    return (fp - fm) / (2 * FD_H), fd_bound(max(abs(fp), abs(fm)))


def term_rows(g, fs, D):
    return [np.array([[t["variance"], t["inv_lengthscale"], t["param"]] + list(t["ard"]) for t in lat]) for lat in g["terms"]]


def gdot(g, pb, v):
    """(g·v in the coordinates of `moved`, Σ |g_j s_j v_j|)."""
    parts = []
    rows = term_rows(g, pb.fs, pb.D)
    for i, f in enumerate(pb.fs):
        for t, j, val in _params(f, pb.D):
            parts.append(rows[i][t, j] * val * v.terms[i][t, j])
    parts += list(np.asarray(g["mean_const"]) * v.mean) + [g["sigma2"] * pb.s2 * v.sigma2] + list(np.asarray(g["y"]) * v.y)
    if pb.oilmm:
        parts += list((np.asarray(g["U"]) * v.U).ravel()) + list(np.asarray(g["S"]) * pb.S * v.S)
    parts = np.array(parts)
    return float(np.sum(parts)), float(np.sum(np.abs(parts)))


def assert_directional(g, pb, v, fd, bound, what=""):
    an, scale = gdot(g, pb, v)
    tol = bound + GPU_RTOL * scale
    assert abs(fd - an) <= tol, (what, fd, an, abs(fd - an), tol)


def projected(pb):
    """(T Y, ν) of the problem: the per-latent data and noise of the bound."""
    if pb.oilmm:
        Tm, nu = o.project_orthogonal(pb.U, pb.S, pb.s2)
    else:
        Tm, nu = np.eye(len(pb.fs)), np.full(len(pb.fs), pb.s2)
    return Tm @ o.reshape_y(pb.y, len(pb.x)), nu


def latent_differences(pb, i):
    """Per-parameter central differences of latent i's hyper-parameters and mean: only ELBO_i depends on them, so each
    difference evaluates `_latent_vfe` of that latent alone.  [((t, j) or "mean", D(h) in the coordinates of `moved`, bound)]"""
    Ty, nu = projected(pb)
    f0 = pb.fs[i]

    def val(g):
        return _latent_vfe(g, pb.x, pb.z, pb.jitter, nu[i], Ty[i])[0]

    out = []
    for t, j, v in _params(f0, pb.D):
        fp, fm = val(_shift(pb.fs, i, t, j, FD_H * v)[i]), val(_shift(pb.fs, i, t, j, -FD_H * v)[i])
        out.append(((t, j), (fp - fm) / (2 * FD_H), fd_bound(max(abs(fp), abs(fm)))))
    fp, fm = (val(dataclasses.replace(f0, mean_const=f0.mean_const + s * FD_H)) for s in (1, -1))
    out.append(("mean", (fp - fm) / (2 * FD_H), fd_bound(max(abs(fp), abs(fm)))))
    return out


def assert_latent_differences(g, pb, i, diffs):
    rows = term_rows(g, pb.fs, pb.D)
    vals = {(t, j): v for t, j, v in _params(pb.fs[i], pb.D)}
    for key, fd, bound in diffs:
        an = g["mean_const"][i] if key == "mean" else rows[i][key] * vals[key]
        assert abs(fd - an) <= bound + GPU_RTOL * abs(an), (i, key, fd, an)


# ------------------------------------------------------------------------------------------------ CPU: the reference
def analytic_gradient(pb):
    """The gradient in the library's layout from the whitened cotangents of `_latent_vfe_grad` (Ḡxz, Ḡz, dELBO/dδ, dELBO/dν),
    contracted with the exact kernel-matrix derivatives of the joint inputs [x; z] (`_contract`), and the closed-form chain rule
    through T Y = S^{-1/2} U' Y, ν = σ²/S and the regulariser -(N Σ log S + N (p-m) log 2πσ² + |R|²/σ²)/2, R = (I - UU') Y."""
    Ty, nu = projected(pb)
    N, M, m = len(pb.x), len(pb.z), len(pb.fs)
    X = np.vstack([o._as2d(pb.x), o._as2d(pb.z)])
    terms, gd, dnu = [], [], []
    for i, f in enumerate(pb.fs):
        Gxz, Gz, d, dn = _latent_vfe_grad(f, pb.x, pb.z, pb.jitter, nu[i], Ty[i])
        G = np.zeros((N + M, N + M))
        G[:N, N:], G[N:, N:] = Gxz, Gz
        G[np.arange(N), np.arange(N)] = -0.5 / nu[i]  # Σ_i k_ii enters as -(Σ_i k_ii)/2ν
        terms.append([{"variance": r[0], "inv_lengthscale": r[1], "param": r[2], "ard": r[3:]} for r in _contract(G, f, X)])
        gd.append(d)
        dnu.append(dn)
    GD, dnu = np.array(gd), np.array(dnu)  # dELBO/d(TY): m x N
    g = {"terms": terms, "mean_const": -GD.sum(axis=1)}
    Y = o.reshape_y(pb.y, N)
    if not pb.oilmm:
        g.update(y=GD.reshape(-1), sigma2=float(np.sum(dnu)))
        return g
    U, S, s2, p = pb.U, pb.S, pb.s2, pb.p
    rS = np.sqrt(S)
    R = Y - U @ (U.T @ Y)
    g["y"] = ((U / rS[None, :]) @ GD - (R - U @ (U.T @ R)) / s2).reshape(-1)
    g["U"] = (Y @ GD.T) / rS[None, :] + (R @ Y.T @ U + Y @ R.T @ U) / s2
    g["S"] = -0.5 * np.sum(GD * Ty, axis=1) / S - dnu * nu / S - N / (2 * S)
    g["sigma2"] = float(np.sum(dnu / S)) - 0.5 * (N * (p - m) / s2 - np.sum(R * R) / s2 ** 2)
    return g


@pytest.mark.parametrize("model,case", [("oilmm", "se_matern52"), ("imogp", "product"), ("oilmm", "ard_D2"), ("imogp", "exponential_ratquad")])
def test_directional_difference_is_within_its_bound_of_the_analytic_gradient(model, case):
    """The reference the GPU cases rely on: at N = 40, M = 9 the central difference along random directions lies within
    `fd_bound` of the analytic derivative, `gdot` of the analytic gradient in the library's layout is that derivative, and the
    bound is small enough to see a relative gradient error of 1e-6."""
    pb = _standard(case, model, 40, 9, 450 + KERNEL_CASES.index(case), 1)
    g = analytic_gradient(pb)
    for seed in range(3):
        v = random_direction(pb, 500 + seed)
        an, scale = gdot(g, pb, v)
        fd, bound = directional_difference(pb, v)
        assert abs(fd - an) <= bound, (seed, fd, an, bound)
        assert bound <= 1e-6 * scale, (bound, scale)
    for b in BLOCKS[:4] + (BLOCKS[4:] if pb.oilmm else ()):  # each block on its own
        v = random_direction(pb, 600, (b,))
        fd, bound = directional_difference(pb, v)
        assert abs(fd - gdot(g, pb, v)[0]) <= bound, b
    for i in range(len(pb.fs)):
        assert_latent_differences(g, pb, i, latent_differences(pb, i))


# ------------------------------------------------------------------------------------------------ which branch each case reaches
OZ = {"off": (0, 7), "S7b8": (7, 8), "S8b7": (8, 7)}
DEFAULTS = {"outer_block": 0, "streams": 4, "lookahead": 1, "chain_fused": 1, "vfe_chunk": 0}
CHAIN_MAX_TILES = 96  # csrc/host_chol.cu:87
OZAKI_MIN_K = 4       # csrc/host_internal.h:95


def sym_tiles(n):
    return n * (n + 1) // 2


def vfe_gram_splits(mt, batch, ntr):  # csrc/vfe.cu:359-363
    sp = -(-2 * 148 // (sym_tiles(mt) * batch))
    return max(1, min(sp, ntr))


def schedule(N, M, m, opts):
    """The branches a VFE call with these options takes, restated from the library (no latent chunking: everything fits):
    the factorisations of K(z, z) and Σ (batch m, mt tile rows), the sweeps, and the Gram's row chunks and splits."""
    o_ = dict(DEFAULTS, **opts)
    mt, nt = math.ceil(M / T), math.ceil(N / T)
    ozaki = o_.get("ozaki", 0)
    ob_user = o_["outer_block"]
    ob = ob_user or 8  # csrc/api.cu:220-228: 0 = the built-in width 8
    out = {"mt": mt, "upper_block_update": mt > ob}  # csrc/host_chol.cu:770-775: trsm_right_lt_upper updates from s0 = ob on
    # csrc/host_chol.cu:609-615: right-looking for batch <= 2 from 12 tile rows (with the int8 update on, not from
    # ozaki_single_nt = 96 tile rows, 64 for two factors, on: out of reach here)
    if o_["lookahead"] and m <= 2 and mt >= 12:
        cf = o_["chain_fused"]
        fused_all = cf == 2 or (cf == 1 and mt <= 32)  # csrc/host_chol.cu:318-321
        rob = ob_user or ((3 if mt <= 112 else 4) if fused_all else (1 if mt <= 32 else 2 if mt <= 48 else 3 if mt <= 112 else 4))
        fused = tuple(jj for jj in range(mt - 1) if fused_all or (cf == 1 and (mt - 1 - jj) * m <= 31))
        out.update(chol="rightlooking", groups=1, fused=fused, ob=rob, int8_chol=False)
    else:
        # csrc/host_chol.cu:639: the int8 update needs mt > outer_block and mt > ozaki_min_k; csrc/host_chol.cu:151,163: a wide
        # update from s0 >= ozaki_min_k at width 2 (no user width)
        int8 = bool(ozaki) and mt > ob and mt > OZAKI_MIN_K
        sob = (ob_user or 2) if int8 else ob
        # csrc/host_chol.cu:658-660: one stream with the fused chain while (mt-1) m <= CHAIN_MAX_TILES, else min(streams, m) groups
        chain_all = o_["chain_fused"] and (mt - 1) * m <= CHAIN_MAX_TILES and mt > 1
        G = 1 if mt <= 1 or chain_all else min(o_["streams"], m)
        bg = -(-m // G)  # the largest group
        # csrc/host_chol.cu:218: inside a block, a column whose TRSM has at most CHAIN_MAX_TILES tiles over the group fuses
        fused = tuple(jj for jj in range(mt - 1) if o_["chain_fused"] and (jj + 1) % sob and (mt - 1 - jj) * bg <= CHAIN_MAX_TILES)
        out.update(chol="chain_all" if chain_all else "leftlooking", groups=G, fused=fused, ob=sob, int8_chol=int8)
    out["int8_sweep"] = bool(ozaki) and mt > 8  # csrc/host_chol.cu:739 (and 688)
    # csrc/host_vfe.cu:69-73: ct tile rows per chunk (0: all of them, as memory allows here), one split count for every chunk
    ct = min(o_["vfe_chunk"] or nt, nt)
    last = nt - ct * ((nt - 1) // ct)
    out["chunks"] = -(-nt // ct)
    out["splits"] = vfe_gram_splits(mt, m, ct)
    out["empty_splits"] = out["splits"] > last  # vfe.cu:368: splits past the last chunk's rows sum empty ranges
    return out


def shape(key):
    _, N, M, m = PROBLEMS[key]
    return N, M, m


# 1. gradient past two inducing tiles: user widths 2 and 3 run trsm_right_lt_upper's block update at mt = 3, 5, 6
GRAD_CASES = [(k, ob) for k in ("oilmm_se_matern52_M300", "imogp_product_M520", "oilmm_ard_D2_M700") for ob in (0, 2, 3)]
# 2. factor schedules: (id, problem, options, the path of chol_factor for K(z, z) and Σ)
SCHED_CASES = [
    ("default_m2", "oilmm_m2_M800", {}, {"chol": "chain_all", "groups": 1}),
    ("unfused_m2", "oilmm_m2_M800", {"chain_fused": 0}, {"chol": "leftlooking", "groups": 2, "fused": ()}),
    ("unfused_one_stream", "oilmm_m2_M800", {"chain_fused": 0, "streams": 1}, {"chol": "leftlooking", "groups": 1, "fused": ()}),
    ("unfused_m6", "imogp_m6_M800", {"chain_fused": 0}, {"chol": "leftlooking", "groups": 4, "fused": ()}),
    ("grouped_m14", "oilmm_m14_M900", {}, {"chol": "leftlooking", "groups": 4, "fused": tuple(range(7))}),
    ("one_stream_m14", "oilmm_m14_M900", {"streams": 1}, {"chol": "leftlooking", "groups": 1, "fused": tuple(range(1, 7))}),
    ("rightlooking", "imogp_m2_M1450", {}, {"chol": "rightlooking", "ob": 3, "fused": tuple(range(11))}),
    ("rightlooking_unfused", "imogp_m2_M1450", {"chain_fused": 0}, {"chol": "rightlooking", "ob": 1, "fused": ()}),
    ("rightlooking_fused_all_w2", "imogp_m2_M1450", {"chain_fused": 2, "outer_block": 2},
     {"chol": "rightlooking", "ob": 2, "fused": tuple(range(11)), "upper_block_update": True}),
    ("no_lookahead", "imogp_m2_M1450", {"lookahead": 0}, {"chol": "chain_all", "groups": 1, "upper_block_update": True}),
]
# 3. row chunks of N = 850 (7 tile rows): 3 -> chunks of 3, 3, 1 rows with 3 splits, two of them empty in the last chunk
CHUNKS = [1, 2, 3, 6, 7, 100]
CHUNK_EMPTY = {1: False, 2: True, 3: True, 6: True, 7: False, 100: False}
# 5. production scale
SCALE_CASES = [(k, z) for k in ("oilmm_m4_M1100", "imogp_m2_M1600") for z in OZ]


def _opts_oz(oz):
    S, bits = OZ[oz]
    return {"ozaki": S, "ozaki_bits": bits} if S else {}


def test_each_gpu_case_reaches_the_branch_it_is_there_for():
    """Shrinking a case, or a change of a selection rule, must fail here instead of quietly dropping a branch."""
    assert [schedule(*shape(k), {})["mt"] for k in dict(GRAD_CASES)] == [3, 5, 6]
    runs = {(k, ob) for k, ob in GRAD_CASES if schedule(*shape(k), {"outer_block": ob})["upper_block_update"]}
    assert runs == {(k, 2) for k in dict(GRAD_CASES)} | {("imogp_product_M520", 3), ("oilmm_ard_D2_M700", 3)}, runs
    paths = set()
    for cid, key, opts, want in SCHED_CASES:
        s = schedule(*shape(key), opts)
        for k, v in want.items():
            assert s[k] == v, (cid, k, s[k], v)
        paths.add((s["chol"], s["groups"], s["fused"], s["ob"]))
    assert len(paths) == len(SCHED_CASES)  # every option set lands on a path of its own
    N, M, m = shape("oilmm_m14_M900")
    assert (math.ceil(M / T) - 1) * m > CHAIN_MAX_TILES  # grouped streams by the rule, not by an option
    N, M, m = shape("imogp_m2_M1450")
    assert m == 2 and M >= 11 * T + 1  # right-looking by the rule: mt >= 12
    assert {k for _, k, _, _ in SCHED_CASES} >= {"oilmm_m2_M800", "imogp_m6_M800"}  # both models at M = 700-900
    N, M, m = shape("oilmm_product_N850")
    assert math.ceil(N / T) == 7 and N % T
    for c in CHUNKS:
        s = schedule(N, M, m, {"vfe_chunk": c})
        assert s["empty_splits"] == CHUNK_EMPTY[c], (c, s)
    assert schedule(N, M, m, {"vfe_chunk": 3})["splits"] == 3
    for key, oz in SCALE_CASES:
        s = schedule(*shape(key), _opts_oz(oz))
        assert s["int8_sweep"] == (oz != "off") and s["mt"] > 8, (key, oz, s)
    assert schedule(*shape("oilmm_m4_M1100"), _opts_oz("S7b8"))["int8_chol"]  # the int8 Cholesky of K(z, z) and Σ
    assert schedule(*shape("imogp_m2_M1600"), _opts_oz("S7b8"))["chol"] == "rightlooking"  # two factors of 13 tile rows stay on DMMA
    for key in dict(GRAD_CASES):  # test points: 3 tile rows, the last one ragged
        assert math.ceil(len(problem(key).xs) / T) == 3 and len(problem(key).xs) % T
    for key in dict(SCALE_CASES):  # 5 tile rows
        assert math.ceil(len(problem(key).xs) / T) == 5 and len(problem(key).xs) % T


# ------------------------------------------------------------------------------------------------ references (once per problem)
_PB = {}
_REF = {}


def problem(key):
    if key not in _PB:
        _PB[key] = PROBLEMS[key][0]()
    return _PB[key]


def reference(key, ndir=0, blocks=(), latents=()):
    """ELBO and marginals at the test points; `ndir` random all-block directions, one direction per entry of `blocks` (a tuple of
    block names) and per-parameter differences of the latents in `latents`, each with its bound."""
    if key not in _REF:
        pb = problem(key)
        val, (Mr, Vr) = vfe_oracle(pb.fs, pb.x, pb.z, pb.jitter, pb.s2, pb.y, pb.U, pb.S, pb.xs)
        _REF[key] = {"val": val, "M": Mr, "V": Vr, "dirs": [], "lat": {}}
    r = _REF[key]
    pb = problem(key)
    want = [random_direction(pb, 700 + k) for k in range(ndir)] + [random_direction(pb, 800 + k, b) for k, b in enumerate(blocks)]
    if len(r["dirs"]) < len(want):
        r["dirs"] = [(v, *directional_difference(pb, v)) for v in want]
    for i in latents:
        if i not in r["lat"]:
            r["lat"][i] = latent_differences(pb, i)
    return r


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def lmm():
    import lmm_b200

    yield lmm_b200
    _restore(lmm_b200.default_context())


def _restore(ctx):
    for k, v in DEFAULTS.items():
        ctx.set_option(k, v)
    ctx.set_option("ozaki", int(os.environ.get("LMM_OZAKI", "0")))  # the library default, or what the whole run was started with
    ctx.set_option("ozaki_bits", int(os.environ.get("LMM_OZAKI_BITS", "7")))


@contextlib.contextmanager
def options(lmm, opts):
    ctx = lmm.default_context()
    _restore(ctx)
    try:
        for k, v in opts.items():
            ctx.set_option(k, v)
        yield
    finally:
        _restore(ctx)


def run(lmm, pb, opts, grad=True):
    """(ELBO, gradient or None, marginal means, variances) of one VFE call with these options."""
    with options(lmm, opts):
        fx = _fx(lmm, pb.fs, pb.x, pb.p, pb.s2, pb.U, pb.S)
        approx = lmm.VFE(_xin(lmm, pb.z), pb.jitter)
        if grad:
            v, g = lmm.elbo_and_gradient(approx, fx, pb.y, with_grad_y=True)
        else:
            v, g = lmm.elbo(approx, fx, pb.y), None
        post = lmm.posterior(approx, fx, pb.y)
        Mg, Vg = lmm.mean_and_var(post(lmm.MOInputIsotopicByOutputs(_xin(lmm, pb.xs), pb.p), pb.s2))
    return v, g, Mg, Vg


def check_value_and_marginals(ref, v, Mg, Vg, rtol=1e-9):
    assert abs(v - ref["val"]) <= rtol * abs(ref["val"]), (v, ref["val"])
    assert_isapprox(Mg, ref["M"], rtol, what="mean")
    assert_isapprox(Vg, ref["V"], rtol, what="var")


def check_directions(g, pb, ref):
    for n, (v, fd, bound) in enumerate(ref["dirs"]):
        assert_directional(g, pb, v, fd, bound, what=n)


@pytest.mark.gpu
@pytest.mark.parametrize("key,ob", GRAD_CASES)
def test_gradient_past_two_inducing_tiles(lmm, key, ob):
    """Every gradient block at 3, 5 and 6 inducing tiles: per-parameter differences of every latent's hyper-parameters and mean,
    and one direction each for σ², y, U and S (a random direction over all of y sees an error in any entry)."""
    pb = problem(key)
    ref = reference(key, blocks=(("sigma2",), ("y",)) + ((("U",), ("S",)) if pb.oilmm else ()), latents=range(len(pb.fs)))
    v, g, Mg, Vg = run(lmm, pb, {"outer_block": ob})
    check_value_and_marginals(ref, v, Mg, Vg)
    for i in range(len(pb.fs)):
        assert_latent_differences(g, pb, i, ref["lat"][i])
    check_directions(g, pb, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("cid,key,opts", [c[:3] for c in SCHED_CASES], ids=[c[0] for c in SCHED_CASES])
def test_factor_schedules(lmm, cid, key, opts):
    pb = problem(key)
    ref = reference(key, ndir=1 if len(pb.fs) > 6 else 2)
    v, g, Mg, Vg = run(lmm, pb, opts)
    check_value_and_marginals(ref, v, Mg, Vg)
    check_directions(g, pb, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", CHUNKS)
def test_row_chunks_and_empty_splits(lmm, chunk):
    """Row chunks of 1 to 7 tile rows of N = 850 against one chunk (only the order of the chunk sums differs: value and marginals
    to 1e-12, the gradient, whose cotangents pass through Σ⁻¹ and Lz⁻¹, to 1e-11 as in test_vfe.py) and against the oracle."""
    key = "oilmm_product_N850"
    pb = problem(key)
    ref = reference(key, ndir=1)
    one, g1, M1, V1 = run(lmm, pb, {})
    v, g, Mg, Vg = run(lmm, pb, {"vfe_chunk": chunk})
    assert abs(v - one) <= 1e-12 * abs(one), (v, one)
    assert_isapprox(Mg, M1, 1e-12, what="mean")
    assert_isapprox(Vg, V1, 1e-12, what="var")
    for k in ("variance", "inv_lengthscale", "mean_const", "ard", "y", "U", "S", "sigma2"):
        assert_isapprox(g[k], g1[k], 1e-11, what=k)
    for a, b in zip(term_rows(g, pb.fs, pb.D), term_rows(g1, pb.fs, pb.D)):
        assert_isapprox(a, b, 1e-11, what="terms")
    check_value_and_marginals(ref, v, Mg, Vg)
    check_directions(g, pb, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["oilmm_m16", "imogp_m16"])
def test_sixteen_latents(lmm, key):
    """16 latents with their own kernels and means: a mixed-up latent offset changes the value, the marginals and the gradient."""
    pb = problem(key)
    ref = reference(key, ndir=2, latents=(0, 7, 15))
    v, g, Mg, Vg = run(lmm, pb, {})
    check_value_and_marginals(ref, v, Mg, Vg)
    check_directions(g, pb, ref)
    for i in (0, 7, 15):
        assert_latent_differences(g, pb, i, ref["lat"][i])


@pytest.mark.gpu
@pytest.mark.parametrize("key,oz", SCALE_CASES)
def test_production_scale_and_the_int8_path(lmm, key, oz):
    """N = 12000 with 9 and 13 inducing tiles, on DMMA and on the int8 path (7 planes of 8 bits, 8 planes of 7 bits): the value
    and the marginals at 600 test points (the int8 sweep over 5 tile rows for Lz and L_Σ) to 1e-9, the gradient along one
    direction."""
    pb = problem(key)
    ref = reference(key, ndir=1)
    v, g, Mg, Vg = run(lmm, pb, _opts_oz(oz))
    check_value_and_marginals(ref, v, Mg, Vg)
    check_directions(g, pb, ref)
