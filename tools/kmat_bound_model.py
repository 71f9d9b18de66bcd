"""NumPy model of the kernel-matrix build's provable envelope (csrc/kmat.cu: kmat_bound_kernel) and of the device arithmetic of
the entries it lets the build skip (stage_points + kmat_tile_body + kappa_eval), for tests/test_kmat_bound_model.py.

fma(x, y, z) is emulated exactly (one rounding of the exact x*y + z through fractions); fma(-2, p, t) is one rounding of t - 2p,
which NumPy's t - 2.0 * p is (2p is exact)."""
from fractions import Fraction

import numpy as np

SQRT3, SQRT5 = 1.7320508075688772, 2.23606797749979


def fma(x, y, z):
    return float(Fraction(x) * Fraction(y) + Fraction(z))


def kappa_zero_d2(kind):
    g = 1.0 + 2.0 ** -40
    return {0: 1416.0 * g, 1: (708.0 / SQRT3) ** 2 * g, 2: (708.0 / SQRT5) ** 2 * g, 3: 708.0 * 708.0 * g}.get(kind, np.inf)


def bound(xs, tile, kind):
    """fb[I] for scaled points xs [N][D] (kmat_bound_kernel, with `tile` points per tile)."""
    N, D = xs.shape
    nt = -(-N // tile)
    lo = np.array([xs[T * tile:(T + 1) * tile].min(0) for T in range(nt)])
    hi = np.array([xs[T * tile:(T + 1) * tile].max(0) for T in range(nt)])
    q = np.maximum(lo * lo, hi * hi).sum(1)
    rel = (D + 4) * 2.0 ** -50
    thr = kappa_zero_d2(kind)
    fb = np.zeros(nt, dtype=np.int64)
    for I in range(nt):
        f = 0
        while f < I:
            g = np.maximum(0.0, np.maximum(lo[I] - hi[f], lo[f] - hi[I]))
            g2 = 0.0
            for k in range(D):
                g2 = fma(g[k], g[k], g2)
            if not (g2 * (1.0 - rel) - rel * (q[I] + q[f]) > thr):
                break
            f += 1
        fb[I] = f
    return fb


def device_d2(a, b, form):
    """The squared distance the build computes for scaled points a, b (D coordinates)."""
    D = len(a)
    if form == 1:
        d2 = 0.0
        for k in range(D):
            df = a[k] - b[k]
            d2 = fma(df, df, d2)
        return d2
    sa = sb = 0.0
    for k in range(D):
        sa = fma(a[k], a[k], sa)
        sb = fma(b[k], b[k], sb)
    t = sa + sb
    if D == 1:
        d2 = t - 2.0 * (a[0] * b[0])  # fma(-2, a0 * b0, t)
    else:
        dot = 0.0
        for k in range(D):
            dot = fma(a[k], b[k], dot)
        d2 = t - 2.0 * dot
    return d2 if d2 > 0.0 else 0.0


def device_kappa_is_zero(kind, d2):
    """kappa_eval(kind, 1, d2) == 0.0 exactly (exp_nonpos flushes arguments below -708)."""
    if kind == 0:
        return -0.5 * d2 < -708.0
    d = np.sqrt(d2)
    s = {1: SQRT3 * d, 2: SQRT5 * d, 3: d}[kind]
    return -s < -708.0
