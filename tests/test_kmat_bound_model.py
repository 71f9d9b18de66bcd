"""CPU model of the kernel-matrix build's provable envelope (tools/kmat_bound_model.py, csrc/kmat.cu: kmat_bound_kernel): on
random and adversarial 1-D and 2-D inputs -- point pairs a few ulps either side of each kind's flush point -- every entry of a
tile the bound lets the build skip evaluates to exactly 0 in the device arithmetic, and the bound never exceeds the value-based
envelope the build records."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import kmat_bound_model as km  # noqa: E402

TILE = 4  # the bound's logic does not depend on the tile size; small tiles keep the exact-arithmetic emulation fast
KINDS = [0, 1, 2, 3]


def flush_distance(kind):
    """The distance |a - b| at which kind's entries flush to 0."""
    return {0: np.sqrt(1416.0), 1: 708.0 / km.SQRT3, 2: 708.0 / km.SQRT5, 3: 708.0}[kind]


def check(xs, kind, form):
    fb = km.bound(xs, TILE, kind)
    nt = len(fb)
    env = np.zeros(nt, dtype=np.int64)
    for I in range(nt):
        env[I] = I
        for k in range(I):
            zero = all(km.device_kappa_is_zero(kind, km.device_d2(a, b, form))
                       for a in xs[I * TILE:(I + 1) * TILE] for b in xs[k * TILE:(k + 1) * TILE])
            if k < fb[I]:
                assert zero, (kind, form, I, k)
            if not zero:
                env[I] = k
                break
    assert np.all(fb <= env)
    return fb


def adversarial_1d(kind, rng, offset_ulps):
    """Tiles of points straddling the flush distance: tile 2j + 1 sits at distance ~flush (+- a few ulps) from tile 2j."""
    d = flush_distance(kind)
    pts = []
    base = 0.0
    for j in range(4):
        a = base + rng.uniform(-1e3, 1e3) * (j % 2)
        b = a + d
        for u in offset_ulps:
            pts.append(a)
        for u in offset_ulps:
            pts.append(np.nextafter(b, np.inf) if u > 0 else b)
            b = b + u * np.spacing(b)
        base = b + 3 * d
    return np.array(pts, dtype=np.float64)[:, None]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("form", [0, 1])
def test_skipped_tiles_are_exact_zeros_1d(kind, form):
    rng = np.random.default_rng(kind)
    for ulps in ([-3, -1, 1, 3], [0, 2, 4, 8], [-8, -4, -2, 0]):
        check(adversarial_1d(kind, rng, ulps), kind, form)
    x = np.sort(rng.uniform(0, 40 * flush_distance(kind), 12 * TILE))[:, None]
    fb = check(x, kind, form)
    assert fb.max() > 0  # the random case skips something: the check above is not vacuous
    check(rng.permutation(x), kind, form)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("form", [0, 1])
def test_skipped_tiles_are_exact_zeros_2d(kind, form):
    rng = np.random.default_rng(10 + kind)
    d = flush_distance(kind)
    x = rng.uniform(0, 20 * d, (10 * TILE, 2))
    x = x[np.argsort(x[:, 0])]
    fb = check(x, kind, form)
    assert fb.max() > 0
    # pairs on the diagonal at the flush distance, a few ulps apart, far from the origin (large |a|² + |b|²)
    pts = []
    for j in range(3):
        c = 1e4 * (j + 1)
        for u in (-2, -1, 1, 2):
            pts.append([c, c])
        for u in (-2, -1, 1, 2):
            e = d / np.sqrt(2.0) + u * np.spacing(d)
            pts.append([c + e + 5 * d * j, c + e])
    check(np.array(pts), kind, form)


def test_rational_quadratic_is_never_skipped():
    x = np.linspace(0, 1e6, 8 * TILE)[:, None]
    assert not km.bound(x, TILE, 4).any()
