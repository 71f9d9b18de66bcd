"""GPU side of the int8 update's digit-plane filter (csrc/ozaki.cu): the slice kernel records each factor tile's first nonzero digit
plane, and the update skips the k-tiles whose digit products are all exactly zero -- whole CTAs, or pass A alone.  OILMM at
N = 4096 with banded SE, Matern52 and dense latents, sorted and tile-shuffled inputs, 7 / 8 planes of 7 / 8 bits, 1 and 4 streams:
logpdf and marginals against the oracle at 1e-9, the factors against the DMMA path, and -- from host digits of the returned factors
-- that CTAs with an empty pass A and a non-empty pass B did run."""
import numpy as np
import pytest

from _tol import assert_isapprox, relnorm
from test_envelope_cholesky import build, lmm, reference  # noqa: F401  (lmm: the fixture that restores the options)
from tools.ozaki_digits import first_planes, update_products

pytestmark = pytest.mark.gpu

# factor against the DMMA path: the truncation of each digit scheme, amplified by the dense SE latent here, which is worse conditioned
# than the random SPD matrices of test_ozaki_gpu.py (measured for it: 8 planes of 8 bits 1.6e-13, 7 planes of 7 bits 3.1e-11)
TOL = {(8, 7): 1e-12, (7, 7): 2e-10, (7, 8): 1e-12, (8, 8): 1e-12}


@pytest.mark.parametrize("streams", [1, 4])
@pytest.mark.parametrize("order", ["sorted", "shuffled"])
@pytest.mark.parametrize("S,bits", [(7, 8), (8, 8), (7, 7), (8, 7)])
def test_digit_skip_matches_oracle_and_dmma(lmm, S, bits, order, streams):  # noqa: F811
    ctx = lmm.default_context()
    ctx.set_option("streams", streams)
    N = 4096
    x, xs, y, lp_ref, M_ref, V_ref, _, envs = reference("oilmm", N, order)
    fx, Oxs, y = build(lmm, "oilmm", N, order)
    ctx.set_option("ozaki", 0)
    post0 = lmm.posterior(fx, y)
    L0 = [f.C for f in post0.f.fs]
    ctx.set_option("ozaki", S)
    ctx.set_option("ozaki_bits", bits)
    post, lp = lmm.posterior(fx, y, with_logpdf=True)
    assert abs(lp - lp_ref) <= 1e-9 * abs(lp_ref), (lp, lp_ref)
    M, V = lmm.mean_and_var(post(Oxs, 0.1))
    assert_isapprox(M, M_ref, 1e-9, "posterior mean")
    np.testing.assert_allclose(V, V_ref, rtol=1e-9)
    empty_a = 0
    for i, f in enumerate(post.f.fs):
        L1 = f.C
        e = relnorm(L1, L0[i])
        assert e < TOL[(S, bits)], (i, e)
        r = update_products(first_planes(L1, S, bits), envs[i], S, bits)
        assert r["pass_b"] <= r["envelope"]
        empty_a += r["ctas_pass_a_empty"]
    assert empty_a > 0  # the empty-pass-A branch of the kernel ran
