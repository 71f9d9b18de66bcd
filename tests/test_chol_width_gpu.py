"""Block width of the batched int8 Cholesky on enveloped factors (csrc/host_chol.cu: chol_factor_stream).  Without a user-set
"outer_block" an enveloped factor of at least 64 tile rows takes width 1, so every update of column J by the k-tiles k < J
(J >= ozaki_min_k) runs in the int8 kernel; smaller ones keep width 2, and a user-set width keeps the in-block updates on DMMA.
With "ozaki_time" the library reports the 128^3 tile products its int8 launches ran: per tile (I, J) of the wide update of block
column [s0, s1), max(0, s0 - max(env[I], env[J])) -- checked at user-set widths 1 and 2 and at the default width on both sides of
the size rule, together with the logpdf against the oracle."""
import os

import numpy as np
import pytest

from test_envelope_cholesky import T, build, reference

pytestmark = pytest.mark.gpu


@pytest.fixture()
def lmm():
    import lmm_b200

    yield lmm_b200
    ctx = lmm_b200.default_context()
    ctx.set_option("ozaki", int(os.environ.get("LMM_OZAKI", "0")))
    ctx.set_option("ozaki_bits", int(os.environ.get("LMM_OZAKI_BITS", "7")))
    ctx.set_option("ozaki_time", 0)
    ctx.set_option("outer_block", 0)
    ctx.set_option("streams", 4)


def int8_products(envs, nt, ob, S, min_k=4):
    want = 0
    for s0 in range(ob, nt, ob):
        if s0 < min_k or s0 * T * S * 16384 >= 2 ** 31:
            continue
        for J in range(s0, min(s0 + ob, nt)):
            for I in range(J, nt):
                kb = np.maximum(envs[:, I], envs[:, J])
                want += int(np.maximum(s0 - kb, 0).sum())
    return want


CASES = [(k, o, 4096, w) for k in ("oilmm", "imogp") for o in ("sorted", "shuffled") for w in (1, 2)] + [
    ("oilmm", "sorted", 4096, 0), ("oilmm", "sorted", 8192, 0)]


@pytest.mark.parametrize("kind,order,N,width", CASES)
def test_int8_update_runs_the_envelope_tile_products_at_the_block_width(lmm, kind, order, N, width):
    ctx = lmm.default_context()
    S, bits = 7, 8
    ctx.set_option("streams", 1)
    ctx.set_option("ozaki", S)
    ctx.set_option("ozaki_bits", bits)
    ctx.set_option("outer_block", width)
    ctx.set_option("ozaki_time", 1)
    x, xs, y, lp_ref, _, _, _, envs = reference(kind, N, order)
    fx, _, y = build(lmm, kind, N, order)
    ctx.last_timings()  # drop what earlier calls recorded
    lp = lmm.logpdf(fx, y)
    tm = ctx.last_timings()
    assert abs(lp - lp_ref) <= 1e-9 * abs(lp_ref), (lp, lp_ref)
    nt = envs.shape[1]
    ob = width or (1 if nt >= 64 else 2)
    want = int8_products(envs, nt, ob, S)
    assert 0 < want < int8_products(np.zeros_like(envs), nt, ob, S)
    assert tm[5] == want, (tm[5], want, ob)
