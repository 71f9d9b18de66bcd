"""Digit planes written by the panel TRSM of the int8 Cholesky (csrc/gemm.cu: gemm_tile_kernel_v2<TRSM, 32, true>, option
"trsm_slice") against the separate slice launch (ozaki_slice_kernel): the planes, first-plane bytes and skipped all-zero tiles are
the same bytes, so the factor, alpha and logpdf are bit-identical.  Enveloped factors (OILMM eval: a band narrower than a tile,
Matern52, SE + Periodic) and dense ones (potrf_batched), both radices, streams 1 and 4, block widths 1, 2 and 4, N a multiple of
128 and not."""
import os

import numpy as np
import pytest

from test_envelope_cholesky import build
from test_ozaki_gpu import spd
from tools.ozaki_digits import first_planes

pytestmark = pytest.mark.gpu
T = 128


@pytest.fixture()
def lmm():
    import lmm_b200

    yield lmm_b200
    ctx = lmm_b200.default_context()
    ctx.set_option("ozaki", int(os.environ.get("LMM_OZAKI", "0")))
    ctx.set_option("ozaki_bits", int(os.environ.get("LMM_OZAKI_BITS", "7")))
    ctx.set_option("trsm_slice", 1)
    ctx.set_option("outer_block", 0)
    ctx.set_option("streams", 4)


def setup(ctx, S, bits, width, streams):
    ctx.set_option("ozaki", S)
    ctx.set_option("ozaki_bits", bits)
    ctx.set_option("outer_block", width)
    ctx.set_option("streams", streams)


@pytest.mark.parametrize("N", [4096, 4000])
@pytest.mark.parametrize("width", [1, 2, 4])
@pytest.mark.parametrize("streams", [1, 4])
@pytest.mark.parametrize("S,bits", [(7, 8), (8, 7)])
def test_enveloped_factor_is_bit_identical(lmm, S, bits, streams, width, N):
    ctx = lmm.default_context()
    setup(ctx, S, bits, width, streams)
    fx, _, y = build(lmm, "oilmm", N, "sorted")
    out = {}
    for ts in (0, 1):
        ctx.set_option("trsm_slice", ts)
        post, lp = lmm.posterior(fx, y, with_logpdf=True)
        lat = post.f.fs
        out[ts] = (lp, [lat[i].C for i in range(len(lat))], [lat[i]._export()[1] for i in range(len(lat))])
    assert out[0][0] == out[1][0]
    for i, (L0, L1) in enumerate(zip(out[0][1], out[1][1])):
        assert np.array_equal(L0, L1), i
    for i, (a0, a1) in enumerate(zip(out[0][2], out[1][2])):
        assert np.array_equal(a0, a1), i
    if width == 1 and streams == 1 and N % T == 0:
        # the batch has tiles outside the envelope and tiles inside it whose digits are all zero (no planes written): the medium
        # band of latent 1 (the narrow band of latent 0 is narrower than a tile, so its envelope tiles all reach the diagonal)
        L = out[1][1][1]
        nt = -(-N // T)
        fp = first_planes(L, S, bits)
        inside = [(I, k) for I in range(nt) for k in range(I + 1) if np.any(L[I * T:(I + 1) * T, k * T:(k + 1) * T])]
        assert len(inside) < nt * (nt + 1) // 2
        assert any(fp[I, k] == S for I, k in inside)


@pytest.mark.parametrize("N", [1700, 2048])
@pytest.mark.parametrize("width", [1, 2, 4])
@pytest.mark.parametrize("streams", [1, 4])
@pytest.mark.parametrize("S,bits", [(7, 8), (8, 7)])
def test_dense_factor_is_bit_identical(lmm, S, bits, streams, width, N):
    ctx = lmm.default_context()
    setup(ctx, S, bits, width, streams)
    A = spd(N, 5, seed=N + width)  # batch >= 3: the batched left-looking schedule
    out = {}
    for ts in (0, 1):
        ctx.set_option("trsm_slice", ts)
        L, ld, info = lmm.potrf_batched(A)
        assert not info.any()
        out[ts] = (np.array(L), np.array(ld))
    assert np.array_equal(out[0][0], out[1][0])
    assert np.array_equal(out[0][1], out[1][1])
