#!/usr/bin/env python
"""NumPy model of the integer-slice (Ozaki) arithmetic of csrc/ozaki.cu -- row scales, digit-plane extraction (radix 128 by
round-to-nearest remainders, radix 256 by exact 64-bit carries), the exact int32 plane products, their FP64 recombination -- with the
same formulas and the same operation order as the CUDA kernels.  Test infrastructure (tests/test_ozaki_model.py, CPU): digit ranges,
exactness of the extraction, the int32 overflow bound, the truncation error of the recombined product."""
import numpy as np


def row_scale(diag):
    """2^(E - 6) with 2^E > sqrt(A_ii)  (ozaki_scale_kernel)."""
    e = np.floor(np.log2(np.sqrt(diag))).astype(np.int64) + 1
    # ilogb semantics: exact powers of two map to their exponent
    e = np.where(np.exp2(e - 1) > np.sqrt(diag), e - 1, e)
    return np.exp2((e - 6).astype(np.float64))


def slice_planes(L, scale, S, bits):
    """L: (rows, K) float64, scale: (rows,).  Returns int8 planes (S, rows, K) with L ~ scale * sum_t q_t * radix^-t."""
    y = L / scale[:, None]  # |y| <= 64 (1 + eps): exact (power-of-two scale)
    planes = np.zeros((S,) + L.shape, dtype=np.int64)
    if bits == 7:
        v = y.copy()
        for t in range(S):
            q = np.rint(v)  # (the kernel rounds by the 1.5 * 2^52 shift: the same round-to-nearest-even)
            planes[t] = q.astype(np.int64)
            v = (v - q) * 128.0  # exact
    else:
        X = np.rint(y * 2.0 ** (8 * (S - 1))).astype(np.int64)
        for t in range(S - 1, 0, -1):
            q = ((X + 128) & 255) - 128
            planes[t] = q
            X = (X - q) >> 8
        planes[0] = X
    assert planes.min() >= -128 and planes.max() <= 127
    return planes.astype(np.int8)


def reconstruct(planes, scale, bits):
    S = planes.shape[0]
    radix = float(1 << bits)
    acc = np.zeros(planes.shape[1:])
    for t in range(S - 1, -1, -1):
        acc = acc / radix + planes[t].astype(np.float64)
    return acc * scale[:, None]


def product(pa, sa, pb, sb, bits):
    """sum_k A(i,k) B(j,k) from the planes: exact int32 sums per d = t + u < S (two passes: d < 4, d >= 4), Horner in 1/radix, scales."""
    S = pa.shape[0]
    radix = float(1 << bits)
    acc = [np.zeros((pa.shape[1], pb.shape[1]), dtype=np.int64) for _ in range(S)]
    for t in range(S):
        for u in range(S - t):
            acc[t + u] += pa[t].astype(np.int64) @ pb[u].astype(np.int64).T
    for a in acc:
        assert np.abs(a).max() < 2 ** 31  # what the int32 accumulators in TMEM must hold
    out = np.zeros(acc[0].shape)
    for lo, hi, pre in ((0, min(S, 4), 1.0), (4, S, radix ** -4)):
        if hi <= lo:
            continue
        h = acc[hi - 1].astype(np.float64)
        for d in range(hi - 2, lo - 1, -1):
            h = h / radix + acc[d].astype(np.float64)
        out += h * (sa[:, None] * pre) * sb[None, :]
    return out


def int32_bound_ok(K, S, bits):
    """the host's check (host_chol.cu: ozaki_wide): pairs per accumulator <= S, each product <= (largest digit)^2."""
    return K * S * (16384 if bits == 8 else 4096) < 2 ** 31


def issue_order(S, pas):
    """The MMAs of one K quarter of pass `pas` in the order oz_issue_quarter<S, PASS> issues them: (t, u, accumulator, collector mode)
    with mode 0 = plain, 1 = fill, 2 = use, 3 = lastuse (same loop bounds as the kernel)."""
    ns = S if pas else min(S, 4)
    dlo, dhi = (4, S - 1) if pas else (0, ns - 1)
    out = []
    for t in range(ns):
        ulo = max(dlo - t, 0)
        uhi = min(dhi - t, ns - 1)
        for u in range(ulo, uhi + 1):
            mode = 0 if uhi == ulo else (1 if u == ulo else (3 if u == uhi else 2))
            out.append((t, u, t + u - dlo, mode))
    return out


def stages(planes, ring=224 * 1024):
    """oz_stages(): stages of a pass in the 224 KB ring (even counts let the two issuing threads own alternate stages)."""
    n = ring // (2 * planes * 4096)
    return 6 if n >= 6 else (4 if n >= 4 else n)
