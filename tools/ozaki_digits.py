"""Host copy of the int8 slicing rule of csrc/ozaki.cu (ozaki_slice_kernel) and of the k-tile filter of ozaki_update_kernel: per
128 x 128 tile (I, k) of a factor, the first digit plane with a nonzero digit (S when every digit is zero), and which products of the
left-looking int8 update then add something to the int32 sums.  Used to recount, from a returned factor, what the kernel skipped."""
import numpy as np

T = 128


def row_scales(L):
    """2^(E_i - 6) with 2^E_i > ||L(i,:)||_2 = sqrt(A_ii) (the kernel takes E_i from the diagonal of A before factoring; the two agree
    unless sqrt(A_ii) is within rounding of a power of two)."""
    nrm = np.sqrt(np.einsum("ij,ij->i", L, L))
    e = np.where(nrm > 0, np.floor(np.log2(np.where(nrm > 0, nrm, 1.0))).astype(np.int64) + 1, 0)
    return np.ldexp(1.0, e - 6)


def digits(y, S, bits):
    """Digit planes [S, ...] (int64) of y = L / row scale, bit for bit as the slice kernel forms them."""
    y = np.asarray(y, dtype=np.float64)
    q = np.empty((S,) + y.shape, dtype=np.int64)
    if bits == 8:  # one rounding to a 64-bit integer, balanced digits in [-128, 127] from the bottom, the top plane keeps the rest
        X = np.rint(y * 2.0 ** (8 * (S - 1))).astype(np.int64)
        for t in range(S - 1, 0, -1):
            q[t] = ((X + 128) & 255) - 128
            X = (X - q[t]) >> 8
        q[0] = X
        return q
    v = y.copy()  # radix 128: round-to-nearest remainders, scaled by 128 each plane (exact)
    for t in range(S):
        r = np.rint(v)
        q[t] = r.astype(np.int64)
        v = (v - r) * 128.0
    return q


def first_planes(L, S, bits, scale=None):
    """fp[I, k] for the lower tiles of the N x N factor L (N a multiple of 128): the first plane with a nonzero digit, S if none."""
    N = L.shape[0]
    nt = N // T
    sc = row_scales(L) if scale is None else scale
    fp = np.full((nt, nt), S, dtype=np.int64)
    for I in range(nt):
        y = L[I * T:(I + 1) * T, :(I + 1) * T] / sc[I * T:(I + 1) * T, None]
        nz = (digits(y, S, bits) != 0).reshape(S, T, I + 1, T).any(axis=(1, 3))  # [plane, k]
        fp[I, :I + 1] = np.where(nz.any(axis=0), nz.argmax(axis=0), S)
    return fp


def update_products(fp, env, S, bits, ob=2, min_k=4):
    """Walk the int8 wide updates of the batched left-looking schedule (block width ob, K >= min_k k-tiles, exact-int32 bound) for one
    factor.  Returns tile products inside the envelope, those in the kernel's pass B set (fp[I,k] + fp[J,k] <= S - 1, i.e. nonzero in
    int32), those in its pass A set (sum <= min(S, 4) - 1), the CTAs (I, J) the kernel runs at all (some pass B member), and those
    among them with an empty pass A."""
    nt = fp.shape[0]
    env = np.zeros(nt, dtype=np.int64) if env is None else np.asarray(env)
    nsA = min(S, 4)
    out = {"envelope": 0, "pass_b": 0, "pass_a": 0, "ctas": 0, "ctas_pass_a_empty": 0}
    for s0 in range(ob, nt, ob):
        if s0 < min_k or s0 * T * S * (16384 if bits == 8 else 4096) >= 2 ** 31:
            continue
        for J in range(s0, min(s0 + ob, nt)):
            for I in range(J, nt):
                kb = max(env[I], env[J])
                if kb >= s0:
                    continue
                s = fp[I, kb:s0] + fp[J, kb:s0]
                nb, na = int(np.sum(s <= S - 1)), int(np.sum(s <= nsA - 1))
                out["envelope"] += s0 - kb
                out["pass_b"] += nb
                out["pass_a"] += na
                out["ctas"] += nb > 0
                out["ctas_pass_a_empty"] += nb > 0 and na == 0
    return out
