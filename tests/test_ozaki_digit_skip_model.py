"""CPU side of the int8 update's digit-plane filter (csrc/ozaki.cu): each pass of ozaki_update_kernel walks only its member k-tiles,
those whose first nonzero digit planes tp(I,k) + tp(J,k) leave a nonzero pair in the pass.  The barrier protocol model
(tools/ozaki_protocol_model.py) with member lists that are empty (pass A), a single k-tile, or have gaps; and the host copy of the
slicing rule (tools/ozaki_digits.py) that the GPU tests and tools/bench_digit_skip.py recount with."""
import numpy as np
import pytest

from tools.ozaki_digits import digits, first_planes, update_products
from tools.ozaki_protocol_model import Violation, explore


@pytest.mark.parametrize("members_a,members_b,nst_a,nst_b", [
    ([], [0, 2], 6, 4),          # pass A empty, pass B not
    ([], [3], 6, 4),             # ... with a single member
    ([], [1, 4, 5], 6, 3),       # ... and a single issuer in pass B
    ([2], [2], 6, 4),            # one member in both passes
    ([0, 5], [0, 3, 5], 6, 4),   # gaps, pass A a strict subset of pass B
    ([1, 6], [1, 2, 6, 9], 4, 2),
])
def test_member_walk_is_safe_and_live(members_a, members_b, nst_a, nst_b):
    res = explore(nst_a=nst_a, nst_b=nst_b, members_a=members_a, members_b=members_b)
    assert res["final_states"] == 1 and res["states"] > 500


def test_empty_pass_without_its_rule_deadlocks():
    """The odd issuer waiting for an init_done nobody arrives on: what the kernel's empty-pass branch avoids."""
    with pytest.raises(Violation, match="deadlock"):
        explore(members_a=[], members_b=[0, 2], empty_pass_fix=False)


@pytest.mark.parametrize("S,bits", [(7, 8), (8, 8), (7, 7), (8, 7), (6, 7)])
def test_digits_reconstruct_and_zero_rule(S, bits):
    """Digits recombine to round(y R^(S-1)) / R^(S-1); an entry has only zero digits iff it rounds to 0 on the finest grid, the rule
    the slice kernel's all-zero pre-pass uses."""
    rng = np.random.default_rng(S * 10 + bits)
    R = 2.0 ** bits
    y = np.concatenate([rng.uniform(-63.9, 63.9, 2000), rng.standard_normal(2000) * 2.0 ** rng.integers(-60, 5, 2000),
                        np.ldexp(np.array([0.5, -0.5, 0.5000001, 1.0, 0.49]), -bits * (S - 1))])
    q = digits(y, S, bits)
    rec = sum(q[t].astype(np.float64) * R ** -t for t in range(S))
    fine = np.rint(y * R ** (S - 1))
    np.testing.assert_array_equal(rec * R ** (S - 1), fine)
    assert np.array_equal((q != 0).any(axis=0), fine != 0)
    if bits == 8:
        assert q[1:].min() >= -128 and q[1:].max() <= 127
    else:
        assert np.abs(q).max() <= 64


def test_first_planes_and_products_of_a_banded_factor():
    """An SE factor decays along its rows: far tiles slice to late planes or all-zero digits, and the pass sets shrink accordingly."""
    N, S, bits = 2048, 7, 8
    x = np.linspace(0, 60, N)
    C = np.exp(-0.5 * (x[:, None] - x[None, :]) ** 2)
    C[np.diag_indices_from(C)] += 0.1
    L = np.linalg.cholesky(C)
    fp = first_planes(L, S, bits)
    nt = N // 128
    assert (np.diag(fp) == 0).all()
    assert fp[nt - 1, 0] == S  # far below the grid
    r = update_products(fp, None, S, bits)
    assert 0 < r["pass_a"] <= r["pass_b"] < r["envelope"]
    assert r["ctas_pass_a_empty"] > 0
