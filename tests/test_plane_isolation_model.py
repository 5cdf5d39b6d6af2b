"""The plane-isolated operands of tests/digit_planes.py, checked on CPU: the construction gives exactly the intended digits,
and the numpy model of the split product keeps a single plane pair (k, l) exactly when k + l <= S - 1 and drops it to exactly
zero otherwise.  tests/test_gpu_oz_planes.py holds oz_gemm_kernel to the same statement."""
import numpy as np
import pytest

import digit_planes as dp
from test_split_scheme import split_digits, split_product


@pytest.mark.parametrize("S", [3, 4, 5, 6, 7])
def test_pure_values_have_one_digit(S):
    """Every plane k < S and every digit value, extremes included, splits into that one digit and nothing else."""
    for k in range(S):
        top = 126 if k == 0 else 127
        d = np.arange(-top, top + 1)
        dp.check_pure(dp.pure_values(d, k), d, k, S)
    # 127 in plane 0 is 0.5 of the scale: the power-of-two scale would double, so plane 0 stops at 126
    assert dp.pure_values(127, 0) == 0.5


@pytest.mark.parametrize("S", [3, 4, 5, 6, 7])
def test_saturated_value_is_a_fixed_point(S):
    planes = split_digits(np.array([dp.SATURATED, -dp.SATURATED]), 1.0, S, dp.R)
    want = [126] * S if S < 7 else [126] * 6 + [125]
    assert [int(p[0]) for p in planes] == want
    assert [int(p[1]) for p in planes] == [-d for d in want]
    # the anchors sit at plane-0 magnitude and leave the power-of-two scale at 1
    assert dp.pure_values(dp.ANCHOR_DIGIT, 0) < 0.5 and dp.pure_values(dp.ANCHOR_DIGIT, 0) >= 0.25
    assert dp.SATURATED < 0.5


@pytest.mark.parametrize("S", [3, 4, 5, 6, 7])
def test_split_product_isolates_each_plane_pair(S):
    """X~ row r in plane k, A row j in plane l: the model's Y[r, j] is the single pair's product where k + l <= S - 1 and
    exactly 0.0 where k + l >= S; the anchors (one column each, the partner's column zero) contribute nothing."""
    rng = np.random.RandomState(S)
    n = 96
    kx, la = np.arange(S), np.arange(S)
    dx = np.stack([dp.random_digits(rng, n, k, zero_fraction=0.0) for k in kx])
    da = np.stack([dp.random_digits(rng, n, l, zero_fraction=0.0) for l in la])
    x = np.stack([dp.pure_values(dx[i], k) for i, k in enumerate(kx)])
    a = np.stack([dp.pure_values(da[j], l) for j, l in enumerate(la)])
    # anchors: X~ in column 0 (A zero there), A in column 1 (X~ zero there)
    x[:, :2] = 0.0
    a[:, :2] = 0.0
    x[0, 0] = dp.pure_values(dp.ANCHOR_DIGIT, 0)
    a[:, 1] = dp.pure_values(dp.ANCHOR_DIGIT, 0)
    dx[:, :2] = 0
    da[:, :2] = 0
    y, px, pa, _ = split_product(x, a, S, dp.R)
    for k in range(S):   # the construction survives the model's own scaling
        np.testing.assert_array_equal(px[k][:, 2:], np.where(kx[:, None] == k, dx, 0)[:, 2:])
        np.testing.assert_array_equal(pa[k][:, 2:], np.where(la[:, None] == k, da, 0)[:, 2:])
    want, want_abs = dp.exact_product(np.stack(px), np.stack(pa), S, 1.0)
    for k in kx:
        for l in la:
            single = float(np.dot(dx[k].astype(np.float64), da[l].astype(np.float64)))
            if k + l >= S:
                assert y[k, l] == 0.0 and want[k, l] == 0.0, (k, l, y[k, l])
            else:
                exact = float(np.longdouble(single) / np.longdouble(dp.R) ** (k + l + 2))
                assert single != 0.0
                assert want[k, l] == exact
                assert abs(y[k, l] - exact) <= (S + 4) * dp.U * abs(exact), (k, l, y[k, l], exact)
    dp.assert_exact(y, want, want_abs, S + 4, "numpy model", zero=np.add.outer(kx, la) >= S)


def test_exact_product_matches_integer_sums():
    """The reference against Python integers and fractions on a small random case (every pair present)."""
    from fractions import Fraction
    rng = np.random.RandomState(7)
    S = 4
    P = rng.randint(-127, 128, size=(S, 3, 50))
    Q = rng.randint(-127, 128, size=(S, 2, 50))
    scale = np.array([[0.5, 4.0]])
    want, want_abs = dp.exact_product(P, Q, S, scale)
    for r in range(3):
        for c in range(2):
            tot = Fraction(0)
            for k in range(S):
                for l in range(S - k):
                    tot += Fraction(int(np.dot(P[k, r], Q[l, c])), dp.R ** (k + l + 2))
            tot *= Fraction(scale[0, c])
            assert abs(Fraction(want[r, c]) - tot) <= abs(tot) * Fraction(1, 2 ** 53)
    assert np.all(want_abs >= np.abs(want))
