"""Operands with known digit planes for the split-integer engine (csrc/ozaki_i8.cuh), and the exact reference of its products.

oz_gemm_kernel multiplies int8 digit planes and adds the plane-pair products in int32 groups g = k + l, weighted R^-(g+2).
Relative to the leading term, group g weighs about R^-g, so a tolerance check on random data cannot see what happens to the
lowest groups.  The operands built here put every row (or column, or block) of an operand into ONE digit plane, so that an
output is a single plane pair (k, l): that pair's product is then the whole output, and a pair with k + l >= S is dropped, so
its outputs are exactly zero.

- `pure_values(d, k)`: binary64 values whose digit expansion is the single digit d in plane k (relative to a power-of-two
  scale of 1).  Dividing d by R in binary64 k + 1 times gives this for every S <= 7, k < S and |d| <= 127 (|d| <= 126 in
  plane 0, so that |v| < 0.5 keeps the scale); `check_pure` verifies it with the numpy restatement of the extraction.
- `SATURATED` = 126/253 is a fixed point of the extraction: its digits are 126 in every plane (the last may be 125).
- Anchors: X~ has one exponent, A, Y and the Gram matrix one per row or column.  An operand whose entries all sit in plane 3
  would be renormalised into plane 0, so every such row or column gets one `ANCHOR` entry at plane-0 magnitude, placed where
  the partner operand is zero so that it contributes no product.
- `exact_product`: the reference, from the digit planes read back from the device.  Each P_k Q_l^T is a float64 matmul of
  integers below 2^53 (exact); the weights and scales are applied in extended precision.
"""
import numpy as np

from test_split_scheme import split_digits

R = 254
ANCHOR_DIGIT = 100                 # plane-0 digit of the anchors: 100 / 254 = 0.39, so the power-of-two scale is 1
SATURATED = 126.0 / 253.0
U = 2.0 ** -53                     # unit roundoff of binary64

# digit count -> (precision mode, LCX_SPLIT_DIGITS override)
MODES = {3: ("fast", None), 4: ("fp64_split", "4"), 5: ("fp64_split5", None), 6: ("fp64_split", None), 7: ("fp64_split7", None)}


def cdiv(a, b):
    return -(-a // b)


def oz_kmax(S):
    """Longest contraction one int32 accumulator group may see (Layout::oz_kmax, csrc/host_session.cuh)."""
    return min(65536, ((1 << 31) // ((R // 2) ** 2 * S)) // 64 * 64)


def bn_max(S):
    return 128 if S <= 4 else 64


def tile_plan(m, S):
    """(n_tiles, bn) of the factor side: m split into equal tiles of a width that is a multiple of 16 (S <= 4) or 8."""
    bnm = bn_max(S)
    n_tiles = cdiv(m, bnm)
    step = 16 if bnm > 64 else 8
    return n_tiles, max(16, cdiv(cdiv(m, n_tiles), step) * step)


def gram_plan(n, m, S):
    """(full, rest, splits) of the Gram product (gram_plan, csrc/host_session.cuh); full = 0: the generic split-K plan."""
    n_tiles, m_tiles, clusters = cdiv(m, bn_max(S)), cdiv(n, 128), 148 // 2
    if n_tiles != 2 or n > oz_kmax(S):
        return 0, 0, 1
    full = (m_tiles // clusters) * clusters
    rest = m_tiles - full
    if full == 0 or rest == 0:
        return 0, 0, 1
    sp = max(1, min(clusters // rest, cdiv(n, 64) // 4))
    chunk = cdiv(cdiv(n, sp), 64) * 64
    return full, rest, cdiv(n, chunk)


def pure_values(d, k):
    """Binary64 values with the single digit d in plane k (scale 1)."""
    v = np.asarray(d, dtype=np.float64)
    for _ in range(k + 1):
        v = v / R
    return v


def random_digits(rng, shape, k, zero_fraction=0.1):
    """Nonzero digits of either sign over the whole range of plane k (|d| <= 126 in plane 0), some entries zero."""
    top = 126 if k == 0 else 127
    d = rng.randint(1, top + 1, size=shape) * rng.choice([-1, 1], size=shape)
    d[rng.random_sample(shape) < zero_fraction] = 0
    return d


def check_pure(values, digits, planes, S):
    """values (any shape) must split at scale 1 into `digits` in plane planes[...] and zero elsewhere."""
    values = np.asarray(values, dtype=np.float64)
    digits = np.broadcast_to(digits, values.shape)
    planes = np.broadcast_to(planes, values.shape)
    got = split_digits(values, 1.0, S, R)
    for k in range(S):
        want = np.where(planes == k, digits, 0)
        bad = np.flatnonzero(got[k] != want)
        assert bad.size == 0, "plane %d of %d: %d values split wrongly (first at %s)" % (k, S, bad.size, bad[:4])


def weights(S):
    """R^-(g+2) for g = 0 .. S-1 in extended precision (exact to far below binary64's rounding)."""
    return [np.longdouble(1) / np.longdouble(R) ** (g + 2) for g in range(S)]


def exact_product(P, Q, S, scale):
    """want[r, c] = scale[r, c] * sum_{k+l <= S-1} R^-(k+l+2) (P_k Q_l^T)[r, c] and want_abs (the same with |P_k|, |Q_l|).

    P: (S, M, K) integer digit planes of the M-side operand, Q: (S, Nc, K) of the factor side; `scale` broadcasts to
    (M, Nc).  Each P_k Q_l^T is a float64 matmul of integers whose partial sums stay below 2^53, so it is exact; only the
    rows of P_k and Q_l that are not all zero take part (the isolated operands are mostly zero in any one plane)."""
    S_, M, K = P.shape
    assert S_ == S and Q.shape[0] == S and Q.shape[2] == K
    assert K * 127 * 127 < 2 ** 53
    Nc = Q.shape[1]
    w = weights(S)
    acc = np.zeros((M, Nc), dtype=np.longdouble)
    acc_abs = np.zeros((M, Nc), dtype=np.longdouble)
    qs = []
    for l in range(S):
        cols = np.flatnonzero(Q[l].any(axis=1))
        qs.append((cols, Q[l][cols].astype(np.float64)))
    for k in range(S):
        rows = np.flatnonzero(P[k].any(axis=1))
        if rows.size == 0:
            continue
        pk = P[k][rows].astype(np.float64)
        for l in range(S - k):
            cols, ql = qs[l]
            if cols.size == 0:
                continue
            ix = np.ix_(rows, cols)
            acc[ix] += (pk @ ql.T).astype(np.longdouble) * w[k + l]
            acc_abs[ix] += (np.abs(pk) @ np.abs(ql).T).astype(np.longdouble) * w[k + l]
    scale = np.broadcast_to(np.asarray(scale, dtype=np.longdouble), (M, Nc))
    return (acc * scale).astype(np.float64), (acc_abs * np.abs(scale)).astype(np.float64)


def assert_exact(got, want, want_abs, c, what, zero=None):
    """|got - want| <= c 2^-53 want_abs everywhere, and got == 0.0 exactly where `zero` is set.

    c counts the binary64 roundings between the exact int32 group sums and the stored output: S - 1 Horner steps, the
    R^-2 and scale multiplications, and one addition per split-K or tail partial.  An isolated output that loses, doubles or
    misplaces its one plane-pair product moves by O(1) of want_abs, far outside this."""
    got = np.asarray(got, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = np.abs(got - want)
    bad = ~(err <= c * U * want_abs)
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, err / np.maximum(want_abs, 1e-300), -1.0)), got.shape)
        raise AssertionError("%s: %d of %d outputs off by more than %g ulps of their magnitude; worst at %s: got %r want %r "
                             "(|want_abs| %r)" % (what, int(bad.sum()), bad.size, c, i, got[i], want[i], want_abs[i]))
    if zero is not None:
        nz = np.flatnonzero(np.asarray(got)[zero] != 0.0)
        assert nz.size == 0, "%s: %d outputs made only of dropped plane pairs are not exactly zero" % (what, nz.size)
