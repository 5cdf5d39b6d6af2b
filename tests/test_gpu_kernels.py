"""GPU unit parity: each C-ABI building block against numpy float64 on seeded operands.
All calls go through liblcx_b200.so (ctypes); nothing here touches /root/reference."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    import torch
    from linearcorex_b200 import _lib
    from linearcorex_b200.corex import _DeviceSession
    sess = _DeviceSession(_lib.PRECISION_FP64)
    yield sess, _lib, torch
    sess.close()


def _dev_mat(torch, a, ld=None):
    """numpy (r x c) -> device tensor with even leading dimension ld >= c (padding filled with NaN on purpose:
    the kernels must never read it)."""
    r, c = a.shape
    ld = ld or (c + (c % 2) + 2)
    t = torch.full((r, ld), float("nan"), dtype=torch.float64, device="cuda")
    t[:, :c] = torch.from_numpy(np.ascontiguousarray(a))
    return t


GEMM_SHAPES = [(128, 104, 160), (1, 1, 1), (5, 3, 7), (257, 100, 333), (300, 13, 50), (100, 100, 1000),
               (130, 260, 40), (64, 500, 96), (1000, 5, 50), (37, 30, 4100)]


@pytest.mark.parametrize("layout", [0, 1, 2])
@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
@pytest.mark.parametrize("variant", ["plain", "trans", "cadd", "split"])
def test_dgemm_matches_numpy(dev, layout, M, N, K, variant):
    sess, L, torch = dev
    rng = np.random.RandomState(M * 131 + N * 17 + K + layout)
    A = rng.randn(M, K)
    B = rng.randn(K, N)
    want = A @ B
    a_store = A if layout in (0, 2) else A.T            # [M][K] or [K][M]
    b_store = B.T if layout == 0 else B                 # [N][K] or [K][N]
    ad, bd = _dev_mat(torch, a_store), _dev_mat(torch, b_store)
    trans = variant == "trans"
    out_shape = (N, M) if trans else (M, N)
    cd = torch.full((out_shape[0], out_shape[1] + (out_shape[1] % 2) + 2), float("nan"), dtype=torch.float64, device="cuda")
    cadd = None
    if variant == "cadd":
        cadd0 = rng.randn(*out_shape)
        cadd = _dev_mat(torch, cadd0, ld=cd.shape[1])
        want = want + cadd0
    max_splits, scratch, nscr = 1, None, 0
    if variant == "split":
        max_splits = 7
        nscr = 7 * cd.numel()
        scratch = torch.empty(nscr, dtype=torch.float64, device="cuda")
    rc = sess.lib.lcx_gemm_f64(sess.h, layout, M, N, K, ad.data_ptr(), ad.stride(0), bd.data_ptr(), bd.stride(0),
                               cd.data_ptr(), cd.stride(0), int(trans), cadd.data_ptr() if cadd is not None else None,
                               max_splits, scratch.data_ptr() if scratch is not None else None, nscr)
    L.check(rc, "lcx_gemm_f64")
    torch.cuda.synchronize()
    got = cd[:, :out_shape[1]].cpu().numpy()
    if trans:
        got = got.T
    scale = np.abs(A) @ np.abs(B)
    assert np.all(np.abs(got - want) <= 1e-14 * scale + 1e-300), np.abs(got - want).max()
    assert torch.isnan(cd[:, out_shape[1]:]).all()  # padding untouched


@pytest.mark.parametrize("m,n", [(1, 7), (2, 33), (5, 64), (30, 100), (100, 257), (160, 40), (161, 300), (257, 1000),
                                 (500, 96), (840, 70)])
def test_solve_matches_numpy(dev, m, n):
    """lcx_solve = np.linalg.solve (linearcorex.py:280, :366): LU with partial pivoting + triangular sweeps.  Covers the
    single-CTA shared-memory factorisation (m <= 160), the cooperative one, and the in-place-in-output sweep (m > 832)."""
    sess, L, torch = dev
    rng = np.random.RandomState(m)
    Wm = rng.randn(m, 3 * m + 5)
    A = Wm @ Wm.T / (3 * m + 5) + 0.05 * rng.randn(m, m) / max(1, m)  # well conditioned, not symmetric
    np.fill_diagonal(A, 1.0)
    A[[0, m - 1]] = A[[m - 1, 0]]  # force row exchanges
    B = rng.randn(m, n)
    ad, bd = _dev_mat(torch, A), _dev_mat(torch, B)
    xd = torch.full((m, n + (n % 2) + 2), float("nan"), dtype=torch.float64, device="cuda")
    nscr = sess.lib.lcx_solve_scratch_doubles(m)
    scr = torch.empty(nscr, dtype=torch.float64, device="cuda")
    L.check(sess.lib.lcx_solve(sess.h, ad.data_ptr(), ad.stride(0), m, bd.data_ptr(), bd.stride(0), xd.data_ptr(),
                               xd.stride(0), n, scr.data_ptr(), nscr))
    got = xd[:, :n].cpu().numpy()
    want = np.linalg.solve(A, B)
    np.testing.assert_allclose(got, want, rtol=1e-10, atol=1e-12 * np.abs(want).max())
    assert torch.isnan(xd[:, n:]).all()  # padding untouched
    if m <= 832:  # in place
        L.check(sess.lib.lcx_solve(sess.h, ad.data_ptr(), ad.stride(0), m, bd.data_ptr(), bd.stride(0), bd.data_ptr(),
                                   bd.stride(0), n, scr.data_ptr(), nscr))
        np.testing.assert_allclose(bd[:, :n].cpu().numpy(), want, rtol=1e-10, atol=1e-12 * np.abs(want).max())


def test_solve_singular_raises(dev):
    sess, L, torch = dev
    A = np.ones((6, 6))
    B = np.ones((6, 3))
    ad, bd = _dev_mat(torch, A), _dev_mat(torch, B)
    xd = torch.zeros((6, 4), dtype=torch.float64, device="cuda")
    nscr = sess.lib.lcx_solve_scratch_doubles(6)
    scr = torch.empty(nscr, dtype=torch.float64, device="cuda")
    with pytest.raises(np.linalg.LinAlgError):
        L.check(sess.lib.lcx_solve(sess.h, ad.data_ptr(), ad.stride(0), 6, bd.data_ptr(), bd.stride(0), xd.data_ptr(),
                                   xd.stride(0), 3, scr.data_ptr(), nscr))


@pytest.mark.parametrize("N,n,m", [(400, 300, 10), (1000, 50, 5), (77, 513, 30), (2000, 5, 1), (130, 1000, 100)])
def test_project_and_colsq(dev, N, n, m):
    sess, L, torch = dev
    rng = np.random.RandomState(N + n + m)
    X = rng.randn(N, n)
    W = rng.randn(m, n) / np.sqrt(n)
    ld = sess.lib.lcx_ld(n)
    xd, wd = _dev_mat(torch, X, ld=ld), _dev_mat(torch, W, ld=ld)
    ldy = sess.lib.lcx_ldy(m)
    y = torch.full((N, ldy), float("nan"), dtype=torch.float64, device="cuda")
    s = torch.zeros(m, dtype=torch.float64, device="cuda")
    nscr = sess.lib.lcx_project_scratch_doubles(N, m)
    scr = torch.empty(nscr, dtype=torch.float64, device="cuda")
    L.check(sess.lib.lcx_project(sess.h, xd.data_ptr(), N, n, ld, wd.data_ptr(), ld, m, y.data_ptr(), ldy, s.data_ptr(),
                                 scr.data_ptr(), nscr))
    torch.cuda.synchronize()
    Y = X @ W.T
    np.testing.assert_allclose(y[:, :m].cpu().numpy(), Y, rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(s.cpu().numpy(), (Y * Y).sum(0), rtol=1e-12)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("mode", ["standard", "outliers"])
@pytest.mark.parametrize("missing", [None, -1e6, float("nan")])
def test_preprocess_matches_oracle(dev, dtype, mode, missing):
    import corex_oracle as oc
    from linearcorex_b200 import Corex
    rng = np.random.RandomState(11)
    x = (rng.randn(9000, 37) * rng.uniform(0.5, 30, size=37) + rng.uniform(-50, 50, size=37))
    x[:, 3] = np.sign(x[:, 3]) * np.abs(x[:, 3]) ** 2.5
    x = x.astype(dtype)
    if missing is not None:
        x = np.where(rng.rand(*x.shape) < 0.05, missing, x).astype(dtype)
    mdl = Corex(n_hidden=2, gaussianize=mode, missing_values=missing, input_dtype="float64")
    xt = mdl.preprocess(x, fit=True)[:, :37].cpu().numpy()
    want, theta, n_obs = oc.standardize(x.astype(np.float64), mode, missing)
    np.testing.assert_allclose(mdl.theta[0], theta[0], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(mdl.theta[1], theta[1], rtol=1e-12)
    np.testing.assert_array_equal(np.asarray(mdl.n_obs), np.asarray(n_obs))
    np.testing.assert_allclose(xt, want, rtol=1e-10, atol=1e-11)
    # transform-time preprocessing imputes with the *new* data's column means but keeps theta (:389, :404)
    x2 = x[:1234]
    xt2 = mdl.preprocess(x2)[:, :37].cpu().numpy()
    want2, _, _ = oc.standardize(x2.astype(np.float64), mode, missing, theta=theta)
    np.testing.assert_allclose(xt2, want2, rtol=1e-10, atol=1e-11)


def _planes(sess, L, torch, which):
    import ctypes as C
    off, rows, cols, ldb, soff = (C.c_longlong() for _ in range(5))
    digits, radix = C.c_int(), C.c_int()
    L.check(sess.lib.lcx_digit_planes_info(sess.h, which, C.byref(off), C.byref(digits), C.byref(rows), C.byref(cols),
                                           C.byref(ldb), C.byref(soff), C.byref(radix)))
    S, R, nr, nc, ld = digits.value, radix.value, rows.value, cols.value, ldb.value
    raw = sess.ws[off.value: off.value + (S * nr * ld + 7) // 8].view(torch.int8)[: S * nr * ld]
    planes = raw.view(S, nr, ld)[:, :, :nc].cpu().numpy().astype(np.int64)
    nscale = 1 if which == 0 else sess.m
    scale = sess.ws[soff.value: soff.value + nscale].cpu().numpy()
    return planes, scale, S, R


@pytest.mark.parametrize("precision", ["fp64_split", "fast", "fp64_split7"])
def test_digit_planes_bit_exact_against_numpy(precision):
    """Integer work is held to bit-exactness: the device's int8 digit planes of X~, A and Y equal the numpy restatement of
    the digit extraction (tests/test_split_scheme.py) digit for digit, and the recombined products are the exact integer sums."""
    import torch
    from linearcorex_b200 import _lib as L
    from linearcorex_b200.corex import _DeviceSession
    from test_split_scheme import pow2_above, split_digits
    rng = np.random.RandomState(3)
    N, n, m = 700, 333, 37
    x = rng.randn(N, n)
    x[5, 17] = -9.25
    u = rng.randn(m, n) * rng.uniform(1e-3, 4.0, size=(m, 1))
    sess = _DeviceSession(L.PRECISIONS[precision])
    ld = sess.lib.lcx_ld(n)
    xt = torch.zeros((N, ld), dtype=torch.float64, device="cuda")
    xt[:, :n] = torch.from_numpy(x)
    sess.bind(xt, N, n, m, None)
    ud = torch.zeros((m, ld), dtype=torch.float64, device="cuda")
    ud[:, :n] = torch.from_numpy(u)
    od = torch.zeros_like(ud)
    L.check(sess.lib.lcx_sig(sess.h, ud.data_ptr(), 0.0, od.data_ptr()))
    torch.cuda.synchronize()
    px, sx, S, R = _planes(sess, L, torch, 0)
    pa, sa, _, _ = _planes(sess, L, torch, 1)
    py, sy, _, _ = _planes(sess, L, torch, 2)
    assert sx[0] == pow2_above(np.abs(x).max())
    np.testing.assert_array_equal(sa, [pow2_above(np.abs(r).max()) for r in u])
    for k, want in enumerate(split_digits(x, sx[0], S, R)):
        np.testing.assert_array_equal(px[k], want)
    for k, want in enumerate(split_digits(u, sa[:, None], S, R)):
        np.testing.assert_array_equal(pa[k], want)
    y_dev = sess.view(L.A_Y).cpu().numpy()
    np.testing.assert_array_equal(sy, [pow2_above(np.abs(c).max()) for c in y_dev.T])
    for k, want in enumerate(split_digits(y_dev, sy[None, :], S, R)):
        np.testing.assert_array_equal(py[k].T, want)  # the Y planes are stored factor-major (K-major for the 2nd contraction)
    # Y itself = the exact integer group sums recombined by the same Horner steps
    groups = [np.zeros((N, m), dtype=np.int64) for _ in range(S)]
    for k in range(S):
        for l in range(S - k):
            groups[k + l] += px[k] @ pa[l].T
    acc = groups[S - 1].astype(np.float64)
    for g in range(S - 2, -1, -1):
        acc = acc * (1.0 / R) + groups[g]
    want_y = acc * ((1.0 / R) * (1.0 / R)) * (sx[0] * sa)[None, :]
    # (binary64 recombination: the device may fuse the multiply-adds, so this part is held to a few ulps of the column scale)
    assert np.all(np.abs(y_dev - want_y) <= 1e-14 * np.abs(want_y).max(axis=0))
    # second contraction: D = (X~^T Y)^T from the exact integer group sums of the X~ and Y digits
    groups = [np.zeros((m, n), dtype=np.int64) for _ in range(S)]
    for k in range(S):
        for l in range(S - k):
            groups[k + l] += py[k] @ px[l]
    acc = groups[S - 1].astype(np.float64)
    for g in range(S - 2, -1, -1):
        acc = acc * (1.0 / R) + groups[g]
    want_d = acc * ((1.0 / R) * (1.0 / R)) * (sx[0] * sy)[:, None]
    d_dev = sess.view(L.A_D).cpu().numpy()
    # (split over samples: the per-split Horner sums are added in binary64, hence a few ulps of the row scale)
    assert np.all(np.abs(d_dev - want_d) <= 1e-13 * np.abs(want_d).max(axis=1, keepdims=True))
    sess.close()


SIG_SHAPES = [(1, 1, 1), (63, 5, 1), (64, 127, 16), (65, 128, 17), (200, 129, 48), (700, 1000, 64), (513, 333, 65),
              (1000, 257, 100), (129, 64, 112), (300, 2049, 128), (4100, 130, 130), (2500, 70, 200)]


@pytest.mark.parametrize("precision,tol", [("fp64", 1e-13), ("fp64_split7", 1e-12), ("fp64_split", 5e-11), ("fp64_split5", 1e-8), ("fast", 5e-4)])
@pytest.mark.parametrize("N,n,m", SIG_SHAPES)
def test_pass_pair_over_tile_edges(precision, tol, N, n, m):
    """`_sig` (:196-213) = one pass pair over X~ at shapes straddling every tile edge of both contractions (128-row and
    128-variable M tiles, 64-wide factor tiles with 16..64-wide tails, padded cluster slots), against numpy float64.
    The tolerances are the digit budgets (48 / 40 / 24 bits below the operand maxima) with margin; a tiling bug is O(1)."""
    import torch
    from linearcorex_b200 import _lib as L
    from linearcorex_b200.corex import _DeviceSession
    rng = np.random.RandomState(N * 7 + n * 3 + m)
    x = rng.randn(N, n)
    u = rng.randn(m, n) * rng.uniform(0.1, 3.0, size=(m, 1))
    eps = 0.36
    sess = _DeviceSession(L.PRECISIONS[precision])
    ld = sess.lib.lcx_ld(n)
    xt = torch.zeros((N, ld), dtype=torch.float64, device="cuda")
    xt[:, :n] = torch.from_numpy(x)
    sess.bind(xt, N, n, m, None)
    ud = torch.zeros((m, ld), dtype=torch.float64, device="cuda")
    ud[:, :n] = torch.from_numpy(u)
    od = torch.full((m, ld), float("nan"), dtype=torch.float64, device="cuda")
    L.check(sess.lib.lcx_sig(sess.h, ud.data_ptr(), eps, od.data_ptr()))
    torch.cuda.synchronize()
    got = od[:, :n].cpu().numpy()
    y = x @ u.T
    want = (1 - eps ** 2) * (x.T @ y).T / N + eps ** 2 * u
    scale = (1 - eps ** 2) * (np.abs(x).T @ np.abs(y)).T / N + eps ** 2 * np.abs(u)
    assert np.all(np.abs(got - want) <= tol * scale.max(axis=1, keepdims=True)), np.abs(got - want).max()
    sess.close()


def _random_shapes(count, seed=20241017):
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(count):
        N = int(rng.choice([rng.randint(1, 70), rng.randint(70, 700), rng.randint(700, 6000)]))
        n = int(rng.choice([rng.randint(1, 70), rng.randint(70, 700), rng.randint(700, 3000)]))
        m = int(rng.choice([rng.randint(1, 20), rng.randint(20, 140), rng.randint(140, 300)]))
        out.append((N, n, m))
    return out


@pytest.mark.parametrize("N,n,m", _random_shapes(24))
def test_pass_pair_random_shapes_fp64_split(N, n, m):
    """The same check as the tile-edge sweep on 24 seeded random shapes (default precision mode)."""
    test_pass_pair_over_tile_edges("fp64_split", 5e-11, N, n, m)


@pytest.mark.parametrize("N,n,m", [(12500, 10000, 100), (9600, 9500, 120), (4000, 20000, 70), (25000, 10000, 100)])
def test_pass_pair_two_level_split(N, n, m, monkeypatch, capfd):
    """Shapes whose units do not fill whole rounds of the 74 resident cluster pairs (config 3's 12 500 samples per rank on 8
    GPUs first): the planner's two-level split (host_session.cuh: plan_two_level; tail units inside the persistent launch,
    ozaki_i8.cuh; tail_fold_kernel) must engage and give the same `_sig` as numpy."""
    from linearcorex_b200 import _lib as L
    monkeypatch.setenv("LCX_PLAN_DEBUG", "1")
    L.load().lcx_workspace_doubles(N, n, m, L.PRECISIONS["fp64_split"])
    plan = capfd.readouterr().err
    assert "[lcx plan]" in plan and plan.count("tail 0 tiles") < 2, plan  # at least one of the two contractions has a tail
    monkeypatch.delenv("LCX_PLAN_DEBUG")
    test_pass_pair_over_tile_edges("fp64_split", 5e-11, N, n, m)
    monkeypatch.setenv("LCX_OZ_TAIL", "0")   # and the uniform plan still works when the tail is switched off
    test_pass_pair_over_tile_edges("fp64_split", 5e-11, N, n, m)
