"""oz_gemm_kernel one digit-plane pair at a time, and at the int32 bound of its group sums.

The tolerance sweeps (test_gpu_kernels.py) compare with numpy at the digit budget; relative to the leading term group g of
the split product weighs about 254^-g, so they cannot see a lost, doubled or misplaced product in the lowest groups (25-50 %
of the plane-pair products in every mode).  Here every row, column or block of an operand sits in ONE digit plane
(tests/digit_planes.py), so an output is a single plane pair (k, l): its product is the whole output, and pairs with
k + l >= S are dropped, so their outputs must be exactly 0.0.  Each use of the kernel is held to the exact integer sums of
the digit planes read back from the device:

- first contraction Y = X~ A^T (KMAJOR = true): X~ row r in plane k_r, A row j in plane l_j;
- second contraction D = (X~^T Y)^T (KMAJOR = false): X~ column i in plane k_i (Y's planes are whatever Y gives);
- Gram build G = X~^T X~ / N (KMAJOR = false): X~ column i in plane k_i, so G[i, i'] is the pair (k_i, k_i');
- Gram product D = (G A^T)^T (KMAJOR = true): a block-diagonal G, each block in one plane, A rows in planes.

Over the digit counts S = 3 (`fast`), 4 (LCX_SPLIT_DIGITS=4), 5, 6 and 7 the shapes reach every tile width of the factor side
(including the spill widths 24, 40, 56 for S >= 5), clusters of 1, 2 and 3 and pairs plus a final three, more work units than
resident clusters, split-K in both contractions and the two-level tails; each test asserts from the planner's
LCX_PLAN_DEBUG line, or from the tile formula of csrc/host_oz.cuh, that it reached what it targets.  The last tests run
near-saturated digits (126 in every plane, one sign) at the planner's int32-exact contraction length oz_kmax and beyond it."""
import re

import numpy as np
import pytest

import digit_planes as dp

pytestmark = pytest.mark.gpu

S_ALL = [3, 4, 5, 6, 7]
SMS = 148
PLAN_RE = re.compile(r"\[lcx plan\] Nl=(\d+) n=(\d+) m=(\d+) gram=(\d) \| K1: splits (\d+) chunk (\d+) tail (\d+) tiles x (\d+) "
                     r"splits \(chunk (\d+)\) \| K2: splits (\d+) chunk (\d+) tail (\d+) tiles x (\d+) splits \(chunk (\d+)\)")
PLAN_KEYS = ["Nl", "n", "m", "gram", "k1_splits", "k1_chunk", "k1_tail_tiles", "k1_tail_splits", "k1_tail_chunk",
             "k2_splits", "k2_chunk", "k2_tail_tiles", "k2_tail_splits", "k2_tail_chunk"]


@pytest.fixture
def env(monkeypatch, capfd):
    """Selects the digit count and returns the planner's LCX_PLAN_DEBUG line of each bind."""
    monkeypatch.setenv("LCX_PLAN_DEBUG", "1")

    class Env:
        def mode(self, S, tail=True):
            prec, digits = dp.MODES[S]
            if digits is None:
                monkeypatch.delenv("LCX_SPLIT_DIGITS", raising=False)
            else:
                monkeypatch.setenv("LCX_SPLIT_DIGITS", digits)
            if tail:
                monkeypatch.delenv("LCX_OZ_TAIL", raising=False)
            else:
                monkeypatch.setenv("LCX_OZ_TAIL", "0")
            return prec

        def plan(self):
            lines = PLAN_RE.findall(capfd.readouterr().err)
            assert lines, "no LCX_PLAN_DEBUG line"
            return dict(zip(PLAN_KEYS, (int(v) for v in lines[-1])))
    return Env()


def _session(prec):
    from linearcorex_b200 import _lib as L
    from linearcorex_b200.corex import _DeviceSession
    return _DeviceSession(L.PRECISIONS[prec]), L


def _to_dev(torch, a, ld):
    t = torch.zeros((a.shape[0], ld), dtype=torch.float64, device="cuda")
    t[:, :a.shape[1]] = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))
    return t


def _planes_dev(sess, L, which):
    """Device view (S, rows, cols) int8 of the digit planes lcx_digit_planes_info describes, and the host copy of their scales."""
    import ctypes as C
    import torch
    off, rows, cols, ldb, soff = (C.c_longlong() for _ in range(5))
    digits, radix = C.c_int(), C.c_int()
    L.check(sess.lib.lcx_digit_planes_info(sess.h, which, C.byref(off), C.byref(digits), C.byref(rows), C.byref(cols),
                                           C.byref(ldb), C.byref(soff), C.byref(radix)))
    S, nr, nc, ld = digits.value, rows.value, cols.value, ldb.value
    assert radix.value == dp.R
    raw = sess.ws[off.value: off.value + (S * nr * ld + 7) // 8].view(torch.int8)[: S * nr * ld]
    nscale = 1 if which == 0 else sess.m
    return raw.view(S, nr, ld)[:, :, :nc], sess.ws[soff.value: soff.value + nscale].cpu().numpy()


def _planes(sess, L, which):
    p, scale = _planes_dev(sess, L, which)
    return p.cpu().numpy(), scale


def _isolated(rng, S, shape, planes_of):
    """Digits and values of a matrix whose entry (r, c) is the single digit d[r, c] in plane planes_of[r, c]."""
    planes_of = np.array(np.broadcast_to(planes_of, shape))
    d = np.zeros(shape, dtype=np.int64)
    for k in range(S):
        sel = planes_of == k
        d[sel] = dp.random_digits(rng, int(sel.sum()), k)
    v = np.zeros(shape)
    for k in range(S):
        sel = planes_of == k
        v[sel] = dp.pure_values(d[sel], k)
    return d, v, planes_of


def _intended(d, planes_of, S):
    return np.stack([np.where(planes_of == k, d, 0) for k in range(S)])


def _assert_planes(got, d, planes_of, S, what):
    want = _intended(d, planes_of, S)
    bad = np.argwhere(got != want)
    assert bad.size == 0, "%s: %d device digits differ from the construction, first (plane, row, col) %s" % (
        what, len(bad), bad[:3].tolist())


# ---- (a) the X pass pair: Y = X~ A^T and D = (X~^T Y)^T ------------------------------------------------------------------
def _pair_operands(rng, S, N, n, m, layout):
    """X~ (N x n) and A (m x n).  layout 'rows': X~ row r in plane kx[r]; 'cols': X~ column i in plane kx[i].  A row j is in
    plane j % S.  Anchors: X~'s at (0, 0), where A is zero; A's in column 1, where X~ is zero."""
    assert n >= 3
    la = np.arange(m) % S
    kx = rng.randint(0, S, size=N if layout == "rows" else n)
    xplanes = np.broadcast_to(kx[:, None] if layout == "rows" else kx[None, :], (N, n)).copy()
    dx, x, _ = _isolated(rng, S, (N, n), xplanes)
    da, a, aplanes = _isolated(rng, S, (m, n), np.broadcast_to(la[:, None], (m, n)).copy())
    for arr in (dx, x, da, a):
        arr[:, :2] = 0
    dx[0, 0], x[0, 0], xplanes[:, 0] = dp.ANCHOR_DIGIT, dp.pure_values(dp.ANCHOR_DIGIT, 0), 0
    da[:, 1], a[:, 1], aplanes[:, 1] = dp.ANCHOR_DIGIT, dp.pure_values(dp.ANCHOR_DIGIT, 0), 0
    dp.check_pure(x, dx, xplanes, S)
    dp.check_pure(a, da, aplanes, S)
    return (dx, x, xplanes, kx), (da, a, aplanes, la)


def _run_pair(env, S, N, n, m, layout, seed, tail=True, check=("Y", "D")):
    """Binds the isolated X~, runs one pass pair (lcx_sig) and checks Y and D against the exact sums of the device's planes."""
    import torch
    prec = env.mode(S, tail)
    rng = np.random.RandomState(seed)
    (dx, x, xplanes, kx), (da, a, aplanes, la) = _pair_operands(rng, S, N, n, m, layout)
    sess, L = _session(prec)
    ld = sess.lib.lcx_ld(n)
    sess.bind(_to_dev(torch, x, ld), N, n, m, None)
    plan = env.plan()
    ad = _to_dev(torch, a, ld)
    od = torch.zeros_like(ad)
    L.check(sess.lib.lcx_sig(sess.h, ad.data_ptr(), 0.0, od.data_ptr()))
    torch.cuda.synchronize()
    px, sx = _planes(sess, L, 0)
    pa, sa = _planes(sess, L, 1)
    assert px.shape[0] == S
    assert sx[0] == 1.0 and np.all(sa == 1.0), "the anchors must keep every scale at 1"
    _assert_planes(px, dx, xplanes, S, "X~ planes")
    _assert_planes(pa, da, aplanes, S, "A planes")
    if "Y" in check:
        y = sess.view(L.A_Y).cpu().numpy()
        want, want_abs = dp.exact_product(px, pa, S, sx[0] * sa[None, :])
        parts = plan["k1_splits"] + (plan["k1_tail_splits"] if plan["k1_tail_tiles"] else 0)
        zero = np.add.outer(kx, la) >= S if layout == "rows" else None
        dp.assert_exact(y, want, want_abs, S + 4 + parts, "Y (S=%d, %s)" % (S, layout), zero=zero)
    if "D" in check:
        py, sy = _planes(sess, L, 2)
        d = sess.view(L.A_D).cpu().numpy()
        want, want_abs = dp.exact_product(py, np.ascontiguousarray(px.transpose(0, 2, 1)), S, sy[:, None] * sx[0])
        parts = plan["k2_splits"] + (plan["k2_tail_splits"] if plan["k2_tail_tiles"] else 0)
        dp.assert_exact(d, want, want_abs, S + 4 + parts, "D (S=%d, %s)" % (S, layout))
    sess.close()
    return plan


def _units_k1(plan, N, m, S):
    """Work units of the first contraction's largest launch and its cluster size (launch_oz_gemm, csrc/ozaki_i8.cuh)."""
    n_tiles, _ = dp.tile_plan(m, S)
    if n_tiles == 1 or n_tiles == 3:
        cl, tiles = n_tiles, n_tiles
    else:                                   # pairs; an odd count's last three run in a launch of their own
        cl, tiles = 2, n_tiles - 3 * (n_tiles % 2)
    return (tiles // cl) * dp.cdiv(N, 128) * plan["k1_splits"], cl


def _coverage_cases():
    cases = []
    for S in S_ALL:
        bnm = dp.bn_max(S)
        step = 16 if bnm > 64 else 8
        for w in range(16, bnm + 1, step):                         # every tile width, one tile (cluster of one)
            cases.append((S, 260, 197, w, "width"))
        two, three, five = (2 * 72, 3 * 112, 5 * 104) if bnm > 64 else (2 * 40, 3 * 56, 5 * 56)
        cases.append((S, 300, 150, two, "pairs"))                  # 2 tiles (S >= 5: spill width 40 in pairs)
        cases.append((S, 300, 150, three, "three"))                # cluster of 3 (S >= 5: spill width 56)
        cases.append((S, 300, 150, five, "pairs+three"))           # 5 tiles: pairs, then a final three
        cases.append((S, 150 * 128 + 5, 70, bnm, "persistent1"))   # more units than resident clusters of one
        cases.append((S, 80 * 128, 70, 2 * bnm, "persistent2"))    # ... of two
        cases.append((S, 60 * 128, 70, 3 * bnm, "persistent3"))    # ... of three
        cases.append((S, 200, 8192, 40, "k1_split"))               # few samples: first contraction split over variables
        cases.append((S, 8192, 256, 40, "k2_split"))               # second contraction split over samples
    return cases


@pytest.mark.parametrize("S,N,n,m,target", _coverage_cases())
def test_pass_pair_planes(env, S, N, n, m, target):
    """Y = X~ A^T with X~ rows and A rows isolated in planes (every Y entry one pair) and D = (X~^T Y)^T against the exact
    digit sums, over the tile widths, cluster shapes, persistent walks and split-K plans of each digit count."""
    n_tiles, bn = dp.tile_plan(m, S)
    if target == "k2_split":   # X~ columns in planes: D isolated on the X~ side
        plan = _run_pair(env, S, N, n, m, "cols", seed=S * 1000 + m + N, check=("D",))
    else:
        plan = _run_pair(env, S, N, n, m, "rows", seed=S * 1000 + m + N,
                         check=("Y", "D") if N * n * m * S * S <= 6e8 else ("Y",))
    if target == "width":
        assert n_tiles == 1 and bn == m
    elif target == "pairs":
        assert n_tiles == 2 and (bn % 16 == 8 if S >= 5 else True)
    elif target == "three":
        assert n_tiles == 3 and (bn % 16 == 8 if S >= 5 else True)
    elif target == "pairs+three":
        assert n_tiles == 5
    elif target.startswith("persistent"):
        units, cl = _units_k1(plan, N, m, S)
        assert cl == int(target[-1]) and units > SMS // cl, (units, cl)
    elif target == "k1_split":
        assert plan["k1_splits"] > 1, plan
    elif target == "k2_split":
        assert plan["k2_splits"] > 1, plan


@pytest.mark.parametrize("S", S_ALL)
@pytest.mark.parametrize("N,n,m_of", [(300, 150, "one"), (300, 150, "two"), (300, 150, "three"), (300, 150, "five"),
                                      (4000, 600, "two")])
def test_second_contraction_planes(env, S, N, n, m_of):
    """D = (X~^T Y)^T with X~ columns isolated in planes: the M-side operand (multicast within clusters of 2 and 3) meets Y's
    planes, every D entry against the exact digit sums."""
    bnm = dp.bn_max(S)
    m = {"one": bnm - 8, "two": 2 * bnm - 8, "three": 3 * bnm - 8, "five": 5 * bnm - 8}[m_of]
    assert dp.tile_plan(m, S)[0] == {"one": 1, "two": 2, "three": 3, "five": 5}[m_of]
    _run_pair(env, S, N, n, m, "cols", seed=S * 77 + m + N, check=("D",))


@pytest.mark.parametrize("S", S_ALL)
def test_two_level_tails(env, S):
    """The two-level split of both contractions (tail units inside the persistent launch, tail_fold_kernel), then the same
    shapes with LCX_OZ_TAIL=0."""
    m = 130 if S <= 4 else 72                      # two tiles: 80 wide, or the spill width 40
    for tail in (True, False):
        plan = _run_pair(env, S, 9500, 500, m, "rows", seed=S, tail=tail, check=("Y",))
        assert (plan["k1_tail_tiles"] > 0 and plan["k1_tail_splits"] > 1) == tail, plan
        plan = _run_pair(env, S, 500, 9500, m, "cols", seed=S + 50, tail=tail, check=("D",))
        assert (plan["k2_tail_tiles"] > 0 and plan["k2_tail_splits"] > 1) == tail, plan


# ---- Gram build: G = X~^T X~ / N ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", S_ALL)
@pytest.mark.parametrize("N,n,block", [(700, 300, 128), (2000, 520, 256)])
def test_gram_build_planes(env, S, N, n, block):
    """X~ column i in plane k_i: G[i, i'] is the single pair (k_i, k_i'), exactly zero for k_i + k_i' >= S.  The anchor is
    X~[0, 0], alone in its row and column."""
    import torch
    prec = env.mode(S)
    rng = np.random.RandomState(S * 31 + n)
    kx = rng.randint(0, S, size=n)
    kx[0] = 0
    xplanes = np.broadcast_to(kx[None, :], (N, n)).copy()
    dx, x, _ = _isolated(rng, S, (N, n), xplanes)
    dx[0, :], x[0, :], dx[:, 0], x[:, 0] = 0, 0.0, 0, 0.0
    dx[0, 0], x[0, 0] = dp.ANCHOR_DIGIT, dp.pure_values(dp.ANCHOR_DIGIT, 0)
    dp.check_pure(x, dx, xplanes, S)
    sess, L = _session(prec)
    ld = sess.lib.lcx_ld(n)
    sess.bind(_to_dev(torch, x, ld), N, n, 4, None)
    plan = env.plan()
    assert plan["k2_tail_tiles"] == 0, plan      # the build walks the uniform split over samples
    g = torch.full((n, ld), float("nan"), dtype=torch.float64, device="cuda")
    nscr = sess.lib.lcx_gram_scratch_doubles(sess.h, block)
    scr = torch.empty(nscr, dtype=torch.float64, device="cuda")
    L.check(sess.lib.lcx_gram_build(sess.h, g.data_ptr(), ld, block, scr.data_ptr(), nscr))
    torch.cuda.synchronize()
    px, sx = _planes(sess, L, 0)
    assert sx[0] == 1.0
    _assert_planes(px, dx, xplanes, S, "X~ planes")
    pt = np.ascontiguousarray(px.transpose(0, 2, 1))
    want, want_abs = dp.exact_product(pt, pt, S, np.longdouble(sx[0]) ** 2 / N)
    dp.assert_exact(g[:, :n].cpu().numpy(), want, want_abs, S + 4 + plan["k2_splits"], "G (S=%d)" % S,
                    zero=np.add.outer(kx, kx) >= S)
    sess.close()


# ---- Gram product: D = (G A^T)^T ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", S_ALL)
@pytest.mark.parametrize("n,route", [(10000, "waves"), (1000, "generic")])
def test_gram_product_planes(env, S, n, route):
    """G block-diagonal with each (symmetric) block in one plane, A rows in planes: D[j, i] is the single pair (k_block(i), l_j).
    Variable 0 carries G's anchor (A is zero there), variable 1 is empty in G and carries A's anchors.  'waves' is the
    gram_plan of whole waves of full-K row tiles plus a split remainder, 'generic' the split-K plan."""
    import torch
    prec = env.mode(S)
    bnm = dp.bn_max(S)
    m = (2 * bnm - 28) if route == "waves" else (3 * bnm - 20)
    full, rest, splits = dp.gram_plan(n, m, S)
    if route == "waves":
        assert full > 0 and rest > 0 and splits > 1, (full, rest, splits)
    else:
        assert full == 0
    rng = np.random.RandomState(S * 7 + n)
    bs = 96
    starts = list(range(2, n, bs))
    kb = rng.randint(0, S, size=len(starts))
    la = np.arange(m) % S
    sess, L = _session(prec)
    ld = sess.lib.lcx_ld(n)
    gd = torch.zeros((n, ld), dtype=torch.float64, device="cuda")
    blocks = []
    for t, i0 in enumerate(starts):
        i1 = min(n, i0 + bs)
        d = np.triu(dp.random_digits(rng, (i1 - i0, i1 - i0), kb[t]))
        d = d + np.triu(d, 1).T
        v = dp.pure_values(d, kb[t])
        dp.check_pure(v, d, kb[t], S)
        gd[i0:i1, i0:i1] = torch.from_numpy(v)
        blocks.append((i0, i1, d))
    gd[0, 0] = float(dp.pure_values(dp.ANCHOR_DIGIT, 0))
    aplanes = np.broadcast_to(la[:, None], (m, n)).copy()
    da, a, _ = _isolated(rng, S, (m, n), aplanes)
    da[:, :2], a[:, :2] = 0, 0.0
    da[:, 1], a[:, 1], aplanes[:, 1] = dp.ANCHOR_DIGIT, dp.pure_values(dp.ANCHOR_DIGIT, 0), 0
    dp.check_pure(a, da, aplanes, S)
    sess.bind_gram(gd, n, m)
    plan = env.plan()
    assert plan["gram"] == 1
    del gd
    ad = _to_dev(torch, a, ld)
    od = torch.zeros_like(ad)
    L.check(sess.lib.lcx_sig(sess.h, ad.data_ptr(), 0.0, od.data_ptr()))
    torch.cuda.synchronize()
    pg_dev, sg = _planes_dev(sess, L, 0)
    pa, sa = _planes(sess, L, 1)
    assert sg[0] == 1.0 and np.all(sa == 1.0)
    _assert_planes(pa, da, aplanes, S, "A planes")
    got = sess.view(L.A_D).cpu().numpy()
    want = np.zeros((m, n))
    want_abs = np.zeros((m, n))
    anchor = pg_dev[:, 0, 0].cpu().numpy()
    assert anchor[0] == dp.ANCHOR_DIGIT and not anchor[1:].any()
    nnz = 1
    for t, (i0, i1, d) in enumerate(blocks):
        pb = pg_dev[:, i0:i1, i0:i1].cpu().numpy()
        _assert_planes(pb, d, np.full(d.shape, kb[t]), S, "G block %d planes" % t)
        nnz += int(np.count_nonzero(pb))
        w, wa = dp.exact_product(pb, np.ascontiguousarray(pa[:, :, i0:i1]), S, sg[0] * sa[None, :])
        want[:, i0:i1], want_abs[:, i0:i1] = w.T, wa.T
    # everything outside the diagonal blocks and the anchor is zero in every plane of G
    assert int(torch.count_nonzero(pg_dev)) == nnz
    parts = splits if route == "waves" else plan["k1_splits"]
    zero = np.zeros((m, n), dtype=bool)
    for t, (i0, i1, _) in enumerate(blocks):
        zero[:, i0:i1] = (la[:, None] + kb[t]) >= S
    dp.assert_exact(got[:, :n], want, want_abs, S + 4 + parts, "Gram D (S=%d, %s)" % (S, route), zero=zero)
    assert np.all(got[:, :2] == 0.0)
    sess.close()


# ---- (c) int32 exactness at the split bound ---------------------------------------------------------------------------
# All operands +126/253 (digits 126 in every plane, one sign): every group sum grows linearly in the contraction length, to
# about 98 % of 2^31 in group S-1 at K = oz_kmax.  148 M tiles of 128 make the planner's cost model pick its minimum split
# cdiv(K, oz_kmax): one split holds all of K = oz_kmax, and at K = 2 oz_kmax + 100 -- where one accumulator would overflow --
# the int32 sums stay exact only because of the split.  Every plane is checked to be constant on the device, so the exact
# sums of one row / column of digits are every output's reference.
BOUND_S = [3, 5, 6, 7]
BIG = 148 * 128


def _saturated_digits(S):
    return [int(p[0]) for p in dp.split_digits(np.array([dp.SATURATED]), 1.0, S, dp.R)]


def _assert_constant(planes_dev, digits, what):
    """planes_dev (S, rows, cols) on the device: plane k is the digit digits[k] everywhere (digits: list, or (S, rows) array)."""
    import torch
    for k in range(planes_dev.shape[0]):
        dk = digits[k]
        if np.ndim(dk) == 0:
            ok = bool((planes_dev[k] == int(dk)).all())
        else:
            ok = bool((planes_dev[k] == torch.as_tensor(np.asarray(dk), device="cuda")[:, None]).all())
        assert ok, "%s: plane %d is not constant" % (what, k)


def _group_top(P, Q, S):
    """Largest |entry| of the unsplit group S-1 sum  sum_{k+l=S-1} P_k Q_l^T  (exact: integers below 2^53)."""
    tot = 0
    for k in range(S):
        tot = tot + P[k].astype(np.float64) @ Q[S - 1 - k].astype(np.float64).T
    return float(np.abs(tot).max())


def _bound_len(S, beyond):
    K = 2 * dp.oz_kmax(S) + 100 if beyond else dp.oz_kmax(S)
    return K, dp.cdiv(K, dp.oz_kmax(S))


def _check_top(top, beyond):
    assert (top > 2 ** 31 - 1) if beyond else (0.97 * 2 ** 31 < top < 2 ** 31), top


@pytest.mark.parametrize("S", BOUND_S)
@pytest.mark.parametrize("beyond", [False, True])
def test_first_contraction_at_int32_bound(env, S, beyond):
    """Y = X~ A^T over K variables, 148 row tiles."""
    import torch
    prec = env.mode(S)
    K, splits = _bound_len(S, beyond)
    N, m = BIG, 16
    sess, L = _session(prec)
    ld = sess.lib.lcx_ld(K)
    xt = torch.zeros((N, ld), dtype=torch.float64, device="cuda")
    xt[:, :K] = dp.SATURATED
    sess.bind(xt, N, K, m, None)
    del xt
    plan = env.plan()
    assert plan["k1_splits"] == splits and plan["k1_tail_tiles"] == 0, plan
    ad = _to_dev(torch, np.full((m, K), dp.SATURATED), ld)
    od = torch.zeros_like(ad)
    L.check(sess.lib.lcx_sig(sess.h, ad.data_ptr(), 0.0, od.data_ptr()))
    torch.cuda.synchronize()
    pxd, sx = _planes_dev(sess, L, 0)
    pad, sa = _planes_dev(sess, L, 1)
    sat = _saturated_digits(S)
    _assert_constant(pxd, sat, "X~")
    _assert_constant(pad, sat, "A")
    px1, pa1 = pxd[:, :1].cpu().numpy(), pad[:, :1].cpu().numpy()
    _check_top(_group_top(px1, pa1, S), beyond)
    want, want_abs = dp.exact_product(px1, pa1, S, sx[0] * sa[None, :1])
    got = sess.view(L.A_Y).cpu().numpy()
    dp.assert_exact(got, np.broadcast_to(want, got.shape), np.broadcast_to(want_abs, got.shape), S + 4 + splits,
                    "Y at K=%d (S=%d)" % (K, S))
    sess.close()


@pytest.mark.parametrize("S", BOUND_S)
@pytest.mark.parametrize("beyond", [False, True])
def test_second_contraction_and_gram_build_at_int32_bound(env, S, beyond):
    """N = K samples over 148 variable tiles.  D = X~^T Y with A = 2^-14 on 16384 of the variables, so that Y = X~ A^T is the
    same near-saturated value and its digits (read back) also sum past 2^31 unsplit; then G = X~^T X~ / N on the same
    session (the build walks the same split over samples)."""
    import torch
    prec = env.mode(S)
    K, splits = _bound_len(S, beyond)
    n, m = BIG, 16
    sess, L = _session(prec)
    ld = sess.lib.lcx_ld(n)
    xt = torch.full((K, ld), dp.SATURATED, dtype=torch.float64, device="cuda")
    sess.bind(xt, K, n, m, None)
    del xt
    plan = env.plan()
    assert plan["k2_splits"] == splits and plan["k2_tail_tiles"] == 0, plan
    a = np.zeros((m, n))
    a[:, :16384] = 2.0 ** -14
    ad = _to_dev(torch, a, ld)
    od = torch.zeros_like(ad)
    L.check(sess.lib.lcx_sig(sess.h, ad.data_ptr(), 0.0, od.data_ptr()))
    torch.cuda.synchronize()
    pxd, sx = _planes_dev(sess, L, 0)
    pyd, sy = _planes_dev(sess, L, 2)
    _assert_constant(pxd, _saturated_digits(S), "X~")
    py1 = pyd[:, :, :1].cpu().numpy()
    _assert_constant(pyd, py1[:, :, 0], "Y")
    px1 = np.ascontiguousarray(pxd[:, :, :1].cpu().numpy().transpose(0, 2, 1))
    py = pyd.cpu().numpy()
    _check_top(_group_top(py[:, :1], px1, S), beyond)
    want, want_abs = dp.exact_product(py, px1, S, sy[:, None] * sx[0])
    got = sess.view(L.A_D).cpu().numpy()
    dp.assert_exact(got, np.broadcast_to(want, got.shape), np.broadcast_to(want_abs, got.shape), S + 4 + splits,
                    "D at N=%d (S=%d)" % (K, S))
    # Gram build on the same planes: every entry K saturated products per plane pair, divided by N
    _check_top(_group_top(px1, px1, S), beyond)
    gw, gwa = dp.exact_product(px1, px1, S, np.longdouble(sx[0]) ** 2 / K)
    g = torch.full((n, ld), float("nan"), dtype=torch.float64, device="cuda")
    nscr = sess.lib.lcx_gram_scratch_doubles(sess.h, 1024)
    scr = torch.empty(nscr, dtype=torch.float64, device="cuda")
    L.check(sess.lib.lcx_gram_build(sess.h, g.data_ptr(), ld, 1024, scr.data_ptr(), nscr))
    torch.cuda.synchronize()
    err = float((g[:, :n] - float(gw[0, 0])).abs().max())
    assert err <= (S + 4 + splits) * dp.U * float(gwa[0, 0]), "G at N=%d (S=%d): max error %r of %r" % (K, S, err, gw[0, 0])
    sess.close()
