"""Corex.sample, impute(return_std=True) and sample_missing on the B200: the generator against tests/philox_ref.py, sample
against numpy from the same normals, bit-identity under splits, blockings, containers, repeats and pickling, statistics of
the draws (fixed seeds, thresholds of at least 5 sigma, so deterministic), conditional standard deviations against the dense
conditional covariance, and every size class and path of the per-row kernel in its sampling mode."""
import pickle

import numpy as np
import pytest

from dense_conditional import dense_conditional, missing_mask
from dense_sampling import dense_conditional_cov, draw_map, lowrank_std
from dense_score import lowrank_parts, woodbury
from philox_ref import normals, stream_words
from test_gpu_conditional import _cond_class, _with_nans
from test_gpu_score import PARITY, _fit, _rel

pytestmark = pytest.mark.gpu


def test_normal_fill_matches_reference():
    import torch
    from linearcorex_b200 import Corex, _lib
    sess = Corex(n_hidden=2, precision="fp64")._session()
    seed, rows, cols = 0x0123456789ABCDEF, 6, 7
    row0 = 2 ** 32 - 3  # the rows cross into the counter's high row word
    for tag, draw in ((0, 0), (1, 5)):
        out = torch.zeros((rows, 8), dtype=torch.float64, device=sess.device)
        words = torch.zeros((rows, 16), dtype=torch.int32, device=sess.device)
        _lib.check(sess.lib.lcx_normal_fill(sess.h, seed, tag, row0, rows, draw, cols, out.data_ptr(), 8, words.data_ptr(), 16),
                   "lcx_normal_fill")
        got_w = words.cpu().numpy().view(np.uint32).reshape(rows, 4, 4)
        want_w = stream_words(seed, tag, np.arange(row0, row0 + rows), draw, cols)
        assert np.array_equal(got_w.astype(np.uint64), want_w)
        got, want = out.cpu().numpy()[:, :cols], normals(seed, tag, np.arange(row0, row0 + rows), draw, cols)
        ulps = np.abs(got - want) / np.spacing(np.maximum(np.abs(want), 1e-300))
        assert ulps.max() <= 8, ulps.max()
    with pytest.raises(_lib.LcxError):
        _lib.check(sess.lib.lcx_normal_fill(sess.h, seed, 0, 0, rows, 0, cols, out.data_ptr(), 4, None, 0), "lcx_normal_fill")


@pytest.mark.parametrize("name", ["readme_demo_f64", "adni_l0_f64"])
def test_sample_matches_numpy(name):
    mdl, _x = _fit(name)
    mean, sd = mdl.theta
    z, delta = lowrank_parts(mdl.moments["rhoinvrho"], mdl.moments["Si"], mdl.eps)
    m, n = z.shape
    for seed, first_row, count in ((3, 0, 40), (2 ** 63 + 11, 2 ** 32 - 5, 9)):
        got = mdl.sample(count, seed=seed, first_row=first_row)
        assert got.shape == (count, n) and got.dtype == np.float64
        eps = normals(seed, 0, np.arange(first_row, first_row + count), 0, m + n)
        want_std = eps[:, :m].dot(z) + np.sqrt(delta) * eps[:, m:]
        assert _rel((got - mean) / sd, want_std) < 1e-12, _rel((got - mean) / sd, want_std)


def test_sample_is_bit_identical_under_splits_blockings_repeats_and_pickling():
    mdl, _x = _fit("syn_400x300x10_f64")
    want = mdl.sample(300, seed=42)
    assert np.array_equal(mdl.sample(300, seed=42), want)
    assert np.array_equal(mdl.sample(7, seed=42, first_row=3), want[3:10])
    assert np.array_equal(np.vstack([mdl.sample(100, seed=42), mdl.sample(200, seed=42, first_row=100)]), want)
    for rows in (7, 128):
        mdl.stream_rows = rows
        assert np.array_equal(mdl.sample(300, seed=42), want), rows
    mdl.stream_rows = None
    dev = mdl.sample(300, seed=42, return_device=True)
    assert dev.is_cuda and tuple(dev.shape) == want.shape and np.array_equal(dev.cpu().numpy(), want)
    clone = pickle.loads(pickle.dumps(mdl))
    assert np.array_equal(clone.sample(300, seed=42), want)
    other = mdl.sample(300, seed=43)
    assert not np.any(other == want)
    np.random.seed(5)
    a = mdl.sample(4)
    np.random.seed(5)
    assert np.array_equal(mdl.sample(4), a) and not np.array_equal(a, mdl.sample(4))
    assert mdl.sample(0, seed=1).shape == (0, want.shape[1])


def test_sample_statistics():
    mdl, _x = _fit("syn_400x300x10_f64")
    cov = mdl.get_covariance()
    mean = mdl.theta[0]
    N = 200000
    x = mdl.sample(N, seed=2024)
    xc = x - mean
    s = xc.T.dot(xc) / N
    d = np.diag(cov)
    zs = (s - cov) / np.sqrt((np.outer(d, d) + cov ** 2) / N)
    assert np.abs(zs).max() < 6, np.abs(zs).max()
    n = x.shape[1]
    q = mdl.mahalanobis(x[:50000])
    assert abs(q.mean() - n) < 6 * np.sqrt(2 * n / len(q)), (q.mean(), n)


def test_sample_errors():
    from linearcorex_b200 import Corex
    from conftest import load_golden
    _z, kw, x = load_golden("readme_demo_f64")
    syn = Corex(**dict(kw, discourage_overlap=False, max_iter=5, precision="fp64")).fit(x)
    with pytest.raises(ValueError, match="discourage_overlap"):
        syn.sample(3, seed=0)
    with pytest.raises(ValueError, match="discourage_overlap"):
        syn.sample_missing(_with_nans(x, 0.1, 1), seed=0)
    none = Corex(**dict(kw, gaussianize="none", max_iter=5)).fit(x)
    with pytest.raises(ValueError, match="theta"):
        none.sample(3, seed=0)
    with pytest.raises(ValueError, match="theta"):
        none.impute(_with_nans(x, 0.1, 1), return_std=True)
    mdl = Corex(**dict(kw, precision="fp64")).fit(x)
    with pytest.raises(ValueError, match="n_draws"):
        mdl.sample_missing(x, n_draws=0)
    with pytest.raises(ValueError, match="seed"):
        mdl.sample(3, seed=-1)
    bad = pickle.loads(pickle.dumps(mdl))
    bad.moments["rhoinvrho"] = bad.moments["rhoinvrho"] * 3.0
    with pytest.raises(np.linalg.LinAlgError, match="positive definite"):
        bad.sample(3, seed=0)
    with pytest.raises(np.linalg.LinAlgError, match="positive definite"):
        bad.sample_missing(_with_nans(x, 0.1, 1), seed=0)
    assert np.all(np.isfinite(mdl.sample(3, seed=0)))  # the session is still usable


@pytest.mark.parametrize("name,precision,algorithm,train_frac", PARITY)
def test_impute_std_parity_with_dense_conditional(name, precision, algorithm, train_frac):
    mdl, held = _fit(name, precision, algorithm, train_frac)
    cov = mdl.get_covariance()
    mean, sd = mdl.theta
    for rate in (0.0, 0.01, 0.3, 0.9):
        x = _with_nans(held[:100], rate, 7)
        x[-1] = np.nan  # one row with nothing observed
        mask = missing_mask(x, mdl.missing_values)
        imp, std = mdl.impute(x, return_std=True)
        assert np.array_equal(imp, mdl.impute(x))
        assert std.shape == x.shape and np.all(std[~mask] == 0.0)
        assert np.abs(std[-1] / sd - 1).max() < 1e-12
        got, want = [], []
        for l in range(len(x) - 1):
            if mask[l].any():
                got.append(std[l, mask[l]] / sd[mask[l]])
                want.append(np.sqrt(np.diag(dense_conditional_cov(cov, sd, mask[l]))))
        if got:
            got, want = np.concatenate(got), np.concatenate(want)
            assert _rel(got, want) < 1e-10, (rate, _rel(got, want))


def _synthetic(m):
    from linearcorex_b200 import Corex
    n = max(50, 6 * m)
    rng = np.random.RandomState(m)
    z = rng.randn(m, n)
    z *= np.sqrt(0.8 * rng.uniform(0.2, 1.0, n)) / np.linalg.norm(z, axis=0)
    si = rng.rand(n)
    mean, sd = rng.randn(n), 0.5 + rng.rand(n)
    mdl = Corex(n_hidden=m, precision="fp64")
    mdl.nv, mdl.eps, mdl.theta = n, 0.0, (mean, sd)
    mdl.moments = {"rhoinvrho": z * (1 + si), "Si": si}
    return mdl, rng


def _sample_class(k, n, m):
    """_cond_class in the sampling mode: a row with nothing observed solves the order-m system of Path B."""
    if k == n:
        return (1 if m <= 64 else 2 if m <= 160 else 3), "B"
    return _cond_class(k, n, m)


@pytest.mark.parametrize("m", [1, 7, 100, 161, 500])
def test_size_classes_std_and_draws_against_numpy(m):
    mdl, rng = _synthetic(m)
    n = mdl.nv
    mean, sd = mdl.theta
    ks = sorted({k for k in (0, 1, 2, 64, 65, 160, 161, 300, m - 1, m, m + 1, n // 2, n - 161, n - 65, n - 2, n - 1, n)
                 if 0 <= k <= n})
    x = mean + sd * rng.randn(len(ks), n)
    for l, k in enumerate(ks):
        x[l, rng.permutation(n)[:k]] = np.nan
    want = np.zeros(8, dtype=np.int64)
    for k in ks:
        cls, path = _sample_class(k, n, m)
        want[cls] += 1
        if path:
            want[4 if path == "A" else 5] += 1
    imp, std = mdl.impute(x, return_std=True)
    assert np.array_equal(mdl._condition_counts, want), (mdl._condition_counts, want)
    seed, first_row, nd = 99, 1000, 17  # 17 draws: a full chunk of 16 and one more
    draws = mdl.sample_missing(x, n_draws=nd, seed=seed, first_row=first_row)
    assert np.array_equal(mdl._condition_counts, want), (mdl._condition_counts, want)
    assert np.array_equal(imp, mdl.impute(x))
    w = woodbury(mdl.moments["rhoinvrho"], mdl.moments["Si"], 0.0, mean, sd)
    for l, k in enumerate(ks):
        mk = np.isnan(x[l])
        assert np.all(std[l, ~mk] == 0.0) and all(np.array_equal(draws[d, l, ~mk], x[l, ~mk]) for d in range(nd))
        if k == 0:
            continue
        _cls, path = _sample_class(k, n, m)
        ref = lowrank_std(w, mk, path)
        assert _rel(std[l, mk] / sd[mk], ref) < 1e-10, (m, k, path, _rel(std[l, mk] / sd[mk], ref))
        mm = draw_map(w, mk, path)
        xh = (imp[l, mk] - mean[mk]) / sd[mk]
        for d in (0, 15, 16):
            eps = normals(seed, 1, [first_row + l], d, mm.shape[1])[0]
            got = (draws[d, l, mk] - mean[mk]) / sd[mk] - xh
            assert _rel(got, mm.dot(eps)) < 1e-9, (m, k, path, d, _rel(got, mm.dot(eps)))


def test_sample_missing_bit_identity(tmp_path):
    import torch
    mdl, x = _fit("syn_400x300x10_f64")
    x = _with_nans(x[:120], 0.3, 2)
    x[5] = np.nan
    mask = np.isnan(x)
    want = mdl.sample_missing(x, n_draws=3, seed=11)
    assert want.shape == (3,) + x.shape and np.all(np.isfinite(want))
    assert all(np.array_equal(want[d][~mask], x[~mask]) for d in range(3))
    assert not np.array_equal(want[0][mask], want[1][mask])
    got = lambda m, xx, **kw: m.sample_missing(xx, n_draws=3, seed=11, **kw)
    for rows in (None, 7, 64):
        mdl.stream_rows = rows
        for _ in range(2):
            assert np.array_equal(got(mdl, x), want), rows
    mdl.stream_rows = 32

    class Rows(object):
        shape = x.shape

        def __getitem__(self, sl):
            return x[sl]
    assert np.array_equal(got(mdl, Rows()), want)
    for alt in (torch.from_numpy(x).cuda(), x.astype(np.float64).tolist()):
        assert np.array_equal(got(mdl, alt), want)
    dev = got(mdl, torch.from_numpy(x).cuda(), return_device=True)
    assert dev.is_cuda and np.array_equal(dev.cpu().numpy(), want)
    assert np.array_equal(np.concatenate([got(mdl, x[:50]), got(mdl, x[50:], first_row=50)], axis=1), want)
    clone = pickle.loads(pickle.dumps(mdl))
    assert np.array_equal(got(clone, x), want)
    x32 = x.astype(np.float32)
    d32 = mdl.sample_missing(x32, n_draws=2, seed=1)
    assert all(np.array_equal(d32[d][~mask], x32.astype(np.float64)[~mask]) for d in range(2))


def test_sample_missing_statistics():
    mdl, x = _fit("syn_400x300x10_f64")
    cov = mdl.get_covariance()
    mean, sd = mdl.theta
    n, m = x.shape[1], mdl.m
    rng = np.random.RandomState(3)
    for k, path in ((5, "A"), (200, "B")):
        assert _cond_class(k, n, m)[1] == path
        row = x[:1].copy()
        mk = np.zeros(n, dtype=bool)
        mk[rng.permutation(n)[:k]] = True
        row[0, mk] = np.nan
        D = 4000
        dr = mdl.sample_missing(row, n_draws=D, seed=8)[:, 0, mk]
        assert mdl._condition_counts[4 if path == "A" else 5] == 1
        xh = mdl.impute(row)[0, mk]
        t = (dr - mean[mk]) / sd[mk]
        th = (xh - mean[mk]) / sd[mk]
        c = dense_conditional_cov(cov, sd, mk)
        zm = (t.mean(axis=0) - th) / np.sqrt(np.diag(c) / D)
        assert np.abs(zm).max() < 6, (path, np.abs(zm).max())
        s = (t - th).T.dot(t - th) / D
        dc = np.diag(c)
        zc = (s - c) / np.sqrt((np.outer(dc, dc) + c ** 2) / D)
        assert np.abs(zc).max() < 6, (path, np.abs(zc).max())
        imp_ref = dense_conditional(cov, mean, sd, row, mk[None])[0][0, mk]
        assert _rel((xh - mean[mk]) / sd[mk], (imp_ref - mean[mk]) / sd[mk]) < 1e-10
