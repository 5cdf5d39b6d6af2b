"""Corex.conditional (ConditionalGaussian) on the B200: parity with the dense conditional Gaussian and with the per-row path
(impute, impute(return_std=True), score_samples(missing='marginalize')), the full-row score when everything is observed,
bit-identity under blockings, containers, repeats, pickling and row splits of the draws, the tag-2 generator against
tests/philox_ref.py, statistics of the draws, every size class of the pattern factor, errors and the two-rank mean."""
import os
import pickle
import sys

import numpy as np
import pytest

from conftest import load_golden
from dense_conditional import dense_conditional
from dense_given import given_parts, given_rows
from dense_sampling import dense_conditional_cov
from philox_ref import normals, stream_words
from test_conditional_given_model import _patterns
from test_gpu_sampling import _synthetic
from test_gpu_score import PARITY, _fit

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300) if np.size(b) else 0.0


def _rows(mdl, x, count):
    """count held-out rows with the fixture's own markers replaced by theta[0]: the tests decide what is observed."""
    x = np.array(x[:count], dtype=np.float64)
    if mdl.missing_values is not None:
        x = np.where(x == mdl.missing_values, mdl.theta[0], x)
    return x


def _split(n, n_obs, seed):
    perm = np.random.RandomState(seed).permutation(n)
    return np.sort(perm[:n_obs]), perm[n_obs:]


@pytest.mark.parametrize("name,precision,algorithm,train_frac", PARITY)
def test_parity_with_dense_and_per_row_paths(name, precision, algorithm, train_frac):
    mdl, held = _fit(name, precision, algorithm, train_frac)
    x = _rows(mdl, held, 100)
    cov = mdl.get_covariance()
    mean, sd = mdl.theta
    n = len(mean)
    for label, obs, tgt in _patterns(n, 5):
        cg = mdl.conditional(obs, tgt)
        miss = np.ones(n, dtype=bool)
        miss[obs] = False
        imp_ref, logp_ref, q_ref = dense_conditional(cov, mean, sd, x, np.broadcast_to(miss, x.shape))
        pred = cg.predict(x[:, obs])
        assert pred.shape == (len(x), len(tgt)) and pred.dtype == np.float64
        st = lambda v: (v - mean[tgt]) / sd[tgt]
        assert _rel(st(pred), st(imp_ref[:, tgt])) < 1e-10, (label, _rel(st(pred), st(imp_ref[:, tgt])))
        pos = np.cumsum(miss) - 1
        ccov = dense_conditional_cov(cov, sd, miss)[np.ix_(pos[tgt], pos[tgt])]
        assert _rel(cg.std / sd[tgt], np.sqrt(np.diag(ccov))) < 1e-10, label
        assert _rel(cg.get_covariance(block_rows=64) / np.outer(sd[tgt], sd[tgt]), ccov) < 1e-10, label
        logp, q = cg.score_samples(x[:, obs]), cg.mahalanobis(x[:, obs])
        if len(obs) == 0:
            assert np.all(logp == 0.0) and np.all(q == 0.0) and np.array_equal(pred, np.broadcast_to(mean[tgt], pred.shape))
        else:
            assert _rel(logp, logp_ref) < 1e-10 and _rel(q, q_ref) < 1e-10, (label, _rel(logp, logp_ref), _rel(q, q_ref))
            assert abs(cg.score(x[:, obs]) - logp_ref.mean()) < 1e-10 * np.abs(logp_ref).max()
        if len(obs) + len(tgt) < n:
            continue
        # the per-row path on the same rows with T set to NaN (T is the whole complement of O)
        holes = x.copy()
        holes[:, tgt] = np.nan
        imp, std = mdl.impute(holes, return_std=True)
        assert _rel(st(pred), st(imp[:, tgt])) < 1e-10, (label, _rel(st(pred), st(imp[:, tgt])))
        assert _rel(cg.std / sd[tgt], std[0, tgt] / sd[tgt]) < 1e-10, label
        assert _rel(logp, mdl.score_samples(holes, missing="marginalize")) < 1e-10, label


def test_everything_observed_is_the_full_score():
    mdl, x = _fit("adni_l0_f64")
    x = _rows(mdl, x, 200)
    n = x.shape[1]
    cg = mdl.conditional(np.arange(n))
    assert len(cg.targets) == 0
    assert _rel(cg.score_samples(x), mdl.score_samples(x)) < 1e-12
    assert _rel(cg.mahalanobis(x), mdl.mahalanobis(x)) < 1e-12
    assert cg.predict(x).shape == (len(x), 0) and cg.sample(x, n_draws=2, seed=1).shape == (2, len(x), 0)
    assert cg.std.shape == (0,) and cg.get_covariance().shape == (0, 0)
    perm = np.random.RandomState(0).permutation(n)  # any order of the observed columns
    assert _rel(mdl.conditional(perm).score_samples(x[:, perm]), mdl.score_samples(x)) < 1e-12


def test_bit_identity_blockings_containers_pickling_and_refit():
    import torch
    mdl, x = _fit("syn_400x300x10_f64")
    obs, tgt = _split(x.shape[1], 200, 1)
    cg = mdl.conditional(obs, tgt)
    xo = np.ascontiguousarray(x[:, obs])
    got = lambda c, xx: (c.predict(xx), c.score_samples(xx), c.mahalanobis(xx), c.sample(xx, n_draws=3, seed=11))
    same = lambda a, b: all(np.array_equal(u, v) for u, v in zip(a, b))
    want = got(cg, xo)
    assert want[3].shape == (3, len(xo), len(tgt)) and not np.array_equal(want[3][0], want[3][1])

    class Rows(object):
        shape = xo.shape

        def __getitem__(self, sl):
            return xo[sl]
    for rows in (None, 7, 128):
        cg.stream_rows = rows
        for _ in range(2):
            assert same(got(cg, xo), want) and same(got(cg, Rows()), want), rows
    cg.stream_rows = None
    for alt in (torch.from_numpy(xo).cuda(), xo.tolist()):
        assert same(got(cg, alt), want)
    x32 = xo.astype(np.float32)
    want32 = got(cg, x32.astype(np.float64))
    assert same(got(cg, x32), want32) and same(got(cg, torch.from_numpy(x32).cuda()), want32)
    dev = cg.predict(torch.from_numpy(xo).cuda(), return_device=True)
    assert dev.is_cuda and np.array_equal(dev.cpu().numpy(), want[0])
    split = np.concatenate([cg.sample(xo[:150], n_draws=3, seed=11), cg.sample(xo[150:], n_draws=3, seed=11, first_row=150)],
                           axis=1)
    assert np.array_equal(split, want[3])
    assert np.array_equal(cg.sample(xo[10:20], n_draws=3, seed=11, first_row=10), want[3][:, 10:20])
    std, cov = cg.std, cg.get_covariance()
    clone = pickle.loads(pickle.dumps(cg))
    assert same(got(clone, xo), want) and np.array_equal(clone.std, std) and np.array_equal(clone.get_covariance(), cov)
    assert same(got(pickle.loads(pickle.dumps(mdl)).conditional(obs, tgt), xo), want)
    np.random.seed(5)
    a = cg.sample(xo[:4])
    np.random.seed(5)
    assert np.array_equal(cg.sample(xo[:4]), a) and not np.array_equal(a, cg.sample(xo[:4]))
    mdl.fit(x[:200])  # refitting the parent leaves an object built before untouched
    assert same(got(cg, xo), want) and np.array_equal(cg.std, std)


def test_draws_match_philox_reference():
    import torch
    from linearcorex_b200 import _lib
    mdl, x = _fit("readme_demo_f64")
    mean, sd = mdl.theta
    obs, tgt = _split(x.shape[1], 7, 2)
    cg = mdl.conditional(obs, tgt)
    m, nt = mdl.m, len(tgt)
    seed, first_row, rows = 2 ** 63 + 5, 2 ** 32 - 3, 6
    xo = np.asarray(x[:rows], dtype=np.float64)[:, obs]
    d = cg.sample(xo, n_draws=2, seed=seed, first_row=first_row)
    g = given_parts(mdl.moments["rhoinvrho"], mdl.moments["Si"], mdl.eps, sd, obs, tgt)
    v = ((xo - mean[obs]) / sd[obs]).dot(g["A"].T)
    for dd in range(2):
        eps = normals(seed, 2, np.arange(first_row, first_row + rows), dd, m + nt)
        want = (v + eps[:, :m]).dot(g["P"]) + np.sqrt(g["delta"][tgt]) * eps[:, m:]
        assert _rel((d[dd] - mean[tgt]) / sd[tgt], want) < 1e-11, _rel((d[dd] - mean[tgt]) / sd[tgt], want)
    sess = cg._session()
    out = torch.zeros((rows, 16), dtype=torch.float64, device=sess.device)
    words = torch.zeros((rows, 32), dtype=torch.int32, device=sess.device)
    _lib.check(sess.lib.lcx_normal_fill(sess.h, seed, 2, first_row, rows, 1, 13, out.data_ptr(), 16, words.data_ptr(), 32),
               "lcx_normal_fill")
    want_w = stream_words(seed, 2, np.arange(first_row, first_row + rows), 1, 13)
    assert np.array_equal(words.cpu().numpy().view(np.uint32)[:, :28].reshape(rows, 7, 4).astype(np.uint64), want_w)


def test_draw_moments():
    mdl, x = _fit("syn_400x300x10_f64")
    mean, sd = mdl.theta
    obs, tgt = _split(x.shape[1], 280, 3)
    cg = mdl.conditional(obs, tgt)
    row = np.asarray(x[:1], dtype=np.float64)[:, obs]
    D = 20000
    t = (cg.sample(row, n_draws=D, seed=8)[:, 0] - mean[tgt]) / sd[tgt]
    th = (cg.predict(row)[0] - mean[tgt]) / sd[tgt]
    c = cg.get_covariance() / np.outer(sd[tgt], sd[tgt])
    dc = np.diag(c)
    zm = (t.mean(axis=0) - th) / np.sqrt(dc / D)  # each a standard normal under the model: 6 sigma over 20 entries
    assert np.abs(zm).max() < 6, np.abs(zm).max()
    s = (t - th).T.dot(t - th) / D
    zc = (s - c) / np.sqrt((np.outer(dc, dc) + c ** 2) / D)
    assert np.abs(zc).max() < 6, np.abs(zc).max()


@pytest.mark.parametrize("m", [1, 7, 100, 161, 500])
def test_sizes_against_numpy_and_impute(m):
    mdl, rng = _synthetic(m)
    n = mdl.nv
    mean, sd = mdl.theta
    x = mean + sd * rng.randn(12, n)
    obs, tgt = _split(n, n - min(300, n // 2), m)
    cg = mdl.conditional(obs, tgt)
    g = given_parts(mdl.moments["rhoinvrho"], mdl.moments["Si"], 0.0, sd, obs, tgt)
    want_mean, want_cov, want_q, want_logp = given_rows(g, ((x - mean) / sd)[:, obs], obs, tgt)
    pred = cg.predict(x[:, obs])
    assert _rel((pred - mean[tgt]) / sd[tgt], want_mean) < 1e-10, m
    assert _rel(cg.get_covariance() / np.outer(sd[tgt], sd[tgt]), want_cov) < 1e-10, m
    assert _rel(cg.std / sd[tgt], np.sqrt(np.diag(want_cov))) < 1e-10, m
    assert _rel(cg.mahalanobis(x[:, obs]), want_q) < 1e-10 and _rel(cg.score_samples(x[:, obs]), want_logp) < 1e-10, m
    holes = x.copy()
    holes[:, tgt] = np.nan
    imp = mdl.impute(holes)
    assert _rel((pred - mean[tgt]) / sd[tgt], (imp[:, tgt] - mean[tgt]) / sd[tgt]) < 1e-10, m
    if m == 500:  # the per-row path took its order-|M| global-slab class (|M| = 300 > 160)
        assert mdl._condition_counts[3] == len(x) and mdl._condition_counts[4] == len(x)


def test_errors():
    from linearcorex_b200 import Corex
    _z, kw, x = load_golden("readme_demo_f64")
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[1]
    syn = Corex(**dict(kw, discourage_overlap=False, max_iter=5, precision="fp64")).fit(x)
    with pytest.raises(ValueError, match="discourage_overlap"):
        syn.conditional([0])
    none = Corex(**dict(kw, gaussianize="none", max_iter=5)).fit(x)
    with pytest.raises(ValueError, match="theta"):
        none.conditional([0])
    mdl = Corex(**dict(kw, precision="fp64", missing_values=-7.5)).fit(x)
    for obs, tgt in (([n], None), ([-1], None), ([0, 0], None), ([0], [1, 1]), ([0], [n]), ([0, 1], [1, 2]), ([[0, 1]], None),
                     ([0.5], None)):
        with pytest.raises(ValueError):
            mdl.conditional(obs, tgt)
    cg = mdl.conditional([0, 2, 4], [1, 3])
    with pytest.raises(ValueError, match="shape"):
        cg.predict(x[:, :4])
    for bad_value in (np.nan, -7.5):
        bad = x[:5, [0, 2, 4]].copy()
        bad[3, 1] = bad_value
        for call in (cg.predict, cg.score_samples, lambda b: cg.sample(b, seed=0)):
            with pytest.raises(ValueError, match="impute"):
                call(bad)
    with pytest.raises(ValueError, match="n_draws"):
        cg.sample(x[:5, [0, 2, 4]], n_draws=0)
    broken = pickle.loads(pickle.dumps(mdl))
    broken.moments["rhoinvrho"] = broken.moments["rhoinvrho"] * 3.0
    with pytest.raises(np.linalg.LinAlgError, match="positive definite"):
        broken.conditional([0, 2, 4])
    assert np.all(np.isfinite(cg.predict(x[:5, [0, 2, 4]])))  # still usable
    empty = mdl.conditional([], [1, 3])
    assert np.array_equal(empty.predict(np.zeros((4, 0))), np.broadcast_to(mdl.theta[0][[1, 3]], (4, 2)))
    assert np.array_equal(empty.score_samples(np.zeros((4, 0))), np.zeros(4))
    assert cg.predict(x[:0, [0, 2, 4]]).shape == (0, 2)


def _two_rank_worker(rank, world, port, ret):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from conftest import load_golden as lg
        from linearcorex_b200 import Corex, shard_rows
        _z, kw, x = lg("syn_400x300x10_f64")
        x = np.asarray(x, dtype=np.float64)
        lo, hi = shard_rows(x.shape[0], rank, world)
        mdl = Corex(comm=True, **dict(kw, precision="fp64")).fit(x[lo:hi])
        obs = np.arange(0, x.shape[1], 3)
        cg = mdl.conditional(obs)
        whole = float(np.mean(cg.score_samples(x[:, obs])))
        got = cg.score(x[lo:hi, obs])
        assert abs(got - whole) < 1e-12 * abs(whole), (got, whole)
        t = torch.tensor([got], dtype=torch.float64, device="cuda")
        lo_t, hi_t = t.clone(), t.clone()
        dist.all_reduce(lo_t, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_t, op=dist.ReduceOp.MAX)
        assert torch.equal(lo_t, hi_t)
        ret[rank] = "ok"
    except Exception:
        import traceback
        ret[rank] = "FAIL: %s" % traceback.format_exc()
    finally:
        dist.destroy_process_group()


def test_two_rank_score():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ret = mp.Manager().dict()
    mp.spawn(_two_rank_worker, args=(2, 30000 + os.getpid() % 1000, ret), nprocs=2, join=True)
    assert len(ret) == 2 and all(v == "ok" for v in ret.values()), dict(ret)
