"""Corex.impute and score_samples / mahalanobis / score(missing='marginalize') on the B200: parity with the dense
conditional Gaussian (tests/dense_conditional.py), bit-identity with scoring on complete rows and with the input on observed
entries, independence of the row blocking, containers and pickling, every size class of the per-row kernel, errors, the
two-rank mean and a held-out imputation property."""
import os
import pickle
import sys

import numpy as np
import pytest

from conftest import load_golden
from dense_conditional import dense_conditional, lowrank_paths, missing_mask
from dense_score import woodbury
from test_gpu_score import PARITY, _fit, _rel

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _with_nans(x, rate, seed):
    x = np.array(x, dtype=np.float64)
    if rate:
        x[np.random.RandomState(seed).rand(*x.shape) < rate] = np.nan
    return x


@pytest.mark.parametrize("name,precision,algorithm,train_frac", PARITY)
def test_parity_with_dense_conditional(name, precision, algorithm, train_frac):
    mdl, held = _fit(name, precision, algorithm, train_frac)
    cov = mdl.get_covariance()
    mean, sd = mdl.theta
    for rate in (0.0, 0.01, 0.3, 0.9):
        x = _with_nans(held[:200], rate, 5)
        mask = missing_mask(x, mdl.missing_values)
        imp_ref, logp_ref, q_ref = dense_conditional(cov, mean, sd, x, mask)
        imp = mdl.impute(x)
        logp = mdl.score_samples(x, missing="marginalize")
        q = mdl.mahalanobis(x, missing="marginalize")
        assert imp.shape == x.shape and imp.dtype == np.float64 and logp.shape == (len(x),)
        assert np.array_equal(imp[~mask], x[~mask])
        if mask.any():
            got, want = ((imp - mean) / sd)[mask], ((imp_ref - mean) / sd)[mask]
            assert _rel(got, want) < 1e-10, (rate, _rel(got, want))
        assert _rel(logp, logp_ref) < 1e-10, (rate, _rel(logp, logp_ref))
        assert _rel(q, q_ref) < 1e-10, (rate, _rel(q, q_ref))
        assert abs(mdl.score(x, missing="marginalize") - logp_ref.mean()) < 1e-10 * np.abs(logp_ref).max()


def test_complete_rows_are_bit_identical_to_scoring():
    mdl, x = _fit("syn_400x300x10_f64")
    part = _with_nans(x, 0.004, 1)  # about 30 % of the rows lose an entry
    full = ~np.isnan(part).any(axis=1)
    assert 0 < full.sum() < len(x)
    assert np.array_equal(mdl.score_samples(part, missing="marginalize")[full], mdl.score_samples(x)[full])
    assert np.array_equal(mdl.mahalanobis(part, missing="marginalize")[full], mdl.mahalanobis(x)[full])
    assert np.array_equal(mdl.score_samples(x, missing="marginalize"), mdl.score_samples(x))
    imp = mdl.impute(part)
    assert np.array_equal(imp[full], x[full]) and np.array_equal(imp[~np.isnan(part)], part[~np.isnan(part)])
    x32 = part.astype(np.float32)
    assert np.array_equal(mdl.impute(x32)[~np.isnan(part)], x32.astype(np.float64)[~np.isnan(part)])


def test_blockings_containers_repeats_and_pickling_are_bit_identical(tmp_path):
    import torch
    mdl, x = _fit("syn_400x300x10_f64")
    x = _with_nans(x, 0.3, 2)
    want = mdl.impute(x), mdl.score_samples(x, missing="marginalize"), mdl.mahalanobis(x, missing="marginalize")
    got = lambda m, xx: (m.impute(xx), m.score_samples(xx, missing="marginalize"), m.mahalanobis(xx, missing="marginalize"))
    same = lambda a, b: all(np.array_equal(u, v, equal_nan=True) for u, v in zip(a, b))
    for rows in (None, 7, 128):
        mdl.stream_rows = rows
        for _ in range(2):
            assert same(got(mdl, x), want), rows
    mdl.stream_rows = 64

    class Rows(object):
        shape = x.shape

        def __getitem__(self, sl):
            return x[sl]
    assert same(got(mdl, Rows()), want)
    np.save(str(tmp_path / "x.npy"), x)
    assert same(got(mdl, np.load(str(tmp_path / "x.npy"), mmap_mode="r")), want)
    for alt in (torch.from_numpy(x).cuda(), torch.from_numpy(x).pin_memory(), x.tolist()):
        assert same(got(mdl, alt), want)
    dev = mdl.impute(torch.from_numpy(x).cuda(), return_device=True)
    assert dev.is_cuda and np.array_equal(dev.cpu().numpy(), want[0])
    clone = pickle.loads(pickle.dumps(mdl))
    assert same(got(clone, x), want)


def test_marker_is_conditioned_on_without_column_means():
    mdl, x = _fit("adni_l0_f64")
    mv = mdl.missing_values
    mask = missing_mask(x, mv)
    assert mask.any()
    as_nan = np.where(mask, np.nan, x)
    assert np.array_equal(mdl.score_samples(x, missing="marginalize"), mdl.score_samples(as_nan, missing="marginalize"))
    imp = mdl.impute(x)
    assert np.array_equal(imp, mdl.impute(as_nan)) and not np.any(imp == mv)


def _cond_class(k, n, m):
    """Python mirror of cond_order / cond_class (lowrank_kernels.cuh): 0 nothing to solve, 1 order <= 64, 2 <= 160, 3 beyond."""
    if k == 0 or k == n:
        return 0, None
    path_a = k * k * m + k ** 3 / 3.0 <= (n - k) * m * m + m ** 3 / 3.0
    p = k if path_a else m
    return (1 if p <= 64 else 2 if p <= 160 else 3), ("A" if path_a else "B")


@pytest.mark.parametrize("m", [1, 7, 100, 161, 500])
def test_size_classes_against_numpy(m):
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
    ks = sorted({k for k in (0, 1, 2, 64, 65, 160, 161, 300, m - 1, m, m + 1, n // 2, n - 161, n - 65, n - 2, n - 1, n)
                 if 0 <= k <= n})
    x = mean + sd * rng.randn(len(ks), n)
    for l, k in enumerate(ks):
        x[l, rng.permutation(n)[:k]] = np.nan
    imp, logp, q = mdl.impute(x), mdl.score_samples(x, missing="marginalize"), mdl.mahalanobis(x, missing="marginalize")
    counts = mdl._condition_counts
    want = np.zeros(8, dtype=np.int64)
    for k in ks:
        cls, path = _cond_class(k, n, m)
        want[cls] += 1
        if path:
            want[4 if path == "A" else 5] += 1
    assert np.array_equal(counts, want), (counts, want)
    w = woodbury(mdl.moments["rhoinvrho"], si, 0.0, mean, sd)
    for l, k in enumerate(ks):
        mk = np.isnan(x[l])
        xt = np.where(mk, 0.0, (x[l] - mean) / sd)
        xh, qq, lp = lowrank_paths(w, xt, mk, w["logdet"], sd, "A" if k <= 1000 else "B")
        if 0 < k < n:
            got = (imp[l, mk] - mean[mk]) / sd[mk]
            assert _rel(got, xh) < 1e-10, (m, k, _rel(got, xh))
        assert abs(q[l] - qq) <= 1e-10 * max(abs(qq), 1.0), (m, k, q[l], qq)
        assert abs(logp[l] - lp) <= 1e-10 * max(abs(lp), 1.0), (m, k, logp[l], lp)
        assert np.array_equal(imp[l, ~mk], x[l, ~mk])


def test_errors():
    from linearcorex_b200 import Corex
    _z, kw, x = load_golden("readme_demo_f64")
    x = _with_nans(x, 0.1, 3)
    syn = Corex(**dict(kw, discourage_overlap=False, max_iter=5, precision="fp64")).fit(np.nan_to_num(x))
    with pytest.raises(ValueError, match="discourage_overlap"):
        syn.impute(x)
    with pytest.raises(ValueError, match="discourage_overlap"):
        syn.score_samples(x, missing="marginalize")
    none = Corex(**dict(kw, gaussianize="none", max_iter=5)).fit(np.nan_to_num(x))
    with pytest.raises(ValueError, match="theta"):
        none.impute(x)
    mdl = Corex(**dict(kw, precision="fp64")).fit(np.nan_to_num(x))
    with pytest.raises(ValueError, match="missing"):
        mdl.score_samples(x, missing="drop")
    with pytest.raises(AssertionError):
        mdl.impute(x[:, :-1])
    bad = pickle.loads(pickle.dumps(mdl))
    bad.moments["rhoinvrho"] = bad.moments["rhoinvrho"] * 3.0
    with pytest.raises(np.linalg.LinAlgError, match="positive definite"):
        bad.impute(x)
    with pytest.raises(np.linalg.LinAlgError, match="positive definite"):
        bad.mahalanobis(x, missing="marginalize")
    assert np.all(np.isfinite(mdl.score_samples(x, missing="marginalize")))  # the session is still usable
    assert mdl.impute(x[:0]).shape == (0, x.shape[1])


def test_impute_beats_column_means_on_held_out_entries():
    from linearcorex_b200 import Corex
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from corex_oracle import latent_factor_data
    x = latent_factor_data(3000, 200, 5, seed=11, snr=1.0, snr_spread=0.3).astype(np.float64)
    train, test = x[:2000], x[2000:]
    mdl = Corex(n_hidden=5, seed=0, precision="fp64").fit(train)
    mask = np.random.RandomState(4).rand(*test.shape) < 0.2
    holes = np.where(mask, np.nan, test)
    err_model = np.mean((mdl.impute(holes)[mask] - test[mask]) ** 2)
    col_means = np.nanmean(holes, axis=0)
    err_means = np.mean((np.broadcast_to(col_means, test.shape)[mask] - test[mask]) ** 2)
    assert err_model < 0.8 * err_means, (err_model, err_means)


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
        holes = x.copy()
        holes[np.random.RandomState(9).rand(*x.shape) < 0.3] = np.nan
        whole = float(np.mean(mdl.score_samples(holes, missing="marginalize")))  # rank-local: no column-mean pass
        got = mdl.score(holes[lo:hi], missing="marginalize")
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


def test_two_rank_marginal_score():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ret = mp.Manager().dict()
    mp.spawn(_two_rank_worker, args=(2, 29900 + os.getpid() % 1000, ret), nprocs=2, join=True)
    assert len(ret) == 2 and all(v == "ok" for v in ret.values()), dict(ret)
