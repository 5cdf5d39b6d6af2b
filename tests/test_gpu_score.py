"""Corex.score_samples / mahalanobis / score / get_precision on the B200: parity with the dense reference in standardised
space (tests/dense_score.py), independence of the row blocking, input containers, pickling, the factor across the one-CTA /
cooperative Cholesky boundary, errors and the two-rank mean."""
import os
import pickle
import sys

import numpy as np
import pytest

from conftest import load_golden
from dense_score import dense_precision, dense_scores, woodbury

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fit(name, precision="fp64", algorithm="auto", train_frac=None):
    from linearcorex_b200 import Corex
    _z, kw, x = load_golden(name)
    x = np.asarray(x, dtype=np.float64)
    held = x
    if train_frac is not None:
        cut = int(train_frac * x.shape[0])
        x, held = x[:cut], x[cut:]
    mdl = Corex(**dict(kw, precision=precision, algorithm=algorithm)).fit(x)
    return mdl, held


def _rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


PARITY = [("readme_demo_f64", "fp64", "auto", None), ("big5_l0_f64", "fp64", "auto", None),
          ("syn_400x300x10_f64", "fp64_split", "stream", None), ("syn_400x300x10_f64", "fp64_split", "gram", None),
          ("syn_400x300x10_f64", "fp64", "stream", 0.8), ("syn_60x400x8_f64", "fp64", "auto", None),
          ("outliers_f64", "fp64", "auto", None), ("standard_missing_f64", "fp64_split", "stream", 0.8),
          ("adni_l0_f64", "fp64", "auto", None)]


@pytest.mark.parametrize("name,precision,algorithm,train_frac", PARITY)
def test_parity_with_dense_reference(name, precision, algorithm, train_frac):
    mdl, x = _fit(name, precision, algorithm, train_frac)
    if algorithm != "auto":
        assert mdl.algorithm_used == algorithm
    cov = mdl.get_covariance()
    mean, sd = mdl.theta
    logp_ref, q_ref = dense_scores(cov, mean, sd, x, mdl.missing_values)
    logp, q = mdl.score_samples(x), mdl.mahalanobis(x)
    assert logp.shape == (x.shape[0],) and logp.dtype == np.float64
    assert _rel(logp, logp_ref) < 1e-10, _rel(logp, logp_ref)
    assert _rel(q, q_ref) < 1e-10, _rel(q, q_ref)
    assert abs(mdl.score(x) - logp_ref.mean()) < 1e-10 * abs(logp_ref.mean())
    ss = np.outer(sd, sd)  # compared in standardised space (adni's column scales span 1e5)
    assert _rel(mdl.get_precision() * ss, dense_precision(cov, sd) * ss) < 1e-10


def test_row_blocks_repeats_and_row_providers_are_bit_identical(tmp_path):
    mdl, x = _fit("syn_400x300x10_f64")
    want = mdl.score_samples(x), mdl.mahalanobis(x)
    for rows in (None, 7, 128):
        mdl.stream_rows = rows
        for _ in range(2):
            assert np.array_equal(mdl.score_samples(x), want[0]) and np.array_equal(mdl.mahalanobis(x), want[1]), rows
    mdl.stream_rows = 64

    class Rows(object):
        shape = x.shape

        def __getitem__(self, sl):
            return x[sl]
    assert np.array_equal(mdl.score_samples(Rows()), want[0])
    np.save(str(tmp_path / "x.npy"), x)
    assert np.array_equal(mdl.score_samples(np.load(str(tmp_path / "x.npy"), mmap_mode="r")), want[0])


def test_input_containers():
    import torch
    mdl, x = _fit("big5_l0_f64")
    want = mdl.score_samples(x)
    for alt in (torch.from_numpy(x).cuda(), torch.from_numpy(x).pin_memory(), x.tolist()):
        assert np.array_equal(mdl.score_samples(alt), want)
    x32 = x.astype(np.float32)
    want32 = mdl.score_samples(x32.astype(np.float64))  # float32 values are exact in binary64
    for alt in (x32, torch.from_numpy(x32).cuda(), torch.from_numpy(x32).pin_memory()):
        assert np.array_equal(mdl.score_samples(alt), want32)
    assert _rel(want32, want) < 1e-5


def test_nan_without_marker_poisons_only_its_row():
    mdl, x = _fit("readme_demo_f64")
    want = mdl.score_samples(x)
    bad = x.copy()
    bad[3, 2] = np.nan
    got = mdl.score_samples(bad)
    assert np.isnan(got[3]) and np.array_equal(np.delete(got, 3), np.delete(want, 3))


def test_unpickled_and_lazy_models(monkeypatch):
    from linearcorex_b200 import Corex
    mdl, x = _fit("syn_400x300x10_f64")
    clone = pickle.loads(pickle.dumps(mdl))
    assert np.array_equal(clone.score_samples(x), mdl.score_samples(x))
    assert np.array_equal(clone.get_precision(), mdl.get_precision())
    monkeypatch.setattr(Corex, "LAZY_MOMENTS_BYTES", 0)
    _z, kw, xs = load_golden("syn_400x300x10_f64")
    lazy = Corex(**dict(kw, precision="fp64")).fit(xs)
    pending = lazy.moments.pending()
    assert "rhoinvrho" in pending
    assert np.array_equal(lazy.score_samples(x), mdl.score_samples(x))
    lazy.get_precision(block_rows=64)
    assert lazy.moments.pending() == pending


def test_precision_outputs_odd_n(tmp_path):
    import torch
    from linearcorex_b200 import Corex
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from corex_oracle import latent_factor_data
    x = latent_factor_data(500, 201, 5, seed=3, snr=1.0, snr_spread=0.3).astype(np.float64)
    mdl = Corex(n_hidden=5, seed=0, precision="fp64").fit(x)
    n = 201
    ref = dense_precision(mdl.get_covariance(), mdl.theta[1])
    full = mdl.get_precision(block_rows=50)
    ss = np.outer(mdl.theta[1], mdl.theta[1])
    assert _rel(full * ss, ref * ss) < 1e-10
    dst = np.zeros((n, n))
    mdl.get_precision(block_rows=50, out=dst)
    mm = np.lib.format.open_memmap(str(tmp_path / "p.npy"), mode="w+", dtype=np.float64, shape=(n, n))
    mdl.get_precision(block_rows=50, out=mm)
    dev = torch.zeros((n, n + 1), dtype=torch.float64, device="cuda")[:, :n]
    mdl.get_precision(block_rows=50, out=dev)
    got = np.zeros((n, n))

    def cb(r0, block):
        got[r0:r0 + block.shape[0]] = block.cpu().numpy()
    mdl.get_precision(block_rows=50, block_callback=cb)
    for other in (dst, np.asarray(mm), dev.cpu().numpy(), got):
        assert np.array_equal(other, full)


@pytest.mark.parametrize("m", [1, 7, 100, 161, 500])
def test_factor_against_numpy_cholesky(m):
    import ctypes as C
    import torch
    from linearcorex_b200 import _lib
    from linearcorex_b200.corex import _DeviceSession
    n = max(50, 6 * m)
    rng = np.random.RandomState(m)
    z = rng.randn(m, n)
    z *= np.sqrt(0.8 * rng.uniform(0.2, 1.0, n)) / np.linalg.norm(z, axis=0)  # sum_j Z_ji^2 in [0.16, 0.8]: Delta > 0
    si = rng.rand(n)
    sd = 0.5 + rng.rand(n)
    rinv = z * (1 + si)
    sess = _DeviceSession(_lib.PRECISION_FP64)
    lib = sess.lib
    ld = lib.lcx_ld(n)
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=sess.device)
    rd = torch.zeros((m, ld), dtype=torch.float64, device=sess.device)
    rd[:, :n] = dev(rinv)
    b = torch.zeros((m, ld), dtype=torch.float64, device=sess.device)
    dinv = torch.empty(n, dtype=torch.float64, device=sess.device)
    logdet = torch.empty(1, dtype=torch.float64, device=sess.device)
    nscr = lib.lcx_lowrank_scratch_doubles(m, n)
    scr = torch.empty(nscr, dtype=torch.float64, device=sess.device)
    sdd, sid = dev(sd), dev(si)
    _lib.check(lib.lcx_lowrank_factor(sess.h, rd.data_ptr(), sid.data_ptr(), ld, m, n, 0.0, sdd.data_ptr(), b.data_ptr(), ld,
                                      dinv.data_ptr(), logdet.data_ptr(), scr.data_ptr(), nscr), "lcx_lowrank_factor")
    w = woodbury(rinv, si, 0.0, None, sd)
    assert _rel(b[:, :n].cpu().numpy(), w["B"]) < 1e-12
    assert _rel(dinv.cpu().numpy(), 1 / w["delta"]) < 1e-14
    assert abs(logdet.item() - w["logdet"]) < 1e-12 * abs(w["logdet"])
    sess.close()


def test_scale_against_woodbury():
    from linearcorex_b200 import Corex
    n, m, rows = 20000, 100, 2000
    rng = np.random.RandomState(7)
    z = rng.randn(m, n) * 0.6 / np.sqrt(m)
    si = rng.rand(n)
    mean, sd = rng.randn(n), 0.5 + rng.rand(n)
    mdl = Corex(n_hidden=m, precision="fp64")
    mdl.nv, mdl.eps, mdl.theta = n, 0.0, (mean, sd)
    mdl.moments = {"rhoinvrho": z * (1 + si), "Si": si}
    x = mean + sd * rng.randn(rows, n)
    w = woodbury(mdl.moments["rhoinvrho"], si, 0.0, mean, sd, x)
    assert _rel(mdl.score_samples(x), w["logp"]) < 1e-10
    assert _rel(mdl.mahalanobis(x), w["q"]) < 1e-10


def test_errors():
    from linearcorex_b200 import Corex
    _z, kw, x = load_golden("readme_demo_f64")
    syn = Corex(**dict(kw, discourage_overlap=False, max_iter=5, precision="fp64")).fit(x)
    with pytest.raises(ValueError, match="discourage_overlap"):
        syn.score_samples(x)
    none = Corex(**dict(kw, gaussianize="none", max_iter=5)).fit(x)
    with pytest.raises(ValueError, match="theta"):
        none.score_samples(x)
    mdl = Corex(**dict(kw, precision="fp64")).fit(x)
    with pytest.raises(AssertionError):
        mdl.score_samples(x[:, :-1])
    bad = pickle.loads(pickle.dumps(mdl))
    bad.moments["rhoinvrho"] = bad.moments["rhoinvrho"] * 3.0
    with pytest.raises(np.linalg.LinAlgError, match="positive definite"):
        bad.score_samples(x)
    assert np.all(np.isfinite(mdl.score_samples(x)))  # the session is still usable


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
        whole = float(np.mean(mdl.score_samples(x)))  # no missing marker: score_samples is rank-local
        got = mdl.score(x[lo:hi])
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
    mp.spawn(_two_rank_worker, args=(2, 29800 + os.getpid() % 1000, ret), nprocs=2, join=True)
    assert len(ret) == 2 and all(v == "ok" for v in ret.values()), dict(ret)
