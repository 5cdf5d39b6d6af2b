"""Per-row sample weights on the device: `Corex.fit(x, sample_weight=w)`.

Weights enter only the column statistics and the one pass that writes X~ (row l scaled by r_l = sqrt(N w_l / W)); the fit
loop is unchanged.  So all-ones weights (and any power-of-two multiple of a weight vector) must give bit-identical fits on
every route and precision, integer weights must match the fit of the repeated rows, and non-integer weights the weighted
reference (tests/weighted_oracle.py).  `algorithm` is pinned in every test: repeating rows changes N and with it what
'auto' would choose."""
import os
import sys

import numpy as np
import pytest

from conftest import load_golden
import weighted_oracle as wo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (golden, constructor overrides): every route, precision, gaussianize mode and preparation path
BIT_CASES = [
    ("syn_400x300x10_f64", dict(precision="fp64", algorithm="stream")),
    ("syn_400x300x10_f64", dict(precision="fp64_split", algorithm="stream")),
    ("syn_400x300x10_f64", dict(precision="fp64_split", algorithm="gram")),
    ("syn_400x300x10_f64", dict(precision="fp64_split7", algorithm="stream")),
    ("syn_400x300x10_f64", dict(precision="fp64_split", algorithm="stream", exact_trials=True)),
    ("syn_400x300x10_f64", dict(precision="fp64_split", algorithm="stream", input_dtype="float32")),
    ("syn_400x300x10_f64", dict(precision="fp64_split", algorithm="stream", stream_rows=96)),
    ("outliers_f64", dict(precision="fp64_split", algorithm="stream")),
    ("outliers_missing_f64", dict(precision="fp64", algorithm="stream")),
    ("standard_missing_f64", dict(precision="fp64_split", algorithm="stream")),
    ("standard_missing_f64", dict(precision="fp64_split", algorithm="gram")),
    # unstandardised, this fit reaches a non-finite TC after ~140 iterations (weighted or not): stop well before
    ("syn_400x300x10_f64", dict(precision="fp64", algorithm="stream", gaussianize="none", max_iter=15)),
    ("syn_400x300x10_f64", dict(precision="fp64_split", algorithm="stream", gaussianize="none", max_iter=15)),
    ("syn_400x300x10_synergy_f64", dict(precision="fp64", algorithm="stream")),
    ("syn_400x300x10_synergy_f64", dict(precision="fp64_split", algorithm="stream")),
]
TOL_CASES = [
    ("syn_400x300x10_f64", dict(precision="fp64", algorithm="stream")),
    ("syn_400x300x10_f64", dict(precision="fp64_split", algorithm="stream")),
    ("syn_400x300x10_f64", dict(precision="fp64_split", algorithm="gram")),
    ("syn_400x300x10_f64", dict(precision="fp64_split7", algorithm="stream")),
    ("outliers_f64", dict(precision="fp64_split", algorithm="stream")),
    ("standard_missing_f64", dict(precision="fp64", algorithm="stream")),
    ("standard_missing_f64", dict(precision="fp64_split", algorithm="stream")),
    ("syn_400x300x10_synergy_f64", dict(precision="fp64", algorithm="stream")),
]
ORACLE_CASES = ["syn_400x300x10_f64", "outliers_f64", "standard_missing_f64", "syn_400x300x10_synergy_f64"]


def _ids(cases):
    return ["%s-%s" % (n, "-".join("%s=%s" % kv for kv in sorted(o.items()))) for n, o in cases]


def _fit(name, w=None, x=None, **over):
    from linearcorex_b200 import Corex
    _, kw, x0 = load_golden(name)
    kw.update(over)
    return Corex(**kw).fit(x0 if x is None else x, sample_weight=w)


def _weights(n, kind, seed=3):
    rng = np.random.RandomState(seed)
    return rng.randint(0, 4, size=n).astype(np.float64) if kind == "int" else rng.uniform(0.1, 3.0, size=n)


def assert_same(a, b):
    """Bit-identical fits: W, every moment, theta, the TC history and the per-iteration trace."""
    np.testing.assert_array_equal(a.ws, b.ws)
    np.testing.assert_array_equal(a.history["TC"], b.history["TC"])
    np.testing.assert_equal(a.trace, b.trace)
    assert set(a.moments.keys()) == set(b.moments.keys())
    for key in a.moments.keys():
        np.testing.assert_array_equal(np.asarray(a.moments[key]), np.asarray(b.moments[key]), err_msg=key)
    if a.theta is None:
        assert b.theta is None
    else:
        for s, t in zip(a.theta, b.theta):
            np.testing.assert_array_equal(s, t)


def _rel(a, b, floor=0.0):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), floor, 1e-300)


def deviation(got, want):
    """Largest relative deviation over W, the TC history and every moment; theta separately."""
    errs = {"ws": _rel(got.ws, want.ws), "TC": _rel(got.history["TC"], want.history["TC"])}
    for key, val in want.moments.items():
        floor = abs(want.tc) if key in ("additivity", "TC_direct", "TC_no_overlap") else 0.0
        errs[key] = _rel(got.moments[key], val, floor)
    theta = max(_rel(s, t) for s, t in zip(got.theta, want.theta)) if want.theta is not None else 0.0
    return max(errs.values()), errs, theta


def assert_close(got, want, tol=1e-9, theta_tol=1e-12):
    assert len(got.history["TC"]) == len(want.history["TC"])
    worst, errs, theta = deviation(got, want)
    assert worst <= tol, {k: v for k, v in errs.items() if v > tol}
    assert theta <= theta_tol, theta
    np.testing.assert_array_equal(got.clusters(), want.clusters())


@pytest.mark.parametrize("name,over", BIT_CASES, ids=_ids(BIT_CASES))
def test_all_ones_and_rescaled_weights_are_bit_identical(name, over):
    n = len(load_golden(name)[2])
    assert_same(_fit(name, np.ones(n), **over), _fit(name, **over))
    w = _weights(n, "real")
    assert_same(_fit(name, 4.0 * w, **over), _fit(name, w, **over))


@pytest.mark.parametrize("name,over", TOL_CASES, ids=_ids(TOL_CASES))
def test_integer_weights_match_repeated_rows(name, over):
    _, _, x = load_golden(name)
    w = _weights(len(x), "int")
    got = _fit(name, w, **over)
    want = _fit(name, x=np.repeat(x, w.astype(np.int64), axis=0), **over)
    assert got.algorithm_used == want.algorithm_used == over["algorithm"]
    assert_close(got, want)
    np.testing.assert_allclose(got.n_obs, want.n_obs, rtol=1e-15)
    assert got.n_samples == len(x)


@pytest.mark.parametrize("name,over", TOL_CASES[:5], ids=_ids(TOL_CASES[:5]))
def test_zero_weights_remove_rows(name, over):
    _, _, x = load_golden(name)
    w = _weights(len(x), "int")
    keep = w > 0
    assert_close(_fit(name, w, **over), _fit(name, w[keep], x=x[keep], **over))


@pytest.mark.parametrize("algorithm", ["stream", "gram"])
def test_zero_weight_outlier_stays_out_of_the_exponent(algorithm):
    name = "syn_400x300x10_f64"
    _, _, x = load_golden(name)
    x = x.copy()
    w = _weights(len(x), "int")
    x[np.flatnonzero(w == 0)[0]] = 1e6
    split = _fit(name, w, x=x, precision="fp64_split", algorithm=algorithm)
    ref = _fit(name, w, x=x, precision="fp64", algorithm="stream")
    assert_close(split, ref)


@pytest.mark.parametrize("name", ORACLE_CASES)
@pytest.mark.parametrize("precision,algorithm", [("fp64", "stream"), ("fp64_split", "stream"), ("fp64_split", "gram")])
def test_real_weights_match_weighted_oracle(name, precision, algorithm):
    z, kw, x = load_golden(name)
    w = _weights(len(x), "real")
    want = wo.WeightedOracleCorex(work_dtype=np.float64, **kw).fit(x, sample_weight=w)
    got = _fit(name, w, precision=precision, algorithm=algorithm)
    assert_close(got, want, theta_tol=1e-12)
    np.testing.assert_allclose(got.n_obs, want.n_obs, rtol=1e-13)


def test_one_row_with_half_the_weight():
    """Very uneven weights raise the shared exponent of X~ in the split modes by log2(max r): fp64 and fp64_split7 hold
    1e-9; fp64_split's deviation is printed (DESIGN.md section 12 records it)."""
    name = "syn_400x300x10_f64"
    z, kw, x = load_golden(name)
    w = np.ones(len(x))
    w[0] = len(x) - 1.0
    want = wo.WeightedOracleCorex(work_dtype=np.float64, **kw).fit(x, sample_weight=w)
    for precision in ("fp64", "fp64_split7", "fp64_split"):
        got = _fit(name, w, precision=precision, algorithm="stream")
        worst, errs, theta = deviation(got, want)
        print("half-weight row: %s max rel dev %.3e (ws %.3e) theta %.3e, %d vs %d iterations"
              % (precision, worst, errs["ws"], theta, len(got.history["TC"]), len(want.history["TC"])))
        if precision != "fp64_split":
            assert_close(got, want, theta_tol=1e-12)
        else:
            assert worst < 1e-6


def test_streamed_preparation_is_bit_identical_to_resident():
    """One 4096-row slab per block: the streamed passes add the same slab partials in the same order."""
    import corex_oracle as oc
    x = oc.latent_factor_data(10000, 96, 6, seed=5, dtype=np.float64)
    w = _weights(len(x), "real")
    for algorithm in ("stream", "gram"):
        kw = dict(n_hidden=6, seed=1, max_iter=30, precision="fp64_split", algorithm=algorithm)
        assert_same(_fit_raw(x, w, stream_rows=4096, **kw), _fit_raw(x, w, **kw))


def _fit_raw(x, w, **kw):
    from linearcorex_b200 import Corex
    return Corex(**kw).fit(x, sample_weight=w)


def test_weight_containers_are_bit_identical():
    import torch
    name = "standard_missing_f64"
    _, _, x = load_golden(name)
    w = _weights(len(x), "real")
    over = dict(precision="fp64_split", algorithm="stream")
    base = _fit(name, w, **over)
    for cont in (list(w), torch.from_numpy(w.copy()), torch.from_numpy(w.copy()).cuda()):
        assert_same(_fit(name, cont, **over), base)


@pytest.mark.parametrize("bad", ["short", "2d", "negative", "nan", "inf", "zeros"])
def test_invalid_weights_raise_and_leave_the_model_untouched(bad):
    from linearcorex_b200 import Corex
    _, kw, x = load_golden("syn_400x300x10_f64")
    n = len(x)
    w = {"short": np.ones(n - 1), "2d": np.ones((n, 1)), "negative": np.r_[-1.0, np.ones(n - 1)],
         "nan": np.r_[np.nan, np.ones(n - 1)], "inf": np.r_[np.inf, np.ones(n - 1)], "zeros": np.zeros(n)}[bad]
    mdl = Corex(precision="fp64", algorithm="stream", **kw).fit(x)
    ws, theta, hist = mdl.ws.copy(), tuple(t.copy() for t in mdl.theta), list(mdl.history["TC"])
    with pytest.raises(ValueError):
        mdl.fit(x, sample_weight=w)
    np.testing.assert_array_equal(mdl.ws, ws)
    np.testing.assert_array_equal(mdl.theta[0], theta[0])
    assert list(mdl.history["TC"]) == hist
    fresh = Corex(precision="fp64", algorithm="stream", **kw)
    with pytest.raises(ValueError):
        fresh.fit(x, sample_weight=w)
    assert fresh.ws.size == 0 and fresh._sess is None


def test_weighted_score():
    name = "syn_400x300x10_f64"
    _, _, x = load_golden(name)
    w = _weights(len(x), "real")
    mdl = _fit(name, w, precision="fp64", algorithm="stream")
    logp = mdl.score_samples(x)
    want = np.average(logp, weights=w)
    assert abs(mdl.score(x, sample_weight=w) - want) <= 1e-13 * abs(want)
    plain = mdl.score(x)
    assert abs(mdl.score(x, sample_weight=np.ones(len(x))) - plain) <= 1e-15 * abs(plain)
    with pytest.raises(ValueError):
        mdl.score(x, sample_weight=-np.ones(len(x)))


def test_fit_layers_passes_weights_to_every_layer():
    from linearcorex_b200 import Corex
    from linearcorex_b200.hierarchy import fit_layers
    _, _, x = load_golden("syn_400x300x10_f64")
    w = _weights(len(x), "real")
    kw = dict(seed=2, max_iter=40, precision="fp64", algorithm="stream")
    models = fit_layers(x, [6, 2], sample_weight=w, **kw)
    assert len(models) == 3
    cur, prev = x, None
    for mdl, width in zip(models, [6, 2, 1]):
        if prev is not None:
            cur = prev.transform(cur, return_device=True)
        prev = Corex(n_hidden=width, **kw).fit(cur, sample_weight=w)
        assert_same(mdl, prev)


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
        from conftest import load_golden
        from linearcorex_b200 import Corex, shard_rows
        for name, prec, algo in (("syn_400x300x10_f64", "fp64", "stream"), ("standard_missing_f64", "fp64_split", "stream"),
                                 ("syn_400x300x10_f64", "fp64_split", "gram")):
            z, kw, x = load_golden(name)
            w = np.random.RandomState(3).uniform(0.1, 3.0, size=len(x))
            kw = dict(kw, precision=prec, algorithm=algo)
            lo, hi = shard_rows(x.shape[0], rank, world)
            mdl = Corex(comm=True, **kw).fit(x[lo:hi], sample_weight=w[lo:hi])
            single = Corex(**kw).fit(x, sample_weight=w)
            assert mdl.n_samples == x.shape[0] and mdl.algorithm_used == algo
            assert len(mdl.history["TC"]) == len(single.history["TC"])
            err = np.abs(mdl.ws - single.ws).max() / np.abs(single.ws).max()
            err_tc = np.abs(mdl.moments["TCs"] - single.moments["TCs"]).max() / np.abs(single.moments["TCs"]).max()
            assert err < 1e-9 and err_tc < 1e-9, (name, prec, algo, err, err_tc)
            t = torch.from_numpy(mdl.ws.copy()).cuda()
            lo_t, hi_t = t.clone(), t.clone()
            dist.all_reduce(lo_t, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi_t, op=dist.ReduceOp.MAX)
            assert torch.equal(lo_t, hi_t)
            s = mdl.score(x[lo:hi], sample_weight=w[lo:hi])
            assert abs(s - single.score(x, sample_weight=w)) <= 1e-9 * abs(s)
        ret[rank] = "ok"
    except Exception:
        import traceback
        ret[rank] = "FAIL: %s" % traceback.format_exc()
    finally:
        dist.destroy_process_group()


def test_two_rank_weighted_fit():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_two_rank_worker, args=(2, 29100 + os.getpid() % 1000, ret), nprocs=2, join=True)
    assert all(str(v) == "ok" for v in ret.values()) and len(ret) == 2, dict(ret)
