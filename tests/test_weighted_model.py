"""Per-row sample weights in the CPU reference (tests/weighted_oracle.py): the defining identity -- an integer-weighted
fit is the fit of the data with row l repeated w_l times -- plus exact invariance under power-of-two rescaling of the
weights and agreement of all-ones weights with the unweighted oracle.  CPU only."""
import numpy as np
import pytest

from conftest import load_golden
import weighted_oracle as wo

CASES = ["syn_400x300x10_f64", "outliers_f64", "standard_missing_f64", "syn_400x300x10_synergy_f64"]


def _fit(name, w=None, repeat=False, max_iter=None):
    _, kw, x = load_golden(name)
    if max_iter is not None:
        kw = dict(kw, max_iter=max_iter)
    mdl = wo.WeightedOracleCorex(work_dtype=np.float64, **kw)
    if repeat:
        return mdl.fit(np.repeat(x, w.astype(np.int64), axis=0))
    return mdl.fit(x, sample_weight=w)


def _weights(name, kind):
    _, _, x = load_golden(name)
    rng = np.random.RandomState(7)
    if kind == "int":
        return rng.randint(0, 4, size=len(x)).astype(np.float64)
    return rng.uniform(0.1, 3.0, size=len(x))


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _compare(got, want, tol, theta_tol):
    assert len(got.history["TC"]) == len(want.history["TC"])
    assert _rel(got.ws, want.ws) <= tol
    assert _rel(got.history["TC"], want.history["TC"]) <= tol
    for key, val in want.moments.items():
        floor = abs(want.tc) if key in ("additivity", "TC_direct", "TC_no_overlap") else 0.0
        err = np.abs(np.asarray(got.moments[key]) - val).max() / max(np.abs(val).max(), floor, 1e-300)
        assert err <= tol, (key, err)
    for a, b in zip(got.theta, want.theta):
        assert _rel(a, b) <= theta_tol
    np.testing.assert_array_equal(got.clusters(), want.clusters())


@pytest.mark.parametrize("name", CASES)
def test_integer_weights_equal_repeated_rows(name):
    w = _weights(name, "int")
    got, want = _fit(name, w), _fit(name, w, repeat=True)
    _compare(got, want, 1e-12, 1e-12)
    np.testing.assert_allclose(got.n_obs, want.n_obs, rtol=0, atol=0)
    assert got.n_samples == len(w) and want.n_samples == int(w.sum())


@pytest.mark.parametrize("name", CASES)
def test_power_of_two_rescaling_is_exact(name):
    w = _weights(name, "real")
    a, b = _fit(name, w, max_iter=20), _fit(name, 4.0 * w, max_iter=20)
    np.testing.assert_array_equal(a.ws, b.ws)
    np.testing.assert_array_equal(a.history["TC"], b.history["TC"])
    for key, val in a.moments.items():
        np.testing.assert_array_equal(b.moments[key], val, err_msg=key)
    for s, t in zip(a.theta, b.theta):
        np.testing.assert_array_equal(s, t)


@pytest.mark.parametrize("name", CASES)
def test_all_ones_match_unweighted(name):
    w = np.ones(len(load_golden(name)[2]))
    got, want = _fit(name, w), _fit(name)
    _compare(got, want, 1e-13, 1e-13)


def test_zero_weight_rows_are_removed():
    name = "outliers_f64"
    w = _weights(name, "int")
    _, kw, x = load_golden(name)
    x = x.copy()
    x[np.flatnonzero(w == 0)[:3]] *= 1e6  # outliers on rows that carry no weight change nothing
    got = wo.WeightedOracleCorex(work_dtype=np.float64, **kw).fit(x, sample_weight=w)
    keep = w > 0
    want = wo.WeightedOracleCorex(work_dtype=np.float64, **kw).fit(x[keep], sample_weight=w[keep])
    _compare(got, want, 1e-12, 1e-12)
