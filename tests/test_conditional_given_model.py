"""CPU checks of the model behind Corex.conditional (ConditionalGaussian): the fixed-pattern factor restated in numpy
(tests/dense_given.py) must give the dense conditional Gaussian's mean, covariance, q and log p (tests/dense_conditional.py,
tests/dense_sampling.py) on every ns float64 golden, for patterns from one target to one observed column, a target set that
is a strict subset of the unobserved columns, and nothing observed."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_golden
from dense_conditional import dense_conditional
from dense_given import given_parts, given_rows
from dense_sampling import dense_conditional_cov

# test_data has duplicate columns (Delta = 2.2e-16: numerically singular, see test_lowrank_model.py)
NS_F64 = sorted(f[:-4] for f in os.listdir(GOLDEN)
                if f.endswith("_f64.npz") and not f.startswith("test_data")
                and "covariance" in np.load(os.path.join(GOLDEN, f)).files
                and bool(np.load(os.path.join(GOLDEN, f)).get("kw_discourage_overlap", True)))


def _patterns(n, seed):
    """(label, observed, targets): |T| = 1, about 3 %, 50 %, n - 1, T a strict subset of the complement, O empty."""
    rng = np.random.RandomState(seed)
    out = []
    for label, nt in (("T=1", 1), ("3%", max(1, int(round(0.03 * n)))), ("50%", n // 2), ("T=n-1", n - 1)):
        perm = rng.permutation(n)
        out.append((label, np.sort(perm[nt:]), perm[:nt]))
    perm = rng.permutation(n)
    out.append(("subset", perm[:n // 3], perm[n // 3 + max(1, n // 10):][::-1]))  # targets in a scrambled order
    out.append(("O empty", np.zeros(0, dtype=np.int64), rng.permutation(n)[:max(1, n // 4)]))
    return out


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def test_fixture_list():
    assert "adni_l0_f64" in NS_F64 and "readme_demo_f64" in NS_F64 and "big5_syn_f64" not in NS_F64


@pytest.mark.parametrize("name", NS_F64)
def test_fixed_pattern_matches_dense_conditional(name):
    z, kw, x = load_golden(name)
    mean, sd, eps = z["theta_mean"], z["theta_std"], float(z["eps_final"])
    x = np.asarray(x, dtype=np.float64)[:4]
    mv = kw.get("missing_values")
    if mv is not None:  # the patterns below decide what is observed
        x = np.where(x == mv, mean, x)
    cov = z["covariance"]
    n = len(mean)
    xt = (x - mean) / sd
    for label, obs, tgt in _patterns(n, 3):
        g = given_parts(z["m_rhoinvrho"], z["m_Si"], eps, sd, obs, tgt)
        got_mean, got_cov, got_q, got_logp = given_rows(g, xt[:, obs], obs, tgt)
        miss = np.ones(n, dtype=bool)
        miss[obs] = False
        imp, logp, q = dense_conditional(cov, mean, sd, x, np.broadcast_to(miss, x.shape))
        want_mean = (imp[:, tgt] - mean[tgt]) / sd[tgt]
        assert _rel(got_mean, want_mean) < 1e-11, (name, label)
        want_cov = dense_conditional_cov(cov, sd, miss)
        pos = np.cumsum(miss) - 1  # position of each unobserved column in the rows of want_cov
        want_cov = want_cov[np.ix_(pos[tgt], pos[tgt])]
        assert _rel(got_cov, want_cov) < 1e-11, (name, label, _rel(got_cov, want_cov))
        if len(obs) == 0:
            assert np.all(got_q == 0.0) and np.all(got_logp == 0.0) and g["logdet"] == 0.0
            continue
        assert np.all(np.abs(got_q - q) < 1e-11 * np.maximum(np.abs(q), 1.0)), (name, label)
        assert np.all(np.abs(got_logp - logp) < 1e-11 * np.abs(logp)), (name, label)


def test_all_observed_is_the_full_score():
    from dense_score import woodbury
    z, _kw, x = load_golden("readme_demo_f64")
    mean, sd, eps = z["theta_mean"], z["theta_std"], float(z["eps_final"])
    n = len(mean)
    obs = np.arange(n)
    g = given_parts(z["m_rhoinvrho"], z["m_Si"], eps, sd, obs, np.zeros(0, dtype=np.int64))
    w = woodbury(z["m_rhoinvrho"], z["m_Si"], eps, mean, sd, x[:5])
    _m, _c, q, logp = given_rows(g, (np.asarray(x[:5], dtype=np.float64) - mean) / sd, obs, [])
    assert _rel(g["A"], w["B"]) < 1e-13 and abs(g["logdet"] - w["logdet"]) < 1e-13 * abs(w["logdet"])
    assert _rel(q, w["q"]) < 1e-12 and _rel(logp, w["logp"]) < 1e-12
