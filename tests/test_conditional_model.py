"""CPU checks of the model behind Corex.impute and score_samples / mahalanobis(missing='marginalize'), on the stored
goldens: both per-row systems of the device path (order |M| and order m, tests/dense_conditional.py) must agree with the
dense conditional Gaussian in standardised space, and with each other."""
import numpy as np
import pytest

from conftest import load_golden
from dense_conditional import dense_conditional, lowrank_paths
from dense_score import woodbury

NAMES = ["readme_demo_f64", "syn_60x400x8_f64", "adni_l0_f64"]


def _setup(name):
    z, kw, x = load_golden(name)
    mean, sd, eps = z["theta_mean"], z["theta_std"], float(z["eps_final"])
    w = woodbury(z["m_rhoinvrho"], z["m_Si"], eps, mean, sd)
    x = np.asarray(x, dtype=np.float64)
    mv = kw.get("missing_values")
    if mv is not None:  # keep the rows free of the golden's own markers; the masks below decide what is missing
        x = np.where(x == mv, mean, x)
    return z, x, mean, sd, w


def _masks(n, m, seed):
    rng = np.random.RandomState(seed)
    out = []
    for k in sorted({0, 1, m - 1, m, m + 1, n - 1, n}):
        mk = np.zeros(n, dtype=bool)
        mk[rng.permutation(n)[:k]] = True
        out.append(("k=%d" % k, mk))
    for rate in (0.01, 0.3, 0.9):
        out.append(("%g" % rate, rng.rand(n) < rate))
    return out


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


@pytest.mark.parametrize("name", NAMES)
def test_paths_match_dense_conditional(name):
    z, x, mean, sd, w = _setup(name)
    m, n = w["B"].shape
    cov = z["covariance"]
    for l, (label, mk) in enumerate(_masks(n, m, 1)):
        row = x[l % len(x)]
        imp, logp, q = dense_conditional(cov, mean, sd, row[None], mk[None])
        xt = (row - mean) / sd
        for path in ("A", "B"):
            xh, qq, lp = lowrank_paths(w, xt, mk, w["logdet"], sd, path)
            if mk.any() and not mk.all():
                want = (imp[0, mk] - mean[mk]) / sd[mk]
                assert _rel(xh, want) < 1e-11, (name, label, path, _rel(xh, want))
            if mk.all():
                assert lp == 0.0 and qq == 0.0
                continue
            assert abs(qq - q[0]) < 1e-11 * max(abs(q[0]), 1.0), (name, label, path, qq, q[0])
            assert abs(lp - logp[0]) < 1e-11 * abs(logp[0]), (name, label, path, lp, logp[0])


@pytest.mark.parametrize("name", NAMES)
def test_paths_agree(name):
    _z, x, mean, sd, w = _setup(name)
    m, n = w["B"].shape
    for l, (label, mk) in enumerate(_masks(n, m, 2)):
        xt = (x[l % len(x)] - mean) / sd
        a = lowrank_paths(w, xt, mk, w["logdet"], sd, "A")
        b = lowrank_paths(w, xt, mk, w["logdet"], sd, "B")
        if mk.any():
            assert _rel(a[0], b[0]) < 1e-11 if not mk.all() else np.array_equal(a[0], b[0]), (name, label)
        assert abs(a[1] - b[1]) < 1e-11 * max(abs(a[1]), 1.0) and abs(a[2] - b[2]) <= 1e-11 * abs(a[2]), (name, label)


def test_complete_row_is_the_full_score_and_empty_row_is_zero():
    z, x, mean, sd, w = _setup("readme_demo_f64")
    n = w["B"].shape[1]
    full = woodbury(z["m_rhoinvrho"], z["m_Si"], float(z["eps_final"]), mean, sd, x[:3])
    for l in range(3):
        xt = (x[l] - mean) / sd
        _xh, q, lp = lowrank_paths(w, xt, np.zeros(n, dtype=bool), w["logdet"], sd, "A")
        assert abs(q - full["q"][l]) < 1e-12 * abs(full["q"][l]) and abs(lp - full["logp"][l]) < 1e-12 * abs(full["logp"][l])
        xh, q, lp = lowrank_paths(w, xt, np.ones(n, dtype=bool), w["logdet"], sd, "B")
        assert lp == 0.0 and q == 0.0 and not xh.any()
    imp, logp, q = dense_conditional(z["covariance"], mean, sd, x[:1], np.ones((1, n), dtype=bool))
    assert logp[0] == 0.0 and q[0] == 0.0 and np.array_equal(imp[0], mean)
