"""CPU checks of the model behind Corex.score_samples / mahalanobis / get_precision, on the stored goldens.

The ns covariance estimate (get_covariance, linearcorex.py:447-451) is S (Z^T Z + Delta) S exactly; the Woodbury /
Sylvester restatement of its log-density, Mahalanobis distance and precision (the identities the device path implements)
must agree with the dense reference in standardised space (tests/dense_score.py), which in turn agrees with scipy wherever
scipy accepts the matrix."""
import numpy as np
import pytest
import scipy.stats

from conftest import GOLDEN, load_golden
from dense_score import dense_precision, dense_scores, lowrank_parts, woodbury

import os

NS_WITH_COV = sorted(f[:-4] for f in os.listdir(GOLDEN)
                     if f.endswith(".npz") and "covariance" in np.load(os.path.join(GOLDEN, f)).files
                     and bool(np.load(os.path.join(GOLDEN, f)).get("kw_discourage_overlap", True)))
# test_data has duplicate columns: Delta = 2.2e-16 there, so the estimate is numerically singular and no dense or low-rank
# evaluation of its inverse is accurate to 1e-12 -- it is kept out of the tolerance checks below (not out of the rebuild).
# The `native` goldens hold float32 moments, so their stored covariance and its rebuild differ by float32 rounding.
WELL_POSED = [name for name in NS_WITH_COV if not name.startswith("test_data") and "native" not in name]


def _parts(name):
    z, kw, x = load_golden(name)
    return z, kw, x, z["theta_mean"], z["theta_std"], float(z["eps_final"])


def test_fixture_list():
    assert len(NS_WITH_COV) == 17 and "adni_l0_f64" in NS_WITH_COV and "big5_syn_f64" not in NS_WITH_COV


@pytest.mark.parametrize("name", NS_WITH_COV)
def test_covariance_is_low_rank_plus_diagonal(name):
    z, _kw, _x, _mean, sd, eps = _parts(name)
    zz, delta = lowrank_parts(z["m_rhoinvrho"], z["m_Si"], eps)
    assert np.all(delta > 0)
    cov = np.outer(sd, sd) * (zz.T.dot(zz) + np.diag(delta))
    # absolute in standardised space (the column scales of adni span 6e-3 .. 1.2e3)
    err = np.abs((cov - z["covariance"]) / np.outer(sd, sd)).max()
    assert err < (1e-6 if "native" in name else 1e-13), (name, err)


@pytest.mark.parametrize("name", WELL_POSED)
def test_dense_reference_matches_scipy(name):
    z, kw, x, mean, sd, _eps = _parts(name)
    try:
        ref = scipy.stats.multivariate_normal(mean, z["covariance"])
    except (ValueError, np.linalg.LinAlgError):
        pytest.skip("scipy rejects this covariance")
    if kw.get("missing_values") is not None:
        pytest.skip("scipy has no imputation")
    logp, _q = dense_scores(z["covariance"], mean, sd, x)
    want = ref.logpdf(np.asarray(x, dtype=np.float64))
    assert np.abs(logp - want).max() < 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("name", WELL_POSED)
def test_woodbury_matches_dense(name):
    z, kw, x, mean, sd, eps = _parts(name)
    mv = kw.get("missing_values")
    logp, q = dense_scores(z["covariance"], mean, sd, x, mv)
    w = woodbury(z["m_rhoinvrho"], z["m_Si"], eps, mean, sd, x, mv)
    assert np.abs(w["logp"] - logp).max() < 1e-12 * np.abs(logp).max()
    assert np.abs(w["q"] - q).max() < 1e-12 * np.abs(q).max()
    # S P S . S^-1 Sigma S^-1 - I: the product in standardised space, free of adni's 1e5 spread of column scales
    ss = np.outer(sd, sd)
    eye = np.eye(len(sd))
    assert np.abs((w["precision"] * ss).dot(z["covariance"] / ss) - eye).max() < 1e-12
    assert np.abs((dense_precision(z["covariance"], sd) * ss).dot(z["covariance"] / ss) - eye).max() < 1e-12


def test_adni_scipy_refuses_but_the_references_agree():
    z, kw, x, mean, sd, eps = _parts("adni_l0_f64")
    with pytest.raises((ValueError, np.linalg.LinAlgError)):
        scipy.stats.multivariate_normal(mean, z["covariance"])
    logp, q = dense_scores(z["covariance"], mean, sd, x, kw["missing_values"])
    w = woodbury(z["m_rhoinvrho"], z["m_Si"], eps, mean, sd, x, kw["missing_values"])
    assert np.all(np.isfinite(logp)) and np.abs(w["logp"] - logp).max() < 1e-12 * np.abs(logp).max()
