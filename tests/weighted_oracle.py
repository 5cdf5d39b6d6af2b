"""Per-row sample weights on top of oracle/corex_oracle.py -- TEST INFRASTRUCTURE ONLY.

The pinned oracle restates the reference, which has no weights.  This module adds them the way the device path does
(DESIGN.md section 12): the column statistics become weighted averages, and row l of X~ is scaled by
r_l = sqrt(N w_l / W) (W = sum of w), so that every average over rows the fit takes -- X~^T Y / N, sum_l Y_lj^2 / N --
is the w-weighted one.  `sample_weight=None` runs the oracle's own code unchanged.
"""
import numpy as np

import corex_oracle as oc


def row_scale(w, n_rows):
    """r_l = sqrt(N w_l / W), the expression lcx_row_scale evaluates."""
    w = np.asarray(w, dtype=np.float64)
    return np.sqrt((float(n_rows) * w) / np.sum(w))


def standardize(x, gaussianize, missing_values, theta=None, sample_weight=None):
    """oracle.standardize with per-row weights (fit only): returns (r-scaled x_tilde, theta, n_obs).

    Missing entries take the weighted mean of the observed entries; 'standard' divides the weighted squared deviations by
    the weighted observed count, 'outliers' by the weight total (np.std's N); n_obs is the weighted observed count."""
    if sample_weight is None:
        return oc.standardize(x, gaussianize, missing_values, theta=theta)
    assert theta is None, "weights only enter fit"
    w = np.asarray(sample_weight, dtype=np.float64)
    x = np.array(x, copy=True)
    w_total = np.sum(w)
    if missing_values is not None:
        if not np.isnan(missing_values):
            x = np.where(x == missing_values, np.nan, x)
        ok = np.isfinite(x)
        n_obs = np.sum(np.where(ok, w[:, None], 0.0), axis=0)
        mu_obs = np.sum(np.where(ok, w[:, None] * np.where(ok, x, 0.0), 0.0), axis=0) / n_obs
        x = np.where(np.isnan(x), mu_obs, x)
    else:
        n_obs = w_total
    if gaussianize in ('standard', 'outliers'):
        mu = np.sum(w[:, None] * x, axis=0) / w_total
        sq = np.sum(w[:, None] * (x - mu) ** 2, axis=0)
        sd = np.sqrt(sq / (n_obs if gaussianize == 'standard' else w_total)).clip(1e-10)
        theta = (mu, sd)
        x = (x - mu) / sd
        if gaussianize == 'outliers':
            x = oc.squash_tails(x)
    elif gaussianize != 'none':
        raise ValueError("gaussianize in {'standard','outliers','none'}")
    return row_scale(w, len(x))[:, None] * x, theta, n_obs


class WeightedOracleCorex(oc.OracleCorex):
    """OracleCorex whose fit takes `sample_weight`; everything after the preparation of X~ is the oracle's own code."""

    _sample_weight = None

    def preprocess(self, x, fit=False):
        if not fit or self._sample_weight is None:
            return super().preprocess(x, fit=fit)
        xt, theta, n_obs = standardize(x, self.gaussianize, self.missing_values, sample_weight=self._sample_weight)
        self.theta = theta
        self.n_obs = n_obs
        return xt

    def fit(self, x, sample_weight=None):
        self._sample_weight = sample_weight
        try:
            return super().fit(x)
        finally:
            self._sample_weight = None
