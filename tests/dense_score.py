"""Reference computations for the scoring methods (Corex.score_samples / mahalanobis / get_precision) -- test helpers only.

dense_*     the dense reference: Gaussian log-density, squared Mahalanobis distance and precision of N(mean, cov) computed
            in standardised space, on C = S^-1 cov S^-1 (S = diag(sd)) with np.linalg.slogdet + np.linalg.solve, then
            log det cov = log det C + 2 sum log sd.  Unlike scipy on the raw covariance it does not mistake widely spread
            column scales (adni: 6e-3 .. 1.2e3) for singularity.
woodbury    a numpy restatement of the low-rank-plus-diagonal identities the device path implements
            (linearcorex_b200/csrc/lowrank_kernels.cuh).
Missing entries of new data are imputed with the new data's column means, as transform does (corex_oracle.impute_missing).
"""
import numpy as np

from corex_oracle import impute_missing

LOG_2PI = np.log(2 * np.pi)


def standardized_rows(x, mean, sd, missing_values=None):
    x = np.asarray(x, dtype=np.float64)
    if missing_values is not None:
        x, _ = impute_missing(x, missing_values)
    return (x - mean) / sd


def dense_scores(cov, mean, sd, x, missing_values=None):
    """(log p, q) of the rows of x under N(mean, cov)."""
    sd = np.asarray(sd, dtype=np.float64)
    c = cov / np.outer(sd, sd)
    sign, logdet_c = np.linalg.slogdet(c)
    assert sign > 0
    xt = standardized_rows(x, mean, sd, missing_values)
    q = np.einsum('li,il->l', xt, np.linalg.solve(c, xt.T))
    logdet = logdet_c + 2 * np.sum(np.log(sd))
    return -0.5 * (cov.shape[0] * LOG_2PI + logdet + q), q


def dense_precision(cov, sd):
    sd = np.asarray(sd, dtype=np.float64)
    c = cov / np.outer(sd, sd)
    return np.linalg.solve(c, np.eye(c.shape[0])) / np.outer(sd, sd)


def lowrank_parts(rhoinvrho, si, eps):
    """Z (m x n) and Delta (n) of Sigma = S (Z^T Z + Delta) S."""
    z = np.asarray(rhoinvrho, dtype=np.float64) / (1 + np.asarray(si, dtype=np.float64)) / np.sqrt(1. - eps ** 2)
    return z, 1. - np.sum(z ** 2, axis=0)


def woodbury(rhoinvrho, si, eps, mean, sd, x=None, missing_values=None):
    """dict with K, G, B, logdet, precision and, given x, logp and q -- the identities of lowrank_kernels.cuh in numpy."""
    import scipy.linalg
    sd = np.asarray(sd, dtype=np.float64)
    z, delta = lowrank_parts(rhoinvrho, si, eps)
    m = z.shape[0]
    k = np.eye(m) + (z / delta).dot(z.T)
    g = np.linalg.cholesky(k)
    b = scipy.linalg.solve_triangular(g, z / delta, lower=True)
    out = {"K": k, "G": g, "B": b, "delta": delta,
           "logdet": 2 * np.sum(np.log(sd)) + np.sum(np.log(delta)) + 2 * np.sum(np.log(np.diag(g))),
           "precision": (np.diag(1. / delta) - b.T.dot(b)) / np.outer(sd, sd)}
    if x is not None:
        xt = standardized_rows(x, mean, sd, missing_values)
        out["q"] = np.sum(xt ** 2 / delta, axis=1) - np.sum(xt.dot(b.T) ** 2, axis=1)
        out["logp"] = -0.5 * (z.shape[1] * LOG_2PI + out["logdet"] + out["q"])
    return out
