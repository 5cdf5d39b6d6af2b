"""Reference computations for conditioning on the observed entries (Corex.impute, score_samples / mahalanobis with
missing='marginalize') -- test helpers only.

dense_conditional   the dense reference: for each row, E[x_M | x_O] = mean_M + Sigma_MO Sigma_OO^-1 (x_O - mean_O), the
                    squared Mahalanobis distance of x_O under Sigma_OO and log N(x_O; mean_O, Sigma_OO), with np.linalg.solve
                    and slogdet on C = S^-1 Sigma S^-1 (standardised space, as tests/dense_score.py, so that adni's column
                    scales do not break it).
lowrank_paths       a numpy restatement of the two per-row systems the device path solves (lowrank_kernels.cuh,
                    condition_rows_kernel): Path A of order |M| and Path B of order m, from woodbury()'s B, Delta and G.
"""
import numpy as np

from dense_score import LOG_2PI


def missing_mask(x, missing_values=None):
    """Missing entries: NaN, or equal to the marker."""
    x = np.asarray(x, dtype=np.float64)
    mask = np.isnan(x)
    if missing_values is not None:
        mask |= x == float(missing_values)
    return mask


def dense_conditional(cov, mean, sd, x, mask):
    """(imputed rows in raw units, log p(x_O), q_O) of the rows of x with missing entries `mask` under N(mean, cov)."""
    sd = np.asarray(sd, dtype=np.float64)
    mean = np.asarray(mean, dtype=np.float64)
    x = np.asarray(x, dtype=np.float64)
    c = cov / np.outer(sd, sd)
    n = c.shape[0]
    imputed, logp, q = x.copy(), np.zeros(len(x)), np.zeros(len(x))
    for l in range(len(x)):
        miss = mask[l]
        obs = ~miss
        if not obs.any():
            imputed[l] = mean
            continue
        xo = (x[l, obs] - mean[obs]) / sd[obs]
        coo = c[np.ix_(obs, obs)]
        sol = np.linalg.solve(coo, xo)
        q[l] = xo.dot(sol)
        sign, logdet = np.linalg.slogdet(coo)
        assert sign > 0
        logp[l] = -0.5 * (obs.sum() * LOG_2PI + logdet + 2 * np.sum(np.log(sd[obs])) + q[l])
        if miss.any():
            imputed[l, miss] = mean[miss] + sd[miss] * c[np.ix_(miss, obs)].dot(sol)
    assert n == x.shape[1]
    return imputed, logp, q


def lowrank_paths(w, xt, miss, logdet_sigma, sd, path):
    """(x^_M, q_O, log p(x_O)) of one standardised row xt by Path 'A' or 'B' from w = woodbury(...)."""
    import scipy.linalg
    b, delta = w["B"], w["delta"]
    n, m = b.shape[1], b.shape[0]
    k = int(miss.sum())
    obs = ~miss
    if k == n:
        return np.zeros(n), 0.0, 0.0
    x0 = np.where(miss, 0.0, xt)
    c = b.dot(x0)
    bm = b[:, miss]
    g = bm.T.dot(c)
    s0 = np.sum(x0[obs] ** 2 / delta[obs])
    if k == 0:
        xh, ldet = np.zeros(0), 0.0
    elif path == "A":
        lam = np.diag(1 / delta[miss]) - bm.T.dot(bm)
        ch = scipy.linalg.cho_factor(lam, lower=True)
        xh = scipy.linalg.cho_solve(ch, g)
        ldet = 2 * np.sum(np.log(np.diag(ch[0])))
    else:
        ginv = scipy.linalg.solve_triangular(w["G"], np.eye(m), lower=True)
        h = ginv.dot(ginv.T)
        bo = b[:, obs]
        e = h + (bo * delta[obs]).dot(bo.T)
        ch = scipy.linalg.cho_factor(e, lower=True)
        dm = delta[miss]
        xh = dm * g + dm * bm.T.dot(scipy.linalg.cho_solve(ch, bm.dot(dm * g)))
        ldet = 2 * np.sum(np.log(np.diag(ch[0]))) - np.sum(np.log(dm))
    q = s0 - c.dot(c) - g.dot(xh)
    logp = -0.5 * ((n - k) * LOG_2PI + logdet_sigma - 2 * np.sum(np.log(sd[miss])) + ldet + q)
    return xh, q, logp
