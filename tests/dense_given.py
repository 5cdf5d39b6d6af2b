"""numpy restatement of conditioning on a fixed column set (Corex.conditional / ConditionalGaussian, lowrank_kernels.cuh:
given_*_kernel) -- test helper only.

With Z and Delta of tests/dense_score.lowrank_parts (Sigma~ = Z^T Z + Delta), observed columns O and targets T:
    E_O = I + Z_O Delta_O^-1 Z_O^T = L L^T,   A = L^-1 Z_O Delta_O^-1,   P = L^-1 Z_T,   v = A x~_O
    E[x~_T | x~_O] = P^T v,   Cov[x~_T | x~_O] = Delta_T + P^T P,   q_O = sum_O x~_i^2 / Delta_i - |v|^2
    log det Sigma_OO = sum_O (2 log sd_i + log Delta_i) + 2 sum log L_kk,   log p(x_O) = -(|O| log 2 pi + log det + q_O) / 2
Draws x~_T = P^T (v + u) + Delta_T^1/2 eps take their normals from tests/philox_ref.py's streams with tag 2: normal j of
stream (seed, 2, row, draw) is u_j for j < m and eps_{j - m} for the targets in their given order.
"""
import numpy as np

from dense_score import LOG_2PI, lowrank_parts


def given_parts(rhoinvrho, si, eps, sd, obs, tgt):
    """dict with A, P, L, delta and logdet (log det Sigma_OO) for the column lists obs and tgt."""
    import scipy.linalg
    z, delta = lowrank_parts(rhoinvrho, si, eps)
    sd = np.asarray(sd, dtype=np.float64)
    zo, do = z[:, obs], delta[obs]
    e = np.eye(z.shape[0]) + (zo / do).dot(zo.T)
    ll = np.linalg.cholesky(e)
    a = scipy.linalg.solve_triangular(ll, zo / do, lower=True)
    p = scipy.linalg.solve_triangular(ll, z[:, tgt], lower=True)
    logdet = np.sum(2 * np.log(sd[obs]) + np.log(do)) + 2 * np.sum(np.log(np.diag(ll)))
    return {"A": a, "P": p, "L": ll, "delta": delta, "logdet": logdet}


def given_rows(g, xt_obs, obs, tgt):
    """(E[x~_T | x~_O] (N, |T|), Cov[x~_T | x~_O], q_O (N,), log p(x_O) (N,)) of standardised observed rows xt_obs."""
    v = xt_obs.dot(g["A"].T)
    mean = v.dot(g["P"])
    cov = np.diag(g["delta"][tgt]) + g["P"].T.dot(g["P"])
    q = np.sum(xt_obs ** 2 / g["delta"][obs], axis=1) - np.sum(v ** 2, axis=1)
    return mean, cov, q, -0.5 * (len(obs) * LOG_2PI + g["logdet"] + q)
