"""Reference computations for the conditional standard deviations and draws of Corex.impute(return_std=True) and
Corex.sample_missing -- test helpers only.

dense_conditional_cov   Sigma~_MM - Sigma~_MO Sigma~_OO^-1 Sigma~_OM in standardised space (C = S^-1 cov S^-1, as
                        tests/dense_conditional.py), by np.linalg.solve.
lowrank_std / draw_map  a numpy restatement of what condition_rows_kernel does in its sampling mode on each path, from
                        woodbury()'s B, Delta and G: W = G_W G_W^T is the row's system (Path A: Lambda_MM = Delta_M^-1 - B_M^T B_M;
                        Path B: E = H + sum_O Delta_i b_i b_i^T), and the kernel's L D L^T of it has L D^1/2 = G_W, so
                        L^-1 v / D^1/2 = G_W^-1 v and L^-T D^-1/2 = G_W^-T.
    Path A  var_a = |G_W^-1 e_a|^2,                     draw map  G_W^-T                                 (eps: k normals)
    Path B  var_a = Delta_a + Delta_a^2 |G_W^-1 b_a|^2,  draw map  [Delta_M^1/2 | Delta_M B_M^T G_W^-T]     (eps: k + m normals)
A row with nothing observed (k = n) is Path B with O empty, W = H.
"""
import numpy as np


def dense_conditional_cov(cov, sd, miss):
    """Conditional covariance of the missing entries `miss` (bool, n) given the others, standardised units."""
    sd = np.asarray(sd, dtype=np.float64)
    c = cov / np.outer(sd, sd)
    obs = ~miss
    cmm = c[np.ix_(miss, miss)]
    if not obs.any():
        return cmm
    cmo = c[np.ix_(miss, obs)]
    return cmm - cmo.dot(np.linalg.solve(c[np.ix_(obs, obs)], cmo.T))


def _system(w, miss, path):
    """(G_W lower Cholesky factor of the row's system, B_M, Delta_M)."""
    b, delta = w["B"], w["delta"]
    bm, dm = b[:, miss], delta[miss]
    if path == "A":
        lam = np.diag(1 / dm) - bm.T.dot(bm)
        return np.linalg.cholesky(lam), bm, dm
    import scipy.linalg
    m = b.shape[0]
    ginv = scipy.linalg.solve_triangular(w["G"], np.eye(m), lower=True)
    bo = b[:, ~miss]
    e = ginv.dot(ginv.T) + (bo * delta[~miss]).dot(bo.T)
    return np.linalg.cholesky(e), bm, dm


def lowrank_std(w, miss, path):
    """Conditional standard deviations of the missing entries by Path 'A' or 'B', standardised units."""
    import scipy.linalg
    gw, bm, dm = _system(w, miss, path)
    if path == "A":
        y = scipy.linalg.solve_triangular(gw, np.eye(len(dm)), lower=True)
        return np.sqrt(np.sum(y ** 2, axis=0))
    y = scipy.linalg.solve_triangular(gw, bm, lower=True)
    return np.sqrt(dm + dm ** 2 * np.sum(y ** 2, axis=0))


def draw_map(w, miss, path):
    """M with v = M eps ~ N(0, Lambda_MM^-1): (k x k) for Path A, (k x (k + m)) for Path B."""
    import scipy.linalg
    gw, bm, dm = _system(w, miss, path)
    gt = scipy.linalg.solve_triangular(gw, np.eye(gw.shape[0]), lower=True).T  # G_W^-T
    if path == "A":
        return gt
    return np.hstack([np.diag(np.sqrt(dm)), (dm[:, None] * bm.T).dot(gt)])
