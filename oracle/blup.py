"""TEST INFRASTRUCTURE ONLY — CPU restatements of the predicted random effects (scilmm_b200.blup).

Three formulations, sharing nothing with the engine beyond the definitions:
  * blup_mme: Henderson's mixed-model equations over all N individuals for ONE relationship matrix plus the residual,
    with a dense A^-1 and the incidence matrix Z that picks the phenotyped rows.  The unphenotyped individuals come
    out of the equations directly; the exact PEV is the random-effect block of the inverse coefficient matrix.
  * blup_vform: the V-form of the same predictor for any K, densely: u = V^-1 (y_s - C beta),
    u_k = s sigma_k A_k[:, obs] u, PEV_k = s^2 (sigma_k diag A_k - sigma_k^2 diag(A_k[:, obs] P A_k[obs, :])).
  * pev_stochastic: the engine's Monte Carlo estimate of the PEV, restated on the same probes: the Philox block of
    the library (tests.util.philox_normals at BLUP_PROBE_STREAM), the engine's permutation, and W = P' L^-T Z from a
    LAPACK factor of V[perm][:, perm].
All outputs are in the units of y (s = y[obs].std(), the scale REML() fits on).
"""
import numpy as np
import scipy.linalg as la
import scipy.sparse as sp

from oracle.estimation import weighted_sum

BLUP_PROBE_STREAM = 2 ** 62       # scilmm_b200.SparseCholesky.BLUP_PROBE_STREAM


def _dense(m):
    return m.toarray() if sp.issparse(m) else np.asarray(m, dtype=float)


def _observed(y):
    obs = ~np.isnan(np.asarray(y, dtype=float))
    return obs, np.flatnonzero(obs), float(np.asarray(y)[obs].std())


def _vsolve(mats, covariates, y, sigmas):
    """(obs, idx, s, V_obs dense, Cholesky of V_obs, C_obs, beta, u = V^-1 (y_s - C beta)) on the observed rows."""
    obs, idx, s = _observed(y)
    ys = np.asarray(y, dtype=float)[idx] / s
    Co = np.asarray(covariates, dtype=float)[idx]
    sub = [sp.csr_matrix(m)[idx][:, idx] for m in mats] + [sp.eye(idx.size).tocsr()]
    V = weighted_sum(sub, sigmas).toarray()
    cV = la.cho_factor(V, lower=True)
    ViC = la.cho_solve(cV, Co)
    M = Co.T @ ViC
    beta = la.solve(M, ViC.T @ ys, assume_a="pos")
    u = la.cho_solve(cV, ys - Co @ beta)
    return obs, idx, s, V, cV, Co, beta, u


def _assemble(covariates, s, obs, beta, U, resid_obs):
    N = obs.size
    resid = np.full(N, np.nan)
    resid[obs] = resid_obs
    fixed = s * (np.asarray(covariates, dtype=float) @ beta)
    return {"u": U, "residual": resid, "fixed": fixed, "yhat": fixed + U.sum(axis=1), "beta": s * beta}


def _reliability(pev, prior):
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(prior != 0, 1.0 - pev / np.where(prior != 0, prior, 1.0), np.nan)


def blup_vform(mats, covariates, y, sigmas, exact_pev=True):
    """Same arguments and keys as scilmm_b200.blup (mats over all N, without the identity; NaN in y = no phenotype),
    plus (exact_pev=True) the exact 'pev' and 'reliability'."""
    obs, idx, s, V, cV, Co, beta, u = _vsolve(mats, covariates, y, sigmas)
    K = len(mats)
    if exact_pev:
        ViC = la.cho_solve(cV, Co)
        P = la.cho_solve(cV, np.eye(idx.size)) - ViC @ la.solve(Co.T @ ViC, ViC.T, assume_a="pos")
    U = np.empty((obs.size, K))
    pev = np.empty((obs.size, K))
    prior = np.empty((obs.size, K))
    for k, m in enumerate(mats):
        Ak = sp.csr_matrix(m)[:, idx]                             # N x n: Cov(u_k, y_s) / sigma_k
        U[:, k] = s * sigmas[k] * (Ak @ u)
        if exact_pev:
            prior[:, k] = s * s * sigmas[k] * sp.csr_matrix(m).diagonal()
            pev[:, k] = prior[:, k] - s * s * sigmas[k] ** 2 * np.sum((Ak @ P) * Ak.toarray(), axis=1)
    out = _assemble(covariates, s, obs, beta, U, s * sigmas[-1] * u)
    if not exact_pev:
        return out
    out["pev"] = pev
    out["reliability"] = _reliability(pev, prior)
    return out


def blup_mme(A, covariates, y, sigmas):
    """Henderson's mixed-model equations for y_s[obs] = C_obs beta + Z a + e, a ~ N(0, sigma_a A) over all N
    individuals, e ~ N(0, sigma_e I); Z (n x N) picks the phenotyped rows.  sigmas = (sigma_a, sigma_e)."""
    obs, idx, s = _observed(y)
    N = obs.size
    ys = np.asarray(y, dtype=float)[idx] / s
    C = np.asarray(covariates, dtype=float)
    Co = C[idx]
    Z = np.zeros((idx.size, N))
    Z[np.arange(idx.size), idx] = 1.0
    sa, se = float(sigmas[0]), float(sigmas[1])
    Ainv = la.inv(_dense(A))
    c = Co.shape[1]
    lhs = np.block([[Co.T @ Co, Co.T @ Z], [Z.T @ Co, Z.T @ Z + (se / sa) * Ainv]])
    rhs = np.concatenate([Co.T @ ys, Z.T @ ys])
    sol = la.solve(lhs, rhs, assume_a="sym")
    beta, a = sol[:c], sol[c:]
    Cinv = la.inv(lhs)
    pev = s * s * se * np.diag(Cinv)[c:]                           # Var(a - a^) = sigma_e (LHS^-1)_aa
    e = ys - Co @ beta - a[idx]
    out = _assemble(C, s, obs, beta, s * a[:, None], s * e)
    out["pev"] = pev[:, None]
    out["reliability"] = _reliability(out["pev"], s * s * sa * np.diag(_dense(A))[:, None])
    return out


def pev_stochastic(mats, covariates, y, sigmas, probes, seed, perm):
    """The engine's estimate of the PEV from `probes` probe columns: W = P' L^-T Z with L = chol(V[perm][:, perm])
    over the observed individuals (perm[new] = old, as SparseCholesky(perm=...)) and Z the library's Philox block
    (key `seed`, stream BLUP_PROBE_STREAM, rows in the factor's order); t = sigma_k A_k[:, obs] W,
    est = sum_j t_ij^2 / p, PEV = sigma_k A_ii - est + (exact fixed-effect term), se from sum_j t_ij^4.
    Returns (pev, pev_se), N x K, in the units of y^2."""
    from tests.util import philox_normals
    obs, idx, s, V, cV, Co, beta, u = _vsolve(mats, covariates, y, sigmas)
    n = idx.size
    perm = np.asarray(perm)
    Z, _ = philox_normals(n, probes, 0, seed, BLUP_PROBE_STREAM)
    L = la.cholesky(V[np.ix_(perm, perm)], lower=True)
    W = np.empty_like(Z)
    W[perm] = la.solve_triangular(L.T, Z, lower=False)
    ViC = la.cho_solve(cV, Co)
    Minv = la.inv(Co.T @ ViC)
    pev = np.empty((obs.size, len(mats)))
    se = np.empty_like(pev)
    for k, m in enumerate(mats):
        Ak = sp.csr_matrix(m)[:, idx]
        t = sigmas[k] * (Ak @ W)
        Y = sigmas[k] * (Ak @ ViC)
        s2, s4 = np.sum(t * t, axis=1), np.sum(t ** 4, axis=1)
        corr = np.sum((Y @ Minv) * Y, axis=1)
        pev[:, k] = s * s * (sigmas[k] * sp.csr_matrix(m).diagonal() - s2 / probes + corr)
        se[:, k] = s * s * np.sqrt(np.maximum(s4 - s2 * s2 / probes, 0.0) / (probes * (probes - 1)))
    return pev, se
