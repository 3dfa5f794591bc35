"""TEST INFRASTRUCTURE ONLY — CPU restatement of the mixed-model association scan (scilmm_b200.association).

The engine takes x~'V^-1 x~ as the squared norm of one forward half-sweep L^-1 P x~; this restatement takes full
solves V^-1 x~ of a dense factor instead, so the two share no formulation beyond the statistic itself:
gamma = x~'P_V y / x~'P_V x~, se = (x~'P_V x~)^-1/2 with P_V = V^-1 - V^-1 C (C'V^-1 C)^-1 C'V^-1.
"""
import numpy as np
import scipy.sparse as sp
from scipy.linalg import cho_solve
import scipy.stats as stats

from oracle.cpu_factor import DenseFactor
from oracle.estimation import fixed_effects, weighted_sum


def decode(G):
    """(centred allele counts with missing entries 0, allele frequency, non-missing count) per column of int8 G."""
    G = np.asarray(G)
    if np.any(G > 2):
        raise ValueError("genotype entries must be 0, 1, 2 or negative (missing)")
    obs = G >= 0
    n_obs = obs.sum(axis=0).astype(np.int64)
    with np.errstate(invalid="ignore", divide="ignore"):
        mu = np.where(obs, G, 0).sum(axis=0) / n_obs
    X = np.where(obs, G - np.nan_to_num(mu)[None, :], 0.0)
    return X, mu / 2.0, n_obs


def association(mats, covariates, y, sigmas, G, factor=DenseFactor):
    """Same arguments and keys as scilmm_b200.association (mats without the identity)."""
    scale = y.std()
    ys = y / scale
    V = weighted_sum(list(mats) + [sp.eye(ys.shape[0]).tocsr()], sigmas)
    f = factor(V)
    ViC, chol, mu, beta = fixed_effects(f, ys, covariates)
    Vir = f(ys - mu)
    X, af, n_obs = decode(G)
    ViX = f(X)
    xVx = np.sum(X * ViX, axis=0)
    q = ViC.T @ X
    t = Vir @ X
    xPx = xVx - np.sum(q * cho_solve(chol, q), axis=0)
    xPx = np.where(xPx > 1e-10 * xVx, xPx, np.nan)
    chi2 = t * t / xPx
    return {"beta": t / xPx * scale, "se": scale / np.sqrt(xPx), "chi2": chi2, "p": stats.chi2.sf(chi2, 1),
            "af": af, "n_obs": n_obs}
