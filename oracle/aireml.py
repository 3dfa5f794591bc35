"""TEST INFRASTRUCTURE ONLY — CPU oracle for AI-REML (REML(..., aireml=True) in scilmm_b200.SparseCholesky).

The reference stubs AI-REML out (SparseCholesky.py:129-130 raises 'AI-REML is broken'), so there is nothing of it to
pin.  What follows restates the engine's AI-REML driver (scilmm_b200.SparseCholesky._aireml_fit) with the same
constants and boundary rule on top of the reference's own gradient (gradient_terms, :62-74) and AI matrix
(average_information, :147-168, negated):
  Gilmour, Thompson & Cullis (1995), Biometrics 51:1440-1450 - average-information REML (Fisher scoring with the
    average of the observed and expected information, AI_ij = 1/2 y'P A_i P A_j P y);
  Loh et al. (2015), Nature Genetics 47:1385-1392 (BOLT-REML) - AI-REML with Monte-Carlo (Hutchinson) traces in the
    score and a fixed probe block for the whole fit.

Nothing under scilmm_b200/ may import this module; tests use it as the checker of the engine's AI-REML fit.
"""
import numpy as np
import scipy.sparse as sp

from oracle.estimation import (average_information, fixed_effects, gradient_terms, he_regression, probe_vectors,
                               varcomp_stderr, weighted_sum)

AIREML_FLOOR = 1e-6       # smallest variance component (y is standardised)
AIREML_TOL = 1e-4         # stop when max |delta log sigma| < AIREML_TOL
AIREML_MAX_ITER = 30


def aireml_step(sig, grad, AI, floor=AIREML_FLOOR, jump=True):
    """One Fisher-scoring step in theta = log sigma: g_t = sigma o grad, H_t = D AI D, delta = -H_t^-1 g_t.
    A component at the floor whose score still points down (grad > 0) is fixed; with jump=True a free component whose
    linearised step is delta_k <= -1 (sigma_k (1 + delta_k) <= 0) is put on the floor in this step and fixed, and the
    others take the step of the reduced system with that move included.  Capped so that max |delta| <= 1.
    Returns (new sigma, max |delta| of the free components before the cap)."""
    sig, grad = np.asarray(sig, dtype=float), np.asarray(grad, dtype=float)
    K = sig.size
    gt = sig * grad
    Ht = sig[:, None] * AI * sig[None, :]
    fixed = (sig <= floor) & (grad > 0)
    while True:
        free = np.flatnonzero(~fixed)
        lin = np.where(fixed, (floor - sig) / sig, 0.0)      # linearised move of the fixed components (0 at the floor)
        delta = np.zeros(K)
        if free.size:
            delta[free] = -np.linalg.solve(Ht[np.ix_(free, free)], gt[free] + Ht[free] @ lin)
        hit = ~fixed & (delta <= -1.0)
        if not (jump and hit.any()):
            break
        fixed |= hit
    size = float(np.max(np.abs(delta[free]))) if free.size else 0.0
    if size > 1.0:
        delta = delta / size
    new = np.where(fixed, np.minimum(sig, floor), np.maximum(sig * np.exp(delta), floor))
    if fixed.any():                                          # a jump to the floor is a step too
        size = max(size, float(np.max(np.log(sig[fixed] / new[fixed]))))
    return new, size


def aireml_fit(cholesky_func, mats, C, y, reml=True, sim_num=100, verbose=False, normal_source=None,
               max_iter=AIREML_MAX_ITER, tol=AIREML_TOL, floor=AIREML_FLOOR, jump=True, trace=None):
    """HE start (reference :120-128) + AI-REML.  The probe block is drawn ONCE (normal_source(n, sim_num), default the
    global numpy stream) and used by every iteration.  Returns (sigma, {'iterations', 'converged'}); `trace` (a list)
    collects (sigma, grad, AI) per iteration."""
    start = he_regression(mats[:-1], C, y, compute_stderr=False)
    start = np.concatenate((start, [1 - start.sum()]))
    if np.any(start < 0):
        start = np.ones(len(mats))
    sig = start / start.sum()
    n = y.shape[0]
    Z = np.random.randn(n, sim_num) if normal_source is None else normal_source(n, sim_num)
    converged, it = False, 0
    while it < max_iter:
        it += 1
        factor = cholesky_func(weighted_sum(mats, sig))
        ViC, chol_CtViC, mu, _ = fixed_effects(factor, y, C)
        Vi_r = factor(y - mu)
        W = probe_vectors(factor, Z, np.argsort(factor.P()))
        grad = gradient_terms(sig, mats, W, Vi_r, reml, ViC, chol_CtViC)
        if reml:
            AI = -average_information(mats, C, factor, y)
        else:                                   # ML: 1/2 (A_i u)' V^-1 (A_j u) with u = V^-1 (y - C beta)
            B = np.column_stack([m.dot(Vi_r) for m in mats])
            AI = 0.5 * B.T.dot(factor(B))
        if trace is not None:
            trace.append((sig.copy(), grad.copy(), AI.copy()))
        sig, size = aireml_step(sig, grad, AI, floor, jump)
        if verbose:
            print('AI-REML iteration %d: sigma %s, max |step| %.3e' % (it, sig, size))
        if size < tol:
            converged = True
            break
    return sig, {"iterations": it, "converged": converged}


def aireml_reml_fit(cholesky_func, mats, C, y, reml=True, sim_num=100, verbose=False, normal_source=None, **kw):
    """REML (reference :177-189) with the AI-REML driver in place of L-BFGS-B; extra key 'aireml'."""
    y = y / y.std()
    mats = list(mats) + [sp.eye(y.shape[0]).tocsr()]
    sig, info = aireml_fit(cholesky_func, mats, C, y, reml, sim_num, verbose, normal_source, **kw)
    factor = cholesky_func(weighted_sum(mats, sig))
    _, _, _, beta = fixed_effects(factor, y, C)
    se = varcomp_stderr(mats, C, factor, y, sim_num)
    return {"covariance coefficients": sig, "covariates coefficients": beta, "covariance std": se, "aireml": info}


def reml_fit(cholesky_func, mats, C, y, reml=True, sim_num=100, verbose=False, normal_source=None):
    """reference: SparseCholesky.py:177-189 (REML).  Extra key 'nll' is not in the reference dict."""
    y = y / y.std()
    mats = list(mats) + [sp.eye(y.shape[0]).tocsr()]
    sig = fit_variance_components(cholesky_func, mats, C, y, reml, sim_num, verbose, normal_source)
    factor = cholesky_func(weighted_sum(mats, sig))
    _, _, _, beta = fixed_effects(factor, y, C)
    se = varcomp_stderr(mats, C, factor, y, sim_num)
    return {"covariance coefficients": sig, "covariates coefficients": beta, "covariance std": se}
