"""TEST INFRASTRUCTURE ONLY — CPU restatement of the binary-trait path (scilmm_b200.glmm / glmm_association).

Nothing under scilmm_b200/ may import this module.  It restates, densely and with the engine's constants:
  the logistic GLM start by IRLS;
  the PQL fit of GMMAT's glmmkin AI scheme (Breslow & Clayton 1993; Chen et al. 2016, AJHG 98:653): per iteration
    the working vector Y~ = eta + (y - mu) / w, Sigma = W^-1 + sum_k tau_k A_k, one REML gradient / AI matrix on
    (Sigma, Y~) with the reference's gradient (gradient_terms) and AI matrix (average_information), an EM step first and
    the AI-REML step (oracle/aireml.py aireml_step) after, and eta = Y~ - W^-1 Sigma^-1 (Y~ - C alpha);
  the score statistics U = x~' P Y~, Var(U) = x~' P x~ by full dense solves;
  the saddlepoint p-value of SAIGE (Zhou et al. 2018, Nat Genet 50:1335) with scipy.optimize.brentq for the root and
    the Lugannani-Rice tail;
  the exact tail of the score for the intercept-only, constant-mu case, a double binomial sum over carriers and
    non-carriers.
"""
import numpy as np
import scipy.linalg as la
import scipy.optimize as optimize
import scipy.sparse as sp
import scipy.special as special
import scipy.stats as stats

from oracle.aireml import AIREML_FLOOR, aireml_step
from oracle.association import decode
from oracle.cpu_factor import DenseFactor
from oracle.estimation import average_information, fixed_effects, gradient_terms, probe_vectors, weighted_sum

MU_EPS = 2.220446049250313e-16     # mu is clamped to [eps, 1 - eps], as R's binomial()
GLMM_TOL = 1e-5
GLMM_MAX_ITER = 50
IRLS_TOL = 1e-10
IRLS_MAX_ITER = 100
SPA_MIN_W = 1e-3


def working(eta, y):
    """(mu, w, Y~) of the logit link at eta."""
    mu = np.clip(special.expit(eta), MU_EPS, 1.0 - MU_EPS)
    w = mu * (1.0 - mu)
    return mu, w, eta + (y - mu) / w


def irls(C, y):
    """Logistic GLM by iteratively reweighted least squares from mu = (y + 1/2) / 2.  Returns alpha."""
    mu = (y + 0.5) / 2.0
    eta = np.log(mu / (1.0 - mu))
    alpha = np.zeros(C.shape[1])
    for _ in range(IRLS_MAX_ITER):
        mu, w, z = working(eta, y)
        new = la.solve(C.T @ (w[:, None] * C), C.T @ (w * z), assume_a="pos")
        step = np.max(np.abs(new - alpha))
        alpha = new
        eta = C @ alpha
        if step < IRLS_TOL * (1.0 + np.max(np.abs(alpha))):
            break
    return alpha


def eta_update(Yt, D, ViR):
    """eta = Y~ - D o Sigma^-1 (Y~ - C alpha) (D = 1 / w): the BLUP identity Y~ - eta = W^-1 Sigma^-1 (Y~ - C alpha)."""
    return Yt - D * ViR


def pql_fit(factor_func, mats, C, y, sim_num=100, normal_source=None, tau_fixed=None, floor=AIREML_FLOOR,
            trace=None):
    """GMMAT glmmkin AI scheme, restated as scilmm_b200.glmm.  factor_func(Sigma) -> a dense factor (e.g.
    lambda M: DenseFactor(M, P) for the engine's permutation P).  The probe block is drawn once, normal_source(n, s) or
    the global numpy stream.  tau_fixed: hold tau at these values (no variance-component step).  Returns the dict of
    scilmm_b200.glmm."""
    n, K = y.shape[0], len(mats)
    alpha = irls(C, y)
    eta = C @ alpha
    mu, w, Yt = working(eta, y)
    tau = np.full(K, np.var(Yt, ddof=1) / (K + 1)) if tau_fixed is None else np.array(tau_fixed, dtype=float)
    Z = np.random.randn(n, sim_num) if normal_source is None else normal_source(n, sim_num)
    converged, it = False, 0
    while it < GLMM_MAX_ITER:
        it += 1
        D = 1.0 / w
        allm = list(mats) + [sp.diags(D).tocsr()]
        sig = np.concatenate([tau, [1.0]])
        f = factor_func(weighted_sum(allm, sig))
        ViC, chol, Cb, a_new = fixed_effects(f, Yt, C)
        ViR = f(Yt - Cb)
        W = probe_vectors(f, Z, np.argsort(f.P()))
        grad = gradient_terms(sig, allm, W, ViR, True, ViC, chol)[:K]
        AI = -average_information(allm, C, f, Yt)[:K, :K]
        if trace is not None:
            trace.append((tau.copy(), grad.copy(), AI.copy()))
        tau_old, alpha_old = tau, alpha
        if tau_fixed is None:
            if it == 1:
                tau = np.maximum(floor, tau - 2.0 * tau * tau * grad / n)
            else:
                tau = aireml_step(tau, grad, AI, floor)[0]
        alpha = a_new
        eta = eta_update(Yt, D, ViR)
        mu, w, Yt = working(eta, y)
        if 2.0 * max(np.max(np.abs(alpha - alpha_old) / (np.abs(alpha) + np.abs(alpha_old) + GLMM_TOL)),
                     np.max(np.abs(tau - tau_old) / (np.abs(tau) + np.abs(tau_old) + GLMM_TOL))) < GLMM_TOL:
            converged = True
            break
    var_a = la.cho_solve(chol, np.eye(C.shape[1]))
    return {"covariance coefficients": tau,
            "covariance std": np.sqrt(np.diag(la.inv(AI)) * (1 + 1.0 / sim_num)),
            "covariates coefficients": alpha, "covariates std": np.sqrt(np.diag(var_a)),
            "latent fractions": tau / (tau.sum() + np.pi ** 2 / 3),
            "mu": mu, "eta": eta, "weights": w, "working y": Yt,
            "glmm": {"iterations": it, "converged": converged}}


def score_statistics(mats, C, fit, G):
    """U = x~' P Y~ and Var(U) = x~' P x~ at the fit, P = Sigma^-1 - Sigma^-1 C (C'Sigma^-1 C)^-1 C'Sigma^-1, by full
    dense solves.  Returns (U, VarU with NaN where monomorphic or in the span of C, af, n_obs)."""
    tau, w, Yt = fit["covariance coefficients"], fit["weights"], fit["working y"]
    f = DenseFactor(weighted_sum(list(mats) + [sp.diags(1.0 / w).tocsr()], np.concatenate([tau, [1.0]])))
    ViC, chol, Cb, _ = fixed_effects(f, Yt, C)
    ViR = f(Yt - Cb)
    X, af, n_obs = decode(G)
    ViX = f(X)
    xVx = np.sum(X * ViX, axis=0)
    q = ViC.T @ X
    xPx = xVx - np.sum(q * la.cho_solve(chol, q), axis=0)
    return ViR @ X, np.where(xPx > 1e-10 * xVx, xPx, np.nan), af, n_obs


def cgf(t, g, mu):
    """K(t), K'(t), K''(t) of S = sum_i g_i (Y_i - mu_i), Y_i ~ Bernoulli(mu_i) independent."""
    a = g * t
    K = np.logaddexp(np.log1p(-mu), np.log(mu) + a) - a * mu
    with np.errstate(over="ignore"):
        p = mu / (mu + (1.0 - mu) * np.exp(-a))
    return K.sum(), np.sum(g * (p - mu)), np.sum(g * g * p * (1.0 - p))


def spa_pvalue(q, g, mu):
    """Two-sided saddlepoint p-value P(|S| >= |q|): roots of K'(zeta) = +-|q| by brentq and the Lugannani-Rice tail of
    each side.  Returns (p, ok); ok is False where |q| is outside the range of K' or |w| < 1e-3 on a side."""
    hi_lim = np.sum(g * ((g > 0) - mu))           # K'(+inf)
    lo_lim = np.sum(g * ((g < 0) - mu))           # K'(-inf)
    total = 0.0
    for side in (1.0, -1.0):
        target = side * abs(q)
        if not (lo_lim < target < hi_lim):
            return np.nan, False
        b = side
        while side * (cgf(b, g, mu)[1] - target) < 0:
            b *= 2.0
        zeta = optimize.brentq(lambda t: cgf(t, g, mu)[1] - target, min(0.0, b), max(0.0, b), xtol=1e-300,
                               rtol=4 * np.finfo(float).eps, maxiter=1000)
        K, _, K2 = cgf(zeta, g, mu)
        w = side * np.sqrt(max(2.0 * (zeta * target - K), 0.0))
        v = zeta * np.sqrt(K2)
        if abs(w) < SPA_MIN_W:
            return np.nan, False
        corr = stats.norm.pdf(w) * (1.0 / v - 1.0 / w)
        total += stats.norm.sf(w) + corr if side > 0 else stats.norm.cdf(w) - corr
    if not (np.isfinite(total) and total >= 0):
        return np.nan, False
    return min(total, 1.0), True


def adjusted_genotype(x, C, w):
    """g~ = x~ - C (C'WC)^-1 C'W x~."""
    return x - C @ la.solve(C.T @ (w[:, None] * C), C.T @ (w * x), assume_a="pos")


def glmm_association(mats, C, fit, G, spa_cutoff=2.0):
    """Same keys as scilmm_b200.glmm_association."""
    U, xPx, af, n_obs = score_statistics(mats, C, fit, G)
    with np.errstate(invalid="ignore", divide="ignore"):
        z = U / np.sqrt(xPx)
        chi2 = z * z
        out = {"beta": U / xPx, "se": 1.0 / np.sqrt(xPx), "score": np.where(np.isfinite(xPx), U, np.nan), "chi2": chi2,
               "p_normal": special.chdtrc(1, chi2), "af": af, "n_obs": n_obs}
    out["p"] = out["p_normal"].copy()
    out["spa"] = np.zeros(G.shape[1], dtype=np.int8)
    X, _, _ = decode(G)
    mu, w = fit["mu"], fit["weights"]
    for j in np.flatnonzero(np.isfinite(z) & (np.abs(np.nan_to_num(z)) > spa_cutoff)):
        g = adjusted_genotype(X[:, j], C, w)
        q = U[j] * np.sqrt(np.sum(g * g * w) / xPx[j])
        p, ok = spa_pvalue(q, g, mu)
        out["spa"][j] = 1 if ok else -1
        if ok:
            out["p"][j] = p
    return out


def exact_tail(n, carriers, mu, s):
    """P(|S| >= s) for S = sum_i g~_i (Y_i - mu), intercept only, Y_i ~ Bernoulli(mu), genotype 1 on `carriers`
    individuals and 0 elsewhere: S = (1 - m) A - m B with m = carriers / n, A ~ Bin(carriers, mu) and
    B ~ Bin(n - carriers, mu) independent (the mean terms cancel)."""
    m = carriers / n
    a = np.arange(carriers + 1)
    b = np.arange(n - carriers + 1)
    pa = stats.binom.pmf(a, carriers, mu)
    pb = stats.binom.pmf(b, n - carriers, mu)
    S = (1.0 - m) * a[:, None] - m * b[None, :]
    return float(np.sum(np.outer(pa, pb)[np.abs(S) >= s * (1.0 - 1e-12)]))
