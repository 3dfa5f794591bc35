"""CPU checks of the binary-trait oracle (oracle/glmm.py) and of the input rules of glmm() / glmm_association(): the
IRLS start against a direct maximisation of the logistic likelihood, the PQL driver with tau held at zero against the
GLM, the BLUP identity of the eta update, and the saddlepoint p-value against the exact tail of the intercept-only,
constant-mu score in two rare-variant cases."""
import sys

import numpy as np
import pytest
import scipy.optimize as optimize
import scipy.sparse as sp
import scipy.special as special
import scipy.stats as stats

from oracle import glmm as og
from oracle import estimation as orc
from oracle.cpu_factor import DenseFactor


def binary_trait(g, q=0.7):
    """The golden y thresholded at its q quantile (1 above), and the covariates."""
    return (g["y"] > np.quantile(g["y"], q)).astype(np.float64), g["cov"]


def test_irls_maximises_the_logistic_likelihood(golden_small):
    y, C = binary_trait(golden_small)
    alpha = og.irls(C, y)

    def nll(a):
        eta = C @ a
        return np.sum(np.logaddexp(0.0, eta) - y * eta)

    def grad(a):
        return C.T @ (special.expit(C @ a) - y)

    def hess(a):
        mu = special.expit(C @ a)
        return C.T @ ((mu * (1 - mu))[:, None] * C)

    ref = optimize.minimize(nll, np.zeros(C.shape[1]), jac=grad, hess=hess, method="trust-exact",
                            options={"gtol": 1e-13})
    assert np.max(np.abs(alpha - ref.x)) < 1e-8 * np.max(np.abs(ref.x))


def test_pql_with_tau_at_zero_is_the_glm(golden_small):
    g = golden_small
    y, C = binary_trait(g)
    fit = og.pql_fit(DenseFactor, [g.csr("A")], C, y, sim_num=4, tau_fixed=[0.0], floor=0.0)
    alpha = og.irls(C, y)
    mu = special.expit(C @ alpha)
    cov = np.linalg.inv(C.T @ ((mu * (1 - mu))[:, None] * C))
    assert fit["glmm"]["converged"]
    assert np.max(np.abs(fit["covariates coefficients"] - alpha)) < 1e-9 * np.max(np.abs(alpha))
    assert np.max(np.abs(fit["covariates std"] - np.sqrt(np.diag(cov)))) < 1e-9 * np.max(np.sqrt(np.diag(cov)))
    assert np.max(np.abs(fit["eta"] - C @ alpha)) < 1e-9 * np.max(np.abs(C @ alpha))


def test_eta_update_is_the_blup_identity(golden_small):
    """Y~ - D o Sigma^-1 (Y~ - C alpha) = C alpha + sum_k tau_k A_k Sigma^-1 (Y~ - C alpha), Sigma = D + sum tau_k A_k."""
    g = golden_small
    y, C = binary_trait(g)
    mats = g.mats("k3")
    alpha = og.irls(C, y)
    _, w, Yt = og.working(C @ alpha, y)
    D = 1.0 / w
    tau = np.array([0.4, 0.15, 0.05])
    f = DenseFactor(orc.weighted_sum(mats + [sp.diags(D).tocsr()], np.concatenate([tau, [1.0]])))
    _, _, Ca, _ = orc.fixed_effects(f, Yt, C)
    ViR = f(Yt - Ca)
    explicit = Ca + sum(t * (m @ ViR) for t, m in zip(tau, mats))
    assert np.max(np.abs(og.eta_update(Yt, D, ViR) - explicit)) < 1e-12 * np.max(np.abs(explicit))


def carrier_case(n, prevalence, carriers):
    m = carriers / n
    g = np.where(np.arange(n) < carriers, 1.0 - m, -m)
    return g, np.full(n, prevalence)


@pytest.mark.parametrize("n, prevalence, carriers, counts, band, normal_off", [
    (5000, 0.02, 100, range(7, 11), (0.80, 0.90), 1e3),
    (2000, 0.01, 6, range(2, 5), (0.33, 0.45), 1e50),
])
def test_spa_against_the_exact_tail(n, prevalence, carriers, counts, band, normal_off):
    """Intercept only, constant mu: S = (1 - m) A - m B with A, B binomial.  At a carrier-case count a (and the
    expected count among the non-carriers) the saddlepoint p is within `band` of the exact two-sided tail, while the
    normal p is more than `normal_off` times too small at the smallest tail."""
    g, mu = carrier_case(n, prevalence, carriers)
    var = np.sum(g * g * mu * (1 - mu))
    b0 = round(prevalence * (n - carriers))
    ratios = []
    for a in counts:
        s = (1.0 - carriers / n) * a - carriers / n * b0
        exact = og.exact_tail(n, carriers, prevalence, s)
        p, ok = og.spa_pvalue(s, g, mu)
        assert ok
        ratios.append(p / exact)
        normal = stats.chi2.sf(s * s / var, 1)
    assert band[0] <= min(ratios) and max(ratios) <= band[1], ratios
    assert exact / normal > normal_off, (exact, normal)
    assert exact < (2.2e-5 if carriers == 100 else 1e-7)


def test_spa_falls_back_outside_the_range_of_K1():
    g, mu = carrier_case(500, 0.1, 3)
    hi = np.sum(g * ((g > 0) - mu))
    p, ok = og.spa_pvalue(1.01 * hi, g, mu)
    assert not ok and np.isnan(p)


def test_refused_inputs_need_no_device(golden_small):
    import scilmm_b200.SparseCholesky  # noqa: F401
    S = sys.modules["scilmm_b200.SparseCholesky"]
    g = golden_small
    y, C = binary_trait(g)
    mats = [g.csr("A")]
    chol = S.SparseCholesky()
    for bad_y in (np.where(y > 0, 2.0, 0.0), np.where(np.arange(g.n) == 3, np.nan, y), np.zeros(g.n), np.ones(g.n),
                  y[1:], y[:, None]):
        with pytest.raises(ValueError):
            S.glmm(chol, mats, C, bad_y)
    bad_C = C.copy()
    bad_C[5, 0] = np.inf
    for args in ((mats, bad_C), (mats, C[1:]), ([g.csr("A")[1:, 1:]], C), ([], C)):
        with pytest.raises(ValueError):
            S.glmm(chol, args[0], args[1], y)
    with pytest.raises(TypeError):
        S.glmm(None, mats, C, y)
    n = g.n
    fit = {"covariance coefficients": np.array([0.3]), "mu": np.full(n, 0.3), "weights": np.full(n, 0.21),
           "working y": np.zeros(n)}
    G = np.zeros((n, 4), dtype=np.int8)
    for kw in (dict(spa_cutoff=-1.0), dict(spa_cutoff=np.nan)):
        with pytest.raises(ValueError):
            S.glmm_association(chol, mats, C, y, fit, G, **kw)
    for bad in (dict(fit, **{"covariance coefficients": np.array([0.3, 0.1])}), dict(fit, mu=np.full(n - 1, 0.3)),
                dict(fit, weights=np.zeros(n))):
        with pytest.raises(ValueError):
            S.glmm_association(chol, mats, C, y, bad, G)
    for bad_G in (G.astype(np.int16), G[1:]):
        with pytest.raises(ValueError):
            S.glmm_association(chol, mats, C, y, fit, bad_G)
    wide = np.hstack([C, np.random.default_rng(0).standard_normal((n, 32 - C.shape[1]))])
    with pytest.raises(ValueError):
        S.glmm_association(chol, mats, wide, y, fit, G)
