"""CPU checks of the association-scan oracle (oracle/association.py): its coefficient and standard error are those of
an explicit GLS refit with the variant as one more covariate, and the genotype decoding rules (missing values, allele
frequency, counts, NaN for monomorphic variants and for variants in the span of the covariates).  Also the input rules
of association(), region_test() and blup(), which need no device."""
import sys

import numpy as np
import pytest

from oracle import association as oa
from oracle import estimation as orc
from oracle.cpu_factor import DenseFactor


def make_genotypes(n, m, seed, missing=0.02):
    """Seeded (n, m) int8 allele counts: per-variant frequencies in 0.05-0.5, `missing` of the entries negative
    (-1 or -9), column 1 monomorphic (all 0), column 2 monomorphic (all 2, with missing entries), column 0 without
    missing entries (tests use it as a covariate)."""
    rng = np.random.default_rng(seed)
    af = rng.uniform(0.05, 0.5, m)
    G = rng.binomial(2, af[None, :], size=(n, m)).astype(np.int8)
    miss = rng.random((n, m)) < missing
    G[miss] = np.where(rng.random(int(miss.sum())) < 0.5, -1, -9).astype(np.int8)
    G[:, 0] = rng.binomial(2, 0.3, n)
    G[:, 1] = 0
    G[:, 2] = np.where(G[:, 2] < 0, G[:, 2], 2)
    return G


def with_variant_covariate(cov, G, j=0):
    """Covariates plus the centred column j of G: that variant then lies in the span of the covariates."""
    X, _, _ = oa.decode(G[:, j:j + 1])
    return np.hstack([cov, X])


def test_oracle_equals_explicit_refit(golden_small):
    g = golden_small
    mats, sig = g.mats("k3"), g["sig_k4"]
    y, cov = g["y"], g["cov"]
    G = make_genotypes(g.n, 12, 3)
    res = oa.association(mats, cov, y, sig, G)
    ys = y / y.std()
    f = DenseFactor(orc.weighted_sum(g.mats("k4"), sig))
    X, _, _ = oa.decode(G)
    checked = 0
    for j in range(G.shape[1]):
        if not np.isfinite(res["beta"][j]):
            continue
        Cj = np.hstack([cov, X[:, j:j + 1]])
        ViC, chol, _, beta = orc.fixed_effects(f, ys, Cj)
        cov_beta = np.linalg.inv(Cj.T @ ViC)
        assert abs(res["beta"][j] - beta[-1] * y.std()) < 1e-9 * abs(beta[-1] * y.std())
        assert abs(res["se"][j] - np.sqrt(cov_beta[-1, -1]) * y.std()) < 1e-9 * res["se"][j]
        assert abs(res["chi2"][j] - beta[-1] ** 2 / cov_beta[-1, -1]) < 1e-9 * res["chi2"][j]
        checked += 1
    assert checked == G.shape[1] - 2


def test_decoding_rules(golden_small):
    g = golden_small
    G = make_genotypes(g.n, 8, 5)
    G[3, 4] = -128
    X, af, n_obs = oa.decode(G)
    obs = G >= 0
    assert np.array_equal(n_obs, obs.sum(axis=0))
    for j in range(G.shape[1]):
        mu = G[obs[:, j], j].astype(float).mean()
        assert af[j] == mu / 2
        assert np.all(X[~obs[:, j], j] == 0.0)
        assert np.allclose(X[obs[:, j], j], G[obs[:, j], j] - mu, rtol=0, atol=1e-15)
    assert n_obs[0] == g.n and n_obs[4] < g.n and af[1] == 0.0 and af[2] == 1.0
    cov = with_variant_covariate(g["cov"], G, 0)
    res = oa.association(g.mats("k3"), cov, g["y"], g["sig_k4"], G)
    nan = ~np.isfinite(res["beta"])
    assert np.array_equal(np.flatnonzero(nan), [0, 1, 2])
    for k in ("se", "chi2", "p"):
        assert np.array_equal(~np.isfinite(res[k]), nan)
    assert np.all((res["p"][~nan] > 0) & (res["p"][~nan] <= 1))
    bad = G.copy()
    bad[7, 6] = 3
    with pytest.raises(ValueError):
        oa.decode(bad)


def test_refused_inputs_need_no_device(golden_small):
    """association(), region_test() and blup() check G, the variance components and the covariates before they look
    for a device: bad input raises ValueError on any host, not the missing-device RuntimeError."""
    import scilmm_b200.SparseCholesky  # noqa: F401
    S = sys.modules["scilmm_b200.SparseCholesky"]
    g = golden_small
    mats, sig, y, cov = g.mats("k3"), g["sig_k4"], g["y"], g["cov"]
    G = make_genotypes(g.n, 40, 5)
    wide = np.hstack([cov, np.random.default_rng(0).standard_normal((g.n, 32 - cov.shape[1]))])
    scans = (lambda C, s, G: S.association(S.SparseCholesky(), mats, C, y, s, G),
             lambda C, s, G: S.region_test(S.SparseCholesky(), mats, C, y, s, G, np.array([0, 20, 40])))
    for call in scans:
        for C, s, bad_G in ((cov, sig, G.astype(np.int16)), (cov, sig, G[1:]), (cov, sig[1:], G), (wide, sig, G)):
            with pytest.raises(ValueError):
                call(C, s, bad_G)
    for C, s in ((cov, sig[1:]), (cov, np.r_[sig, 0.1]), (wide, sig)):
        with pytest.raises(ValueError):
            S.blup(S.SparseCholesky(), mats, C, y, s)
