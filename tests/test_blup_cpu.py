"""CPU checks of the BLUP oracle (oracle/blup.py): the V-form predictor against Henderson's mixed-model equations over
all individuals (with and without unphenotyped ones), the identity sum_k u_k + e = y - C beta on the phenotyped rows,
the exact PEV of the two formulations, the masked prediction against Cov(u_new, y) P y formed densely, and the Monte
Carlo PEV estimate against the exact PEV."""
import numpy as np
import pytest
import scipy.linalg as la
import scipy.sparse as sp

from oracle import blup as ob
from tests.util import rel_err

KEYS = ("u", "residual", "fixed", "yhat", "beta")


def masked_y(y, ncov, mask):
    """y with NaN at the unphenotyped individuals of one of the named masks."""
    y = np.array(y, dtype=float)
    n = y.size
    if mask == "random":
        y[np.random.default_rng(3).random(n) < 0.2] = np.nan
    elif mask == "first":
        y[0] = np.nan
    elif mask == "last":
        y[-1] = np.nan
    elif mask == "few":                      # only c + 1 individuals keep a phenotype
        keep = np.random.default_rng(4).choice(n, ncov + 1, replace=False)
        drop = np.ones(n, dtype=bool)
        drop[keep] = False
        y[drop] = np.nan
    return y


MASKS = ["none", "random", "first", "last", "few"]


def assert_close(a, b, tol, keys=KEYS):
    for k in keys:
        fin = np.isfinite(b[k])
        assert np.array_equal(np.isfinite(a[k]), fin), k
        assert rel_err(a[k][fin], b[k][fin]) <= tol, (k, rel_err(a[k][fin], b[k][fin]))


@pytest.mark.parametrize("case", ["small", "c1mini"])
@pytest.mark.parametrize("mask", MASKS)
def test_vform_equals_mme(golden_small, golden_c1mini, case, mask):
    g = golden_small if case == "small" else golden_c1mini
    mats, sig = g.mats("k2")[:-1], g["sig_k2"]
    y = masked_y(g["y"], g["cov"].shape[1], mask)
    v = ob.blup_vform(mats, g["cov"], y, sig)
    m = ob.blup_mme(mats[0], g["cov"], y, sig)
    assert_close(v, m, 1e-10, KEYS + ("pev", "reliability"))
    assert np.array_equal(np.isnan(v["residual"]), np.isnan(y))


@pytest.mark.parametrize("case", ["small", "c1mini"])
@pytest.mark.parametrize("mask", MASKS)
def test_components_and_residual_add_up(golden_small, golden_c1mini, case, mask):
    """On the phenotyped rows sum_k u_k + e = s V u = y - s C beta (V u = y_s - C beta)."""
    g = golden_small if case == "small" else golden_c1mini
    y = masked_y(g["y"], g["cov"].shape[1], mask)
    out = ob.blup_vform(g.mats("k4")[:-1], g["cov"], y, g["sig_k4"])
    obs = ~np.isnan(y)
    lhs = out["u"][obs].sum(axis=1) + out["residual"][obs]
    assert rel_err(lhs, y[obs] - out["fixed"][obs]) <= 1e-12
    assert np.allclose(out["yhat"], out["fixed"] + out["u"].sum(axis=1), rtol=0, atol=1e-14 * np.abs(y[obs]).max())


@pytest.mark.parametrize("mask", ["none", "random"])
def test_masked_prediction_is_conditional_mean(golden_c1mini, mask):
    """u_k = Cov(u_k, y) P y with P = V^-1 - V^-1 C (C'V^-1 C)^-1 C'V^-1 formed from a dense inverse of V."""
    g = golden_c1mini
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    y = masked_y(g["y"], g["cov"].shape[1], mask)
    out = ob.blup_vform(mats, g["cov"], y, sig)
    idx = np.flatnonzero(~np.isnan(y))
    s = y[idx].std()
    V = sum(sig[k] * mats[k].toarray()[np.ix_(idx, idx)] for k in range(3)) + sig[3] * np.eye(idx.size)
    Vi = la.inv(V)
    C = g["cov"][idx]
    P = Vi - Vi @ C @ la.inv(C.T @ Vi @ C) @ C.T @ Vi
    for k in range(3):
        ref = s * sig[k] * mats[k].toarray()[:, idx] @ (P @ (y[idx] / s))
        assert rel_err(out["u"][:, k], ref) <= 1e-10


def test_stochastic_pev_tracks_the_exact_pev(golden_small):
    """The Monte Carlo estimate is unbiased with the standard error it reports: z = (est - exact) / se."""
    g = golden_small
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    y = masked_y(g["y"], g["cov"].shape[1], "random")
    n = int(np.sum(~np.isnan(y)))
    exact = ob.blup_vform(mats, g["cov"], y, sig)["pev"]
    est, se = ob.pev_stochastic(mats, g["cov"], y, sig, 1024, 7, np.arange(n))
    # no phenotyped relative through A_k (a household whose members all lack a phenotype): nothing to estimate
    none = se == 0
    assert 0 < none.sum() < 0.2 * none.size
    assert rel_err(est[none], exact[none]) <= 1e-12
    est, se, exact = est[~none], se[~none], exact[~none]
    z = (est - exact) / se
    assert np.mean(np.abs(z) > 4) < 0.005 and abs(np.mean(z)) < 0.2, (np.mean(np.abs(z) > 4), np.mean(z))
    # a different order of the factor changes the probes, not the quantity estimated
    est2, se2 = ob.pev_stochastic(mats, g["cov"], y, sig, 1024, 7, np.arange(n)[::-1])
    est2, se2 = est2[~none], se2[~none]
    assert not np.array_equal(est, est2)
    assert np.mean(np.abs(est2 - exact) / se2 > 4) < 0.005


def test_identity_component_is_predicted_like_any_other(golden_small):
    g = golden_small
    mats = [g.mats("k2")[0], sp.eye(g.n).tocsr()]
    sig = np.array([0.4, 0.2, 0.4])
    y = masked_y(g["y"], g["cov"].shape[1], "random")
    out = ob.blup_vform(mats, g["cov"], y, sig)
    obs = ~np.isnan(y)
    assert np.all(out["u"][~obs, 1] == 0.0)               # no phenotype, no covariance with y through I
    assert rel_err(out["u"][obs, 1], out["residual"][obs] * sig[1] / sig[2]) <= 1e-12
