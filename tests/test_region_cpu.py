"""CPU checks of the region tests: the oracle (oracle/region.py) burden statistic against an explicit GLS refit with the
burden score as one more covariate, one-variant regions against the association oracle, the tail function of the chi2
mixture (exact branch, closed form of the (a, a, b, b) mixture, the point q = sum lam, monotonicity), the null
calibration of the SKAT p-value, and the input rules."""
import numpy as np
import pytest
import scipy.stats as stats

from oracle import association as oa
from oracle import estimation as orc
from oracle import region as oreg
from oracle.cpu_factor import DenseFactor
import scilmm_b200 as slmm
from scilmm_b200.SparseCholesky import chi2_mixture_sf
from tests.test_association_cpu import make_genotypes, with_variant_covariate

BOUNDS = np.array([0, 1, 3, 4, 10, 25, 26, 40])      # regions of 1, 2 (monomorphic), 1, 6, 15, 1 and 14 variants


def closed_form(q, a, b):
    """P(a chi2_2 + b chi2_2 > q), a != b."""
    return (a * np.exp(-q / (2 * a)) - b * np.exp(-q / (2 * b))) / (a - b)


@pytest.mark.parametrize("weights", ["default", "random"])
def test_burden_equals_explicit_refit(golden_small, weights):
    g = golden_small
    mats, sig, y, cov = g.mats("k3"), g["sig_k4"], g["y"], g["cov"]
    G = make_genotypes(g.n, 40, 31)
    w = None if weights == "default" else np.random.default_rng(2).uniform(0.1, 3.0, 40)
    res = oreg.region_test(mats, cov, y, sig, G, BOUNDS, w)
    X, af, _ = oa.decode(G)
    if w is None:
        w = stats.beta.pdf(np.minimum(af, 1 - af), 1, 25)
    ys = y / y.std()
    f = DenseFactor(orc.weighted_sum(g.mats("k4"), sig))
    assert np.array_equal(res["n_variants"], np.diff(BOUNDS))
    assert np.isnan(res["burden_beta"][1]) and np.isnan(res["skat_p"][1]) and res["n_poly"][1] == 0
    checked = 0
    for r in range(BOUNDS.size - 1):
        if not np.isfinite(res["burden_beta"][r]):
            continue
        score = X[:, BOUNDS[r]:BOUNDS[r + 1]] @ w[BOUNDS[r]:BOUNDS[r + 1]]
        Cs = np.hstack([cov, score[:, None]])
        ViC, _, _, beta = orc.fixed_effects(f, ys, Cs)
        cov_beta = np.linalg.inv(Cs.T @ ViC)
        assert abs(res["burden_beta"][r] - beta[-1] * y.std()) <= 1e-9 * abs(beta[-1] * y.std())
        assert abs(res["burden_se"][r] - np.sqrt(cov_beta[-1, -1]) * y.std()) <= 1e-9 * res["burden_se"][r]
        assert abs(res["burden_chi2"][r] - beta[-1] ** 2 / cov_beta[-1, -1]) <= 1e-9 * res["burden_chi2"][r]
        checked += 1
    assert checked == BOUNDS.size - 2


def test_one_variant_regions_match_the_association_oracle(golden_small):
    g = golden_small
    mats, sig = g.mats("k3"), g["sig_k4"]
    G = make_genotypes(g.n, 12, 32)
    cov = with_variant_covariate(g["cov"], G, 0)
    w = np.random.default_rng(5).uniform(0.5, 2.0, 12)
    res = oreg.region_test(mats, cov, g["y"], sig, G, np.arange(13), w)
    ref = oa.association(mats, cov, g["y"], sig, G)
    nan = ~np.isfinite(ref["chi2"])
    assert np.array_equal(np.flatnonzero(nan), [0, 1, 2])
    for k in ("burden_chi2", "burden_p", "skat_p"):
        assert np.array_equal(~np.isfinite(res[k]), nan), k
    fin = ~nan
    for got, want in ((res["burden_chi2"], ref["chi2"]), (res["burden_p"], ref["p"]), (res["skat_p"], ref["p"]),
                      (res["burden_beta"] * w, ref["beta"]), (res["burden_se"] * w, ref["se"])):
        assert np.all(np.abs(got[fin] - want[fin]) <= 1e-12 * np.abs(want[fin]))
    xPx = (g["y"].std() / ref["se"][fin]) ** 2           # x~'P_V x~ in the standardised units
    assert np.allclose(res["skat_q"][fin], (w * w)[fin] * ref["chi2"][fin] * xPx, rtol=1e-12, atol=0)


@pytest.mark.parametrize("r", [1, 5, 40])
def test_tail_exact_for_equal_weights(r):
    lam = np.full(r, 0.7)
    for q in (1e-3, 0.5, r * 0.7, 10.0, 200.0, 2000.0):
        want = stats.chi2.sf(q / 0.7, r)
        assert abs(chi2_mixture_sf(q, lam) - want) <= 1e-12 * want


@pytest.mark.parametrize("ratio", [1.5, 3, 10, 100, 1000])
def test_tail_against_closed_form(ratio):
    a, b = ratio, 1.0
    lam = [a, a, b, b]
    for p in np.logspace(np.log10(0.99), -300, 120):
        lo, hi = 1e-9, 2.0 * a * (np.log(a / (a - b)) - np.log(p)) + 10 * a
        for _ in range(200):                  # q with closed_form(q) = p, bisected in log p
            mid = 0.5 * (lo + hi)
            lo, hi = (mid, hi) if closed_form(mid, a, b) > p else (lo, mid)
        q = 0.5 * (lo + hi)
        want = closed_form(q, a, b)
        band = 0.0063 if want > 0.5 else (0.040 if want > 1e-6 else 0.073)
        assert abs(chi2_mixture_sf(q, lam) / want - 1) <= band, (ratio, q, want)


@pytest.mark.parametrize("ratio", [1.5, 10, 1000])
def test_tail_at_the_mean(ratio):
    lam = np.array([ratio, ratio, 1.0, 1.0])
    for q in lam.sum() * np.array([1 - 1e-9, 1.0, 1 + 1e-9]):
        p = chi2_mixture_sf(q, lam)
        assert np.isfinite(p) and abs(p / closed_form(q, ratio, 1.0) - 1) <= 0.01


def test_tail_monotone_and_q_nonpositive():
    lam = np.array([5.0, 2.0, 1.0, 0.3, 0.01])
    grid = np.concatenate([np.linspace(1e-6, 3 * lam.sum(), 400), np.geomspace(3 * lam.sum(), 5000, 200)])
    p = np.array([chi2_mixture_sf(q, lam) for q in grid])
    assert np.all(np.diff(p) <= 0) and np.all((p >= 0) & (p <= 1))
    assert chi2_mixture_sf(0.0, lam) == 1.0 and chi2_mixture_sf(-1.0, lam) == 1.0


def test_skat_null_calibration():
    rng = np.random.default_rng(11)
    A = rng.standard_normal((6, 6))
    U = np.linalg.qr(A)[0]
    Phi = U @ np.diag([4.0, 2.5, 1.5, 1.0, 0.6, 0.2]) @ U.T
    lam = np.linalg.eigvalsh(Phi)
    t = rng.multivariate_normal(np.zeros(6), Phi, size=20000)
    p = np.array([chi2_mixture_sf(q, lam) for q in np.sum(t * t, axis=1)])
    assert stats.kstest(p, "uniform").pvalue > 1e-3


def test_input_rules(golden_small):
    g = golden_small
    mats, sig, y, cov = g.mats("k3"), g["sig_k4"], g["y"], g["cov"]
    G = make_genotypes(g.n, 600, 33)
    bad = [np.array([1, 600]), np.array([0, 599]), np.array([0, 10, 10, 600]), np.array([0, 20, 10, 600]),
           np.array([0, 513, 600]), np.array([0.0, 600.0])]
    ok = np.array([0, 512, 600])
    bad_w = (np.ones(599), -np.ones(600), np.r_[np.ones(599), np.nan], np.r_[np.ones(599), np.inf])
    for call in (oreg.region_test, lambda *a: slmm.region_test(slmm.SparseCholesky(), *a)):
        for b in bad:
            with pytest.raises(ValueError):
                call(mats, cov, y, sig, G, b)
        for w in bad_w:
            with pytest.raises(ValueError):
                call(mats, cov, y, sig, G, ok, w)
