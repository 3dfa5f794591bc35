"""TEST INFRASTRUCTURE ONLY — CPU restatement of the region tests (scilmm_b200.region_test).

The engine forms each region's Phi = X~'P_V X~ as F'F - q'M^-1 q from one forward half-sweep F = L^-1 P X~ and a device
Gram; this restatement builds P_V = V^-1 - V^-1 C (C'V^-1 C)^-1 C'V^-1 explicitly from full solves of a dense factor
and takes Phi = X~' P_V X~ and t = X~' P_V y.  The input rules, default weights, burden and SKAT statistics and NaN rules
are restated here from their definitions; only the tail probability of the chi2 mixture (chi2_mixture_sf) is shared
with the engine.  (It lives beside oracle/association.py rather than in it, which stays as the scan's record.)
"""
import numpy as np
import scipy.sparse as sp
import scipy.stats as stats

from oracle.association import decode
from oracle.cpu_factor import DenseFactor
from oracle.estimation import weighted_sum
from scilmm_b200.SparseCholesky import chi2_mixture_sf

KEYS = ("n_variants", "n_poly", "burden_beta", "burden_se", "burden_chi2", "burden_p", "skat_q", "skat_p")


def check(bounds, weights, m):
    b = np.asarray(bounds)
    if b.ndim != 1 or b.size < 2 or b.dtype.kind not in "iu":
        raise ValueError("bounds must be a 1-D int array")
    b = b.astype(np.int64)
    width = np.diff(b)
    if b[0] != 0 or b[-1] != m or np.any(width < 1) or np.any(width > 512):
        raise ValueError("bounds must go from 0 to m in steps of 1 to 512")
    if weights is not None:
        weights = np.asarray(weights, dtype=float)
        if weights.shape != (m,) or not np.all(np.isfinite(weights)) or np.any(weights < 0):
            raise ValueError("weights must be m finite values >= 0")
    return b, weights


def region_test(mats, covariates, y, sigmas, G, bounds, weights=None, factor=DenseFactor):
    """Same arguments and keys as scilmm_b200.region_test (mats without the identity)."""
    bounds, weights = check(bounds, weights, np.shape(G)[1])
    scale = y.std()
    ys = y / scale
    C = np.asarray(covariates, dtype=np.float64)
    V = weighted_sum(list(mats) + [sp.eye(ys.shape[0]).tocsr()], sigmas)
    Vi = factor(V)(np.eye(ys.shape[0]))
    ViC = Vi @ C
    PV = Vi - ViC @ np.linalg.solve(C.T @ ViC, ViC.T)
    X, af, _ = decode(G)
    if weights is None:
        maf = np.minimum(af, 1.0 - af)
        weights = np.where(np.isnan(af), 0.0, stats.beta.pdf(np.nan_to_num(maf), 1, 25))
    R = bounds.size - 1
    out = {k: np.full(R, np.nan) for k in KEYS}
    out["n_variants"] = np.diff(bounds)
    out["n_poly"] = np.zeros(R, dtype=np.int64)
    for r in range(R):
        Xr = X[:, bounds[r]:bounds[r + 1]]
        w = weights[bounds[r]:bounds[r + 1]]
        xVx = Xr.T @ Vi @ Xr
        Phi = Xr.T @ PV @ Xr
        t = Xr.T @ PV @ ys
        out["n_poly"][r] = np.count_nonzero(np.diag(xVx) > 0)
        score = Xr @ w                             # the burden column: GLS of y on [C | score]
        v = score @ PV @ score
        if v > 1e-10 * (score @ Vi @ score):
            s = score @ PV @ ys
            out["burden_beta"][r] = s / v * scale
            out["burden_se"][r] = scale / np.sqrt(v)
            out["burden_chi2"][r] = s * s / v
            out["burden_p"][r] = stats.chi2.sf(s * s / v, 1)
        lam = np.linalg.eigvalsh(np.diag(w) @ Phi @ np.diag(w))
        if lam[-1] > 1e-10 * np.trace(np.diag(w) @ xVx @ np.diag(w)):
            q = float(np.sum((w * t) ** 2))
            out["skat_q"][r] = q
            out["skat_p"][r] = chi2_mixture_sf(q, lam[lam > 1e-10 * lam[-1]])
    return out
