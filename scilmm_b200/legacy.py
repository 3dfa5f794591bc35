"""Drop-ins for the reference's legacy estimation entry points (scilmm/Estimation/LMM.py, scilmm/Estimation/HE.py),
which scilmm/SciLMM.py:185-189 still calls.  Same signatures and return values; all sparse / factorization
arithmetic runs in libscilmm_b200.so through the engine of scilmm_b200.SparseCholesky (no CPU fallback).

    LMM(cholesky, mats, covariates, y, with_intercept=True, reml=True, sim_num=100, verbose=False)   LMM.py:154-171
    compute_HE(y, covariates, covariance_matrices, fit_intercept=False)                              HE.py:22-40

Differences of the legacy path against SparseCholesky.REML that are preserved here: the intercept column comes
FIRST (LMM.py:157), the optimiser starts from equal components instead of the HE estimate (LMM.py:113-114), y is
not standardised, fixed-effect p-values are returned (LMM.py:127-131), and compute_HE regresses the covariates out
with an (optional) intercept, uses only off-diagonal moments and appends 1 - sum as the residual component.
"""
import numpy as np
import scipy.linalg as la
import scipy.optimize as optimize
import scipy.sparse as sparse
import scipy.stats as stats

import importlib
from . import engine as _eng

_mod = importlib.import_module("scilmm_b200.SparseCholesky")   # the module (the package attribute is the class)


def compute_sigmas(cholesky, mats, covariates, y, reml=True, sim_num=100, verbose=True):
    """LMM.py:111-124: L-BFGS-B over log sigma from equal starting components."""
    x0 = np.ones(len(mats))
    x0 = np.log(x0 / x0.sum())
    opt = optimize.minimize(_mod.bolt_gradient_estimation, x0,
                            args=(cholesky, mats, covariates, y, reml, sim_num, verbose, True),
                            jac=True, method='L-BFGS-B', options={'eps': 1e-5, 'ftol': 1e-7})
    return np.exp(opt.x)


def compute_fixed_effects_p_value(y, covariates, fixed_effects, L_CT_invV_C):
    """LMM.py:127-131."""
    var_fixedeffects = la.cho_solve(L_CT_invV_C, np.eye(covariates.shape[1]))
    test_stats = fixed_effects ** 2 / np.diag(var_fixedeffects)
    return stats.f(1, y.shape[0] - 1).sf(test_stats)


def LMM(cholesky, mats, covariates, y, with_intercept=True, reml=True, sim_num=100, verbose=False):
    """LMM.py:154-171 on the GPU engine."""
    functor = _mod._need_functor(cholesky)
    y = np.asarray(y, dtype=np.float64)
    mats = list(mats) + [sparse.eye(y.size).tocsr()]
    covariates = np.asarray(covariates, dtype=np.float64)
    if with_intercept:
        covariates = np.hstack((np.ones((y.size, 1)), covariates))
    mats_coefficients = compute_sigmas(functor, mats, covariates, y, reml, sim_num, verbose)
    ses = functor._session(mats, covariates, y)
    ses.factor_at(mats_coefficients)
    _, chol, fixed_effects, _, _ = ses.fixed_effects()
    p_values = compute_fixed_effects_p_value(y, covariates, fixed_effects, chol)
    sigmas_sigmas = compute_sig_of_sig(ses, sim_num)
    return {"covariance coefficients": mats_coefficients,
            "covariates coefficients": fixed_effects,
            "covariance std": sigmas_sigmas,
            "covariates p-values": p_values}


def compute_sig_of_sig(ses, sim_num):
    """LMM.py:134-151 on the device.  Unlike SparseCholesky.compute_hess (:147-168) only the innermost vector is
    projected: hess[i,j] = -0.5 y' V^-1 A_i V^-1 A_j P y; the K solves of each stage are batched as one multi-RHS
    solve."""
    torch = ses.torch
    K, C, y, eng = ses.K, ses.C, ses.y, ses.eng
    B = torch.cat([C, y.unsqueeze(1)], dim=1).contiguous()
    eng.solve_(B)
    c = C.shape[1]
    ViC, Viy = B[:, :c].contiguous(), B[:, c].contiguous()
    M = torch.linalg.inv(C.t() @ ViC)
    Py = Viy - ViC @ (M @ (C.t() @ Viy))
    F = eng.solve_(torch.cat([ses.matset.spmm(j, Py.unsqueeze(1)) for j in range(K)], dim=1).contiguous())
    hess = np.empty((K, K))
    for i in range(K):
        G = eng.solve_(ses.matset.spmm(i, F[:, i:].contiguous()))
        vals = (-0.5 * (y @ G)).cpu().numpy()
        for t, j in enumerate(range(i, K)):
            hess[i, j] = hess[j, i] = vals[t]
    return np.sqrt(np.diag(la.inv(-hess)) * (1 + 1.0 / sim_num))


def regress_beta_out(y, covariates, fit_intercept):
    """HE.py:8-19 (sklearn LinearRegression restated as a least-squares solve; same residuals and coefficients)."""
    y = np.asarray(y, dtype=np.float64)
    C = np.asarray(covariates, dtype=np.float64)
    X = np.hstack((C, np.ones((C.shape[0], 1)))) if fit_intercept else C
    coefs, *_ = np.linalg.lstsq(X, y, rcond=None)
    return y - X.dot(coefs), coefs.tolist()


def compute_HE(y, covariates, covariance_matrices, fit_intercept=False):
    """HE.py:22-40: off-diagonal Haseman-Elston moments on the GPU, residual component appended."""
    if any(not sparse.issparse(m) for m in covariance_matrices):
        raise TypeError("scilmm_b200.legacy.compute_HE takes scipy.sparse matrices")
    y, cov_coefs = regress_beta_out(y, covariates, fit_intercept)
    torch = _eng.require_cuda()
    ms = _eng.MatSet(list(covariance_matrices))
    out = ms.he_moments_device(_eng.to_device(y, torch)).cpu().numpy()
    q_off, _, S_off, _ = _eng.MatSet.split_moments(out, ms.K)
    coef = np.linalg.inv(S_off).dot(q_off)
    coef = np.append(coef, 1 - coef.sum())
    return coef, cov_coefs
