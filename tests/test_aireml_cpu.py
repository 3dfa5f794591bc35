"""AI-REML on the CPU: the Gram form of the average-information matrix the engine computes, and the oracle's AI-REML
driver (oracle/aireml.py aireml_fit) against the optimum of the exact REML likelihood.  No GPU needed."""
import importlib

import numpy as np
import pytest
import scipy.linalg as la
import scipy.optimize as optimize
import scipy.sparse as sp

from oracle import aireml as air
from oracle import estimation as orc
from oracle.cpu_factor import DenseFactor
from tests.util import rel_err


def exact_probes(n, s):
    """sqrt(s) I: W W' / s = V^-1 exactly, so the Monte-Carlo traces of gradient_terms are exact (s = n)."""
    return np.sqrt(s) * np.eye(n, s)


def exact_reml_optimum(mats, C, y, floor):
    """Minimiser of the exact REML nll (dense V^-1) over sigma >= floor, by bounded L-BFGS-B on sigma itself."""
    dense = [m.toarray() for m in mats]

    def nll_grad(s):
        V = sum(sk * m for sk, m in zip(s, dense))
        Vi = la.inv(V)
        ViC = Vi @ C
        M = C.T @ ViC
        P = Vi - ViC @ la.solve(M, ViC.T)
        Py = P @ y
        nll = 0.5 * (y @ Py + np.linalg.slogdet(V)[1] + np.linalg.slogdet(M)[1])
        return nll, np.array([0.5 * (np.sum(P * m) - Py @ m @ Py) for m in dense])
    res = optimize.minimize(nll_grad, np.full(len(mats), 1.0 / len(mats)), jac=True, method="L-BFGS-B",
                            bounds=[(floor, None)] * len(mats), options=dict(ftol=1e-16, gtol=1e-12, maxiter=1000))
    return res.x


@pytest.mark.parametrize("case", ["golden_small", "golden_c1mini"])
@pytest.mark.parametrize("tag", ["k2", "k4"])
def test_gram_form_of_the_ai_matrix(case, tag, request):
    """AI_ij = 1/2 [F_i'F_j - (ViC'b_i)' (C'V^-1C)^-1 (ViC'b_j)] with F = L^-1 P B (a forward solve only, rows in the
    permuted order) equals -average_information (reference compute_hess)."""
    g = request.getfixturevalue(case)
    mats, sig = g.mats(tag), g["sig_" + tag]
    ys = g["y"] / g["y"].std()
    C = g["cov"]
    perm = np.random.default_rng(7).permutation(g.n).astype(np.int32)
    f = DenseFactor(orc.weighted_sum(mats, sig), perm)
    ViC, chol, mu, _ = orc.fixed_effects(f, ys, C)
    u = f(ys - mu)
    B = np.column_stack([m.dot(u) for m in mats])
    F = la.solve_triangular(f._Lp, B[perm], lower=True)
    CtB = ViC.T @ B
    AI = 0.5 * (F.T @ F - CtB.T @ la.cho_solve(chol, CtB))
    assert rel_err(AI, -orc.average_information(mats, C, f, ys)) < 1e-12


@pytest.mark.parametrize("base", ["k1", "k3"])
def test_exact_trace_fit_reaches_the_exact_optimum(base, golden_c1mini):
    """Exact traces (n = 1 720): the AI-REML fit lands on the bounded optimum of the exact REML likelihood, the k4
    component whose optimum is 0 on the floor."""
    g = golden_c1mini
    ys = g["y"] / g["y"].std()
    mats = g.mats(base) + [sp.eye(g.n).tocsr()]
    sig, info = air.aireml_fit(lambda M: DenseFactor(M), mats, g["cov"], ys, True, g.n, normal_source=exact_probes)
    ref = exact_reml_optimum(mats, g["cov"], ys, air.AIREML_FLOOR)
    assert info["converged"]
    assert np.max(np.abs(sig - ref)) < 1e-6, (sig, ref)
    if base == "k3":
        assert sig[1] == air.AIREML_FLOOR and np.all(sig[[0, 2, 3]] > 1e-2)


def test_floor_jump_shortens_the_fit(golden_small):
    """The linearised-step rule puts the boundary component on the floor in one step instead of a walk of capped
    steps; both versions reach the same optimum."""
    g = golden_small
    ys = g["y"] / g["y"].std()
    mats = g.mats("k4")
    out = {}
    for jump in (False, True):
        out[jump] = air.aireml_fit(lambda M: DenseFactor(M), mats, g["cov"], ys, True, g.n, normal_source=exact_probes,
                                   jump=jump)
        assert out[jump][1]["converged"]
    assert out[True][1]["iterations"] + 5 <= out[False][1]["iterations"]
    assert np.max(np.abs(out[True][0] - out[False][0])) < 1e-5


@pytest.mark.parametrize("tag", ["k2", "k4"])
def test_fixed_probe_block_fit_stops_on_the_step_rule(tag, golden_small):
    """Monte-Carlo traces from ONE probe block: the fit is a deterministic root-finding problem and stops with a
    step below the tolerance; the block is drawn once."""
    g = golden_small
    ys = g["y"] / g["y"].std()
    draws = []

    def source(n, s):
        draws.append(s)
        return np.random.default_rng(11).standard_normal((n, s))
    trace = []
    sig, info = air.aireml_fit(lambda M: DenseFactor(M), g.mats(tag), g["cov"], ys, True, 20, normal_source=source,
                               trace=trace)
    assert draws == [20] and info["converged"] and info["iterations"] == len(trace) < air.AIREML_MAX_ITER
    s, grad, AI = trace[-1]
    new, size = air.aireml_step(s, grad, AI)
    assert size < air.AIREML_TOL and np.array_equal(new, sig)


def test_engine_step_rule_is_the_oracles():
    """The engine's host step (scilmm_b200.SparseCholesky._aireml_step) and the oracle's restatement agree bit for
    bit, boundary cases included; the engine's constants are the oracle's."""
    S = importlib.import_module("scilmm_b200.SparseCholesky")
    assert (S.AIREML_FLOOR, S.AIREML_TOL, S.AIREML_MAX_ITER) == (air.AIREML_FLOOR, air.AIREML_TOL,
                                                                  air.AIREML_MAX_ITER)
    rng = np.random.default_rng(0)
    jumps = 0
    for _ in range(500):
        K = int(rng.integers(2, 6))
        sig = np.exp(rng.normal(size=K) - 1)
        sig[rng.random(K) < 0.2] = air.AIREML_FLOOR
        grad = 3 * rng.normal(size=K)
        M = rng.normal(size=(K, K))
        AI = M @ M.T + 0.1 * np.eye(K)
        a, b = S._aireml_step(sig, grad, AI), air.aireml_step(sig, grad, AI)
        assert np.array_equal(a[0], b[0]) and a[1] == b[1]
        assert np.all(a[0] >= air.AIREML_FLOOR)
        jumps += int(np.any((a[0] == air.AIREML_FLOOR) & (sig > air.AIREML_FLOOR)))
    assert jumps > 0
