"""AI-REML on the GPU: the average-information matrix of RemlSession.evaluate(ai=True) against compute_hess, whole
REML(aireml=True) fits against the oracle's AI-REML driver on the engine's own permutation, the fixed probe block of
a fit, the symmetric-components rule and the two-rank NCCL fit."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import aireml as air
from oracle import estimation as orc
from oracle.cpu_factor import DenseFactor
from tests.util import philox_normals, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def slmm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import scilmm_b200  # noqa: F401
    import scilmm_b200.SparseCholesky  # noqa: F401
    return sys.modules["scilmm_b200.SparseCholesky"]


@pytest.mark.parametrize("tag", ["k2", "k4"])
def test_ai_matrix_equals_minus_compute_hess_c1(golden_c1, slmm, tag):
    """evaluate(ai=True) at C1 size: AI = -compute_hess to 1e-10, and nll / gradient are those of evaluate()."""
    g = golden_c1
    mats, sig = g.mats(tag), g["sig_" + tag]
    ys = g["y"] / g["y"].std()
    chol = slmm.SparseCholesky()
    ses = chol._session(mats, g["cov"], ys)
    Z = np.random.default_rng(3).standard_normal((g.n, 16))
    nll, grad = ses.evaluate(sig, True, 16, Z=Z)
    nll_a, grad_a, AI = ses.evaluate(sig, True, 16, Z=Z, ai=True)
    assert nll_a == nll and np.array_equal(grad_a, grad)
    hess = slmm.compute_hess(mats, g["cov"], ses.factor_at(sig), ys)
    assert rel_err(AI, -hess) < 1e-10
    assert np.array_equal(AI, AI.T)


def test_ai_matrix_ml_drops_the_projection(golden_small, slmm):
    """reml=False: AI = 1/2 (A_i u)' V^-1 (A_j u) with u = V^-1 (y - C beta)."""
    g = golden_small
    mats, sig = g.mats("k4"), g["sig_k4"]
    ys = g["y"] / g["y"].std()
    ses = slmm.SparseCholesky()._session(mats, g["cov"], ys)
    _, _, AI = ses.evaluate(sig, False, 8, Z=np.ones((g.n, 8)), ai=True)
    f = DenseFactor(orc.weighted_sum(mats, sig))
    _, _, mu, _ = orc.fixed_effects(f, ys, g["cov"])
    u = f(ys - mu)
    B = np.column_stack([m.dot(u) for m in mats])
    assert rel_err(AI, 0.5 * B.T @ f(B)) < 1e-10


@pytest.mark.parametrize("base", ["k1", "k3"])
def test_c1_aireml_fit_on_the_engines_own_permutation(golden_c1, slmm, base):
    """Whole REML(aireml=True) fit at C1 size (7 108 individuals) against oracle/aireml.py aireml_reml_fit, forced onto
    the engine's nested-dissection permutation and the same numpy probe block: sigma, beta and standard errors to
    1e-6, the same number of iterations (k3: the epistasis component ends on the floor)."""
    g = golden_c1
    chol = slmm.SparseCholesky()
    np.random.seed(41)
    out = slmm.REML(chol, g.mats(base), g["cov"], g["y"].copy(), reml=True, sim_num=g.sim_num, aireml=True)
    ses = next(iter(chol._sessions.values()))
    P = ses.eng.perm()
    assert not np.array_equal(P, np.arange(g.n))
    np.random.seed(41)
    ref = air.aireml_reml_fit(lambda M: DenseFactor(M, P), g.mats(base), g["cov"], g["y"].copy(), reml=True,
                              sim_num=g.sim_num)
    assert out["aireml"]["converged"] and ref["aireml"]["converged"]
    assert out["aireml"]["iterations"] == ref["aireml"]["iterations"]
    assert ses.n_eval == out["aireml"]["iterations"]
    for key in ("covariance coefficients", "covariates coefficients", "covariance std"):
        assert rel_err(out[key], ref[key]) < 1e-6, (key, out[key], ref[key])


def test_device_probes_one_stream_per_fit(golden_small, slmm):
    """rng='device': two fresh functors with one seed give bit-identical fits, and the fit equals one driven by the host
    copy of stream 0 of the Philox generator (every iteration draws the same block)."""
    g = golden_small
    fits = [slmm.REML(slmm.SparseCholesky(rng="device", seed=5), g.mats("k3"), g["cov"], g["y"].copy(), sim_num=24,
                      aireml=True) for _ in range(2)]
    for key in ("covariance coefficients", "covariates coefficients", "covariance std"):
        assert np.array_equal(fits[0][key], fits[1][key])
    assert fits[0]["aireml"] == fits[1]["aireml"] and fits[0]["aireml"]["iterations"] > 1
    host = slmm.SparseCholesky(rng="host_buffer", seed=5)
    calls = []
    host.probe_source = lambda n, s: calls.append(s) or philox_normals(n, s, 0, 5, 0)[0]
    fit_h = slmm.REML(host, g.mats("k3"), g["cov"], g["y"].copy(), sim_num=24, aireml=True)
    assert calls == [24]
    assert fit_h["aireml"] == fits[0]["aireml"]
    assert rel_err(fit_h["covariance coefficients"], fits[0]["covariance coefficients"]) < 1e-9


def test_asymmetric_component_is_refused(golden_small, slmm):
    g = golden_small
    A = g.csr("A")
    Aj = (sp.tril(A) + 0.5 * sp.triu(A, 1)).tocsr()
    chol = slmm.SparseCholesky()
    with pytest.raises(ValueError):
        slmm.REML(chol, [Aj], g["cov"], g["y"].copy(), sim_num=8, aireml=True)
    with pytest.raises(ValueError):
        slmm.estimate_var_comps(chol, [Aj, sp.eye(g.n).tocsr()], g["cov"], g["y"] / g["y"].std(), sim_num=8,
                                verbose=False, aireml=True)
    ses = chol._session([Aj, sp.eye(g.n).tocsr()], g["cov"], g["y"] / g["y"].std())
    with pytest.raises(ValueError):
        ses.evaluate(np.array([0.4, 0.6]), True, 8, ai=True)


def test_two_rank_nccl_aireml_fit():
    """Sharded AI-REML fits (probe columns split over two ranks, one all-reduce of K doubles per iteration) equal the
    unsharded ones, and both ranks end with the same sigma bit for bit.  Needs two GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29573", os.path.join(ROOT, "tests", "nccl_two_rank_aireml.py")]
    out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "TWO_RANK_AIREML_OK" in out.stdout, out.stdout[-4000:]
