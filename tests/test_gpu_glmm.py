"""Binary traits on the GPU (glmm() / glmm_association()): the PQL fit against oracle/glmm.py on the engine's own
permutation, device probes, the fixed point of the fit, the score statistics and the saddlepoint kernel against the
oracle, bitwise independence of the saddlepoint block, a planted effect, refused inputs, device memory and the sharded
fit and scan over two ranks."""
import gc
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import glmm as og
from oracle.association import decode
from oracle.cpu_factor import DenseFactor
from tests.test_association_cpu import make_genotypes
from tests.util import philox_normals, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIT_KEYS = ("covariance coefficients", "covariates coefficients", "covariance std", "covariates std")


@pytest.fixture(scope="module")
def slmm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import scilmm_b200.SparseCholesky  # noqa: F401
    return sys.modules["scilmm_b200.SparseCholesky"]


def binary(g, prevalence):
    """The golden y thresholded so that a fraction `prevalence` are cases; the golden covariates carry the intercept."""
    return (g["y"] > np.quantile(g["y"], 1.0 - prevalence)).astype(np.float64)


def rare_genotypes(n, m, seed):
    """make_genotypes with low-frequency columns from column 3 on (allele frequency 0.002 - 0.03)."""
    G = make_genotypes(n, m, seed)
    rng = np.random.default_rng(seed + 1)
    af = rng.uniform(0.002, 0.03, m - 3)
    G[:, 3:] = np.where(G[:, 3:] < 0, G[:, 3:], rng.binomial(2, af[None, :], size=(n, m - 3)))
    return G


@pytest.fixture(scope="module")
def c1_fit(golden_c1, slmm):
    """One K = 1 fit on case_c1 at prevalence 0.05 and its functor."""
    g = golden_c1
    y = binary(g, 0.05)
    chol = slmm.SparseCholesky()
    np.random.seed(7)
    fit = slmm.glmm(chol, [g.csr("A")], g["cov"], y, sim_num=g.sim_num)
    assert fit["glmm"]["converged"]
    return chol, y, fit


@pytest.mark.parametrize("tag", ["k1", "k3"])
def test_fit_matches_oracle_on_the_engines_permutation(golden_c1, slmm, tag):
    g = golden_c1
    y = binary(g, 0.3)
    chol = slmm.SparseCholesky()
    np.random.seed(41)
    out = slmm.glmm(chol, g.mats(tag), g["cov"], y, sim_num=g.sim_num)
    P = chol._glmm.eng.perm()
    assert not np.array_equal(P, np.arange(g.n))
    np.random.seed(41)
    ref = og.pql_fit(lambda M: DenseFactor(M, P), g.mats(tag), g["cov"], y, sim_num=g.sim_num)
    assert out["glmm"]["converged"] and ref["glmm"]["converged"]
    assert out["glmm"]["iterations"] == ref["glmm"]["iterations"]
    for key in FIT_KEYS:
        assert rel_err(out[key], ref[key]) < 1e-6, (key, out[key], ref[key])
    for key in ("mu", "eta", "working y", "weights"):
        assert rel_err(out[key], ref[key]) < 1e-6, key
    mu, w, Yt = og.working(out["eta"], y)
    assert rel_err(out["mu"], mu) < 1e-14 and np.array_equal(out["weights"], out["mu"] * (1 - out["mu"]))
    assert rel_err(out["working y"], Yt) < 1e-12
    tau = out["covariance coefficients"]
    assert np.allclose(out["latent fractions"], tau / (tau.sum() + np.pi ** 2 / 3), rtol=1e-15)


def test_device_probes_one_stream_per_fit(golden_small, slmm):
    g = golden_small
    y = binary(g, 0.3)
    mats = g.mats("k1")
    fits = [slmm.glmm(slmm.SparseCholesky(rng="device", seed=5), mats, g["cov"], y, sim_num=24) for _ in range(2)]
    for key in FIT_KEYS + ("mu", "working y"):
        assert np.array_equal(fits[0][key], fits[1][key]), key
    assert fits[0]["glmm"] == fits[1]["glmm"] and fits[0]["glmm"]["iterations"] > 1
    host = slmm.SparseCholesky(rng="host_buffer", seed=5)
    calls = []
    host.probe_source = lambda n, s: calls.append(s) or philox_normals(n, s, 0, 5, 0)[0]
    fit_h = slmm.glmm(host, mats, g["cov"], y, sim_num=24)
    assert calls == [24]
    assert fit_h["glmm"] == fits[0]["glmm"]
    for key in FIT_KEYS:
        assert rel_err(fit_h[key], fits[0][key]) < 1e-9, key


def test_fixed_point_and_phase1_against_the_oracle(golden_c1, slmm, c1_fit):
    """At the returned state the scan's U is x~'(y - mu) up to the PQL tolerance; U and Var(U) equal the oracle's dense
    score statistics to 1e-9; the call reuses the fit's session."""
    g = golden_c1
    chol, y, fit = c1_fit
    ses = chol._glmm
    G = make_genotypes(g.n, 60, 31)
    out = slmm.glmm_association(chol, [g.csr("A")], g["cov"], y, fit, G, spa_cutoff=np.inf)
    assert chol._glmm is ses
    assert set(out) == set(slmm.GLMM_ASSOC_KEYS) and all(out[k].shape == (60,) for k in slmm.GLMM_ASSOC_KEYS)
    assert out["spa"].dtype == np.int8 and not out["spa"].any()
    assert np.array_equal(out["p"], out["p_normal"], equal_nan=True)
    X, af, n_obs = decode(G)
    direct = X.T @ (y - fit["mu"])
    fin = np.isfinite(out["score"])
    assert np.array_equal(np.flatnonzero(~fin), [1, 2])
    assert np.max(np.abs(out["score"][fin] - direct[fin])) < 1e-3 * np.max(np.abs(direct[fin]))
    U, V, af_o, n_obs_o = og.score_statistics([g.csr("A")], g["cov"], fit, G)
    assert rel_err(out["score"][fin], U[fin]) < 1e-9
    assert rel_err(out["se"][fin], 1 / np.sqrt(V[fin])) < 1e-9
    assert rel_err(out["beta"][fin], U[fin] / V[fin]) < 1e-9
    assert np.array_equal(out["n_obs"], n_obs_o) and np.array_equal(out["af"], af_o, equal_nan=True)


def test_phase1_memory_order_and_block_width(golden_c1, slmm, c1_fit):
    g = golden_c1
    chol, y, fit = c1_fit
    m = 300
    G = make_genotypes(g.n, m, 32)
    base = slmm.glmm_association(chol, [g.csr("A")], g["cov"], y, fit, G, spa_cutoff=np.inf)
    ses = chol._glmm
    sig = np.concatenate([fit["covariance coefficients"], [1.0]])
    for order in ("C", "F"):
        Go = np.asarray(G, order=order)
        for block in (7, 128, m):
            part = ses.association(sig, Go, block)
            fin = np.isfinite(base["score"])
            assert rel_err(part["score"][fin], base["score"][fin]) < 1e-12
            assert rel_err(part["var"][fin], 1 / base["se"][fin] ** 2) < 1e-12


def test_spa_kernel_matches_oracle_and_is_blocking_independent(golden_c1, slmm, c1_fit):
    g = golden_c1
    chol, y, fit = c1_fit
    mats = [g.csr("A")]
    G = rare_genotypes(g.n, 160, 33)
    out = slmm.glmm_association(chol, mats, g["cov"], y, fit, G, spa_cutoff=1.0)
    ref = og.glmm_association(mats, g["cov"], fit, G, spa_cutoff=1.0)
    assert np.array_equal(out["spa"], ref["spa"])
    applied = out["spa"] == 1
    assert applied.sum() >= 20, out["spa"]
    assert rel_err(out["p"][applied] / ref["p"][applied], np.ones(applied.sum())) < 1e-8
    assert np.array_equal(out["p"][~applied], out["p_normal"][~applied], equal_nan=True)
    # the saddlepoint block: widths 7 / 128 / all, and other cutoffs that change which variants share a block
    ses = chol._glmm
    sig = np.concatenate([fit["covariance coefficients"], [1.0]])
    part = ses.association(sig, G, 512)
    z = part["score"] / np.sqrt(part["var"])
    flag = np.flatnonzero(np.isfinite(z) & (np.abs(np.nan_to_num(z)) > 1.0))
    runs = {}
    for block in (7, 128, flag.size):
        runs[block] = ses.spa(G, flag, part["score"][flag], part["var"][flag], fit["mu"], fit["weights"], block)
    for block in (7, 128):
        for a, b in zip(runs[block], runs[flag.size]):
            assert np.array_equal(a, b, equal_nan=True)
    done = runs[7][1] == 1
    assert np.array_equal(runs[7][1], out["spa"][flag]) and np.array_equal(runs[7][0][done], out["p"][flag][done])
    for cutoff in (0.5, 1.5):
        other = slmm.glmm_association(chol, mats, g["cov"], y, fit, G, spa_cutoff=cutoff)
        both = (other["spa"] != 0) & (out["spa"] != 0)
        assert both.any()
        assert np.array_equal(other["p"][both], out["p"][both], equal_nan=True)
        assert np.array_equal(other["spa"][both], out["spa"][both])


def test_planted_effect_is_recovered(golden_c1, slmm):
    g = golden_c1
    G = make_genotypes(g.n, 20, 34)
    j, gamma = 0, 0.5
    rng = np.random.default_rng(35)
    ys = (g["y"] - g["y"].mean()) / g["y"].std()
    eta = -1.0 + gamma * (G[:, j] - G[:, j].mean()) + 0.7 * ys + g["cov"][:, 0] * 0.3
    y = (rng.random(g.n) < 1 / (1 + np.exp(-eta))).astype(np.float64)
    chol = slmm.SparseCholesky()
    np.random.seed(3)
    fit = slmm.glmm(chol, [g.csr("A")], g["cov"], y, sim_num=50)
    out = slmm.glmm_association(chol, [g.csr("A")], g["cov"], y, fit, G)
    assert abs(out["beta"][j] - gamma) < 4 * out["se"][j], (out["beta"][j], gamma, out["se"][j])
    assert out["p"][j] < 1e-6 and out["spa"][j] != 0


def test_rebuilt_session_errors_and_memory(golden_small, slmm):
    """A fit from another functor is scanned without a refit and gives the same result; invalid genotypes raise
    SlmmError in both phases and the session survives; y outside {0, 1} is refused by the working-vector kernel; repeated
    fits and scans hold no more device memory."""
    import torch
    from scilmm_b200 import engine
    g = golden_small
    y = binary(g, 0.2)
    mats = [g.csr("A")]
    G = rare_genotypes(g.n, 40, 36)
    chol = slmm.SparseCholesky()
    np.random.seed(2)
    fit = slmm.glmm(chol, mats, g["cov"], y, sim_num=16)
    first = slmm.glmm_association(chol, mats, g["cov"], y, fit, G, spa_cutoff=1.0)
    other = slmm.SparseCholesky()
    again = slmm.glmm_association(other, mats, g["cov"], y, fit, G, spa_cutoff=1.0)
    assert other._glmm is not None and other._sessions == {}
    assert np.array_equal(first["spa"], again["spa"]) and np.array_equal(first["n_obs"], again["n_obs"])
    for k in ("beta", "se", "score", "p", "p_normal"):
        fin = np.isfinite(first[k])
        assert np.array_equal(fin, np.isfinite(again[k])) and rel_err(again[k][fin], first[k][fin]) < 1e-12, k
    bad = np.array(G, order="F")
    bad[10, 5] = 3
    with pytest.raises(slmm.SlmmError):
        slmm.glmm_association(chol, mats, g["cov"], y, fit, bad)
    ses = chol._glmm
    flag = np.flatnonzero(first["spa"] != 0)
    with pytest.raises(slmm.SlmmError):
        ses.spa(bad, np.array([5]), first["score"][:1], 1 / first["se"][:1] ** 2, fit["mu"], fit["weights"], 4)
    res = slmm.glmm_association(chol, mats, g["cov"], y, fit, G, spa_cutoff=1.0)
    for k in slmm.GLMM_ASSOC_KEYS:
        assert np.array_equal(res[k], first[k], equal_nan=True), k
    assert flag.size > 0
    n = g.n
    f64 = dict(dtype=torch.float64, device="cuda")
    with pytest.raises(slmm.SlmmError):
        engine.glmm_working(torch.zeros(n, **f64), torch.zeros(n, **f64), torch.ones(n, **f64),
                            torch.full((n,), 2.0, **f64), torch.empty(n, **f64), torch.empty(n, **f64))

    def cycle():
        np.random.seed(2)
        f = slmm.glmm(chol, mats, g["cov"], y, sim_num=16)
        slmm.glmm_association(chol, mats, g["cov"], y, f, G, spa_cutoff=1.0)
        torch.cuda.synchronize()

    def free():
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]

    cycle()
    base = free()
    for _ in range(3):
        cycle()
        assert base - free() <= 32 << 20


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_rank_fit_and_scan(backend):
    """Two ranks: probe columns of the fit and the variants of both scan phases split over the ranks; both equal the
    single-GPU results to 1e-12.  nccl needs two GPUs; gloo runs both ranks on one."""
    import torch
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", SLMM_TWO_RANK_BACKEND=backend)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29591", os.path.join(ROOT, "tests", "nccl_two_rank_glmm.py")]
    out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "TWO_RANK_GLMM_OK" in out.stdout, out.stdout[-4000:]
