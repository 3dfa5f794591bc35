"""Association scan on the GPU (association() / RemlSession.association): against the CPU oracle on the golden cases,
independence of the memory order and block width, the device-side genotype check, reuse of the REML session, a
planted effect, and the sharded scan over two ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import association as oa
from tests.test_association_cpu import make_genotypes, with_variant_covariate
from tests.util import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("beta", "se", "chi2", "p", "af", "n_obs")


@pytest.fixture(scope="module")
def slmm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import scilmm_b200.SparseCholesky  # noqa: F401
    return sys.modules["scilmm_b200.SparseCholesky"]


def assert_same(a, b, tol):
    for k in ("beta", "se", "chi2"):
        fin = np.isfinite(b[k])
        assert np.array_equal(np.isfinite(a[k]), fin), k
        assert rel_err(a[k][fin], b[k][fin]) <= tol, (k, rel_err(a[k][fin], b[k][fin]))
    assert np.array_equal(np.isfinite(a["p"]), np.isfinite(b["p"]))
    assert np.array_equal(a["n_obs"], b["n_obs"])
    assert np.array_equal(a["af"], b["af"], equal_nan=True)


@pytest.mark.parametrize("case", ["small", "c1"])
@pytest.mark.parametrize("tag", ["k2", "k4"])
def test_scan_matches_oracle(golden_small, golden_c1, slmm, case, tag):
    g = golden_small if case == "small" else golden_c1
    G = make_genotypes(g.n, 70, 11)
    cov = with_variant_covariate(g["cov"], G, 0)
    mats, sig = g.mats(tag)[:-1], g["sig_" + tag]
    out = slmm.association(slmm.SparseCholesky(), mats, cov, g["y"], sig, G)
    ref = oa.association(mats, cov, g["y"], sig, G)
    assert set(out) == set(KEYS) and all(out[k].shape == (70,) for k in KEYS)
    assert np.array_equal(np.flatnonzero(~np.isfinite(out["beta"])), [0, 1, 2])
    assert_same(out, ref, 1e-9)
    fin = np.isfinite(ref["p"])
    assert np.allclose(out["p"][fin], ref["p"][fin], rtol=1e-8, atol=1e-300)


def test_memory_order_and_block_width(golden_c1, slmm):
    g = golden_c1
    m = 620                                     # a whole-width Fortran block is 4.4 MB: the staged ring upload
    G = make_genotypes(g.n, m, 12)
    cov = with_variant_covariate(g["cov"], G, 0)
    ys = g["y"] / g["y"].std()
    ses = slmm.SparseCholesky()._session(g.mats("k4"), cov, ys)
    base = ses.association(g["sig_k4"], G, m)
    for order in ("C", "F"):
        Go = np.asarray(G, order=order)
        for block in (7, 128, m):
            assert_same(ses.association(g["sig_k4"], Go, block), base, 1e-12)
    part = ses.association(g["sig_k4"], np.asfortranarray(G), 64, 45, 250)
    assert_same(part, {k: v[45:250] for k, v in base.items()}, 1e-12)


def test_invalid_entry_raises_and_session_survives(golden_small, slmm):
    g = golden_small
    G = make_genotypes(g.n, 20, 13)
    chol = slmm.SparseCholesky()
    mats, sig = g.mats("k3"), g["sig_k4"]
    good = slmm.association(chol, mats, g["cov"], g["y"], sig, G)
    for order in ("C", "F"):
        bad = np.array(G, order=order)
        bad[100, 17] = 3
        with pytest.raises(slmm.SlmmError):
            slmm.association(chol, mats, g["cov"], g["y"], sig, bad)
    assert_same(slmm.association(chol, mats, g["cov"], g["y"], sig, G), good, 0.0)
    with pytest.raises(ValueError):
        slmm.association(chol, mats, g["cov"], g["y"], sig, G.astype(np.int16))
    with pytest.raises(ValueError):
        slmm.association(chol, mats, g["cov"], g["y"], sig, G[1:])
    with pytest.raises(ValueError):
        slmm.association(chol, mats, g["cov"], g["y"], sig[:-1], G)
    with pytest.raises(TypeError):
        slmm.association(None, mats, g["cov"], g["y"], sig, G)
    wide = np.hstack([g["cov"], np.random.default_rng(0).standard_normal((g.n, 29))])
    with pytest.raises(ValueError):
        slmm.association(chol, mats, wide, g["y"], sig, G)
    assert_same(slmm.association(chol, mats, wide[:, :31], g["y"], sig, G),
                oa.association(mats, wide[:, :31], g["y"], sig, G), 1e-9)


def test_association_after_reml_reuses_the_session(golden_small, slmm):
    g = golden_small
    chol, mats, cov = slmm.SparseCholesky(), g.mats("k3"), g["cov"]
    np.random.seed(5)
    fit = slmm.REML(chol, mats, cov, g["y"].copy(), sim_num=16, aireml=True)
    ses = next(iter(chol._sessions.values()))
    G = make_genotypes(g.n, 10, 14)
    out = slmm.association(chol, mats, cov, g["y"], fit["covariance coefficients"], G)
    assert len(chol._sessions) == 1 and next(iter(chol._sessions.values())) is ses
    ref = oa.association(mats, cov, g["y"], fit["covariance coefficients"], G)
    assert_same(out, ref, 1e-9)


def test_planted_effect_is_recovered(golden_c1, slmm):
    g = golden_c1
    G = make_genotypes(g.n, 30, 15)
    j, gamma = 0, 0.25 * g["y"].std()
    y2 = g["y"] + gamma * G[:, j]
    out = slmm.association(slmm.SparseCholesky(), g.mats("k2")[:-1], g["cov"], y2, g["sig_k2"], G)
    assert abs(out["beta"][j] - gamma) < 4 * out["se"][j], (out["beta"][j], gamma, out["se"][j])
    assert out["chi2"][j] > 30


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_rank_scan(backend):
    """Two ranks each scan half of the variants and one all-reduce gives both the single-GPU arrays to 1e-12.  nccl
    needs two GPUs; gloo runs both ranks on one."""
    import torch
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", SLMM_TWO_RANK_BACKEND=backend)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29581", os.path.join(ROOT, "tests", "nccl_two_rank_assoc.py")]
    out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "TWO_RANK_ASSOC_OK" in out.stdout, out.stdout[-4000:]
