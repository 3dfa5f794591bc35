"""Predicted random effects on the GPU (blup() / RemlSession.blup / slmm_blup_*): against the CPU oracle on the golden
cases with and without unphenotyped individuals, the identity sum_k u_k + e = y - C beta, the column-mapped product
against scipy, reuse of the REML session, bitwise repeatability, the stochastic PEV against the oracle's estimate on
the same probes and against the exact PEV, the refused inputs, device memory, and the PEV over two ranks."""
import gc
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import blup as ob
from tests.test_blup_cpu import MASKS, masked_y
from tests.util import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("u", "residual", "fixed", "yhat", "beta")


@pytest.fixture(scope="module")
def slmm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import scilmm_b200.SparseCholesky  # noqa: F401
    return sys.modules["scilmm_b200.SparseCholesky"]


def assert_close(a, b, tol, keys=KEYS):
    for k in keys:
        assert a[k].shape == b[k].shape, k
        fin = np.isfinite(b[k])
        assert np.array_equal(np.isfinite(a[k]), fin), k
        assert rel_err(a[k][fin], b[k][fin]) <= tol, (k, rel_err(a[k][fin], b[k][fin]))


@pytest.mark.parametrize("case", ["small", "c1"])
@pytest.mark.parametrize("tag", ["k2", "k4"])
@pytest.mark.parametrize("mask", MASKS)
def test_blup_matches_oracle(golden_small, golden_c1, slmm, case, tag, mask):
    g = golden_small if case == "small" else golden_c1
    mats, sig = g.mats(tag)[:-1], g["sig_" + tag]
    y = masked_y(g["y"], g["cov"].shape[1], mask)
    out = slmm.blup(slmm.SparseCholesky(), mats, g["cov"], y, sig)
    ref = ob.blup_vform(mats, g["cov"], y, sig, exact_pev=False)
    assert set(out) == set(KEYS)
    assert_close(out, ref, 1e-10)
    assert np.array_equal(np.isnan(out["residual"]), np.isnan(y))
    assert not np.any(np.isnan(out["u"])) and not np.any(np.isnan(out["yhat"]))
    obs = ~np.isnan(y)
    # sum_k u_k + e = s V u = s (y_s - C beta) on the phenotyped rows
    lhs = out["u"][obs].sum(axis=1) + out["residual"][obs]
    assert rel_err(lhs, y[obs] - out["fixed"][obs]) <= 1e-12


@pytest.mark.parametrize("mask", ["none", "random"])
def test_identity_component_is_predicted_like_any_other(golden_c1, slmm, mask):
    """An identity among `mats` (an extra i.i.d. effect) shares its pattern with the residual identity REML() appends,
    so the in-sample session groups the two; blup() predicts the user's one like any other column."""
    import scipy.sparse as sp
    g = golden_c1
    mats, sig = [g.mats("k2")[0], sp.eye(g.n).tocsr()], np.array([0.35, 0.15, 0.5])
    y = masked_y(g["y"], 3, mask)
    chol = slmm.SparseCholesky()
    out = slmm.blup(chol, mats, g["cov"], y, sig, pev_probes=128)
    if mask == "none":
        ses = next(iter(chol._sessions.values()))
        assert [1, 2] in ses._groups
    ref = ob.blup_vform(mats, g["cov"], y, sig)
    assert_close(out, ref, 1e-10)
    obs = ~np.isnan(y)
    assert np.all(out["u"][~obs, 1] == 0.0)
    assert rel_err(out["u"][obs, 1], out["residual"][obs] * sig[1] / sig[2]) <= 1e-12
    ok = out["pev_se"] > 0
    assert np.median(np.abs(out["pev"] - ref["pev"])[ok] / out["pev_se"][ok]) < 1.5


def test_masked_equals_in_sample_on_the_cut_blocks(golden_c1, slmm):
    g = golden_c1
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    y = masked_y(g["y"], 3, "random")
    obs = ~np.isnan(y)
    idx = np.flatnonzero(obs)
    chol = slmm.SparseCholesky()
    masked = slmm.blup(chol, mats, g["cov"], y, sig)
    inner = slmm.blup(chol, [m[idx][:, idx] for m in mats], g["cov"][idx], y[idx], sig)
    for k in KEYS:
        a = masked[k] if k == "beta" else masked[k][obs]
        assert rel_err(a, inner[k]) <= 1e-12, k


def test_identity_map_equals_the_session_matset(golden_c1, slmm):
    """The masked path (matrices of their own, a column map) with nothing masked gives the unmasked path's bits."""
    from scilmm_b200 import engine as E
    g = golden_c1
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    chol = slmm.SparseCholesky()
    ys = g["y"] / g["y"].std()
    ses = slmm._scan_session(chol, mats, g["cov"], ys)
    own = [[k for k in ks if k < 3] for ks in ses._groups]
    own = [ks for ks in own if ks]
    a = ses.blup(sig, ses.matset, own, None, 256)
    ms = E.MatSet(mats)
    assert ms.pattern_groups(2) == own
    b = ses.blup(sig, ms, own, np.arange(g.n, dtype=np.int32), 256)
    for k in ("U", "corr"):
        assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy()), k
    for pa, pb in zip(a["parts"], b["parts"]):
        assert np.array_equal(pa.cpu().numpy(), pb.cpu().numpy())
    full = slmm.blup(chol, mats, g["cov"], g["y"], sig)
    assert np.array_equal(full["u"], a["U"].cpu().numpy() * g["y"].std())


@pytest.mark.parametrize("ncols", [1, 7, 12, 32])
@pytest.mark.parametrize("G", [1, 2])
def test_blup_spmm_against_scipy(golden_c1, slmm, ncols, G):
    import torch
    from scilmm_b200 import engine as E
    g = golden_c1
    A, Ep, H = g.mats("k3")
    ms = E.MatSet([A, Ep, H])
    ks = [0, 1][:G]
    assert ms.pattern_id(1) == ms.pattern_id(0)
    sig = [0.7, -1.3][:G]
    rng = np.random.default_rng(ncols)
    obs = rng.random(g.n) < 0.8
    idx = np.flatnonzero(obs)
    colmap = np.full(g.n, -1, dtype=np.int32)
    colmap[idx] = np.arange(idx.size)
    X = rng.standard_normal((idx.size, ncols))
    Y = ms.blup_spmm(ks, sig, torch.from_numpy(X).cuda(), colmap).cpu().numpy()
    for gi, k in enumerate(ks):
        ref = sig[gi] * (g.mats("k3")[k][:, idx] @ X)
        assert rel_err(Y[gi], ref) <= 1e-13
    # the identity map (NULL) over all rows
    Xf = rng.standard_normal((g.n, ncols))
    Yf = ms.blup_spmm(ks, sig, torch.from_numpy(Xf).cuda()).cpu().numpy()
    for gi, k in enumerate(ks):
        assert rel_err(Yf[gi], sig[gi] * (g.mats("k3")[k] @ Xf)) <= 1e-13


def test_map_skips_and_empty_rows(golden_c1, slmm):
    """Households (H) whose members all lack a phenotype have no observed neighbour: their rows come out exactly 0,
    in the product and in the probe sums; a map that is all -1 gives zeros everywhere."""
    import torch
    from scilmm_b200 import engine as E
    g = golden_c1
    H = g.mats("k3")[2]
    ms = E.MatSet([H])
    rng = np.random.default_rng(1)
    obs = rng.random(g.n) < 0.5
    idx = np.flatnonzero(obs)
    colmap = np.full(g.n, -1, dtype=np.int32)
    colmap[idx] = np.arange(idx.size)
    empty = np.asarray(H[:, idx].getnnz(axis=1) == 0).ravel()
    assert empty.sum() > 10
    X = torch.from_numpy(rng.standard_normal((idx.size, 3))).cuda()
    Y = ms.blup_spmm([0], [1.0], X, colmap).cpu().numpy()[0]
    assert np.all(Y[empty] == 0.0) and np.all(np.any(Y[~empty] != 0.0, axis=1))
    W = torch.from_numpy(rng.standard_normal((idx.size, 128))).cuda()
    s2 = torch.empty(g.n, 1, dtype=torch.float64, device="cuda")
    s4 = torch.empty_like(s2)
    ms.blup_rowsumsq([0], [1.0], W, s2, s4, colmap)
    t = H[:, idx] @ W.cpu().numpy()
    assert rel_err(s2.cpu().numpy()[:, 0], np.sum(t * t, axis=1)) <= 1e-13
    assert rel_err(s4.cpu().numpy()[:, 0], np.sum(t ** 4, axis=1)) <= 1e-13
    assert np.all(s2.cpu().numpy()[empty] == 0.0)
    Z = ms.blup_spmm([0], [1.0], X[:1], np.full(g.n, -1, dtype=np.int32)).cpu().numpy()
    assert np.all(Z == 0.0)
    # map entries are checked on the device, whether the map comes from the host or is already there
    past = np.where(obs, 0, idx.size).astype(np.int32)             # an entry past the rows of X
    below = colmap.copy()
    below[7] = -2
    for bad in (past, below, torch.from_numpy(past).cuda()):
        with pytest.raises(slmm.SlmmError):
            ms.blup_spmm([0], [1.0], X, bad)
        with pytest.raises(slmm.SlmmError):
            ms.blup_rowsumsq([0], [1.0], W, s2, s4, bad)
    with pytest.raises(slmm.SlmmError):
        ms.blup_spmm([0], [1.0], X)                   # no map needs X over all n rows
    with pytest.raises(ValueError):
        ms.blup_spmm([0], [1.0], X, colmap[:-1])      # a map has n entries


def test_blup_after_reml_reuses_the_session(golden_small, slmm):
    g = golden_small
    chol, mats, cov = slmm.SparseCholesky(), g.mats("k3"), g["cov"]
    np.random.seed(5)
    fit = slmm.REML(chol, mats, cov, g["y"].copy(), sim_num=16, aireml=True)
    ses = next(iter(chol._sessions.values()))
    out = slmm.blup(chol, mats, cov, g["y"], fit["covariance coefficients"], pev_probes=128)
    assert len(chol._sessions) == 1 and next(iter(chol._sessions.values())) is ses
    ref = ob.blup_vform(mats, cov, g["y"], fit["covariance coefficients"], exact_pev=False)
    assert_close(out, ref, 1e-10)
    assert np.allclose(out["beta"], fit["covariates coefficients"] * g["y"].std(), rtol=1e-12, atol=0)


def test_repeatable_bit_for_bit(golden_c1, slmm):
    g = golden_c1
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    y = masked_y(g["y"], 3, "random")
    a = slmm.blup(slmm.SparseCholesky(seed=3), mats, g["cov"], y, sig, pev_probes=200)
    b = slmm.blup(slmm.SparseCholesky(seed=3), mats, g["cov"], y, sig, pev_probes=200)
    assert set(a) == set(KEYS) | {"pev", "pev_se", "reliability"}
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    c = slmm.blup(slmm.SparseCholesky(seed=4), mats, g["cov"], y, sig, pev_probes=200)
    assert np.array_equal(a["u"], c["u"]) and not np.array_equal(a["pev"], c["pev"])


@pytest.mark.parametrize("probes", [128, 256])
@pytest.mark.parametrize("setup", ["natural", "perm"])
def test_pev_matches_the_same_probe_oracle(golden_c1mini, slmm, probes, setup):
    """Same Philox block, same permutation: the engine's estimate is the oracle's to 1e-10, whatever rng says."""
    g = golden_c1mini
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    if setup == "natural":
        y = g["y"]
        chol = slmm.SparseCholesky(ordering_method="natural", rng="numpy", seed=11)
        perm = np.arange(g.n)
    else:
        y = masked_y(g["y"], 3, "random")
        n = int(np.sum(~np.isnan(y)))
        perm = np.random.default_rng(2).permutation(n).astype(np.int32)
        chol = slmm.SparseCholesky(perm=perm, rng="device", seed=11)
    out = slmm.blup(chol, mats, g["cov"], y, sig, pev_probes=probes)
    assert np.array_equal(next(iter(chol._sessions.values())).eng.perm(), perm)
    pev, se = ob.pev_stochastic(mats, g["cov"], y, sig, probes, 11, perm)
    assert rel_err(out["pev"], pev) <= 1e-10
    assert rel_err(out["pev_se"], se) <= 1e-10
    exact = ob.blup_vform(mats, g["cov"], y, sig)
    ok = se > 0
    assert np.median(np.abs(out["pev"] - exact["pev"])[ok] / se[ok]) < 1.5
    prior = out["pev"] / (1.0 - out["reliability"])
    assert rel_err(prior, exact["pev"] / (1.0 - exact["reliability"])) <= 1e-10


def test_pev_statistics_against_the_exact_pev(golden_c1, slmm):
    """1024 probes on c1 (7 108 individuals, three components): z = (est - exact) / pev_se exceeds 4 in fewer than
    0.5 % of the entries and averages to within 0.1 of 0.  Fixed seed: the outcome does not vary between runs."""
    g = golden_c1
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    out = slmm.blup(slmm.SparseCholesky(seed=0), mats, g["cov"], g["y"], sig, pev_probes=1024)
    exact = ob.blup_vform(mats, g["cov"], g["y"], sig)["pev"]
    ok = out["pev_se"] > 0
    z = (out["pev"] - exact)[ok] / out["pev_se"][ok]
    assert ok.mean() > 0.99
    assert np.mean(np.abs(z) > 4) < 0.005, np.mean(np.abs(z) > 4)
    assert abs(np.mean(z)) < 0.1, np.mean(z)


def test_refused_inputs(golden_small, slmm):
    g = golden_small
    chol = slmm.SparseCholesky()
    mats, sig, cov, y = g.mats("k3"), g["sig_k4"], g["cov"], g["y"]
    with pytest.raises(ValueError):
        slmm.blup(chol, mats, cov, y, sig[:-1])
    with pytest.raises(ValueError):
        slmm.blup(chol, mats, cov, y[1:], sig)
    with pytest.raises(ValueError):
        slmm.blup(chol, [mats[0], mats[1][:, 1:], mats[2]], cov, y, sig)
    with pytest.raises(ValueError):
        slmm.blup(chol, [mats[0][1:, 1:]] + mats[1:], cov, y, sig)
    with pytest.raises(ValueError):
        slmm.blup(chol, mats, cov, np.full(g.n, np.nan), sig)
    few = np.full(g.n, np.nan)
    few[:3] = y[:3]                                   # c = 3 covariates need 4 phenotypes
    with pytest.raises(ValueError):
        slmm.blup(chol, mats, cov, few, sig)
    bad = cov.copy()
    bad[5, 1] = np.nan
    with pytest.raises(ValueError):
        slmm.blup(chol, mats, bad, y, sig)
    wide = np.hstack([cov, np.random.default_rng(0).standard_normal((g.n, 29))])
    with pytest.raises(ValueError):
        slmm.blup(chol, mats, wide, y, sig)
    with pytest.raises(ValueError):
        slmm.blup(chol, mats, cov, y, sig, pev_probes=1)
    with pytest.raises(TypeError):
        slmm.blup(None, mats, cov, y, sig)
    out = slmm.blup(chol, mats, wide[:, :31], y, sig)
    assert_close(out, ob.blup_vform(mats, wide[:, :31], y, sig, exact_pev=False), 1e-9)


def test_masked_calls_with_pev_return_device_memory(golden_c1, slmm):
    """Three masked calls with PEV (a MatSet over all individuals, a session on the cut blocks, probe blocks and
    partial sums) give free device memory back to the baseline once their functors are gone."""
    import torch

    def free():
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]

    g = golden_c1
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    y = masked_y(g["y"], 3, "random")
    slmm.blup(slmm.SparseCholesky(), mats, g["cov"], y, sig, pev_probes=256)      # first-call work
    base = free()
    for _ in range(3):
        slmm.blup(slmm.SparseCholesky(), mats, g["cov"], y, sig, pev_probes=256)
        assert free() >= base - (32 << 20)


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_rank_pev(backend):
    """Two ranks each sweep half of the probe blocks: pev and pev_se are bit-identical to one rank, u equal.  nccl
    needs two GPUs; gloo runs both ranks on one."""
    import torch
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", SLMM_TWO_RANK_BACKEND=backend)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29583", os.path.join(ROOT, "tests", "nccl_two_rank_blup.py")]
    out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "TWO_RANK_BLUP_OK" in out.stdout, out.stdout[-4000:]
