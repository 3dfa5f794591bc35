"""Region tests on the GPU (region_test() / RemlSession.region_test / slmm_assoc_region_gram): the region Gram kernel
against numpy and its bitwise rules, parity with the CPU oracle on the golden cases, one-variant regions against the
association scan, independence of the memory order and block width, session reuse and the device-side genotype check,
a planted rare-variant region, and the sharded call over two ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import region as oreg
from tests.test_association_cpu import make_genotypes, with_variant_covariate
from tests.util import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLOAT_KEYS = ("burden_beta", "burden_se", "burden_chi2", "burden_p", "skat_q", "skat_p")
# column 0 (in the span of C when it is added as a covariate), columns 1-2 (monomorphic), then regions of 1-100
SIZES = [1, 2, 1, 5, 17, 40, 100, 2, 64, 30, 37, 9]
BOUNDS = np.concatenate([[0], np.cumsum(SIZES)])


@pytest.fixture(scope="module")
def slmm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import scilmm_b200.SparseCholesky  # noqa: F401
    return sys.modules["scilmm_b200.SparseCholesky"]


def assert_same(a, b, tol, ptol=None):
    assert np.array_equal(a["n_variants"], b["n_variants"]) and np.array_equal(a["n_poly"], b["n_poly"])
    for k in FLOAT_KEYS:
        fin = np.isfinite(b[k])
        assert np.array_equal(np.isfinite(a[k]), fin), k
        t = ptol if (ptol is not None and k.endswith("_p")) else tol
        assert rel_err(a[k][fin], b[k][fin]) <= t, (k, rel_err(a[k][fin], b[k][fin]))


# ------------------------------------------------------------------------------------------------ the Gram kernel
def gram(torch, E, F, bounds):
    out = torch.empty(int(np.sum(np.diff(bounds) ** 2)), dtype=torch.float64, device="cuda")
    E.assoc_region_gram(F, bounds, out)
    res, off = [], 0
    for w in np.diff(bounds):
        res.append(out[off:off + w * w].view(w, w).cpu().numpy())
        off += w * w
    return res


def test_region_gram_kernel(slmm):
    import torch
    from scilmm_b200 import engine as E
    n = 5001                                     # not a multiple of the row chunk
    rng = np.random.default_rng(41)
    widths = [1, 7, 63, 64, 65, 130, 512]
    bounds = np.concatenate([[0], np.cumsum(widths)])
    Fh = rng.standard_normal((n, bounds[-1]))
    F = torch.from_numpy(Fh).cuda()
    squares = gram(torch, E, F, bounds)
    ss = torch.empty(bounds[-1], dtype=torch.float64, device="cuda")
    diag = E.assoc_colsumsq(F, ss).cpu().numpy()
    for r, S in enumerate(squares):
        cols = Fh[:, bounds[r]:bounds[r + 1]]
        ref = cols.T @ cols
        scale = np.sqrt(np.outer(np.diag(ref), np.diag(ref)))
        assert np.max(np.abs(S - ref) / scale) <= 1e-13, widths[r]
        assert np.array_equal(S, S.T)
        d = diag[bounds[r]:bounds[r + 1]]
        assert np.max(np.abs(np.diag(S) - d) / d) <= 1e-14
    # the same columns at other offsets, alone or packed with other regions, in blocks of odd width: the same bits
    for r in range(len(widths)):
        cols = Fh[:, bounds[r]:bounds[r + 1]]
        for lead in (0, 3, 61):
            tail = 5
            G2 = np.hstack([rng.standard_normal((n, lead)), cols, rng.standard_normal((n, tail))])
            b2 = [0] + ([lead] if lead else []) + [lead + cols.shape[1], G2.shape[1]]
            got = gram(torch, E, torch.from_numpy(G2).cuda(), np.array(b2))
            assert np.array_equal(got[1 if lead else 0], squares[r]), (widths[r], lead)
    out = torch.empty(1 << 20, dtype=torch.float64, device="cuda")
    for b, bad in ((10, [0, 5, 5, 10]), (10, [0, 6, 4, 10]), (10, [0, 5, 9]), (10, [1, 5, 10]), (520, [0, 513, 520])):
        with pytest.raises(slmm.SlmmError):
            E.assoc_region_gram(torch.zeros(n, b, dtype=torch.float64, device="cuda"), np.array(bad), out)


# ------------------------------------------------------------------------------------------------ statistics
@pytest.mark.parametrize("case", ["small", "c1"])
@pytest.mark.parametrize("tag", ["k2", "k4"])
def test_region_test_matches_oracle(golden_small, golden_c1, slmm, case, tag):
    g = golden_small if case == "small" else golden_c1
    m = int(BOUNDS[-1])
    G = make_genotypes(g.n, m, 42)
    cov = with_variant_covariate(g["cov"], G, 0)
    mats, sig = g.mats(tag)[:-1], g["sig_" + tag]
    chol = slmm.SparseCholesky()
    for weights in (None, np.random.default_rng(7).uniform(0.0, 4.0, m)):
        out = slmm.region_test(chol, mats, cov, g["y"], sig, G, BOUNDS, weights)
        ref = oreg.region_test(mats, cov, g["y"], sig, G, BOUNDS, weights)
        assert set(out) == set(ref) and all(out[k].shape == (BOUNDS.size - 1,) for k in out)
        assert np.isnan(out["burden_p"][0]) and np.isnan(out["burden_p"][1]) and np.isnan(out["skat_p"][1])
        assert out["n_poly"][1] == 0 and np.all(np.isfinite(out["burden_p"][2:]))
        assert_same(out, ref, 1e-9, 1e-8)


def test_one_variant_regions_match_the_scan(golden_c1, slmm):
    g = golden_c1
    G = make_genotypes(g.n, 300, 43)
    cov = with_variant_covariate(g["cov"], G, 0)
    mats, sig = g.mats("k4")[:-1], g["sig_k4"]
    chol = slmm.SparseCholesky()
    reg = slmm.region_test(chol, mats, cov, g["y"], sig, G, np.arange(301), np.ones(300))
    scan = slmm.association(chol, mats, cov, g["y"], sig, G)
    fin = np.isfinite(scan["chi2"])
    assert np.array_equal(np.flatnonzero(~fin), [0, 1, 2])
    for k, s in (("burden_chi2", "chi2"), ("burden_p", "p"), ("skat_p", "p"), ("burden_beta", "beta"),
                 ("burden_se", "se")):
        assert np.array_equal(np.isfinite(reg[k]), fin), k
        assert rel_err(reg[k][fin], scan[s][fin]) <= 1e-9, (k, rel_err(reg[k][fin], scan[s][fin]))


def test_memory_order_and_block_width(golden_c1, slmm):
    g = golden_c1
    sizes = np.random.default_rng(44).integers(1, 65, 40)
    bounds = np.concatenate([[0], np.cumsum(sizes)])
    G = make_genotypes(g.n, int(bounds[-1]), 45)
    ys = g["y"] / g["y"].std()
    ses = slmm.SparseCholesky()._session(g.mats("k4"), g["cov"], ys)
    base = ses.region_test(g["sig_k4"], G, bounds, None, 512)
    for order in ("C", "F"):
        Go = np.asarray(G, order=order)
        for block in (64, 128, 512):
            assert_same(ses.region_test(g["sig_k4"], Go, bounds, None, block), base, 1e-12)
    part = ses.region_test(g["sig_k4"], np.asfortranarray(G), bounds, None, 128, 7, 31)
    assert_same(part, {k: v[7:31] for k, v in base.items()}, 1e-12)


def test_session_reuse_and_invalid_genotype(golden_small, slmm):
    g = golden_small
    chol, mats, cov = slmm.SparseCholesky(), g.mats("k3"), g["cov"]
    np.random.seed(5)
    fit = slmm.REML(chol, mats, cov, g["y"].copy(), sim_num=16, aireml=True)
    ses = next(iter(chol._sessions.values()))
    sig = fit["covariance coefficients"]
    G = make_genotypes(g.n, 60, 46)
    bounds = np.array([0, 3, 10, 25, 60])
    good = slmm.region_test(chol, mats, cov, g["y"], sig, G, bounds)
    assert len(chol._sessions) == 1 and next(iter(chol._sessions.values())) is ses
    assert_same(good, oreg.region_test(mats, cov, g["y"], sig, G, bounds), 1e-9, 1e-8)
    for order in ("C", "F"):
        bad = np.array(G, order=order)
        bad[100, 17] = 3
        with pytest.raises(slmm.SlmmError):
            slmm.region_test(chol, mats, cov, g["y"], sig, bad, bounds)
    assert_same(slmm.region_test(chol, mats, cov, g["y"], sig, G, bounds), good, 0.0)


def test_planted_rare_variant_region(golden_c1, slmm):
    g = golden_c1
    rng = np.random.default_rng(47)
    G = make_genotypes(g.n, 200, 48)
    hit = slice(80, 88)                          # one region of 8 rare variants, af 0.5-2 %, with one common effect
    af = rng.uniform(0.005, 0.02, 8)
    G[:, hit] = rng.binomial(2, af[None, :], size=(g.n, 8)).astype(np.int8)
    y2 = g["y"] + 0.5 * g["y"].std() * G[:, hit].sum(axis=1)
    bounds = np.arange(0, 201, 8)
    out = slmm.region_test(slmm.SparseCholesky(), g.mats("k2")[:-1], g["cov"], y2, g["sig_k2"], G, bounds)
    r = 80 // 8
    assert out["burden_p"][r] < 1e-6, out["burden_p"][r]
    assert out["burden_p"][r] == np.nanmin(out["burden_p"])


@pytest.mark.parametrize("backend", ["nccl", "gloo"])
def test_two_rank_region_test(backend):
    """Two ranks each test half of the regions and one all-reduce gives both the single-GPU arrays to 1e-12.  nccl
    needs two GPUs; gloo runs both ranks on one."""
    import torch
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", SLMM_TWO_RANK_BACKEND=backend)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29585", os.path.join(ROOT, "tests", "nccl_two_rank_region.py")]
    out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "TWO_RANK_REGION_OK" in out.stdout, out.stdout[-4000:]
