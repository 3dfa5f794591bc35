"""Solve mode 3, the backward half-sweep from the factor's row order (P' L^-T Z), and the REML probe block it computes.

The reference draws W = V^-1 (L Z)[argsort P] (SparseCholesky.py:49-52).  With P V P' = L L' and lmul returning
P' L Z, V^-1 P' L Z = P' L^-T L^-1 L Z = P' L^-T Z: one backward half-sweep on Z, without L Z and the forward sweep.
  * mode 3 is mode 2 with only the input gather removed: bit for bit at every front shape of test_gpu_front_shapes
    and at every RHS-width class of the solve schedules (streaming kernels, tiles, look-ahead, > 160 columns);
  * on the c1mini golden set, natural and nesdis ordering: against the old composition solve_(lmul(Z)) and LAPACK's
    P' L^-T Z, and bit-identical across calls;
  * at the 250K config: evaluate() gives the same nll and the same fixed-effect arrays bit for bit as with the old
    composition, and the gradient to rounding."""
import sys

import numpy as np
import pytest
import scipy.linalg as la
import scipy.sparse as sp

from tests.test_gpu_front_shapes import SHAPES, assert_front, front_matrix
from tests.util import rel_err

pytestmark = pytest.mark.gpu

WIDTHS = (1, 2, 4, 8, 12, 16, 32, 33, 64, 128, 161)


@pytest.fixture(scope="module")
def slmm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import scilmm_b200  # noqa: F401
    import scilmm_b200.SparseCholesky  # noqa: F401
    return sys.modules["scilmm_b200.SparseCholesky"]


@pytest.fixture(scope="module")
def eng():
    from scilmm_b200 import engine
    return engine


def backward_ref(V, P, Z):
    """LAPACK: P' L^-T Z with L = chol(V[P][:, P]) and Z in the factor's row order."""
    L = la.cholesky(V[np.ix_(P, P)], lower=True)
    out = np.empty_like(Z)
    out[P] = la.solve_triangular(L.T, Z, lower=False)
    return out


def mode3_against_mode2(dev, eng, P, n, widths, seed):
    """mode 3 on Z equals mode 2 on the block whose row gather gives Z (B[P] = Z), bit for bit.  Returns the
    (width, Z, mode-3 result) triples."""
    out = []
    for k in widths:
        Z = np.random.default_rng(seed + k).standard_normal((n, k))
        B = np.empty_like(Z)
        B[P] = Z
        got = dev.solve_(eng.to_device(Z), 3).cpu().numpy()
        want = dev.solve_(eng.to_device(B), 2).cpu().numpy()
        assert np.array_equal(got, want), ("mode 3 != mode 2 on the gathered block", k)
        out.append((k, Z, got))
    return out


@pytest.mark.parametrize("ns,rs", SHAPES, ids=["ns%d_rs%d" % s for s in SHAPES])
def test_mode3_is_mode2_without_the_gather(ns, rs, slmm, eng):
    V = front_matrix(ns, rs)
    assert_front(eng, V, ns, rs)
    f = slmm.SparseCholesky(ordering_method="natural")(sp.csc_matrix(V))
    P = f.P()
    for k, Z, got in mode3_against_mode2(f._chol, eng, P, V.shape[0], WIDTHS, 1000 * ns + rs):
        if k in (1, 33, 161):
            assert rel_err(got, backward_ref(V, P, Z)) < 1e-10, k


@pytest.mark.parametrize("ordering", ["natural", "nesdis"])
def test_probe_block_on_c1mini(ordering, golden_c1mini, slmm, eng):
    """V^-1 (L Z)[argsort P] by one backward half-sweep: against solve_(lmul(Z)), against LAPACK's P' L^-T Z on the
    permuted dense matrix, bit-identical across calls, and mode 3 against mode 2 on the gathered block."""
    Vs = golden_c1mini.csc("V_k4")
    V = Vs.toarray()
    n = V.shape[0]
    f = slmm.SparseCholesky(ordering_method=ordering)(Vs)
    P = f.P()
    if ordering == "nesdis":
        assert not np.array_equal(P, np.arange(n))
    dev = f._chol
    for k in (1, 16, 33, 128):
        Z = np.random.default_rng(k).standard_normal((n, k))
        Zd = eng.to_device(Z)
        W = dev.solve_(Zd.clone(), 3)
        old = dev.solve_(dev.lmul(Zd)).cpu().numpy()
        Wh = W.cpu().numpy()
        assert rel_err(Wh, old) < 1e-11, k
        assert rel_err(Wh, backward_ref(V, P, Z)) < 1e-11, k
        assert np.array_equal(dev.solve_(Zd.clone(), 3).cpu().numpy(), Wh), k
    mode3_against_mode2(dev, eng, P, n, (2, 128), 7)


def test_caller_probe_block_is_not_overwritten(golden_c1mini, slmm, eng):
    """The probe solve works in place on its own copy: a device block handed to evaluate() (whole or sliced) and a
    host block keep their values, and all three give the same evaluation."""
    import torch
    g = golden_c1mini
    mats, sig = g.mats("k4"), g["sig_k4"]
    ys = g["y"] / g["y"].std()
    ses = slmm.SparseCholesky()._session(mats, g["cov"], ys)
    Zh = np.random.default_rng(4).standard_normal((ses.n, 24))
    Zd = eng.to_device(Zh)
    Zd_before = Zd.clone()
    outs = [ses.evaluate(sig, True, 24, Z=Z) for Z in (Zd, Zh, torch.from_numpy(Zh))]
    assert torch.equal(Zd, Zd_before)
    for nll, grad in outs[1:]:
        assert nll == outs[0][0] and np.array_equal(grad, outs[0][1])
    W = ses.probes(24, Z=Zd, col_begin=5, col_end=17)
    assert torch.equal(Zd, Zd_before)
    old = ses.eng.solve_(ses.eng.lmul(Zd[:, 5:17].contiguous()))
    assert float((W - old).abs().max() / old.abs().max()) < 1e-11


def test_evaluate_at_250k_against_the_old_composition(slmm, eng):
    """250K config, rng='device': evaluate() with the probe block by one backward half-sweep against the same
    evaluation with W = solve_(lmul(Z)) on the same Philox block.  nll and every array of ses.last but W bit for bit,
    W and the gradient to rounding.  A solve mode outside 0-3 is refused."""
    import torch
    import bench
    from scilmm_b200 import pedigree as Ped
    A, _, cov, y, info = bench.make_inputs(250000, 1e-3, 10)
    n = A.shape[0]
    mats = [A, Ped.epistasis(A), sp.eye(n).tocsr()]
    sig = np.array([0.3, 0.15, 0.55])
    ses = slmm.SparseCholesky(rng="device", seed=12345)._session(mats, cov, y / y.std())
    stream = 11
    nll, grad = ses.evaluate(sig, True, 128, probe_stream=stream)
    new = dict(ses.last)

    def old_probes(sim_num, Z=None, col_begin=0, col_end=None, pre=None, probe_stream=None):
        col_end = sim_num if col_end is None else col_end
        Zd = ses.eng.probe_normals(ses.n, col_end - col_begin, col_begin, ses.functor.seed, probe_stream)
        return ses.eng.solve_(ses.eng.lmul(Zd))

    ses.probes = old_probes
    try:
        nll_o, grad_o = ses.evaluate(sig, True, 128, probe_stream=stream)
    finally:
        del ses.probes
    old = ses.last
    assert nll == nll_o
    assert rel_err(grad, grad_o) < 1e-10, (grad, grad_o)
    assert new["logdet"] == old["logdet"]
    assert np.array_equal(new["beta"], old["beta"])
    assert np.array_equal(new["chol"][0], old["chol"][0])
    for k in ("ViC", "Vir", "Viy"):
        assert bool((new[k] == old[k]).all()), k
    Wn, Wo = new["W"], old["W"]
    assert float((Wn - Wo).abs().max() / Wo.abs().max()) < 1e-11
    from scilmm_b200._lib import SlmmError
    for mode in (7, -1):
        B = Wn[:, :4].clone()
        with pytest.raises(SlmmError, match="mode"):
            ses.eng.solve_(B, mode=mode)
        assert torch.equal(B, Wn[:, :4]), mode
