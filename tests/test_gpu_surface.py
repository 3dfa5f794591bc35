"""GPU parity tests, part 2: the public surface round 1 left untested (MINQUE, run_estimates(reml=True),
run_estimates_from_paths, the stand-alone wrappers, slmm_matset_upload / slmm_he_moments_host), the BASELINE
configs at their stated sizes (C1 = 10,000 simulated individuals against the unmodified reference; C2 = 100,000
against a CPU oracle with an INDEPENDENT symbolic analysis), and the behaviours added in round 2 (solve plans per
stream section, CHOLMOD's lower-triangle rule, session fingerprints, counter-based probe stream, row-block shards,
dense / exact / fixed-index HE branches).  Tolerances are the north-star ones."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg as la
import scipy.sparse as sp

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


@pytest.fixture(scope="module")
def eng():
    from scilmm_b200 import engine
    return engine


# ------------------------------------------------------------------------------------------ config 1 at its size
def test_c1_he_factor_and_evaluation_vs_reference(golden_c1, slmm):
    """BASELINE config 1 (simulate_tree(10000, 1e-3, 1.4, 0.8), 7,108 kept) against the UNMODIFIED reference."""
    g = golden_c1
    for tag in ("k1", "k3"):
        est = slmm.HE(g.mats(tag), g["cov"], g["y"].copy())
        assert rel_err(est, g["he_" + tag]) < 1e-9
        est = slmm.HE(g.mats(tag), g["cov"], g["y"].copy(), MQS=True)
        assert rel_err(est, g["he_mqs_" + tag]) < 1e-9
    ys = g["y"] / g["y"].std()
    for tag in ("k2", "k4"):
        V = g.csc("V_" + tag)
        for ordering in ("natural", "nesdis"):
            f = slmm.SparseCholesky(ordering_method=ordering)(V)
            assert abs(f.logdet() - g["logdet_" + tag]) < 1e-10 * abs(g["logdet_" + tag])
            assert rel_err(f(ys), g["Viy_" + tag]) < 1e-10
            assert rel_err(f(g["cov"]), g["ViC_" + tag]) < 1e-10
        mats, sig = g.mats(tag), g["sig_" + tag]
        chol = slmm.SparseCholesky(ordering_method="natural")      # the golden stream was frozen with P = identity
        for reml in (False, True):
            np.random.seed(g.seed + 4)
            nll, grad = slmm.bolt_gradient_estimation(np.log(sig), chol, mats, g["cov"], ys, reml, g.sim_num, False)
            assert abs(nll - g["bolt_nll_%s_%d" % (tag, reml)]) < 1e-10 * abs(nll)
            assert rel_err(grad, g["bolt_grad_%s_%d" % (tag, reml)]) < 1e-8
        fac = chol._session(mats, g["cov"], ys).factor_at(sig)
        assert rel_err(slmm.compute_hess(mats, g["cov"], fac, ys), g["hess_" + tag]) < 1e-9


def test_c1_full_fit_vs_reference_identity_permutation(golden_c1, slmm):
    """Whole REML() fit at config-1 size against the unmodified reference (frozen numpy stream, P = I)."""
    g = golden_c1
    np.random.seed(g.seed + 5)
    out = slmm.REML(slmm.SparseCholesky(ordering_method="natural"), g.mats("k1"), g["cov"], g["y"].copy(),
                    reml=True, sim_num=g.sim_num)
    assert rel_err(out["covariance coefficients"], g["reml_sig_k2"]) < 1e-6
    assert rel_err(out["covariates coefficients"], g["reml_beta_k2"]) < 1e-6
    assert rel_err(out["covariance std"], g["reml_se_k2"]) < 1e-6


@pytest.mark.parametrize("base", ["k1", "k3"])
def test_c1_full_fit_on_the_engines_own_permutation(golden_c1, slmm, base):
    """Final variance components to 1e-6 with the engine's OWN nested-dissection permutation over a whole fit: the
    oracle (pinned to the reference by tests/test_oracle_golden.py) is forced onto the same P and the same Z stream."""
    g = golden_c1
    chol = slmm.SparseCholesky()                                   # default ordering: nested dissection
    np.random.seed(41)
    out = slmm.REML(chol, g.mats(base), g["cov"], g["y"].copy(), reml=True, sim_num=g.sim_num)
    ses = next(iter(chol._sessions.values()))
    P = ses.eng.perm()
    assert not np.array_equal(P, np.arange(g.n))
    np.random.seed(41)
    ref = orc.reml_fit(lambda M: DenseFactor(M, P), g.mats(base), g["cov"], g["y"].copy(), reml=True,
                       sim_num=g.sim_num)
    assert rel_err(out["covariance coefficients"], ref["covariance coefficients"]) < 1e-6
    assert rel_err(out["covariates coefficients"], ref["covariates coefficients"]) < 1e-6
    assert rel_err(out["covariance std"], ref["covariance std"]) < 1e-6


# ------------------------------------------------------------------------------------------ config 2
def test_c2_100k_against_independent_symbolic_oracle(slmm, eng):
    """BASELINE config 2: 100,000 simulated individuals, K = 3 (IBD, A o A, I), 10 covariates.  The CPU checker takes
    ONLY the permutation from the engine; elimination tree, column counts, supernodes and scatter maps come from
    oracle/symbolic_ref.py (no product code), the numerics from LAPACK.  nnz(L) / column counts / logdet / solves /
    nll / gradient of one evaluation must agree."""
    import bench
    from oracle.supernodal_cpu import SupernodalCPUFactor
    from oracle.symbolic_ref import IndependentPlan
    from scilmm_b200 import pedigree as P
    A, _, cov, y, info = bench.make_inputs(100000, 1e-3, 10)
    n = A.shape[0]
    mats = [A, P.epistasis(A), sp.eye(n).tocsr()]
    sig = np.array([0.3, 0.15, 0.55])
    ys = y / y.std()
    chol = slmm.SparseCholesky(rng="numpy")
    sim_num = 16
    np.random.seed(7)
    nll, grad = slmm.bolt_gradient_estimation(np.log(sig), chol, mats, cov, ys, True, sim_num, False)
    ses = chol._session(mats, cov, ys)
    st = ses.eng.stats()
    perm = ses.eng.perm()
    plan = IndependentPlan(ses.union, perm)
    assert plan.sym.nnzL == st["nnzL"] and plan.sym.flops == st["flops"]
    a = eng.SymbolicView(ses.union, perm=perm).arrays()
    assert np.array_equal(plan.colcount, a["colcount"]) and np.array_equal(plan.parent, a["parent"])
    V = orc.weighted_sum(mats, sig)
    ref = SupernodalCPUFactor(V, plan=plan)
    assert abs(ses.last["logdet"] - ref.logdet()) < 1e-10 * abs(ref.logdet())
    B = np.random.default_rng(1).standard_normal((n, 5))
    X = ses.eng.solve_(eng.to_device(B)).cpu().numpy()
    assert rel_err(X, ref(B)) < 1e-10
    np.random.seed(7)
    nll_o, grad_o = orc.reml_evaluation(np.log(sig), lambda M: SupernodalCPUFactor(M, plan=plan), mats, cov, ys,
                                        True, sim_num)
    assert abs(nll - nll_o) < 1e-10 * abs(nll_o)
    assert rel_err(grad, grad_o) < 1e-8


# ------------------------------------------------------------------------------------------ untested surface
@pytest.mark.parametrize("case", ["golden_small", "golden_c1mini"])
def test_minque_vs_reference(case, request, slmm):
    g = request.getfixturevalue(case)
    for tag in ("k1", "k3"):
        np.random.seed(g.seed + 6)
        est = slmm.MINQUE(slmm.SparseCholesky(ordering_method="natural"), g.mats(tag), g["cov"], g["y"].copy(),
                          num_iter=2, sim_num=g.sim_num)
        assert rel_err(est, g["minque_" + tag]) < 1e-7
    est, se = slmm.MINQUE(slmm.SparseCholesky(ordering_method="natural"), g.mats("k1"), g["cov"], g["y"].copy(),
                          compute_stderr=True, num_iter=1)
    assert se == 0.0 and est.shape == (1,)


def test_minque_indefinite_h_raises_like_cholmod(golden_small, slmm):
    """A third MINQUE iteration makes H indefinite on this input (the reference dies in CHOLMOD with
    CholmodNotPositiveDefiniteError): the engine raises its analogue, it never returns NaNs."""
    g = golden_small
    np.random.seed(g.seed + 6)
    with pytest.raises(slmm.NotPositiveDefiniteError):
        slmm.MINQUE(slmm.SparseCholesky(ordering_method="natural"), g.mats("k1"), g["cov"], g["y"].copy(),
                    num_iter=3, sim_num=g.sim_num)


def test_run_estimates_reml_branch_and_from_paths(golden_c1mini, slmm, tmp_path):
    import pandas as pd
    from scipy.io import mmwrite
    g = golden_c1mini
    A, n = g.csr("A"), g.n
    cov = pd.DataFrame({"c0": g["cov"][:, 0], "c1": g["cov"][:, 1]})
    phe = pd.Series(g["y"])
    np.random.seed(9)
    out = slmm.run_estimates(A.copy(), phe, cov, reml=True, ignore_indices=True)
    covm = np.hstack([g["cov"][:, :2], np.ones((n, 1))])
    covm[:, :-1] -= covm[:, :-1].mean(axis=0)
    covm[:, :-1] /= covm[:, :-1].std(axis=0)
    P = np.arange(n)        # run_estimates builds its own SparseCholesky(): fetch its permutation through a twin fit
    chol = slmm.SparseCholesky()
    np.random.seed(9)
    twin = slmm.REML(chol, [A], covm, g["y"].copy(), reml=True, sim_num=100)
    assert rel_err(out["covariance coefficients"], twin["covariance coefficients"]) < 1e-12
    P = next(iter(chol._sessions.values())).eng.perm()
    np.random.seed(9)
    ref = orc.reml_fit(lambda M: DenseFactor(M, P), [A], covm, g["y"].copy(), reml=True, sim_num=100)
    assert rel_err(out["covariance coefficients"], ref["covariance coefficients"]) < 1e-6
    assert rel_err(out["covariance std"], ref["covariance std"]) < 1e-6
    # file-based entry point (reference :398-403): MatrixMarket + csv, HE branch
    mmwrite(str(tmp_path / "A.mtx"), A)
    cov.to_csv(tmp_path / "cov.csv", index=False)
    phe.to_csv(tmp_path / "phe.csv", index=False, header=False)
    np.random.seed(5)
    est, se = slmm.run_estimates_from_paths(str(tmp_path / "A.mtx"), str(tmp_path / "phe.csv"),
                                            str(tmp_path / "cov.csv"), reml=False, ignore_indices=True)
    np.random.seed(5)
    est_o, se_o = orc.he_regression([A], covm, g["y"].copy(), compute_stderr=True)
    assert rel_err(est, est_o) < 1e-9 and rel_err(se, se_o) < 1e-7


def test_standalone_wrappers_vs_reference(golden_c1mini, slmm):
    """estimate_fixed_effects / negative_log_likelihood / simulate_vector / compute_gradients called the way the
    reference's bolt_gradient_estimation calls them (:96-108), on a B200Factor."""
    g = golden_c1mini
    mats, sig = g.mats("k4"), g["sig_k4"]
    ys = g["y"] / g["y"].std()
    cov = g["cov"]
    f = slmm.SparseCholesky(ordering_method="natural")(g.csc("V_k4"))
    ViC, Lc, mu, beta = slmm.estimate_fixed_effects(f, ys, cov)
    assert rel_err(ViC, g["ViC_k4"]) < 1e-10 and rel_err(beta, g["beta_k4"]) < 1e-10
    Vir = f(ys - mu)
    assert rel_err(Vir, g["Vir_k4"]) < 1e-10
    for reml, key in ((False, "nll_ml_k4"), (True, "nll_reml_k4")):
        nll = slmm.negative_log_likelihood(f, ys, Vir, mu, Lc, reml)
        assert abs(nll - g[key]) < 1e-10 * abs(g[key])
    np.random.seed(g.seed + 4)
    W = slmm.simulate_vector(f, g.n, g.sim_num, np.argsort(f.P()))
    np.random.seed(g.seed + 4)
    Z = np.random.randn(g.n, g.sim_num)
    d = DenseFactor(g.csc("V_k4"))
    assert rel_err(W, d(d.L().dot(Z))) < 1e-9
    for reml in (False, True):
        grad = slmm.compute_gradients(sig, mats, W, Vir, reml, ViC, Lc) * sig
        assert rel_err(grad, g["bolt_grad_k4_%d" % reml]) < 1e-8


def test_matset_upload_and_he_moments_host_cabi(golden_c1mini, eng):
    """The host-buffer entry points of the C-ABI (slmm_matset_upload, slmm_he_moments_host), called directly."""
    from scilmm_b200._lib import check, lib, np_ptr
    g = golden_c1mini
    mats = [eng.canonical_csr(m) for m in g.mats("k3")]
    K, n = len(mats), g.n
    h = C.c_void_p()
    check(lib().slmm_matset_create(n, K, C.byref(h)))
    try:
        for k, m in enumerate(mats):
            check(lib().slmm_matset_upload(h, k, np_ptr(m.indptr), np_ptr(m.indices), np_ptr(m.data)))
        pid = [C.c_int32(-1) for _ in range(K)]
        for k in range(K):
            check(lib().slmm_matset_pattern_id(h, k, C.byref(pid[k])))
        assert pid[0].value == pid[1].value == 0 and pid[2].value == 2     # A and A o A share one pattern
        y = np.random.default_rng(2).standard_normal(n)
        out = np.zeros(2 * K + 2 * K * K)
        check(lib().slmm_he_moments_host(h, np_ptr(y), np_ptr(out)))
        q_off, q_diag, S_off, S_diag = eng.MatSet.split_moments(out, K)
        qo, So = orc.he_moments(mats, y)
        assert rel_err(q_off, qo) < 1e-11 and rel_err(S_off, So) < 1e-11
        qm, Sm = orc.he_moments(mats, y, MQS=True)
        assert rel_err(q_off + q_diag - y.dot(y), qm) < 1e-11 and rel_err(S_off + S_diag - (n - 1), Sm) < 1e-11
    finally:
        check(lib().slmm_matset_destroy(h))


# ------------------------------------------------------------------------------------------ round-2 behaviours
def test_aux_solve_with_the_same_width_as_the_probe_block(golden_c1mini, slmm):
    """sim_num == c + 1: the fixed-effect solve on the auxiliary stream and the probe solve on stream 0 have the
    same RHS width.  Their plans (work buffers, graphs) must be distinct: results equal the serial run bit for bit."""
    g = golden_c1mini
    mats, sig = g.mats("k4"), g["sig_k4"]
    ys = g["y"] / g["y"].std()
    c = g["cov"].shape[1]
    Z = np.random.default_rng(0).standard_normal((g.n, c + 1))
    res = []
    for overlap in (True, False, True):
        chol = slmm.SparseCholesky()
        ses = chol._session(mats, g["cov"], ys)
        ses.overlap = overlap
        for _ in range(3):
            nll, grad = ses.evaluate(sig, True, c + 1, Z=Z)
        res.append((nll, grad.copy(), ses.last["beta"].copy()))
    for r in res[1:]:
        assert r[0] == res[0][0] and np.array_equal(r[1], res[0][1]) and np.array_equal(r[2], res[0][2])
    nll_o, grad_o = orc.reml_evaluation(sig, lambda M: DenseFactor(M, ses.eng.perm()), mats, g["cov"], ys, True,
                                        c + 1, take_exp=False, normal_source=lambda n, s: Z)
    assert abs(res[0][0] - nll_o) < 1e-10 * abs(nll_o) and rel_err(res[0][1], grad_o) < 1e-8


def test_graph_replay_equals_launch_by_launch(golden_c1mini, slmm, eng):
    """Schedules replayed from CUDA graphs give bit-identical factors / solves to the launch-by-launch walk
    (profiling mode walks the list eagerly on one stream), and so does the same solve replayed on the auxiliary
    stream inside an auxiliary section."""
    g = golden_c1mini
    f = slmm.SparseCholesky()(g.csc("V_k4"))
    B = np.random.default_rng(4).standard_normal((g.n, 40))
    x1, ld1 = f(B), f.logdet()
    e = f._chol
    e.set_profiling(True)
    e.add_values(e._self_map, eng.to_device(eng.canonical_csr(sp.csr_matrix(g.csc("V_k4"))).data).data_ptr(), 1.0, True)
    e.factorize()
    f2 = slmm.B200Factor(e)
    x2, ld2 = f2(B), f2.logdet()
    e.set_profiling(False)
    assert ld1 == ld2 and np.array_equal(x1, x2)
    Bd = eng.to_device(B)
    e.aux_begin()
    try:
        e.solve_(Bd)
    finally:
        e.aux_end()
    e.aux_join()
    assert np.array_equal(Bd.cpu().numpy(), x1), "solve in an auxiliary section"


def test_cholmod_lower_triangle_rule(golden_small, slmm):
    """sksparse.cholmod.cholesky reads only the lower triangle of the CSC matrix it is given (reference :23-26).
    A triangular-only V, or one whose upper triangle holds garbage, factors like the symmetric V."""
    g = golden_small
    V = g.csc("V_k4")
    b = np.random.default_rng(0).standard_normal(g.n)
    chol = slmm.SparseCholesky()
    f = chol(V)
    x, ld = f(b), f.logdet()
    low = sp.tril(V, format="csc")
    f = chol(low)
    assert abs(f.logdet() - ld) < 1e-12 * abs(ld) and rel_err(f(b), x) < 1e-12
    junk = (low + 3.0 * sp.triu(V, 1, format="csc")).tocsc()
    f = chol(junk)
    assert abs(f.logdet() - ld) < 1e-12 * abs(ld) and rel_err(f(b), x) < 1e-12


def test_asymmetric_component_uses_its_lower_triangle(golden_small, slmm):
    """A relationship matrix whose upper triangle differs from its lower one: V is defined by the lower triangles (what
    CHOLMOD reads from the CSC sum), the gradient products use the stored matrix as the reference does."""
    g = golden_small
    A, eye = g.csr("A"), sp.eye(g.n).tocsr()
    Aj = (sp.tril(A) + 0.5 * sp.triu(A, 1)).tocsr()
    mats, sig = [Aj, eye], np.array([0.4, 0.6])
    ys = g["y"] / g["y"].std()
    chol = slmm.SparseCholesky()
    Z = np.random.default_rng(1).standard_normal((g.n, 12))
    ses = chol._session(mats, g["cov"], ys)
    nll, grad = ses.evaluate(sig, True, 12, Z=Z)
    P = ses.eng.perm()

    def lower_factor(M):
        low = sp.tril(sp.csc_matrix(M))
        return DenseFactor(low + sp.tril(low, -1).T, P)
    nll_o, grad_o = orc.reml_evaluation(sig, lower_factor, mats, g["cov"], ys, True, 12, take_exp=False,
                                        normal_source=lambda n, s: Z)
    assert abs(nll - nll_o) < 1e-10 * abs(nll_o) and rel_err(grad, grad_o) < 1e-8


def test_session_cache_notices_in_place_edits(golden_small, slmm):
    g = golden_small
    mats, sig = [m.copy() for m in g.mats("k2")], g["sig_k2"]
    ys = (g["y"] / g["y"].std()).copy()
    cov = g["cov"].copy()
    chol = slmm.SparseCholesky(ordering_method="natural")
    Z = np.random.default_rng(2).standard_normal((g.n, 8))

    def run(c, m, cv, yy):
        c.rng, c.probe_source = "host_buffer", (lambda n, s: Z)
        return slmm.bolt_gradient_estimation(np.log(sig), c, m, cv, yy, True, 8, False)
    base = run(chol, mats, cov, ys)
    ys[:] = np.roll(ys, 3)                                  # same object, new content
    edited = run(chol, mats, cov, ys)
    fresh = run(slmm.SparseCholesky(ordering_method="natural"), mats, cov, ys)
    assert edited[0] != base[0] and edited[0] == fresh[0] and np.array_equal(edited[1], fresh[1])
    mats[0].data *= 1.25
    edited = run(chol, mats, cov, ys)
    fresh = run(slmm.SparseCholesky(ordering_method="natural"), mats, cov, ys)
    assert edited[0] == fresh[0] and np.array_equal(edited[1], fresh[1])
    chol.invalidate()
    assert not chol._sessions


def test_probe_stream_is_counter_based(golden_small, slmm):
    """Device probes: Philox4x32-10 keyed by (seed, evaluation, row, global column).  Uniforms bit-exact against the
    numpy restatement, normals to 1e-13, and a column slice drawn alone equals the slice of the whole block."""
    g = golden_small
    f = slmm.SparseCholesky()(g.csc("V_k2"))
    e = f._chol
    full = e.probe_normals(g.n, 24, 0, 12345, 3).cpu().numpy()
    ref, _ = philox_normals(g.n, 24, 0, 12345, 3)
    assert np.max(np.abs(full - ref)) < 1e-13
    part = e.probe_normals(g.n, 7, 11, 12345, 3).cpu().numpy()
    assert np.array_equal(part, full[:, 11:18])
    other = e.probe_normals(g.n, 24, 0, 12345, 4).cpu().numpy()
    assert not np.array_equal(other, full)
    assert abs(full.mean()) < 0.05 and abs(full.std() - 1) < 0.05
    # an evaluation with rng='device' is reproducible given (seed, evaluation index)
    mats, sig = g.mats("k2"), g["sig_k2"]
    ys = g["y"] / g["y"].std()
    outs = []
    for _ in range(2):
        chol = slmm.SparseCholesky(rng="device", seed=99)
        outs.append(slmm.bolt_gradient_estimation(np.log(sig), chol, mats, g["cov"], ys, True, 16, False))
    assert outs[0][0] == outs[1][0] and np.array_equal(outs[0][1], outs[1][1])


def test_he_row_block_shards_hold_only_their_rows(golden_c1, eng):
    """Row-block sharded storage (what every rank does at N > 1): three shards, each uploading only its rows, the
    symmetry decided from summed hashes, partial moments adding up to the unsharded result."""
    import torch
    from scilmm_b200 import sharding
    g = golden_c1
    mats = g.mats("k3")
    K, n = len(mats), g.n
    y = np.random.default_rng(5).standard_normal(n)
    yd = eng.to_device(y)
    whole = eng.MatSet(mats)
    ref = whole.he_moments_device(yd).cpu().numpy().copy()
    bounds = sharding.row_blocks_by_lower_nnz(mats[0], 3)
    shards = [eng.MatSet(mats, row_range=(int(bounds[r]), int(bounds[r + 1]))) for r in range(3)]
    assert sum(s.h2d_bytes for s in shards) < whole.h2d_bytes + 3 * 3 * 4 * (n + 1)
    assert all(s.nnz[0] < whole.nnz[0] for s in shards)
    # emulate the all-reduce of the symmetry hashes: collect every shard's partial sums, add, hand the total back
    parts = []
    for s in shards:
        s.resolve_symmetry_sharded(lambda t: parts.append(t.clone()) or t)
        s._sym_known = False
    total = torch.stack(parts).sum(dim=0)
    for s in shards:
        s.resolve_symmetry_sharded(lambda t: t.copy_(total))
    out = sum(s.he_moments_device(yd).cpu().numpy().copy() for s in shards)
    assert rel_err(out, ref) < 1e-12
    with pytest.raises(Exception):
        shards[0].spmm(0, torch.zeros(n, 2, dtype=torch.float64, device="cuda"))
    # an asymmetric matrix is recognised from the summed hashes too (then full rows are read: still exact)
    Aj = (sp.tril(mats[0]) + 0.5 * sp.triu(mats[0], 1)).tocsr()
    sh = [eng.MatSet([Aj], row_range=(int(bounds[r]), int(bounds[r + 1]))) for r in range(3)]
    parts = []
    for s in sh:
        s.resolve_symmetry_sharded(lambda t: parts.append(t.clone()) or t)
        s._sym_known = False
    total = torch.stack(parts).sum(dim=0)
    assert total[0].item() != total[1].item()
    for s in sh:
        s.resolve_symmetry_sharded(lambda t: t.copy_(total))
    out = sum(s.he_moments_device(yd).cpu().numpy().copy() for s in sh)
    q_off, _, S_off, _ = eng.MatSet.split_moments(out, 1)
    qo, So = orc.he_moments([Aj], y)
    assert rel_err(q_off, qo) < 1e-11 and rel_err(S_off, So) < 1e-11


def test_he_dense_exact_and_fixed_index_branches(golden_small, slmm):
    g = golden_small
    mats = g.mats("k3")
    # dense inputs (reference :224-231)
    est_d = slmm.HE([m.toarray() for m in mats], g["cov"], g["y"].copy())
    assert rel_err(est_d, g["he_k3"]) < 1e-9
    # exact sampling variance, sim_num=None (reference :260-268), K = 1 and K = 3 with the reference's index slips
    for tag in ("k1", "k3"):
        est, se = slmm.HE(g.mats(tag), g["cov"], g["y"].copy(), compute_stderr=True, sim_num=None)
        est_o, se_o = orc.he_regression(g.mats(tag), g["cov"], g["y"].copy(), compute_stderr=True, sim_num=None)
        assert rel_err(est, est_o) < 1e-9
        assert np.allclose(se, se_o, rtol=1e-7, equal_nan=True)
    # fix_indices: identical to the reference for K = 1 ...
    np.random.seed(3)
    a = slmm.HE(g.mats("k1"), g["cov"], g["y"].copy(), compute_stderr=True, sim_num=20)
    np.random.seed(3)
    b = slmm.HE(g.mats("k1"), g["cov"], g["y"].copy(), compute_stderr=True, sim_num=20, fix_indices=True)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    # ... and for K = 3 equal to the intended formula evaluated with scipy on the same stream
    np.random.seed(4)
    est, se = slmm.HE(mats, g["cov"], g["y"].copy(), compute_stderr=True, sim_num=20, fix_indices=True)
    det = {}
    orc.he_regression(mats, g["cov"], g["y"].copy(), detail=det)
    K, n = 3, g.n
    H = sum(est[k] * mats[k] for k in range(K)) + (1 - est.sum()) * sp.eye(n)
    Vq = np.empty((K, K))
    np.random.seed(4)
    for i in range(K):
        for j in range(i + 1):
            Z = np.random.randn(n, 20)
            t2 = H.dot(mats[j].dot(Z) - Z)
            t4 = H.dot(mats[i].dot(t2) - t2)
            Vq[i, j] = Vq[j, i] = 2 * np.mean(np.einsum('ij,ij->j', Z, t4))
    var = np.linalg.solve(det["S"], np.linalg.solve(det["S"], Vq).T).T
    assert np.allclose(se, np.sqrt(np.diag(var)), rtol=1e-7, equal_nan=True)


# ------------------------------------------------------------------------------------------ two ranks over NCCL
def test_two_rank_nccl_equals_one_rank():
    """Sharded == unsharded on real GPUs: REML evaluation with rng='numpy' (probe columns sharded, one all-reduce of
    K doubles), rng='device' (counter-based stream), and the row-block sharded HE fit.  Needs two GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29571", os.path.join(ROOT, "tests", "nccl_two_rank.py")]
    out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-4000:]
    assert "TWO_RANK_OK" in out.stdout, out.stdout[-4000:]


# ------------------------------------------------------------------------------------------ IBD builder (8f-1)
@pytest.mark.parametrize("case", ["golden_small", "golden_c1mini", "golden_c1"])
def test_device_ibd_builder_bit_exact_vs_reference(case, request):
    """csrc/ibd.cu against the UNMODIFIED reference's LD / simple_numerator (Matrices/Numerator.py:5-43) frozen in the
    golden files: L, D and A = L D L' bit for bit, pattern included."""
    from scilmm_b200 import ibd
    g = request.getfixturevalue(case)
    rel = g.csr("rel")
    A, L, D = ibd.simple_numerator(rel)
    Ag, Lg = g.csr("ibd_full"), g.csr("ibd_Lfac")
    assert np.array_equal(A.indptr, Ag.indptr) and np.array_equal(A.indices, Ag.indices)
    assert np.array_equal(A.data, Ag.data)
    assert np.array_equal(L.indptr, Lg.indptr) and np.array_equal(L.indices, Lg.indices)
    assert np.array_equal(L.data, Lg.data)
    assert np.array_equal(D.diagonal(), g["ibd_D"])
    L2, D2, F = ibd.LD(rel, return_inbreeding_coefficient=True)
    assert np.array_equal(A.diagonal(), 1.0 + F)          # a_ii = 1 + F_i, exactly (same sums)
    A2 = ibd.create_numerator(L2, D2)
    A2.sort_indices()
    assert np.array_equal(A2.data, A.data)


def test_device_ibd_builder_known_answers_and_errors():
    from scilmm_b200 import ibd, pedigree as P
    from scilmm_b200._lib import SlmmError
    # the reference's 10-individual fixture in topological order (Tests/Examples/relationship_example.csv)
    par = {3: (0, 1), 4: (0, 1), 6: (2, 3), 7: (4, 5), 8: (6, 7), 9: (6, 7)}
    rows, cols = zip(*[(c, p) for c, ps in par.items() for p in ps])
    rel = sp.csr_matrix((np.ones(len(rows), bool), (rows, cols)), shape=(10, 10))
    A, T, D, F = ibd.numerator(rel)
    Ad = A.toarray()
    assert Ad[3, 4] == 0.5 and Ad[6, 7] == 0.125 and Ad[8, 9] == 0.5625 and Ad[9, 9] == 1.0625
    assert np.array_equal(D, [1, 1, 1, .5, .5, 1, .5, .5, .5, .5])
    # a larger simulated pedigree against the host generator (itself bit-identical to the reference on the goldens)
    ped = P.simulate_pedigree(30000, 1e-3, seed=4)
    Ah, Th, Dh, Fh = P.numerator(ped["rel"])
    A, T, D, F = ibd.numerator(ped["rel"])
    assert np.array_equal(A.indptr, Ah.indptr) and np.array_equal(A.indices, Ah.indices)
    assert np.array_equal(A.data, Ah.data) and np.array_equal(D, Dh) and np.array_equal(F, Fh)
    assert abs(T - Th).max() == 0
    bad = sp.csr_matrix((np.ones(3, bool), ([3, 3, 3], [0, 1, 2])), shape=(4, 4))         # three parents
    with pytest.raises(SlmmError):
        ibd.numerator(bad)
    bad = sp.csr_matrix((np.ones(1, bool), ([0], [2])), shape=(4, 4))                    # parent after child
    with pytest.raises(SlmmError):
        ibd.numerator(bad)


# ------------------------------------------------------------------------------------------ narrow-RHS kernels
def test_narrow_rhs_streaming_kernels(slmm, eng):
    """nrhs <= 32 takes the HBM-streaming kernels (csrc/skinny_ops.cuh): every row template (1, 2, 4 register-blocked;
    8, 16, 32 rows on the tensor pipe; each at its top edge and inside it), both flavours, split-K with the triangular
    bound (L*Z of a 2,500-column front), gathered rows with K > 512 (700 coupled rows below the dense front); 33, 48
    and 64 columns take the DMMA tile path.  Against LAPACK and bit-reproducible."""
    rng = np.random.default_rng(12)
    nd, nt, nc = 2500, 900, 700
    B = rng.standard_normal((nd, nd))
    D = B @ B.T / nd + 2.0 * np.eye(nd)
    T = sp.random(nt, nt, 0.02, random_state=2)
    T = (T + T.T + 20 * sp.eye(nt)).toarray()
    T[:nc, :nc] += 0.01
    V = np.zeros((nd + nt, nd + nt))
    C = 0.01 * rng.standard_normal((nd, nc))
    V[:nd, :nd] = D
    V[nd:, nd:] = T
    V[:nd, nd:nd + nc] = C
    V[nd:nd + nc, :nd] = C.T
    Vs = sp.csc_matrix(V)
    n = nd + nt
    for ordering in ("natural", "nesdis"):
        f = slmm.SparseCholesky(ordering_method=ordering)(Vs)
        P = f.P()
        Lref = la.cholesky(V[P][:, P], lower=True)
        for k in (1, 2, 3, 4, 5, 8, 9, 12, 13, 16, 17, 24, 32, 33, 48, 64):
            Bm = rng.standard_normal((n, k)) if k > 1 else rng.standard_normal(n)
            X1, X2 = f(Bm), f(Bm)
            assert np.array_equal(X1, X2)
            assert rel_err(X1, np.linalg.solve(V, Bm)) < 1e-10, (ordering, k)
            Z = rng.standard_normal((n, k))
            got = f.lmul(eng.to_device(Z)).cpu().numpy()
            want = (Lref @ Z)[np.argsort(P)]
            assert rel_err(got, want) < 1e-11, (ordering, k)
        # the two half sweeps on their own (mode 1: L^-1 P b, mode 2: P' L^-T)
        Bm = rng.standard_normal((n, 6))
        y = f._chol.solve_(eng.to_device(Bm), mode=1).cpu().numpy()
        # mode 1 leaves the permuted forward solution scattered back through P
        want = np.empty_like(Bm)
        want[P] = la.solve_triangular(Lref, Bm[P], lower=True)
        assert rel_err(y, want) < 1e-10


# ------------------------------------------------------------------------------------------ tiled quadratic forms
@pytest.mark.parametrize("case", ["golden_c1mini", "golden_c1"])
def test_tiled_quadforms_and_gram(case, request, slmm, eng):
    """csrc/quadform_tiled.cu against scipy and against the row-per-warp kernels: column quadratic forms of a wide
    block and the Gram matrix of the narrow block, K = 2 matrices on one pattern (A, A o A), ragged widths, a
    permutation from the factor; bit-reproducible."""
    import torch
    g = request.getfixturevalue(case)
    A, E_ = g.csr("A"), g.csr("E")
    n = g.n
    ms = eng.MatSet([A, E_])
    f = slmm.SparseCholesky()(g.csc("V_k2"))
    ms.build_tiles(0, f._chol)
    ms.build_tiles(1, f._chol)
    st = ms.tile_stats(0)
    low = sp.tril(A).nnz
    assert st["entries"] == low and 0 < st["distinct"] <= low and st["tiles"] >= (n + 63) // 64
    rng = np.random.default_rng(8)
    for ncols, nb in ((140, 12), (29, 12), (128, 0), (33, 3), (160, 16), (5, 5)):
        X = rng.standard_normal((n, ncols))
        Xd = eng.to_device(X)
        for ks, mats in (([0, 1], [A, E_]), ([1], [E_])):
            d1, G1 = ms.quadform_tiled(ks, Xd, nb)
            d2, G2 = ms.quadform_tiled(ks, Xd, nb)
            assert torch.equal(d1, d2) and (nb == 0 or torch.equal(G1, G2))
            for gi, M in enumerate(mats):
                want = np.sum(M.dot(X) * X, axis=0)
                assert rel_err(d1[gi].cpu().numpy(), want) < 1e-12
                if nb:
                    wantG = X[:, :nb].T.dot(M.dot(X[:, :nb]))
                    assert rel_err(G1[gi].cpu().numpy(), wantG) < 1e-12
    # one REML evaluation with and without the tiled pass
    mats, sig = g.mats("k4"), g["sig_k4"]
    ys = g["y"] / g["y"].std()
    Z = rng.standard_normal((n, 40))
    out = []
    for tiles in (True, False):
        ses = slmm.SparseCholesky()._session(mats, g["cov"], ys)
        assert ses.matset.has_tiles([0, 1]) and not ses.matset.has_tiles([3])
        ses.use_tiles = tiles
        out.append(ses.evaluate(sig, True, 40, Z=Z))
    assert out[0][0] == out[1][0] and rel_err(out[0][1], out[1][1]) < 1e-11


def test_wide_front_after_odd_sized_inverse_block(slmm, eng):
    """A wide front (> 1024 columns: blocked panel chain, in-place triangular panel multiply through W) that FOLLOWS
    a supernode whose block inverse has an odd number of entries.  The TMA tile grid is shifted by one column for an
    operand on an odd element; an in-place multiply split over two tile columns reads what the other column
    overwrites (seen as a 4e-3 solve residual at the 250K bench size, never below 100K individuals: no wide fronts
    there).  Against LAPACK, on both orderings, for the logdet, a solve and L*Z."""
    rng = np.random.default_rng(21)
    n1, n2 = 333, 2601
    def spd(m):
        B = rng.standard_normal((m, m))
        return B @ B.T / m + 2.0 * np.eye(m)
    V = np.zeros((n1 + n2, n1 + n2))
    V[:n1, :n1] = spd(n1)
    V[n1:, n1:] = spd(n2)
    Vs = sp.csc_matrix(V)
    sign, ld = np.linalg.slogdet(V)
    Bm = rng.standard_normal((n1 + n2, 7))
    want = np.linalg.solve(V, Bm)
    for ordering in ("natural", "nesdis"):
        f = slmm.SparseCholesky(ordering_method=ordering)(Vs)
        assert abs(f.logdet() - ld) < 1e-9 * abs(ld), ordering
        assert rel_err(f(Bm), want) < 1e-10, ordering
        P = f.P()
        Lref = la.cholesky(V[P][:, P], lower=True)
        Z = rng.standard_normal((n1 + n2, 130))
        got = f.lmul(eng.to_device(Z)).cpu().numpy()
        assert rel_err(got, (Lref @ Z)[np.argsort(P)]) < 1e-11, ordering


def test_headline_size_250k_properties(slmm, eng):
    """BASELINE config 1 as simulated for the headline metric (250,000 individuals, K = 3, 10 covariates, wide
    fronts of several thousand columns): size-independent properties of the factor at FULL size - V x = b for every
    RHS-width class of the solve schedules (narrow streaming kernels, DMMA tiles), L*Z undone by the forward sweep,
    bitwise repeatability of logdet and (LZ)' V^-1 (LZ) = Z'Z.  (scripts/solve_check.py prints the same residuals
    for a chosen size.)"""
    import torch, bench
    from scilmm_b200 import pedigree as P
    A, _, cov, y, info = bench.make_inputs(250000, 1e-3, 10)
    n = A.shape[0]
    mats = [A, P.epistasis(A), sp.eye(n).tocsr()]
    sig = np.array([0.3, 0.15, 0.55])
    chol = slmm.SparseCholesky(rng="device")
    ses = chol._session(mats, cov, y / y.std())
    ses.factor_at(sig)
    ld1 = ses.eng.logdet()
    ses.factor_at(sig)
    assert ses.eng.logdet() == ld1
    assert ses.eng.stats()["max_super_cols"] > 1024          # the blocked wide-front path is exercised
    torch.manual_seed(0)
    for k in (1, 2, 4, 8, 12, 16, 32, 128):
        B = torch.randn(n, k, dtype=torch.float64, device="cuda")
        X = ses.eng.solve_(B.clone())
        VX = sum(float(sig[j]) * ses.matset.spmm(j, X) for j in range(3))
        assert float((VX - B).abs().max() / B.abs().max()) < 1e-11, k
        LZ = ses.eng.lmul(B.clone())
        Y = ses.eng.solve_(LZ.clone(), mode=1)                 # L^-1 (L Z): Z with its rows permuted
        assert float(((Y * Y).sum(0) - (B * B).sum(0)).abs().max() / (B * B).sum(0).max()) < 1e-12, k
        # (L Z)' V^-1 (L Z) = Z'Z column by column (lmul returns P'LZ; V^-1 = P' L^-T L^-1 P)
        q1, q2 = (LZ * ses.eng.solve_(LZ.clone())).sum(0), (B * B).sum(0)
        assert float(((q1 - q2).abs() / q2).max()) < 1e-11, k


def test_upload_columns_pitched_copy(eng):
    """slmm_upload_h2d_2d: a column slice of a host block (ndarray, pageable and pinned CPU tensors) arrives as a
    contiguous device block, bit for bit; degenerate and full-width slices; bad layouts are refused."""
    import torch
    rng = np.random.default_rng(3)
    Z = rng.standard_normal((5003, 37))
    for lo, hi in ((0, 37), (5, 19), (36, 37), (0, 1), (7, 7)):
        for src in (Z, torch.from_numpy(Z), torch.from_numpy(Z).pin_memory()):
            got = eng.upload_columns(src, lo, hi)
            assert got.is_cuda and got.is_contiguous() and tuple(got.shape) == (5003, hi - lo)
            assert np.array_equal(got.cpu().numpy(), Z[:, lo:hi])
    with pytest.raises(ValueError):
        eng.upload_columns(np.asfortranarray(Z), 0, 3)
    with pytest.raises(ValueError):
        eng.upload_columns(Z.astype(np.float32), 0, 3)


def test_symmetry_detection_by_hash_sums(golden_c1mini, eng):
    """MatSet.is_symmetric (one streaming pass of hash sums): symmetric matrices pass; a single off-diagonal value
    changed in its last bit, a single missing mirror entry, and a pair of swapped values are all recognised."""
    g = golden_c1mini
    A = g.csr("A")
    B = A.copy(); C_ = A.copy(); D = A.copy()
    rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
    off = np.flatnonzero(rows != A.indices)
    B.data[off[5]] = np.nextafter(B.data[off[5]], 2.0)
    C_.data[off[7]] = 0.0; C_.eliminate_zeros()
    up = off[rows[off] < A.indices[off]]
    D.data[up[0]], D.data[up[1]] = D.data[up[1]] + 0.25, D.data[up[0]] + 0.25
    ms = eng.MatSet([A, B, C_.tocsr(), D])
    assert ms.is_symmetric(0) and not ms.is_symmetric(1) and not ms.is_symmetric(2) and not ms.is_symmetric(3)
