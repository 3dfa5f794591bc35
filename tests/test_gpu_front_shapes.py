"""The supernodal factor and the three solve modes at every front shape the schedules of csrc/chol.cu treat
differently, against LAPACK on the permuted matrix (L is unique given P).

`build_factor_schedule` and `get_plan` branch on the width ns of a front: one 64-column POTRF block (ns <= 64), a
narrow front whose 1024-column diagonal block is inverted by the batched W pass (64 < ns <= 1024), and a wide front
(ns > 1024: a chain of 1024-column outer blocks, each inverted by recursive doubling, then CPANEL / OUTER).  A last
outer block of at most 64 columns keeps its inverse in the 64 x 64 POTRF slot (`outer_block`, ldw = 64) and has no
doubling steps.  The golden pedigrees never reach a front wider than 64 columns, so every case here builds a matrix
with one front of a chosen (ns, rs) = (columns, rows below) and asserts that the analysis really has it.

Every check runs on the functor's own device factor:
  * L against scipy.linalg.cholesky, logdet against slogdet; the panels of a second factorization, of a profiled one
    (one stream, launch by launch) and of a timeline one (look-ahead streams with timed events) bit for bit;
  * per RHS width (every streaming-kernel family, the tile path, look-ahead from 64 columns, more than 160 columns):
    mode 0 (V^-1 B), mode 1 (forward half L^-1 P B), mode 2 (backward half P' L^-T B) and L*Z against LAPACK,
    mode 2 after mode 1 equal to mode 0 bit for bit;
  * the width list a second time, bit for bit: it has more widths than `get_plan` keeps, so its plans and their
    captured graphs are rebuilt in between;
  * a non-positive (or NaN) pivot raises NotPositiveDefiniteError at the column LAPACK reports, and the same functor
    then factors the good matrix exactly as a fresh one does."""
import functools
import sys

import numpy as np
import pytest
import scipy.linalg as la
import scipy.sparse as sp
from scipy.linalg import lapack

from tests.util import rel_err

pytestmark = pytest.mark.gpu

WIDTHS = (1, 2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 64, 65, 128, 161)
SIBLING = 40          # columns of the second child of the tail: keeps the target front from merging into the tail


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


# ------------------------------------------------------------------------------------------ matrices and references
def _spd(rng, m):
    G = rng.standard_normal((m, m))
    return G @ G.T / m + 2.0 * np.eye(m)


@functools.lru_cache(maxsize=None)
def _front_matrix(ns, rs):
    """Dense V (natural order): a dense SPD block of ns columns, a sibling dense SPD block of SIBLING columns, both
    coupled densely (0.01 N(0,1)) to a dense SPD tail of rs rows.  The tail's first column has two children, so the
    first block stays a front of its own: (ns, rs)."""
    rng = np.random.default_rng(1000 * ns + rs)
    n0 = ns + SIBLING
    V = np.zeros((n0 + rs, n0 + rs))
    V[:ns, :ns] = _spd(rng, ns)
    V[ns:n0, ns:n0] = _spd(rng, SIBLING)
    if rs:
        V[n0:, n0:] = _spd(rng, rs)
        C = 0.01 * rng.standard_normal((n0, rs))
        V[:n0, n0:] = C
        V[n0:, :n0] = C.T
    V.setflags(write=False)
    return V


def front_matrix(ns, rs):
    return _front_matrix(ns, rs).copy()


def front_shapes(eng, V, ordering="natural"):
    a = eng.SymbolicView(sp.csr_matrix(V), ordering=ordering).arrays()
    ns = np.diff(a["sn_first"])
    return set(zip(ns.tolist(), (a["sn_nrow"] - ns).tolist()))


def assert_front(eng, V, ns, rs):
    """The case covers what it claims: the analysis has a supernode of exactly ns columns and rs rows below."""
    shapes = front_shapes(eng, V)
    assert (ns, rs) in shapes, ("front (%d, %d) not in the analysis" % (ns, rs), sorted(shapes)[-6:])


class DenseRef(object):
    """LAPACK on the permuted matrix V[P][:, P]."""

    def __init__(self, V, P):
        self.V, self.P = V, P
        self.L = la.cholesky(V[np.ix_(P, P)], lower=True)
        self.lu = la.lu_factor(V)                      # dgetrf: what np.linalg.solve factors, once for all widths

    def solve(self, B):
        return la.lu_solve(self.lu, B)

    def forward(self, B):
        out = np.empty_like(B)
        out[self.P] = la.solve_triangular(self.L, B[self.P], lower=True)
        return out

    def backward(self, B):
        out = np.empty_like(B)
        out[self.P] = la.solve_triangular(self.L.T, B[self.P], lower=False)
        return out

    def lmul(self, Z):
        return (self.L @ Z)[np.argsort(self.P)]

    def logdet(self):
        sign, ld = np.linalg.slogdet(self.V)
        assert sign > 0
        return ld

    def L_err(self, Lgot):
        return rel_err(Lgot.toarray(), self.L)


def block_diag_csc(blocks):
    nb = blocks.shape[0]
    return sp.bsr_matrix((blocks, np.arange(nb), np.arange(nb + 1)), shape=(nb * blocks.shape[1],) * 2).tocsc()


class BlockDiagRef(object):
    """LAPACK per diagonal block of a block-diagonal V in natural order (P = identity): blocks (nb, b, b)."""

    def __init__(self, blocks):
        self.blocks = blocks
        self.Lb = np.linalg.cholesky(blocks)
        self.nb, self.b = blocks.shape[0], blocks.shape[1]
        self.P = np.arange(self.nb * self.b)

    def _split(self, B):
        return B.reshape(self.nb, self.b, -1)

    def solve(self, B):
        return np.linalg.solve(self.blocks, self._split(B)).reshape(B.shape)

    def forward(self, B):
        return np.linalg.solve(self.Lb, self._split(B)).reshape(B.shape)

    def backward(self, B):
        return np.linalg.solve(self.Lb.transpose(0, 2, 1), self._split(B)).reshape(B.shape)

    def lmul(self, Z):
        return np.matmul(self.Lb, self._split(Z)).reshape(Z.shape)

    def logdet(self):
        return 2.0 * float(np.sum(np.log(np.diagonal(self.Lb, axis1=1, axis2=2))))

    def L_err(self, Lgot):
        want = block_diag_csc(self.Lb)
        return float(abs(Lgot.tocsr() - want).max() / abs(want).max())


def check_factor_and_solves(slmm, eng, Vs, make_ref):
    """Factor Vs (natural order) twice with one functor, then profiled and in timeline mode, all bit for bit; check the
    factor and every solve mode at every width against LAPACK, then once more bit for bit after the solve plans were
    evicted and rebuilt."""
    chol = slmm.SparseCholesky(ordering_method="natural")
    f = chol(Vs)
    panels = f._chol.panels()
    f = chol(Vs)
    assert np.array_equal(f._chol.panels(), panels), "two factorizations differ"
    dev = f._chol
    vals = eng.to_device(eng.canonical_csr(sp.csr_matrix(Vs)).data)
    for run in ("profiled", "timeline"):
        dev.add_values(dev._self_map, vals.data_ptr(), 1.0, True)
        if run == "profiled":
            dev.set_profiling(True)
            dev.factorize()
            dev.set_profiling(False)
        else:
            dev.timeline()
        assert np.array_equal(dev.panels(), panels), "%s factorization differs" % run
    f = slmm.B200Factor(dev)
    ref = make_ref(f.P())
    n = Vs.shape[0]
    ld = ref.logdet()
    assert abs(f.logdet() - ld) <= 1e-10 * abs(ld), (f.logdet(), ld)
    assert ref.L_err(f.L()) < 1e-11
    first = {}
    for rep in range(2):
        for k in WIDTHS:
            rng = np.random.default_rng(k)
            B, Z = rng.standard_normal((n, k)), rng.standard_normal((n, k))
            Bd = eng.to_device(B)
            x0 = dev.solve_(Bd.clone(), 0).cpu().numpy()
            y1d = dev.solve_(Bd.clone(), 1)
            y1 = y1d.cpu().numpy()
            x12 = dev.solve_(y1d, 2).cpu().numpy()
            y2 = dev.solve_(Bd.clone(), 2).cpu().numpy()
            lz = dev.lmul(eng.to_device(Z)).cpu().numpy()
            got = (x0, y1, y2, x12, lz)
            if rep == 0:
                assert rel_err(x0, ref.solve(B)) < 1e-10, ("mode 0", k)
                assert rel_err(y1, ref.forward(B)) < 1e-10, ("mode 1", k)
                assert rel_err(y2, ref.backward(B)) < 1e-10, ("mode 2", k)
                assert np.array_equal(x12, x0), ("mode 2 after mode 1 != mode 0", k)
                assert rel_err(lz, ref.lmul(Z)) < 1e-11, ("L*Z", k)
                first[k] = got
            else:
                for what, a, b in zip(("mode 0", "mode 1", "mode 2", "mode 1+2", "L*Z"), got, first[k]):
                    assert np.array_equal(a, b), ("second pass, rebuilt plan", what, k)


# ------------------------------------------------------------------------------------------ 1. front shapes
# (ns, rs): 64 is one POTRF block; 65 the first front with a batched W (its last 64-row step has 1 row); 128 / 129 the
# edges of a 128-column tile; 1023 / 1024 the largest narrow fronts (1024: a full batched W); 1025 a wide front whose
# last outer block has 1 column; 1035 / 1072 last blocks of 11 / 48 columns (the 250K config's fronts 2059 and 1072);
# 1088 / 1089 last blocks of 64 / 65 columns (both sides of the POTRF-slot fallback; 65 doubles with a 1-column second
# half); 2048 a full last block; 2059 two outer blocks and an 11-column tail.  rs = 0 is a root front (no Schur step),
# rs = 700 takes the CTA-per-item extend-add (>= 512 rows).
SHAPES = [(64, 130), (65, 0), (128, 700), (129, 1), (1023, 130), (1024, 700), (1025, 0), (1035, 130), (1072, 700),
          (1088, 1), (1089, 130), (2048, 0), (2059, 700)]


@pytest.mark.parametrize("ns,rs", SHAPES, ids=["ns%d_rs%d" % s for s in SHAPES])
def test_front_shape_against_lapack(ns, rs, slmm, eng):
    V = front_matrix(ns, rs)
    assert_front(eng, V, ns, rs)
    check_factor_and_solves(slmm, eng, sp.csc_matrix(V), lambda P: DenseRef(V, P))


# ------------------------------------------------------------------------------------------ degenerate sizes
@pytest.mark.parametrize("n", [1, 2, 3, 7])
def test_tiny_dense_matrices(n, slmm, eng):
    """n = 1, 2, 3, 7: one dense front; the width list runs from below n to far above it."""
    V = _spd(np.random.default_rng(n), n)
    check_factor_and_solves(slmm, eng, sp.csc_matrix(V), lambda P: DenseRef(V, P))


def test_diagonal_matrix(slmm, eng):
    """A diagonal V of 5,000 rows: 5,000 single-column supernodes, all in one level, no update anywhere."""
    d = np.random.default_rng(5).uniform(0.5, 3.0, 5000)
    Vs = sp.diags(d, format="csc")
    view = eng.SymbolicView(Vs, ordering="natural")
    assert view.nsuper == 5000 and view.nlevels == 1
    check_factor_and_solves(slmm, eng, Vs, lambda P: BlockDiagRef(d.reshape(-1, 1, 1)))


def test_many_2x2_components(slmm, eng):
    """3,000 disjoint 2 x 2 blocks: 3,000 two-column supernodes side by side in one level."""
    rng = np.random.default_rng(6)
    a, b = rng.uniform(1.0, 3.0, 3000), rng.uniform(1.0, 3.0, 3000)
    c = rng.uniform(-0.9, 0.9, 3000) * np.sqrt(a * b)
    blocks = np.stack([np.stack([a, c], 1), np.stack([c, b], 1)], 1)
    Vs = block_diag_csc(blocks)
    view = eng.SymbolicView(Vs, ordering="natural")
    arr = view.arrays()
    assert view.nsuper == 3000 and view.nlevels == 1 and np.all(np.diff(arr["sn_first"]) == 2)
    check_factor_and_solves(slmm, eng, Vs, lambda P: BlockDiagRef(blocks))


# ------------------------------------------------------------------------------------------ 3. where a factorization fails
def lapack_fail_column(M):
    """0-based column of the first non-positive or NaN pivot of dpotrf on M, -1 if none.  OpenBLAS's dpotrf does not
    test for NaN (it reports success with NaNs in the factor); reference LAPACK stops at the first NaN pivot, which is
    the first NaN on the diagonal of the factor."""
    c, info = lapack.dpotrf(M, lower=1, clean=0)
    cols = [info - 1] if info > 0 else []
    nan = np.flatnonzero(np.isnan(np.diag(c)))
    if nan.size:
        cols.append(int(nan[0]))
    return min(cols) if cols else -1


def check_failure_and_reuse(slmm, V_good, V_bad, ordering, want_col):
    """V_bad raises at want_col; the same functor then factors V_good (same pattern) bit for bit like a fresh one."""
    chol = slmm.SparseCholesky(ordering_method=ordering)
    with pytest.raises(slmm.NotPositiveDefiniteError) as err:
        chol(sp.csc_matrix(V_bad))
    assert err.value.column == want_col, (err.value.column, want_col)
    f = chol(sp.csc_matrix(V_good))
    assert len(chol._engines) == 1, "the good matrix must reuse the failed factorization's engine"
    fresh = slmm.SparseCholesky(ordering_method=ordering)(sp.csc_matrix(V_good))
    assert f.logdet() == fresh.logdet()
    B = np.random.default_rng(3).standard_normal((V_good.shape[0], 5))
    assert np.array_equal(f(B), fresh(B))
    return f


# (label, ns, rs, column, how):  "neg" sets V[c, c] = -1; "schur" sets V[c, c] just below |L[c, :c]|^2 of the good
# factor (positive entry, the pivot goes negative only after the updates of earlier columns)
FAILURES = [
    ("column_0", 1023, 130, 0, "neg"),
    ("tail_column", 1023, 130, 1023 + SIBLING + 77, "neg"),
    ("narrow_front_64k_plus_r", 1023, 130, 64 * 7 + 13, "neg"),
    ("wide_second_outer_block", 2059, 130, 1024 + 301, "neg"),
    ("wide_11_column_last_block", 2059, 130, 2048 + 6, "neg"),
    ("last_block_48_columns", 1072, 700, 1024 + 40, "neg"),
    ("tail_after_children_updates", 1072, 700, 1072 + SIBLING, "schur"),
    ("wide_after_outer_update", 2059, 130, 1024 + 500, "schur"),
    ("wide_last_block_after_updates", 2059, 130, 2048 + 9, "schur"),
]


@pytest.mark.parametrize("label,ns,rs,col,how", FAILURES, ids=[f[0] for f in FAILURES])
def test_failing_column_matches_lapack(label, ns, rs, col, how, slmm, eng):
    V = front_matrix(ns, rs)
    assert_front(eng, V, ns, rs)
    bad = V.copy()
    if how == "neg":
        bad[col, col] = -1.0
    else:
        L = la.cholesky(V, lower=True)
        s = float(L[col, :col] @ L[col, :col])
        bad[col, col] = s * (1.0 - 1e-6)
        assert 0.0 < bad[col, col] and V[col, col] - s > 0.0
    want = lapack_fail_column(bad)
    assert want == col                   # natural ordering: the permuted column is the column
    check_failure_and_reuse(slmm, V, bad, "natural", want)


def test_nan_entry_fails_at_the_lapack_column(slmm, eng):
    """One NaN as a symmetric off-diagonal pair inside a wide front (1089 columns, last block of 65): the pivot of its
    later column is the first NaN."""
    V = front_matrix(1089, 130)
    bad = V.copy()
    bad[1050, 300] = bad[300, 1050] = np.nan
    want = lapack_fail_column(bad)
    assert want == 1050
    check_failure_and_reuse(slmm, V, bad, "natural", want)


def test_failing_column_is_the_permuted_one(slmm, eng):
    """Under nesdis the reported column is the column of the PERMUTED matrix (SymbolicView's permutation)."""
    V = front_matrix(1089, 130)
    P = eng.SymbolicView(sp.csr_matrix(V), ordering="nesdis").arrays()["perm"]
    cp = next(c for c in range(700, V.shape[0]) if P[c] != c)     # a column the ordering moved
    bad = V.copy()
    bad[P[cp], P[cp]] = -1.0
    want = lapack_fail_column(bad[np.ix_(P, P)])
    assert want == cp and lapack_fail_column(bad) == P[cp] != cp
    f = check_failure_and_reuse(slmm, V, bad, "nesdis", want)
    assert np.array_equal(f.P(), P)
