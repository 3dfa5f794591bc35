"""Device memory comes back: failed calls leak nothing and destroying a handle frees all it allocated.

Free memory is read for the whole device (cudaMemGetInfo through torch), so every leak these tests look for is sized
at 100 MB or more against a tolerance of 32 MB."""
import ctypes as C
import gc

import numpy as np
import pytest
import scipy.sparse as sp

from tests.util import rel_err

pytestmark = pytest.mark.gpu
TOL = 32 << 20


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import scilmm_b200  # noqa: F401
    return torch


def free_bytes(torch):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info()[0]


def banded(n, lo, hi, rng):
    """CSR with the entries i + lo .. i + hi of every row i (clipped to [0, n)), random values, sorted rows."""
    rows = np.repeat(np.arange(n), hi - lo + 1)
    cols = rows + np.tile(np.arange(lo, hi + 1), n)
    keep = (cols >= 0) & (cols < n)
    m = sp.csr_matrix((rng.standard_normal(int(keep.sum())), (rows[keep], cols[keep])), shape=(n, n))
    m.sort_indices()
    return m


def symmetric_banded(n, half, rng):
    m = banded(n, -half, 0, rng)
    m = (m + m.T).tocsr()
    m.sort_indices()
    return m


def upload(h, k, m):
    from scilmm_b200._lib import check, lib, np_ptr
    ip = np.ascontiguousarray(m.indptr, dtype=np.int32)
    ix = np.ascontiguousarray(m.indices, dtype=np.int32)
    dt = np.ascontiguousarray(m.data, dtype=np.float64)
    check(lib().slmm_matset_upload(h, k, np_ptr(ip), np_ptr(ix), np_ptr(dt)))


def test_failed_tile_build_leaks_nothing(torch):
    """A matrix with no entry on or below the diagonal cannot be tiled.  Each failed build used to keep its sort
    buffers (24 bytes per stored entry: about 350 MB here)."""
    from scilmm_b200._lib import check, lib, np_ptr
    n = 8192
    rng = np.random.default_rng(0)
    upper = banded(n, 1, 2048, rng)                      # strictly upper: ~14.7M entries
    good = symmetric_banded(n, 40, rng)
    ident = torch.arange(n, dtype=torch.int32, device="cuda")
    h = C.c_void_p()
    check(lib().slmm_matset_create(n, 2, C.byref(h)))
    try:
        upload(h, 0, upper)
        upload(h, 1, good)
        base = free_bytes(torch)
        for _ in range(5):
            assert lib().slmm_matset_build_tiles(h, 0, ident.data_ptr(), ident.data_ptr()) == 1   # SLMM_ERR_INVALID
            assert base - free_bytes(torch) <= TOL
        check(lib().slmm_matset_build_tiles(h, 1, ident.data_ptr(), ident.data_ptr()))
        X = torch.randn(n, 24, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
        ks = np.array([1], dtype=np.int32)
        tiled = torch.empty(1, 24, dtype=torch.float64, device="cuda")
        multi = torch.empty(1, 24, dtype=torch.float64, device="cuda")
        check(lib().slmm_quadform_tiled(h, 1, np_ptr(ks), X.data_ptr(), 24, 0, tiled.data_ptr(), None))
        check(lib().slmm_quadform_multi(h, 1, np_ptr(ks), X.data_ptr(), 24, 0, n, multi.data_ptr()))
        assert rel_err(tiled.cpu().numpy(), multi.cpu().numpy()) < 1e-12
    finally:
        check(lib().slmm_matset_destroy(h))


def cycles(torch, make_and_use):
    """One warm-up cycle loads the kernels it launches; then three create / use / destroy cycles must each hand
    every byte back."""
    make_and_use()
    gc.collect()
    base = free_bytes(torch)
    for _ in range(3):
        make_and_use()
        gc.collect()
        assert base - free_bytes(torch) <= TOL


def test_chol_engine_teardown_frees_everything(torch):
    from scilmm_b200 import engine
    g = 32                                               # 3-D 7-point grid: n = 32,768, panels ~280 MB
    t = sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(g, g))
    eye = sp.eye(g)
    lap = sp.kron(sp.kron(t, eye), eye) + sp.kron(sp.kron(eye, t), eye) + sp.kron(sp.kron(eye, eye), t)
    V = engine.canonical_csr((lap + 0.5 * sp.eye(g ** 3)).tocsr())
    n = V.shape[0]

    def run():
        e = engine.CholEngine(V)
        ptr_t, idx_t, val_t = (engine.to_device(a, torch) for a in (V.indptr, V.indices, V.data))
        mid = e.register_pattern_device(ptr_t, idx_t, V.nnz)
        e.add_values(mid, val_t.data_ptr(), 1.0, True)
        e.factorize()
        for w in (1, 8, 33, 128):
            for mode in (0, 1, 2):
                e.solve_(torch.ones(n, w, dtype=torch.float64, device="cuda"), mode)
        e.lmul(torch.ones(n, 8, dtype=torch.float64, device="cuda"))
        e.aux_begin()
        e.solve_(torch.ones(n, 12, dtype=torch.float64, device="cuda"))
        e.aux_end()
        e.aux_join()
        e.set_profiling(True)
        e.add_values(mid, val_t.data_ptr(), 1.0, True)
        e.factorize()
        e.set_profiling(False)
        e.add_values(mid, val_t.data_ptr(), 1.0, True)
        e.timeline()
        torch.cuda.synchronize()
        del e

    cycles(torch, run)


def test_matset_teardown_frees_everything(torch):
    from scilmm_b200 import engine
    from scilmm_b200._lib import check, lib
    n = 200_000
    rng = np.random.default_rng(3)
    A = symmetric_banded(n, 30, rng)                     # 12M entries: values and tiles ~100 MB each
    B = symmetric_banded(n, 4, rng)                      # a second pattern: HE builds a cross map between the two
    ident = torch.arange(n, dtype=torch.int32, device="cuda")
    y = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    X = torch.randn(n, 64, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(5))

    def run():
        ms = engine.MatSet([A, B])
        ms.he_moments_device(y)
        check(lib().slmm_matset_build_tiles(ms._h, 0, ident.data_ptr(), ident.data_ptr()))
        ms.quadform_tiled([0], X, 8)
        ms.quadform_gram_multi([0], X[:, 8:], X[:, :8])
        torch.cuda.synchronize()
        del ms

    cycles(torch, run)


def test_ibd_teardown_frees_everything(torch):
    from scilmm_b200 import ibd
    from tests.util import load_golden
    rel = load_golden("case_c1").csr("rel")

    def run():
        ibd.simple_numerator(rel)

    cycles(torch, run)
