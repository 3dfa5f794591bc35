"""N>1 host logic on CPU: two gloo ranks run the same partition + combine code the GPU path uses
(scilmm_b200/sharding.py); the per-rank partial results are produced by the oracle restricted to the rank's
shard, all-reduced, and compared with the unsharded oracle."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from scilmm_b200 import sharding
from tests.util import load_golden


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _pack(q_off, q_diag, S_off, S_diag):
    return np.concatenate([q_off, q_diag, S_off.ravel(), S_diag.ravel()])


def _partial_he(mats, y, lo, hi):
    """Moments of rows [lo,hi) in the device layout [q_off | q_diag | S_off | S_diag] (lower triangle filled)."""
    K = len(mats)
    q_off, q_diag = np.zeros(K), np.zeros(K)
    S_off, S_diag = np.zeros((K, K)), np.zeros((K, K))
    for i in range(K):
        Ai = mats[i][lo:hi]
        di = mats[i].diagonal()[lo:hi]
        q_diag[i] = di.dot(y[lo:hi] ** 2)
        q_off[i] = y[lo:hi].dot(Ai.dot(y)) - q_diag[i]
        for j in range(i + 1):
            S_diag[i, j] = di.dot(mats[j].diagonal()[lo:hi])
            S_off[i, j] = Ai.multiply(mats[j][lo:hi]).sum() - S_diag[i, j]
    return _pack(q_off, q_diag, S_off, S_diag)


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        assert sharding.rank_world() == (rank, world)
        g = load_golden("case_c1mini")
        mats = g.mats("k3")
        y = np.random.default_rng(0).standard_normal(g.n)
        bounds = sharding.row_blocks_by_nnz(mats[0].indptr, world)
        part = torch.from_numpy(_partial_he(mats, y, int(bounds[rank]), int(bounds[rank + 1])))
        sharding.allreduce_sum_(part)
        # REML probe columns: partial trace sums over this rank's column slice
        s = 11
        W = np.random.default_rng(1).standard_normal((g.n, s))
        lo, hi = sharding.column_block(s, rank, world)
        comp1 = torch.tensor([np.sum(m.dot(W[:, lo:hi]) * W[:, lo:hi]) for m in mats])
        sharding.allreduce_sum_(comp1)
        if rank == 0:
            out["he"] = part.numpy().copy()
            out["comp1"] = comp1.numpy().copy()
            out["bounds"] = bounds
    finally:
        dist.destroy_process_group()


def test_two_rank_partition_and_allreduce():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    g = load_golden("case_c1mini")
    mats = g.mats("k3")
    y = np.random.default_rng(0).standard_normal(g.n)
    full = _partial_he(mats, y, 0, g.n)
    assert np.allclose(out["he"], full, rtol=1e-12, atol=1e-9)
    W = np.random.default_rng(1).standard_normal((g.n, 11))
    assert np.allclose(out["comp1"], [np.sum(m.dot(W) * W) for m in mats], rtol=1e-12)
    b = out["bounds"]
    assert b[0] == 0 and b[-1] == g.n and np.all(np.diff(b) >= 0)
    nnz = mats[0].indptr[b[1:]] - mats[0].indptr[b[:-1]]
    assert abs(nnz[0] - nnz[1]) <= 2 * np.diff(mats[0].indptr).max()      # balanced by nonzeros


def _scan_result(total):
    """A per-variant result as the scans return it: float64 with NaN slots, int64 counts, int8 flags with -1."""
    rng = np.random.default_rng(2)
    x = rng.standard_normal(total)
    x[[0, 3, total - 1]] = np.nan
    return {"p": x, "n_obs": rng.integers(0, 1 << 40, total), "spa": rng.integers(-1, 2, total).astype(np.int8)}


def _gather_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        total = 7
        lo, hi = sharding.column_block(total, rank, world)
        part = {k: v[lo:hi].copy() for k, v in _scan_result(total).items()}
        out[rank] = sharding.gather_slices(part, ("p", "n_obs", "spa"), total, lo, hi, "cpu")
    finally:
        dist.destroy_process_group()


def test_two_rank_gather_slices():
    """Slices of 3 and 4 entries: every rank gets the unsharded arrays, NaN slots and dtypes included."""
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gather_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    full = _scan_result(7)
    assert (full["spa"] == -1).any()
    for rank in range(world):
        for k, v in full.items():
            assert out[rank][k].dtype == v.dtype, (rank, k)
            assert np.array_equal(out[rank][k], v, equal_nan=True), (rank, k)


def test_partition_helpers_edge_cases():
    assert sharding.rank_world() == (0, 1)
    assert sharding.active_group() is None
    t = torch.ones(3)
    assert sharding.allreduce_sum_(t) is t and torch.all(t == 1)
    part = _scan_result(5)
    assert sharding.gather_slices(part, tuple(part), 5, 0, 5, "cpu") is part
    for s, w in ((128, 8), (100, 8), (3, 8), (0, 2)):
        blocks = [sharding.column_block(s, r, w) for r in range(w)]
        assert blocks[0][0] == 0 and blocks[-1][1] == s
        assert all(blocks[r][1] == blocks[r + 1][0] for r in range(w - 1))
        sizes = [b - a for a, b in blocks]
        assert max(sizes) - min(sizes) <= 1
    indptr = np.array([0, 0, 0, 10, 10, 11, 30])
    for w in (1, 2, 4, 8):
        b = sharding.row_blocks_by_nnz(indptr, w)
        assert b.size == w + 1 and b[0] == 0 and b[-1] == 6 and np.all(np.diff(b) >= 0)
    assert sharding.row_blocks_by_nnz(np.zeros(5, dtype=np.int32), 3).tolist() == [0, 0, 0, 4]


def test_row_blocks_balance_the_lower_triangle():
    """HE row blocks are cut by the entries on/below the diagonal (what the symmetric kernels read)."""
    import scipy.sparse as sp
    from scilmm_b200 import sharding
    from tests.util import load_golden
    A = load_golden("case_c1").csr("A")
    low = sp.tril(A).tocsr()
    for world in (2, 4, 8):
        b = sharding.row_blocks_by_lower_nnz(A, world)
        assert b[0] == 0 and b[-1] == A.shape[0] and np.all(np.diff(b) >= 0)
        work = np.array([low.indptr[b[i + 1]] - low.indptr[b[i]] for i in range(world)], dtype=float)
        assert work.max() / work.mean() < 1.10
    assert list(sharding.row_blocks_by_lower_nnz(A, 1)) == [0, A.shape[0]]
