"""Multi-GPU partitioning of the path (one process per GPU, torch.distributed).

The path shards in exactly two places (SURVEY.md §8e); everything else is replicated:
  * REML probe / RHS columns: every rank assembles and factors V itself (inputs are replicated, recomputing
    is cheaper than broadcasting the factor), takes a contiguous slice of the sim_num probe columns through
    the backward half-sweep and the fused SpMM reductions, and the K partial trace sums are combined with ONE
    all-reduce of K doubles per evaluation.
  * HE row blocks: contiguous row ranges balanced by nonzeros; ONE all-reduce of 2K + 2K^2 doubles.
The helpers work on CPU tensors with the gloo backend as well, which is how the host logic is tested.
"""
import numpy as np


def active_group():
    """torch.distributed module if a process group with more than one rank is initialised, else None."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return dist
    except Exception:
        pass
    return None


def rank_world():
    dist = active_group()
    return (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)


def column_block(ncols, rank, world):
    """Contiguous slice [lo, hi) of `ncols` probe columns owned by `rank` (sizes differ by at most one)."""
    return (ncols * rank) // world, (ncols * (rank + 1)) // world


def row_blocks_by_nnz(indptr, world):
    """world+1 row boundaries such that every block holds about nnz/world nonzeros (contiguous rows)."""
    indptr = np.asarray(indptr, dtype=np.int64)
    n = indptr.size - 1
    targets = indptr[-1] * np.arange(1, world, dtype=np.float64) / world
    cuts = np.searchsorted(indptr, targets, side="left")
    bounds = np.concatenate(([0], np.clip(cuts, 0, n), [n])).astype(np.int64)
    return np.maximum.accumulate(bounds)


def row_blocks_by_lower_nnz(m, world, sample_stride=16):
    """world+1 row boundaries balancing the entries ON AND BELOW THE DIAGONAL, which is what the HE kernels read for
    symmetric matrices (rows near the end of a symmetric matrix hold most of the lower triangle: balancing the
    stored entries would leave the last rank ~2x the work of the first).  The lower-triangle length is measured
    exactly on every sample_stride-th row (a vectorised bisection on the sorted row, no scan of the 10^8-entry
    index array) and interpolated in between."""
    indptr = np.asarray(m.indptr, dtype=np.int64)
    n = indptr.size - 1
    if world <= 1 or n == 0:
        return np.array([0, n], dtype=np.int64)
    rows = np.unique(np.concatenate((np.arange(0, n, sample_stride), [n - 1]))).astype(np.int64)
    lo, hi = indptr[rows].copy(), indptr[rows + 1].copy()
    idx = m.indices
    while True:                                   # first position with col > row, per sampled row
        act = lo < hi
        if not act.any():
            break
        mid = (lo + hi) // 2
        col = idx[np.minimum(mid, idx.size - 1)]
        go = act & (col <= rows)
        lo = np.where(go, mid + 1, lo)
        hi = np.where(act & ~go, mid, hi)
    length = np.maximum(indptr[rows + 1] - indptr[rows], 1)
    frac = (lo - indptr[rows]) / length
    lower = np.interp(np.arange(n), rows, frac) * np.diff(indptr)
    cum = np.concatenate(([0.0], np.cumsum(lower)))
    targets = cum[-1] * np.arange(1, world, dtype=np.float64) / world
    cuts = np.searchsorted(cum, targets, side="left")
    bounds = np.concatenate(([0], np.clip(cuts, 0, n), [n])).astype(np.int64)
    return np.maximum.accumulate(bounds)


def allreduce_sum_(t):
    """In-place sum over ranks (no-op without a process group).  Tiny payloads: latency, not bandwidth."""
    dist = active_group()
    if dist is not None:
        dist.all_reduce(t)
    return t


def gather_slices(part, keys, total, lo, hi, device):
    """Whole length-`total` result arrays on every rank from each rank's slice [lo, hi): part[k] holds this rank's
    entries of key k.  One all-reduce of a float64 (len(keys), total) tensor on `device`, zero outside each rank's
    slice (NaN entries survive the sum); every array comes back with the dtype of its part[k].  Without a process
    group, part itself."""
    dist = active_group()
    if dist is None:
        return part
    import torch
    full = torch.zeros(len(keys), total, dtype=torch.float64, device=device)
    full[:, lo:hi] = torch.from_numpy(np.stack([part[k].astype(np.float64) for k in keys]))
    dist.all_reduce(full)
    full = full.cpu().numpy()
    return {k: full[i].astype(part[k].dtype, copy=False) for i, k in enumerate(keys)}
