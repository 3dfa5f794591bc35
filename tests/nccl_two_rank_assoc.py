"""Launched by tests/test_gpu_association.py::test_two_rank_scan under torchrun (2 ranks): every rank runs the
association scan with the process group active (each rank scans half of the variants, one all-reduce assembles the
arrays), then the unsharded scan with the collective layer bypassed, and asserts that both ranks hold the unsharded
arrays to 1e-12.  Prints TWO_RANK_ASSOC_OK on rank 0.  SLMM_TWO_RANK_BACKEND=gloo runs the same check with both ranks
on one GPU."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    backend = os.environ.get("SLMM_TWO_RANK_BACKEND", "nccl")
    torch.cuda.set_device(local % torch.cuda.device_count())
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist.init_process_group(backend)
    import scilmm_b200.SparseCholesky  # noqa: F401
    S = sys.modules["scilmm_b200.SparseCholesky"]
    from scilmm_b200 import sharding
    from tests.test_association_cpu import make_genotypes, with_variant_covariate
    from tests.util import load_golden, rel_err
    g = load_golden("case_c1")
    G = np.asfortranarray(make_genotypes(g.n, 101, 21))        # odd split: 50 + 51 variants
    cov = with_variant_covariate(g["cov"], G, 0)

    def scan():
        return S.association(S.SparseCholesky(), g.mats("k4")[:-1], cov, g["y"], g["sig_k4"], G)

    sharded = scan()
    real = sharding.active_group
    sharding.active_group = lambda: None           # same process, collectives bypassed: the 1-rank computation
    try:
        single = scan()
    finally:
        sharding.active_group = real
    for k in ("beta", "se", "chi2", "p"):
        fin = np.isfinite(single[k])
        assert np.array_equal(np.isfinite(sharded[k]), fin), k
        assert rel_err(sharded[k][fin], single[k][fin]) <= 1e-12, (k, rel_err(sharded[k][fin], single[k][fin]))
    assert np.array_equal(sharded["n_obs"], single["n_obs"]) and sharded["n_obs"].dtype == np.int64
    assert np.array_equal(sharded["af"], single["af"])
    dist.barrier()
    if rank == 0:
        print("TWO_RANK_ASSOC_OK", int(np.isfinite(sharded["beta"]).sum()), "finite of", G.shape[1])
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
