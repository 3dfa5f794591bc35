"""Launched by tests/test_gpu_region.py::test_two_rank_region_test under torchrun (2 ranks): every rank runs the region
tests with the process group active (each rank tests a contiguous half of the regions, one all-reduce assembles the
arrays), then the unsharded call with the collective layer bypassed, and asserts that both ranks hold the unsharded
arrays to 1e-12.  Prints TWO_RANK_REGION_OK on rank 0.  SLMM_TWO_RANK_BACKEND=gloo runs the same check with both
ranks on one GPU."""
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
    sizes = [1, 2, 1, 9, 30, 4, 70, 3, 12, 5, 25]              # odd split: 5 + 6 regions
    bounds = np.concatenate([[0], np.cumsum(sizes)])
    G = np.asfortranarray(make_genotypes(g.n, int(bounds[-1]), 22))
    cov = with_variant_covariate(g["cov"], G, 0)

    def call():
        return S.region_test(S.SparseCholesky(), g.mats("k4")[:-1], cov, g["y"], g["sig_k4"], G, bounds)

    sharded = call()
    real = sharding.active_group
    sharding.active_group = lambda: None           # same process, collectives bypassed: the 1-rank computation
    try:
        single = call()
    finally:
        sharding.active_group = real
    for k in ("burden_beta", "burden_se", "burden_chi2", "burden_p", "skat_q", "skat_p"):
        fin = np.isfinite(single[k])
        assert np.array_equal(np.isfinite(sharded[k]), fin), k
        assert rel_err(sharded[k][fin], single[k][fin]) <= 1e-12, (k, rel_err(sharded[k][fin], single[k][fin]))
    for k in ("n_variants", "n_poly"):
        assert np.array_equal(sharded[k], single[k]) and sharded[k].dtype == np.int64, k
    dist.barrier()
    if rank == 0:
        print("TWO_RANK_REGION_OK", int(np.isfinite(sharded["skat_p"]).sum()), "finite of", len(sizes))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
