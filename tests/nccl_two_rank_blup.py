"""Launched by tests/test_gpu_blup.py::test_two_rank_pev under torchrun (2 ranks): every rank calls blup() with the
process group active (each rank sweeps half of the probe blocks, one all-reduce assembles the partial sums), then the
unsharded call with the collective layer bypassed, and asserts that pev and pev_se are bit-identical and u equal.
Prints TWO_RANK_BLUP_OK on rank 0.  SLMM_TWO_RANK_BACKEND=gloo runs the same check with both ranks on one GPU."""
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
    from tests.test_blup_cpu import masked_y
    from tests.util import load_golden
    g = load_golden("case_c1")
    y = masked_y(g["y"], g["cov"].shape[1], "random")

    def call():
        # 3 probe blocks (128 + 128 + 44 columns): an odd split, 1 + 2
        return S.blup(S.SparseCholesky(seed=9), g.mats("k4")[:-1], g["cov"], y, g["sig_k4"], pev_probes=300)

    sharded = call()
    real = sharding.active_group
    sharding.active_group = lambda: None           # same process, collectives bypassed: the 1-rank computation
    try:
        single = call()
    finally:
        sharding.active_group = real
    for k in ("pev", "pev_se", "reliability", "u", "residual", "fixed", "yhat", "beta"):
        assert np.array_equal(sharded[k], single[k], equal_nan=True), k
    dist.barrier()
    if rank == 0:
        print("TWO_RANK_BLUP_OK", sharded["pev"].shape)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
