"""Launched by tests/test_gpu_aireml.py::test_two_rank_nccl_aireml_fit under torchrun (2 ranks, NCCL): every rank runs
the AI-REML fit with the process group active (probe columns sharded, the AI matrix computed in full on every rank),
then the unsharded fit on its own GPU with the collective layer bypassed, and asserts they agree and that both ranks
hold the same sigma bit for bit.  Prints TWO_RANK_AIREML_OK on rank 0.  SLMM_TWO_RANK_BACKEND=gloo runs the same
check with both ranks on one GPU (gloo all-reduces CUDA tensors through the host)."""
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
    from tests.util import load_golden, rel_err
    g = load_golden("case_c1")
    sim_num = 25                                   # odd split: 12 + 13 columns

    def fit(rng_mode):
        np.random.seed(17)
        return S.REML(S.SparseCholesky(rng=rng_mode, seed=2024), g.mats("k3"), g["cov"], g["y"].copy(),
                      sim_num=sim_num, aireml=True)

    sharded = {m: fit(m) for m in ("numpy", "device")}
    real = sharding.active_group
    sharding.active_group = lambda: None           # same process, collectives bypassed: the 1-rank computation
    try:
        single = {m: fit(m) for m in ("numpy", "device")}
    finally:
        sharding.active_group = real
    for m in ("numpy", "device"):
        assert sharded[m]["aireml"]["converged"], (m, sharded[m]["aireml"])
        assert sharded[m]["aireml"] == single[m]["aireml"], (m, sharded[m]["aireml"], single[m]["aireml"])
        for key in ("covariance coefficients", "covariates coefficients", "covariance std"):
            assert rel_err(sharded[m][key], single[m][key]) < 1e-9, (m, key, sharded[m][key], single[m][key])
        # every rank took the same steps
        t = torch.tensor(list(sharded[m]["covariance coefficients"]), dtype=torch.float64, device="cuda")
        lo, hi = t.clone(), t.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert torch.equal(lo, hi), (m, lo, hi)
    dist.barrier()
    if rank == 0:
        print("TWO_RANK_AIREML_OK", {m: (sharded[m]["covariance coefficients"], sharded[m]["aireml"])
                                     for m in sharded})
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
