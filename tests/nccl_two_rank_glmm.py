"""Launched by tests/test_gpu_glmm.py::test_two_rank_fit_and_scan under torchrun (2 ranks): every rank runs the PQL
fit (probe columns sharded) and the saddlepoint-calibrated scan (variants of both phases sharded, one all-reduce) with
the process group active, then both unsharded with the collective layer bypassed, and asserts that they agree to 1e-12
and that both ranks hold the same tau bit for bit.  Prints TWO_RANK_GLMM_OK on rank 0.  SLMM_TWO_RANK_BACKEND=gloo
runs the same check with both ranks on one GPU."""
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
    from tests.test_gpu_glmm import binary, rare_genotypes
    from tests.util import load_golden, rel_err
    g = load_golden("case_c1")
    y = binary(g, 0.1)
    mats = [g.csr("A")]
    G = np.asfortranarray(rare_genotypes(g.n, 101, 41))      # odd split: 50 + 51 variants
    sim_num = 25                                             # odd split: 12 + 13 probe columns

    def run():
        chol = S.SparseCholesky(rng="device", seed=11)
        fit = S.glmm(chol, mats, g["cov"], y, sim_num=sim_num)
        return fit, S.glmm_association(chol, mats, g["cov"], y, fit, G, spa_cutoff=1.0)

    sharded = run()
    real = sharding.active_group
    sharding.active_group = lambda: None           # same process, collectives bypassed: the 1-rank computation
    try:
        single = run()
    finally:
        sharding.active_group = real
    assert sharded[0]["glmm"] == single[0]["glmm"] and sharded[0]["glmm"]["converged"], sharded[0]["glmm"]
    for key in ("covariance coefficients", "covariates coefficients", "covariance std", "covariates std", "mu"):
        assert rel_err(sharded[0][key], single[0][key]) < 1e-12, (key, sharded[0][key], single[0][key])
    a, b = sharded[1], single[1]
    assert np.array_equal(a["spa"], b["spa"]) and a["spa"].dtype == np.int8 and (a["spa"] == 1).any()
    assert np.array_equal(a["n_obs"], b["n_obs"]) and a["n_obs"].dtype == np.int64
    for k in ("beta", "se", "score", "chi2", "p", "p_normal", "af"):
        fin = np.isfinite(b[k])
        assert np.array_equal(np.isfinite(a[k]), fin), k
        assert rel_err(a[k][fin], b[k][fin]) <= 1e-12, (k, rel_err(a[k][fin], b[k][fin]))
    t = torch.tensor(list(sharded[0]["covariance coefficients"]), dtype=torch.float64, device="cuda")
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    assert torch.equal(lo, hi), (lo, hi)
    dist.barrier()
    if rank == 0:
        print("TWO_RANK_GLMM_OK", sharded[0]["covariance coefficients"], sharded[0]["glmm"],
              int((a["spa"] == 1).sum()), "saddlepoint p of", G.shape[1])
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
