"""Binary-trait fit and scan at the 250K config (one B200): the trait of bench.make_inputs thresholded at prevalence
0.1 and 0.01, mats = [A] (K = 1; --epistasis adds A o A), 11 covariates with the intercept, the seeded int8 variants
of scripts/assoc_scan.py.  Per prevalence: glmm() wall time, iterations and time per PQL iteration; phase 1
(RemlSession.association on the fit's session) variants/s against association() on the same variants; the fraction of
variants flagged for the saddlepoint at |z| > 2; phase 2 time per flagged variant, its histogram of CGF passes (Newton
and bracket steps, both sides) and the saddlepoint kernel's achieved rate against its FP64 bound; one whole
glmm_association() call.  Prints one JSON record.
usage: python scripts/glmm_scan.py [--variants 50176] [--epistasis] [--out profiles/r08_glmm.json]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

# FP64 instructions (DFMA + DADD + DMUL) of the loop body of spa_cgf in the sm_100a SASS, every branch of expm1 / log1p
# counted: 55 DFMA, 21 DADD, 17 DMUL.  The bound below issues all of them at the DFMA rate of the data sheet.
SPA_FP64_INSTR_PER_ELEMENT = 93
B200_FP64_TFLOPS = 37.0          # data sheet, FP64 (one GPU of an HGX B200): 18.5 T DFMA/s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--individuals", type=int, default=250000)
    ap.add_argument("--variants", type=int, default=50176)
    ap.add_argument("--prevalences", default="0.1,0.01")
    ap.add_argument("--sim-num", type=int, default=100)
    ap.add_argument("--epistasis", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from assoc_scan import genotypes, gpu_info
    from scilmm_b200 import pedigree as Ped
    import scilmm_b200.SparseCholesky  # noqa: F401
    S = sys.modules["scilmm_b200.SparseCholesky"]
    assert torch.cuda.is_available(), "this script measures on the GPU"
    torch.cuda.set_device(0)
    info = gpu_info()

    A, _, cov, yq, cfg = bench.make_inputs(args.individuals, 1e-3, 10)
    n = A.shape[0]
    mats = [A, Ped.epistasis(A)] if args.epistasis else [A]
    G = genotypes(torch, n, args.variants, 7)
    m = G.shape[1]
    out = {}
    for prev in [float(v) for v in args.prevalences.split(",")]:
        y = (yq > np.quantile(yq, 1.0 - prev)).astype(np.float64)
        chol = S.SparseCholesky(rng="device", seed=12345)
        torch.cuda.synchronize()
        t0 = time.time()
        fit = S.glmm(chol, mats, cov, y, sim_num=args.sim_num)
        torch.cuda.synchronize()
        fit_s = time.time() - t0
        ses = chol._glmm
        sig = np.concatenate([fit["covariance coefficients"], [1.0]])
        block = S.ASSOC_BLOCK
        ses.association(sig, G, block, 0, 2 * block)                 # warm-up: solve plan, copy stream, scratch
        torch.cuda.synchronize()
        t0 = time.time()
        part = ses.association(sig, G, block)
        torch.cuda.synchronize()
        p1_s = time.time() - t0
        z = part["score"] / np.sqrt(part["var"])
        flag = np.flatnonzero(np.isfinite(z) & (np.abs(np.nan_to_num(z)) > 2.0))
        sblock = S._scan_width(n, S.SPA_BYTES_PER_ENTRY, 1)
        ses.spa(G, flag[:8], part["score"][flag[:8]], part["var"][flag[:8]], fit["mu"], fit["weights"], 8)  # warm-up
        timing = []
        torch.cuda.synchronize()
        t0 = time.time()
        ps, status, iters = ses.spa(G, flag, part["score"][flag], part["var"][flag], fit["mu"], fit["weights"], sblock,
                                    timing=timing)
        torch.cuda.synchronize()
        p2_s = time.time() - t0
        kernel_ms = float(sum(a.elapsed_time(b) for a, b in timing))
        passes = int(iters.sum())
        bound_ms = 1e3 * passes * n * SPA_FP64_INSTR_PER_ELEMENT / (B200_FP64_TFLOPS * 1e12 / 2)
        hist = np.bincount(iters)
        # association() on the same variants: the REML-type session of the same matrices with an identity
        torch.cuda.synchronize()
        t0 = time.time()
        S.association(S.SparseCholesky(rng="device", seed=1), mats, cov, y, np.full(len(mats) + 1, 0.5), G)
        torch.cuda.synchronize()
        assoc_s = time.time() - t0
        torch.cuda.synchronize()
        t0 = time.time()
        res = S.glmm_association(chol, mats, cov, y, fit, G)
        torch.cuda.synchronize()
        whole_s = time.time() - t0
        out[str(prev)] = {
            "fit": {"wall_s": round(fit_s, 2), "iterations": fit["glmm"]["iterations"],
                    "converged": fit["glmm"]["converged"], "s_per_iteration": round(fit_s / fit["glmm"]["iterations"], 3),
                    "tau": fit["covariance coefficients"].tolist(), "tau_std": fit["covariance std"].tolist(),
                    "latent_fractions": fit["latent fractions"].tolist()},
            "phase1": {"wall_s": round(p1_s, 3), "variants_per_s": round(m / p1_s, 1),
                       "association_wall_s_incl_setup": round(assoc_s, 3),
                       "association_variants_per_s_incl_setup": round(m / assoc_s, 1)},
            "flagged": int(flag.size), "flagged_fraction": round(flag.size / m, 5),
            "phase2": {"wall_s": round(p2_s, 3), "block": sblock, "kernel_ms": round(kernel_ms, 2),
                       "ms_per_flagged_variant": round(1e3 * p2_s / max(flag.size, 1), 4),
                       "kernel_ms_per_flagged_variant": round(kernel_ms / max(flag.size, 1), 4),
                       "status_counts": {str(k): int(np.sum(status == k)) for k in (1, -1)},
                       "cgf_passes_histogram": {str(i): int(c) for i, c in enumerate(hist) if c},
                       "cgf_passes_total": passes,
                       "element_passes_per_s": round(passes * n / (kernel_ms * 1e-3), 1) if kernel_ms else None,
                       "fp64_bound_ms": round(bound_ms, 3),
                       "share_of_fp64_bound": round(bound_ms / kernel_ms, 4) if kernel_ms else None},
            "glmm_association_wall_s": round(whole_s, 3),
            "min_p": float(np.nanmin(res["p"])), "min_p_normal": float(np.nanmin(res["p_normal"]))}
        print(json.dumps({str(prev): out[str(prev)]}), flush=True)
        del chol, ses
        torch.cuda.empty_cache()
    rec = {"script": "scripts/glmm_scan.py",
           "config": {"individuals": args.individuals, "n": n, "K": len(mats), "ncov": 11, "sf": 1e-3, "variants": m,
                      "sim_num": args.sim_num, "spa_cutoff": 2.0, "missing": 0.01, "allele_freq": [0.05, 0.5]},
           "gpu": info, "device": torch.cuda.get_device_name(0),
           "timing": "wall clock around whole calls ending in a device synchronise; phase 1 after a 2-block warm-up; "
                     "saddlepoint kernel time from CUDA events around each launch",
           "fp64_bound": "passes x n x %d FP64 instructions (SASS of the CGF loop) at %.1f TFLOP/s / 2 (data sheet)"
                         % (SPA_FP64_INSTR_PER_ELEMENT, B200_FP64_TFLOPS),
           "prevalence": out}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
