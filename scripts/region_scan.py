"""Region tests at the 250K config (one B200): regions/s and variants/s of RemlSession.region_test over the seeded
50 176-variant genotype matrix of scripts/assoc_scan.py in two groupings, (a) gene-like regions with geometric sizes of
mean 25 capped at 512 and (b) 512-wide regions; per-block CUDA-event medians of the pipeline's phases against the
same-width solve_(., mode=1) alone; the host time of each block's finish (median, max) and of its per-region
statistics; and the region Gram kernel (slmm_assoc_region_gram) alone on a 512-column block against its flop and byte
bounds.  Prints one JSON record.
usage: python scripts/region_scan.py [--variants 50176] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

DGEMM_TFLOPS = 35.4      # cuBLAS DGEMM on one B200 (DESIGN.md 6)
HBM_TBS = 7.7            # HGX B200 data sheet, one GPU


def groupings(m, seed=3):
    rng = np.random.default_rng(seed)
    sizes = []
    while sum(sizes) < m:
        sizes.append(int(min(512, rng.geometric(1.0 / 25))))
    sizes[-1] -= sum(sizes) - m
    if sizes[-1] == 0:
        sizes.pop()
    gene = np.concatenate([[0], np.cumsum(sizes)])
    wide = np.concatenate([np.arange(0, m, 512), [m]])
    return {"a_gene_like": gene, "b_512_wide": wide}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--individuals", type=int, default=250000)
    ap.add_argument("--variants", type=int, default=50176)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from assoc_scan import genotypes, gpu_info
    from scilmm_b200 import engine as E
    from scilmm_b200 import pedigree as Ped
    import scilmm_b200.SparseCholesky  # noqa: F401
    S = sys.modules["scilmm_b200.SparseCholesky"]
    assert torch.cuda.is_available(), "this script measures on the GPU"
    torch.cuda.set_device(0)
    info = gpu_info()

    A, _, cov, y, cfg = bench.make_inputs(args.individuals, 1e-3, 10)
    n = A.shape[0]
    mats = [A, Ped.epistasis(A), sp.eye(n).tocsr()]
    sig = np.array([0.3, 0.15, 0.55])
    ses = S.SparseCholesky(rng="device", seed=12345)._session(mats, cov, y / y.std())
    G = genotypes(torch, n, args.variants, 7)
    m = G.shape[1]
    block = S.ASSOC_BLOCK

    host_s = [0.0]
    stats_fn = S.region_statistics

    def timed_stats(*a):
        t0 = time.perf_counter()
        try:
            return stats_fn(*a)
        finally:
            host_s[0] += time.perf_counter() - t0

    def ms(a, b):
        return a.elapsed_time(b)

    # the sweep alone at the block width, on the factor of V at sig
    ses.factor_at(sig)
    X = torch.empty(n, block, dtype=torch.float64, device="cuda")
    X.normal_()
    Xw = torch.empty_like(X)
    solo = []
    for r in range(3 + args.reps):
        Xw.copy_(X)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        ses.eng.solve_(Xw, mode=1)
        b.record()
        torch.cuda.synchronize()
        if r >= 3:
            solo.append(a.elapsed_time(b))
    sweep_ms = float(np.median(solo))

    runs = {}
    for name, bounds in groupings(m).items():
        R = bounds.size - 1
        warm = int(np.searchsorted(bounds, 2 * block, side="right")) - 1
        ses.region_test(sig, G, bounds, None, block, 0, max(warm, 1))      # warm-up: plans, copy stream, scratch
        torch.cuda.synchronize()
        S.region_statistics = timed_stats
        host_s[0] = 0.0
        timing = []
        t0 = time.time()
        try:
            res = ses.region_test(sig, G, bounds, None, block, timing=timing)
            torch.cuda.synchronize()
        finally:
            S.region_statistics = stats_fn
        wall = time.time() - t0
        full = timing[1:-1]
        phase = np.median(np.array([[ms(t[0], t[1]), ms(t[1], t[2]), ms(t[2], t[3]), ms(t[3], t[4])] for t in full]),
                          axis=0)
        blocks_ms = [ms(timing[i][0], timing[i + 1][0]) for i in range(1, len(timing) - 1)]
        nblocks = len(timing)
        widths = np.diff(bounds)
        runs[name] = {
            "regions": int(R), "blocks": nblocks, "region_size_mean": round(float(widths.mean()), 2),
            "region_size_max": int(widths.max()), "wall_s": round(wall, 3),
            "variants_per_s": round(m / wall, 1), "regions_per_s": round(R / wall, 1),
            "block_ms_median": round(float(np.median(blocks_ms)), 3),
            "block_over_sweep_alone": round(float(np.median(blocks_ms)) / sweep_ms, 4),
            "phase_ms_median": {"upload_wait": round(float(phase[0]), 4), "genotype_kernel": round(float(phase[1]), 4),
                                "sweep": round(float(phase[2]), 3), "region_gram": round(float(phase[3]), 4)},
            "host_statistics_ms_per_block": round(1e3 * host_s[0] / nblocks, 3),
            "host_finish_ms_per_block": [round(1e3 * float(np.median(ses.last["finish_s"])), 3),
                                         round(1e3 * float(np.max(ses.last["finish_s"])), 3)],
            "nan_burden": int(np.sum(~np.isfinite(res["burden_p"]))),
            "nan_skat": int(np.sum(~np.isfinite(res["skat_p"]))),
            "min_burden_p": float(np.nanmin(res["burden_p"])), "min_skat_p": float(np.nanmin(res["skat_p"]))}

    # the region Gram alone on one 512-column block.  F (0.83 GB at 202K) is far larger than L2, so the byte bound is
    # F read once from HBM; the tiles of one row chunk re-read its strips (bytes_strip_reads), mostly from L2
    kern = {}
    gene = groupings(m)["a_gene_like"]
    first = gene[:int(np.searchsorted(gene, block, side="right"))]
    cases = {"gene_like_first_block": np.r_[first, block] if first[-1] != block else first,
             "one_512_region": np.array([0, block])}
    for name, bounds in cases.items():
        w = np.diff(bounds)
        jmin = np.arange(block // 64)            # strip I pairs with strips jmin[I]..I (as slmm_assoc_region_gram)
        for r in range(w.size):
            for s in range(bounds[r] // 64, (bounds[r + 1] - 1) // 64 + 1):
                jmin[s] = min(jmin[s], bounds[r] // 64)
        ntiles = int(np.sum(np.arange(block // 64) - jmin + 1))
        strip_reads = 2 * ntiles - block // 64   # a diagonal tile reads one strip, an off-diagonal tile two
        out = torch.empty(int(np.sum(w.astype(np.int64) ** 2)), dtype=torch.float64, device="cuda")
        for _ in range(3):
            E.assoc_region_gram(X, bounds, out)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.reps)]
        torch.cuda.synchronize()
        for r in range(args.reps):
            ev[2 * r].record()
            E.assoc_region_gram(X, bounds, out)
            ev[2 * r + 1].record()
        torch.cuda.synchronize()
        t = np.array([ms(ev[2 * r], ev[2 * r + 1]) for r in range(args.reps)])
        flop = 2.0 * n * 64 * 64 * ntiles
        byts = 8.0 * n * block
        t_flop, t_byte = flop / (DGEMM_TFLOPS * 1e12) * 1e3, byts / (HBM_TBS * 1e12) * 1e3
        kern[name] = {"regions": int(w.size), "tiles": ntiles, "ms_median": round(float(np.median(t)), 4),
                      "ms_min": round(float(t.min()), 4), "ms_max": round(float(t.max()), 4),
                      "flop": flop, "bytes_F_once": byts, "bytes_strip_reads": 8.0 * n * 64 * strip_reads,
                      "tflops_achieved": round(flop / np.median(t) / 1e9, 2),
                      "flop_bound_ms_at_dgemm_rate": round(t_flop, 4), "byte_bound_ms_at_hbm_peak": round(t_byte, 4),
                      "bound_by": "flop" if t_flop > t_byte else "bytes",
                      "over_larger_bound": round(float(np.median(t)) / max(t_flop, t_byte), 3)}

    rec = {"script": "scripts/region_scan.py",
           "config": {"individuals": args.individuals, "n": n, "K": 3, "ncov": int(cov.shape[1]), "sf": 1e-3,
                      "sigmas": sig.tolist(), "variants": m, "block": block, "weights": "beta(maf; 1, 25)"},
           "gpu": info, "device": torch.cuda.get_device_name(0),
           "timing": "wall clock of whole calls after a 2-block warm-up per grouping; per-block phases are CUDA-event "
                     "medians over the steady-state blocks; sweep alone and the Gram kernel: medians of %d after 3 "
                     "warm-up; host statistics: perf_counter around the per-region statistics" % args.reps,
           "sweep_mode1_alone_ms": round(sweep_ms, 3), "groupings": runs, "region_gram_kernel": kern}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
