"""Predicted random effects at the 250K config (one B200): phases of blup() with a seeded 20 % of the phenotypes masked.
K = 3 (A, A∘A and the residual identity), 11 covariates.  Records the host cut of the phenotyped blocks, the session
set-up with and without a cached analysis, the factorization, the (c+1)-column solve, slmm_blup_spmm per pattern group
(CUDA-event medians next to its HBM byte count), the PEV at 128 and 1024 probes split into backward half-sweeps and
rowsumsq passes (CUDA events per block), and whole blup() calls by wall clock.  Prints one JSON record.
usage: python scripts/blup_predict.py [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--individuals", type=int, default=250000)
    ap.add_argument("--masked", type=float, default=0.2)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from assoc_scan import gpu_info
    from scilmm_b200 import engine as E
    from scilmm_b200 import pedigree as Ped
    import scilmm_b200.SparseCholesky  # noqa: F401
    S = sys.modules["scilmm_b200.SparseCholesky"]
    assert torch.cuda.is_available(), "this script measures on the GPU"
    torch.cuda.set_device(0)
    info = gpu_info()

    A, _, cov, y, cfg = bench.make_inputs(args.individuals, 1e-3, 10)
    N = A.shape[0]
    mats = [A, Ped.epistasis(A)]
    sig = np.array([0.3, 0.15, 0.55])
    y = y.copy()
    y[np.random.default_rng(2024).random(N) < args.masked] = np.nan
    obs = ~np.isnan(y)
    idx = np.flatnonzero(obs)
    n = idx.size
    scale = y[obs].std()

    def events(fn, reps):
        """Median / min / max ms of fn() between CUDA events, after 2 warm-up calls."""
        out = []
        for r in range(2 + reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            if r >= 2:
                out.append(a.elapsed_time(b))
        return [round(float(np.median(out)), 4), round(float(np.min(out)), 4), round(float(np.max(out)), 4)]

    rec = {"script": "scripts/blup_predict.py",
           "config": {"individuals": args.individuals, "N": N, "n_phenotyped": n, "masked": args.masked,
                      "nnz_A": int(A.nnz), "K": 3, "ncov": cov.shape[1], "sigmas": sig.tolist()},
           "gpu": info, "device": torch.cuda.get_device_name(0),
           "timing": "host phases by wall clock; device phases by CUDA events, median/min/max of %d after 2 warm-up "
                     "calls unless stated" % args.reps}

    # host cut of the phenotyped blocks
    t0 = time.time()
    sub = [E.canonical_csr(m)[idx][:, idx] for m in mats]
    rec["host_subblock_cut_s"] = round(time.time() - t0, 3)

    # session set-up on the cut blocks: new analysis, then the cached one (the functor keeps its engines by pattern)
    chol = S.SparseCholesky(rng="device", seed=7)
    ys = y[idx] / scale
    torch.cuda.synchronize()
    t0 = time.time()
    ses = S._scan_session(chol, sub, cov[idx], ys)
    torch.cuda.synchronize()
    rec["session_setup_new_analysis_s"] = round(time.time() - t0, 3)
    rec["session_timings_new_analysis"] = {k: round(v, 3) for k, v in ses.timings.items()}
    chol.invalidate()
    del ses
    sub = [E.canonical_csr(m)[idx][:, idx] for m in mats]
    torch.cuda.synchronize()
    t0 = time.time()
    ses = S._scan_session(chol, sub, cov[idx], ys)
    torch.cuda.synchronize()
    rec["session_setup_cached_analysis_s"] = round(time.time() - t0, 3)
    rec["session_timings_cached_analysis"] = {k: round(v, 3) for k, v in ses.timings.items()}

    reps = args.reps
    rec["factorization_ms"] = events(lambda: ses.factor_at(sig), reps)
    ses.factor_at(sig)
    rec["fixed_effect_solve_ms"] = events(lambda: ses.fixed_effects(), reps)

    # slmm_blup_spmm on [u | V^-1 C] per pattern group of the full-N matrices
    t0 = time.time()
    ms = E.MatSet(mats)
    torch.cuda.synchronize()
    rec["full_matset_upload_s"] = round(time.time() - t0, 3)
    colmap = np.full(N, -1, dtype=np.int32)
    colmap[idx] = np.arange(n, dtype=np.int32)
    cm = E.to_device(colmap, torch)
    ViC, _, _, _, u = ses.fixed_effects()
    X = torch.cat([u.unsqueeze(1), ViC], dim=1).contiguous()
    spmm = {}
    for ks in ms.pattern_groups(2):
        G = len(ks)
        nnz = ms.nnz[ks[0]]
        for ncols in (1, X.shape[1]):
            Xc = X[:, :ncols].contiguous()
            t = events(lambda: ms.blup_spmm(ks, sig[ks], Xc, cm), reps)
            hbm = 4 * (N + 1) + 8 * nnz + 8 * nnz * G + 8 * n * ncols
            out_b = 8 * N * ncols * G
            spmm["ks=%s,ncols=%d" % (ks, ncols)] = {
                "ms": t, "hbm_bytes": hbm, "out_bytes": out_b,
                "GB_per_s_at_median": round((hbm + out_b) / (t[0] * 1e-3) / 1e9, 1)}
    rec["blup_spmm"] = spmm

    # the PEV passes: one 128-column probe block = Philox draw + backward half-sweep (mode 3), then rowsumsq
    groups = ms.pattern_groups(2)
    Wb = ses.eng.solve_(ses.eng.probe_normals(n, S.BLUP_BLOCK, 0, 7, S.BLUP_PROBE_STREAM), mode=3)
    sums = [(torch.empty(N, len(ks), dtype=torch.float64, device="cuda"),
             torch.empty(N, len(ks), dtype=torch.float64, device="cuda")) for ks in groups]
    rec["probe_block_sweep_ms"] = events(
        lambda: ses.eng.solve_(ses.eng.probe_normals(n, S.BLUP_BLOCK, 0, 7, S.BLUP_PROBE_STREAM), mode=3), reps)
    rows = {}
    for ks, (s2, s4) in zip(groups, sums):
        nnz = ms.nnz[ks[0]]
        t = events(lambda: ms.blup_rowsumsq(ks, sig[ks], Wb, s2, s4, cm), reps)
        gather = 8 * S.BLUP_BLOCK * nnz
        rows["ks=%s" % ks] = {"ms": t, "nnz": nnz, "gathered_W_bytes": gather, "W_bytes": 8 * n * S.BLUP_BLOCK,
                              "gathered_GB_per_s_at_median": round(gather / (t[0] * 1e-3) / 1e9, 1)}
    rec["rowsumsq_per_block"] = rows

    # PEV split into sweeps and rowsumsq over all blocks of one call, and whole blup() calls by wall clock
    pev = {}
    for p in (128, 1024):
        sweep, rsq = [], []
        for b in range(-(-p // S.BLUP_BLOCK)):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
            W = ses.eng.solve_(ses.eng.probe_normals(n, S.BLUP_BLOCK, b * S.BLUP_BLOCK, 7, S.BLUP_PROBE_STREAM),
                               mode=3)
            e[1].record()
            for ks, (s2, s4) in zip(groups, sums):
                ms.blup_rowsumsq(ks, sig[ks], W, s2, s4, cm)
            e[2].record()
            torch.cuda.synchronize()
            sweep.append(e[0].elapsed_time(e[1]))
            rsq.append(e[1].elapsed_time(e[2]))
        pev[str(p)] = {"sweeps_ms": round(float(np.sum(sweep)), 3), "rowsumsq_ms": round(float(np.sum(rsq)), 3),
                       "blocks": len(sweep)}
    rec["pev_device_phases"] = pev
    del Wb, W, sums, ms
    torch.cuda.empty_cache()

    calls = {}
    for p in (0, 128, 1024):
        walls = []
        for r in range(3):
            torch.cuda.synchronize()
            t0 = time.time()
            out = S.blup(chol, mats, cov, y, sig, pev_probes=p)
            torch.cuda.synchronize()
            walls.append(time.time() - t0)
        calls["masked_p%d" % p] = [round(w, 3) for w in walls]
        if p == 1024:
            ok = out["pev_se"] > 0
            rec["pev_relative_se_median_p1024"] = [round(float(np.median(out["pev_se"][ok[:, k], k] / out["pev"][ok[:, k], k])), 5)
                                                   for k in range(2)]
            rec["reliability_median_p1024"] = {
                "phenotyped": [round(float(np.median(out["reliability"][obs, k])), 4) for k in range(2)],
                "unphenotyped": [round(float(np.median(out["reliability"][~obs, k])), 4) for k in range(2)]}
    # in-sample: the session of a fit on all N individuals
    yall = np.where(obs, y, np.nanmean(y))
    chol2 = S.SparseCholesky(rng="device", seed=7)
    S.blup(chol2, mats, cov, yall, sig)
    walls = []
    for r in range(3):
        torch.cuda.synchronize()
        t0 = time.time()
        S.blup(chol2, mats, cov, yall, sig)
        torch.cuda.synchronize()
        walls.append(time.time() - t0)
    calls["in_sample_p0_session_reused"] = [round(w, 3) for w in walls]
    rec["blup_call_wall_s"] = calls
    rec["blup_call_note"] = ("masked calls cut the blocks on the host and set up a session on them each time (cached "
                             "analysis); the first masked p=0 call follows the measurements above on the same functor")
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
