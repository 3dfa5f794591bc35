"""Association scan at the 250K config (one B200): variants/s of RemlSession.association at block widths 128, 256 and
512 over a seeded int8 genotype matrix (Fortran order, per-variant allele frequencies 0.05-0.5, 1 % missing), per-block
CUDA-event medians of the pipeline's phases (upload wait, genotype kernel, forward half-sweep, sum of squares), the
device memory a width holds, against the same-width solve_(., mode=1) alone, the same scan from a C-ordered
copy of the first variants, and the largest relative difference of beta on the first block against a device full
solve (mode 0).  Prints one JSON record.  usage: python scripts/assoc_scan.py [--variants 50176] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.linalg as la
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [s.strip() for s in out.strip().split(",")]))
    except (OSError, subprocess.SubprocessError):
        return {}


def genotypes(torch, n, m, seed, missing=0.01, chunk=1024):
    """(n, m) Fortran-ordered int8 host matrix drawn on the device chunk by chunk: binomial(2, p_j) with p_j uniform in
    0.05-0.5, `missing` of the entries -1."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    G = np.empty((m, n), dtype=np.int8)           # G.T is the Fortran-ordered (n, m) matrix
    for j0 in range(0, m, chunk):
        j1 = min(m, j0 + chunk)
        p = 0.05 + 0.45 * torch.rand(j1 - j0, 1, generator=g, device="cuda", dtype=torch.float64)
        a = (torch.rand(j1 - j0, n, generator=g, device="cuda", dtype=torch.float64) < p).to(torch.int8)
        b = (torch.rand(j1 - j0, n, generator=g, device="cuda", dtype=torch.float64) < p).to(torch.int8)
        x = a + b
        x[torch.rand(j1 - j0, n, generator=g, device="cuda") < missing] = -1
        G[j0:j1] = x.cpu().numpy()
    return G.T


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--individuals", type=int, default=250000)
    ap.add_argument("--variants", type=int, default=50176)
    ap.add_argument("--widths", default="128,256,512")
    ap.add_argument("--c-order-variants", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
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
    eng = ses.eng
    t0 = time.time()
    G = genotypes(torch, n, args.variants, 7)
    gen_s = time.time() - t0
    m = G.shape[1]

    def ms(a, b):
        return a.elapsed_time(b)

    widths = {}
    first_block = None
    for w in [int(v) for v in args.widths.split(",")]:
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        ses.association(sig, G, w, 0, 2 * w)                     # warm-up: solve plan, copy stream, scratch
        torch.cuda.synchronize()
        timing = []
        t0 = time.time()
        res = ses.association(sig, G, w, timing=timing)
        torch.cuda.synchronize()
        wall = time.time() - t0
        held = free0 - torch.cuda.mem_get_info()[0]              # solve plan of width w + the scan's buffers (cached)
        full = [t for t in timing[1:-1]]                         # whole blocks in steady state
        phase = np.array([[ms(t[0], t[1]), ms(t[1], t[2]), ms(t[2], t[3]), ms(t[3], t[4]), ms(t[0], t[4])]
                          for t in full])
        blocks_ms = [ms(timing[i][0], timing[i + 1][0]) for i in range(1, len(timing) - 1)]
        X = torch.empty(n, w, dtype=torch.float64, device="cuda")
        X.normal_()
        Xw = torch.empty_like(X)
        solo = []
        for r in range(3 + args.reps):
            Xw.copy_(X)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            eng.solve_(Xw, mode=1)
            b.record()
            torch.cuda.synchronize()
            if r >= 3:
                solo.append(a.elapsed_time(b))
        med = np.median(phase, axis=0)
        rec = {"variants": m, "wall_s": round(wall, 3), "variants_per_s": round(m / wall, 1),
               "block_ms_median": round(float(np.median(blocks_ms)), 3),
               "phase_ms_median": {"upload_wait": round(float(med[0]), 4), "genotype_kernel": round(float(med[1]), 4),
                                   "sweep": round(float(med[2]), 3), "sumsq": round(float(med[3]), 4),
                                   "first_to_last_event": round(float(med[4]), 3)},
               "device_bytes_held": int(held), "device_bytes_per_entry": round(held / (n * w), 2),
               "solve_mode1_alone_ms": [round(float(np.median(solo)), 3), round(float(np.min(solo)), 3),
                                        round(float(np.max(solo)), 3)],
               "nan_variants": int(np.sum(~np.isfinite(res["beta"])))}
        rec["block_over_sweep_alone"] = round(rec["block_ms_median"] / rec["solve_mode1_alone_ms"][0], 4)
        widths[str(w)] = rec
        if first_block is None:
            first_block = (w, res)
        del X, Xw
        torch.cuda.empty_cache()

    # first block against a device full solve: gamma = t / (x'V^-1 x - q' M^-1 q) with V^-1 x from mode 0
    w, res = first_block
    ViC, chol, beta, Viy = ses.fixed_effects()
    Vir = Viy - ViC @ torch.from_numpy(beta).to("cuda")
    P = torch.cat([ViC, Vir.unsqueeze(1)], dim=1).contiguous()
    g8 = torch.empty(n * w, dtype=torch.int8, device="cuda")
    strides = E.upload_genotype_block(G, 0, w, g8)
    Xt = torch.empty(n, w, dtype=torch.float64, device="cuda")
    proj = torch.empty(P.shape[1] * w, dtype=torch.float64, device="cuda")
    nobs, gsum = (torch.empty(w, dtype=torch.int64, device="cuda") for _ in range(2))
    E.assoc_genotypes(g8, n, w, strides, P, Xt, proj, nobs, gsum)
    xVx = (Xt * eng.solve_(Xt.clone(), mode=0)).sum(dim=0).cpu().numpy()
    proj = proj.view(P.shape[1], w).cpu().numpy()
    q, t = proj[:-1], proj[-1]
    gamma = t / (xVx - np.sum(q * la.cho_solve(chol, q), axis=0))
    fin = np.isfinite(res["beta"][:w])
    beta_rel = float(np.max(np.abs(res["beta"][:w][fin] - gamma[fin]) / np.abs(gamma[fin])))

    # the same scan from a C-ordered host matrix (pitched DMA of n rows x width bytes)
    Gc = np.ascontiguousarray(G[:, :args.c_order_variants])
    wc = 256
    ses.association(sig, Gc, wc, 0, 2 * wc)
    torch.cuda.synchronize()
    t0 = time.time()
    res_c = ses.association(sig, Gc, wc)
    torch.cuda.synchronize()
    wall_c = time.time() - t0
    ref = res["beta"][:Gc.shape[1]]
    fin = np.isfinite(ref)
    c_vs_f = float(np.max(np.abs(res_c["beta"][fin] - ref[fin])) / np.max(np.abs(ref[fin])))
    same_nan = bool(np.array_equal(np.isfinite(res_c["beta"]), fin))

    rec = {"script": "scripts/assoc_scan.py",
           "config": {"individuals": args.individuals, "n": n, "K": 3, "ncov": 10, "sf": 1e-3, "sigmas": sig.tolist(),
                      "variants": m, "missing": 0.01, "allele_freq": [0.05, 0.5], "order": "F"},
           "gpu": info, "device": torch.cuda.get_device_name(0),
           "timing": "wall clock of whole scans after a 2-block warm-up per width; per-block phases are CUDA-event "
                     "medians over the steady-state blocks; solve alone: median/min/max of %d after 3 warm-up"
                     % args.reps,
           "genotype_generation_s": round(gen_s, 1), "widths": widths,
           "first_block_beta_max_rel_diff_vs_full_solve": beta_rel, "first_block_width": w,
           "c_order": {"variants": int(Gc.shape[1]), "width": wc, "wall_s": round(wall_c, 3),
                       "variants_per_s": round(Gc.shape[1] / wall_c, 1), "same_nan_pattern": same_nan,
                       "beta_max_rel_diff_vs_F_order": c_vs_f}}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
