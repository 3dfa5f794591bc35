"""The REML probe block two ways at the 250K config (one B200): the old composition solve_(lmul(Z)) split into L*Z,
the forward half (mode 1) and the backward half (mode 2), against one backward half-sweep from the factor's row order,
solve_(Z, mode=3) = P' L^-T Z.  Widths 128, 64, 32 and 16 (the local probe block at 1, 2, 4 and 8 GPUs), then
evaluate() and evaluate(ai=True), and the largest relative difference of W between the two formulations.

CUDA-event medians after warm-up; every timed solve starts from a fresh copy of its input (copied outside the timed
window).  Prints one JSON record.  usage: python scripts/probe_solve_ab.py [--reps 20] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--individuals", type=int, default=250000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--eval-reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from scilmm_b200 import pedigree as Ped
    import scilmm_b200.SparseCholesky  # noqa: F401
    S = sys.modules["scilmm_b200.SparseCholesky"]
    assert torch.cuda.is_available(), "this script measures on the GPU"
    torch.cuda.set_device(0)

    A, _, cov, y, info = bench.make_inputs(args.individuals, 1e-3, 10)
    n = A.shape[0]
    mats = [A, Ped.epistasis(A), sp.eye(n).tocsr()]
    sig = np.array([0.3, 0.15, 0.55])
    ses = S.SparseCholesky(rng="device", seed=12345)._session(mats, cov, y / y.std())
    eng = ses.eng
    ses.factor_at(sig)

    def median_ms(fn, prep=None, reps=args.reps, warm=3):
        times = []
        for i in range(warm + reps):
            arg = prep() if prep is not None else None
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn(arg)
            b.record()
            torch.cuda.synchronize()
            if i >= warm:
                times.append(a.elapsed_time(b))
        return round(float(np.median(times)), 3), round(float(np.min(times)), 3), round(float(np.max(times)), 3)

    widths = {}
    W_diff = None
    for k in (128, 64, 32, 16):
        Z = eng.probe_normals(n, k, 0, 12345, 1)
        work = torch.empty_like(Z)
        LZ = eng.lmul(Z)
        Y = eng.solve_(LZ.clone(), mode=1)

        def fresh(src):
            return lambda: work.copy_(src)
        rec = {
            "lmul_ms": median_ms(lambda _: eng.lmul(Z)),
            "mode1_ms": median_ms(lambda w: eng.solve_(w, mode=1), fresh(LZ)),
            "mode2_ms": median_ms(lambda w: eng.solve_(w, mode=2), fresh(Y)),
            "old_composition_ms": median_ms(lambda _: eng.solve_(eng.lmul(Z))),
            "mode3_ms": median_ms(lambda w: eng.solve_(w, mode=3), fresh(Z)),
        }
        rec["old_parts_sum_ms"] = round(rec["lmul_ms"][0] + rec["mode1_ms"][0] + rec["mode2_ms"][0], 3)
        rec["saved_ms"] = round(rec["old_composition_ms"][0] - rec["mode3_ms"][0], 3)
        W_old = eng.solve_(eng.lmul(Z))
        W_new = eng.solve_(Z.clone(), mode=3)
        rec["W_max_rel_diff"] = float((W_new - W_old).abs().max() / W_old.abs().max())
        if k == 128:
            W_diff = rec["W_max_rel_diff"]
        widths[str(k)] = rec
        del Z, work, LZ, Y, W_old, W_new

    for _ in range(3):
        ses.evaluate(sig, True, 128)
        ses.evaluate(sig, True, 128, ai=True)
    evaluate_ms = median_ms(lambda _: ses.evaluate(sig, True, 128), reps=args.eval_reps, warm=1)
    evaluate_ai_ms = median_ms(lambda _: ses.evaluate(sig, True, 128, ai=True), reps=args.eval_reps, warm=1)

    rec = {"script": "scripts/probe_solve_ab.py", "config": {"individuals": args.individuals, "n": n, "K": 3,
                                                             "ncov": 10, "sf": 1e-3, "rng": "device"},
           "gpu": gpu_info(), "device": torch.cuda.get_device_name(0),
           "timing": "CUDA-event [median, min, max] ms over %d reps after 3 warm-up; evaluate over %d"
                     % (args.reps, args.eval_reps),
           "widths": widths, "evaluate_ms": evaluate_ms, "evaluate_ai_ms": evaluate_ai_ms,
           "W_max_rel_diff_128": W_diff}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
