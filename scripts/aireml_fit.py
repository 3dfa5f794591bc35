"""AI-REML against L-BFGS-B on the flagship configuration (BASELINE.json config 3: 250,000 simulated individuals,
K = 3: IBD A, A o A, I; 10 covariates + intercept; 128 probes, rng='device'), in one process on one GPU:

  * both whole REML() fits through the public API with fresh functors (setup included): wall time, setup,
    evaluations / iterations, sigma, standard errors, and max |delta sigma| / SE between the two;
  * the Monte-Carlo spread of the AI-REML estimate: --spread more AI-REML fits on the same session with other probe
    blocks, each with its distance to the L-BFGS-B estimate in SE units and the exact REML nll at its estimate (the
    nll does not depend on the probes, so it ranks the estimates);
  * the cost of evaluate(ai=True) against evaluate() at the AI-REML estimate, the two alternated in one loop
    (host clock around work that ends in a device synchronise), and compute_hess for scale.

A small fit on the golden pedigree runs first, so that neither timed fit pays for the CUDA context or the pinned
upload ring.  Prints the card name and power limit and the record as one JSON line; --out also writes it to a file.
    python scripts/aireml_fit.py [--individuals 250000] [--reps 20] [--out results/aireml_fit.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [v.strip() for v in q.split(",")][:2]
    except Exception as e:          # the record says so rather than guessing
        info["power_limit"] = "unavailable (%s)" % type(e).__name__
    return info


def fit(S, mats, cov, y, sim_num, aireml):
    import torch
    chol = S.SparseCholesky(rng="device", seed=777)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = S.REML(chol, mats, cov, y, reml=True, sim_num=sim_num, verbose=False, aireml=aireml)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ses = next(iter(chol._sessions.values()))
    rec = {"wall_s": round(wall, 3), "setup_s": round(ses.setup_s, 3), "evaluations": int(ses.n_eval),
           "sigma2": [float(v) for v in out["covariance coefficients"]],
           "se": [float(v) for v in out["covariance std"]], "nll": float(out["nll"])}
    if aireml:
        rec["aireml"] = out["aireml"]
    return rec, chol, ses


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--individuals", type=int, default=250000)
    ap.add_argument("--sf", type=float, default=1e-3)
    ap.add_argument("--ncov", type=int, default=10)
    ap.add_argument("--sim-num", type=int, default=128)
    ap.add_argument("--reps", type=int, default=20, help="alternated evaluate() / evaluate(ai=True) pairs")
    ap.add_argument("--spread", type=int, default=4, help="extra AI-REML fits with other probe blocks")
    ap.add_argument("--out", default=None, help="also write the JSON record to this file")
    args = ap.parse_args()

    import torch
    import bench
    import scilmm_b200.SparseCholesky  # noqa: F401
    from tests.util import load_golden
    S = sys.modules["scilmm_b200.SparseCholesky"]
    from scilmm_b200 import pedigree as P
    if not torch.cuda.is_available():
        raise SystemExit("aireml_fit.py measures on a CUDA device; none found")
    rec = {"card": card(), "config": {"individuals": args.individuals, "sf": args.sf, "ncov": args.ncov,
                                      "sim_num": args.sim_num, "K": 3, "rng": "device"}}
    print("card:", rec["card"], flush=True)

    g = load_golden("case_small")                     # warm-up: context, pinned ring, module loads
    for aireml in (False, True):
        S.REML(S.SparseCholesky(rng="device"), g.mats("k1"), g["cov"], g["y"].copy(), sim_num=8, aireml=aireml)

    A, _, cov, y, info = bench.make_inputs(args.individuals, args.sf, args.ncov)
    rec["config"].update(n=info["n"], nnz_A=info["nnz"])
    base = [A, P.epistasis(A)]

    lbfgs, chol, ses = fit(S, base, cov, y, args.sim_num, aireml=False)
    print("L-BFGS-B fit:", lbfgs, flush=True)
    del chol, ses
    ai, chol, ses = fit(S, base, cov, y, args.sim_num, aireml=True)
    print("AI-REML fit:", ai, flush=True)
    se = np.asarray(lbfgs["se"])
    diff = np.abs(np.asarray(ai["sigma2"]) - np.asarray(lbfgs["sigma2"])) / se
    rec.update(lbfgs=lbfgs, aireml=ai, max_abs_diff_over_se=float(diff.max()), diff_over_se=diff.tolist(),
               speedup_wall=round(lbfgs["wall_s"] / ai["wall_s"], 3))

    # Monte-Carlo spread: the same session (y standardised as REML() does), other probe streams
    import scipy.sparse as sp
    mats = ses._refs[0]
    ys = ses._refs[2]
    assert len(mats) == 3 and sp.issparse(mats[2])
    sl, sa = np.asarray(lbfgs["sigma2"]), np.asarray(ai["sigma2"])
    spread = []
    for r in range(args.spread):
        chol.seed = 1000 + r
        s_r, info_r = S._aireml_fit(chol, mats, cov, ys, True, args.sim_num, False)
        spread.append({"sigma2": s_r.tolist(), "iterations": info_r["iterations"],
                       "max_abs_diff_vs_lbfgs_over_se": float(np.max(np.abs(s_r - sl) / se)),
                       "max_abs_diff_vs_first_aireml_over_se": float(np.max(np.abs(s_r - sa) / se)),
                       "nll": float(ses.evaluate(s_r, True, 8, probe_stream=0)[0])})
        print("AI-REML fit, probe seed %d:" % chol.seed, spread[-1], flush=True)
    rec["aireml_spread"] = spread
    rec["nll_at_estimate"] = {"lbfgs": float(ses.evaluate(sl, True, 8, probe_stream=0)[0]),
                              "aireml": float(ses.evaluate(sa, True, 8, probe_stream=0)[0])}

    # evaluate() vs evaluate(ai=True) at the AI-REML estimate, alternated; same probe stream for both
    sig = np.asarray(ai["sigma2"])
    stream = ses.n_eval
    times = {"plain": [], "ai": []}

    def one(with_ai):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ses.evaluate(sig, True, args.sim_num, ai=with_ai, probe_stream=stream)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3
    for _ in range(2):                                # warm-up of both shapes
        one(False), one(True)
    for r in range(args.reps):
        order = (False, True) if r % 2 == 0 else (True, False)
        for with_ai in order:
            times["ai" if with_ai else "plain"].append(one(with_ai))
    nll0, grad0 = ses.evaluate(sig, True, args.sim_num, probe_stream=stream)
    nll1, grad1, AI = ses.evaluate(sig, True, args.sim_num, ai=True, probe_stream=stream)
    factor = ses.factor_at(sig)
    hess_ms = []
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        H = S._hess_device(ses, factor._chol)
        torch.cuda.synchronize()
        hess_ms.append((time.perf_counter() - t0) * 1e3)
    med = {k: float(np.median(v)) for k, v in times.items()}
    rec["evaluate_ms"] = {"plain_median": round(med["plain"], 3), "ai_median": round(med["ai"], 3),
                          "added_median": round(med["ai"] - med["plain"], 3),
                          "plain_min": round(min(times["plain"]), 3), "ai_min": round(min(times["ai"]), 3),
                          "reps": args.reps, "plain_all": [round(v, 3) for v in times["plain"]],
                          "ai_all": [round(v, 3) for v in times["ai"]]}
    rec["compute_hess_ms"] = {"median": round(float(np.median(hess_ms[1:])), 3), "all": [round(v, 3) for v in hess_ms]}
    rec["ai_check"] = {"same_nll_and_grad": bool(nll0 == nll1 and np.array_equal(grad0, grad1)),
                       "max_rel_diff_ai_vs_minus_hess": float(np.max(np.abs(AI + H)) / np.max(np.abs(H)))}
    print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
