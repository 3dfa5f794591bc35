#!/usr/bin/env python
"""bench.py - headline benchmark of the SparseCholesky path on B200 (contract: one JSON line on rank 0).

Workload (BASELINE.json config 3): simulated pedigree of 250,000 individuals (sparsity_factor 1e-3,
gen_exp 1.4, init_keep_rate 0.8, seed 0) -> IBD A, epistasis A o A, identity; 10 covariates + intercept;
one "step" = one REML evaluation (`bolt_gradient_estimation`, reference scilmm/SparseCholesky.py:77-117):
V assembly, supernodal LL' factorization, logdet, c+1 deterministic solve columns, 128 Hutchinson probe
columns through L*Z + solve, fused SpMM quadratic forms, REML trace correction.  Symbolic analysis happens
once before the loop and is reported separately.  A Haseman-Elston fit (BASELINE.json config 4, K=3) is
timed as a secondary result in the same line (`he`).

  value      seconds per REML evaluation with every input resident in HBM (probes drawn on the device)
  e2e        the same evaluation through the public API with host buffers: host sigma + host probe block
             (pinned) copied in, nll + gradient copied out, every step
  roofline   the dominant kernel (FP64 DMMA tile GEMM): issued dense flops / device time of its launches,
             measured with CUDA events on the launching stream in a separate profiled pass
  cpu_baseline  the oracle port (oracle/estimation.py + oracle/supernodal_cpu.py) on the host cores: a BOUNDED
             sample (deterministic part in full, probe pipeline on --cpu-cols columns); the measured seconds and
             the value scaled to all columns are reported as separate fields

Multi-GPU (torchrun): factor replicated, probe columns sharded, one NCCL allreduce of K doubles per
evaluation ("strong" scaling: total work fixed).

--impl reference: the reference's algorithm on the host cores, nothing extrapolated - every step is one full
`bolt_gradient_estimation` as oracle/estimation.py restates it (scipy sparse kernels, factor.L().dot(Z) and all 128
probe columns), on the multifrontal LAPACK factor with the analysis repeated per evaluation as the reference does.
A step takes ~1-2 minutes, so the arm runs one warm-up (none with --warmup 0) and then --steps timed steps; with
--ref-budget SECONDS it stops early once the next step would exceed the budget (at least one runs).  It prints the
number it EXECUTED in "steps" (the request is kept in "steps_requested").

--dump-outputs DIR writes what the last timed step computed (nll, gradient and, in the GPU arm, logdet, fixed
effects, V^-1 y, V^-1 r, V^-1 C and the probe block W on a seeded sample of rows) as DIR/<name>.npy.  The inputs
are generated from fixed seeds, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

_RESULT_OUT = None          # set by main(): importing this module leaves the process's stdout alone


def emit(obj):
    _RESULT_OUT.write(json.dumps(obj) + "\n")
    _RESULT_OUT.flush()


# removal fractions found once by simulate_pedigree's bisection (seed 0); avoids repeating the search
REMOVE_FRAC = {(250000, 1e-3): 0.065625, (100000, 1e-3): 0.084375, (20000, 1e-3): None,
               (1000000, 1e-4): 0.103125, (3000000, 3.3e-5): 0.1125,
               (3000000, 1e-5): 0.16875, (3000000, 2e-5): 0.13125}


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print("[bench]", *a, file=sys.stderr, flush=True)


def host_mem():
    try:
        import psutil
        vm = psutil.virtual_memory()
        return "rss %.1f GB, host avail %.0f of %.0f GB" % (psutil.Process().memory_info().rss / 2 ** 30,
                                                            vm.available / 2 ** 30, vm.total / 2 ** 30)
    except Exception:
        return "n/a"


def release_host_caches(torch):
    """Drop what the previous phase pinned / cached (N ranks share one host: 8 x several GB of pinned staging and
    matrices would otherwise stay resident while the next workload is generated)."""
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    try:
        torch._C._host_emptyCache()
    except Exception:
        pass


def make_inputs(n, sf, ncov, seed=0, with_household=False):
    from scilmm_b200 import pedigree as P
    t0 = time.time()
    ped = P.simulate_pedigree(n, sf, seed=seed, remove_frac=REMOVE_FRAC.get((n, sf)))
    A, T, D, F = P.numerator(ped["rel"])
    extra = []
    if with_household:
        extra.append(P.household_matrix(ped["household"]))
    keep, out = P.drop_unrelated(A, *extra)
    A = out[0]
    nn = A.shape[0]
    rng = np.random.default_rng(seed + 1)
    cov = rng.standard_normal((nn, ncov))
    y = P.quick_phenotype(T, D, np.zeros((n, 0)), 0.4, np.zeros(0), rng)[keep]
    cov = np.hstack([cov, np.ones((nn, 1))])
    cov[:, :-1] -= cov[:, :-1].mean(axis=0)
    cov[:, :-1] /= cov[:, :-1].std(axis=0)
    y = y + cov[:, :-1].dot(np.full(ncov, 0.05))
    info = dict(n_sim=n, n=nn, nnz=int(A.nnz), sf=sf, seed=seed, remove_frac=ped["remove_frac"])
    log("inputs generated in %.1f s" % (time.time() - t0), info)
    return A, (out[1] if with_household else None), cov, y, info


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[4 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def gemm_traffic_record():
    """DRAM traffic of the dominant kernel comes from an ncu --set full capture (never from a literal in this file):
    profiles/gemm_traffic.json is written by scripts/ncu_summary.py from the .ncu-rep of one representative launch
    and names the launch and the capture it came from.  Absent file -> traffic null."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "gemm_traffic.json")))
        return {"traffic": rec["dram_bytes"], "traffic_launch": rec["launch"], "traffic_source": rec["source"]}
    except Exception:
        return {"traffic": None, "traffic_source": "no ncu capture on file (profiles/gemm_traffic.json)"}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(path, values, per_row=None, n=0):
    """--dump-outputs: writes every array as <path>/<name>.npy in float64, so that two builds run with the same
    arguments can be compared output for output.  `values` are written whole; the device tensors of `per_row` (n rows
    each) are cut to one fixed, seeded sample of rows, the same rows for every tensor, as many as the 64 MB the whole
    dump may take allow."""
    os.makedirs(path, exist_ok=True)
    out = {k: np.atleast_1d(np.asarray(v, dtype=np.float64)) for k, v in values.items()}
    if per_row:
        import torch
        row_bytes = sum(8 * int(np.prod(v.shape[1:])) for v in per_row.values())
        room = DUMP_BYTES - sum(a.nbytes for a in out.values()) - 1024 * (len(out) + len(per_row))   # npy headers
        m = min(n, room // row_bytes)
        rows = np.sort(np.random.default_rng(0).choice(n, m, replace=False)) if m < n else np.arange(n)
        for k, v in per_row.items():
            out[k] = v[torch.from_numpy(rows).to(v.device)].double().cpu().numpy()
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)
    log("outputs of the last step written to %s: %s" % (path, {k: a.shape for k, a in out.items()}))


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reml_sample(mats, cov, y, sig, reml, sim_num, sample_cols):
    """BOUNDED sample of one oracle REML evaluation on the host: assembly, analysis, factorization, logdet and
    the deterministic solves in full; the probe pipeline (L*Z, solve, SpMM reductions) on `sample_cols` of the
    sim_num columns.  Returns the seconds actually measured and, separately, the value scaled to all columns."""
    from oracle import estimation as orc
    from oracle.supernodal_cpu import SupernodalCPUFactor, SupernodalPlan
    import scipy.linalg as la
    t = {}
    t0 = time.time()
    V = orc.weighted_sum(mats, sig)
    t["assemble"] = time.time() - t0
    t0 = time.time()
    plan = SupernodalPlan(sp.csr_matrix((V.data, V.indices, V.indptr), shape=V.shape))
    t["analyze"] = time.time() - t0           # the reference repays this on every evaluation (:22-26 from :92)
    t0 = time.time()
    f = SupernodalCPUFactor(V, plan=plan)
    logdet = f.logdet()
    t["factor"] = time.time() - t0
    t0 = time.time()
    ViC, chol, mu, beta = orc.fixed_effects(f, y, cov)
    Vir = f(y - mu)
    nll = orc.nll_value(f, y, Vir, mu, chol, reml)
    t["fixed"] = time.time() - t0
    t0 = time.time()
    rng = np.random.default_rng(7)
    Z = rng.standard_normal((y.size, sample_cols))
    W = f(f.lmul_unperm(Z))
    for k in range(len(mats)):
        _ = np.sum(mats[k].dot(W) * W, axis=0)
    t["probe_sample"] = time.time() - t0
    t0 = time.time()
    for k in range(len(mats)):
        _ = Vir.dot(mats[k].dot(Vir))
        if reml:
            _ = la.cho_solve(chol, ViC.T.dot(mats[k].dot(ViC)))
    t["quad"] = time.time() - t0
    scale = float(sim_num) / sample_cols
    measured = sum(t.values())
    scaled = measured + (scale - 1.0) * t["probe_sample"]
    return dict(measured_s=measured, scaled_s=scaled, parts=t, nll=nll, logdet=logdet, flops=plan.sym.flops)


def cpu_reml_full(mats, cov, y, sig, reml, sim_num, seed):
    """One FULL oracle evaluation: oracle.estimation.reml_evaluation is the line-by-line restatement of the
    reference's bolt_gradient_estimation (:77-117), here on the multifrontal LAPACK Factor with the analysis
    repeated inside the call (reanalyze=True), scipy's single-threaded sparse kernels and factor.L().dot(Z)."""
    from oracle import estimation as orc
    from oracle.supernodal_cpu import supernodal_cholesky_func
    np.random.seed(seed)
    t0 = time.time()
    nll, grad = orc.reml_evaluation(np.log(sig), supernodal_cholesky_func(reanalyze=True), mats, cov, y, reml,
                                    sim_num, False, True)
    return time.time() - t0, nll, grad


def cpu_he(mats, cov, y):
    from oracle import estimation as orc
    t0 = time.time()
    est = orc.he_regression(list(mats), cov, y.copy(), compute_stderr=False)
    return time.time() - t0, est


# ------------------------------------------------------------------------------------------------ main
def main():
    # The contract is ONE JSON line on stdout.  Libraries write to file descriptor 1 behind Python's back (NCCL prints
    # its version banner there on the first collective), so fd 1 is pointed at stderr for the whole run and the result
    # line goes to a private duplicate of the original stdout.
    global _RESULT_OUT
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--individuals", dest="n", type=int, default=250000)   # not "--n": torchrun's parser treats it as an ambiguous abbreviation
    ap.add_argument("--sf", type=float, default=1e-3)
    ap.add_argument("--probes", type=int, default=128)
    ap.add_argument("--ncov", type=int, default=10)
    ap.add_argument("--he-n", type=int, default=1000000)
    ap.add_argument("--he-sf", type=float, default=1e-4)
    ap.add_argument("--skip-he", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--cpu-cols", type=int, default=8)
    ap.add_argument("--ref-budget", type=float, default=None,
                    help="--impl reference: stop early once the next timed step would take the steps past this many "
                         "seconds (at least one runs); by default all --steps run")
    ap.add_argument("--skip-fit", action="store_true", help="skip the full REML() fit (wall time incl. setup)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64, at most 64 MB; arrays "
                         "with one row per individual are cut to a fixed, seeded sample of rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.ref_budget is not None:
        # the probes are reseeded per step: a wall-time cut would make the dumped step depend on the machine's speed
        ap.error("--dump-outputs cannot be combined with --ref-budget")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    sig = np.array([0.3, 0.15, 0.55])
    workload = "REML evaluation, simulated pedigree %d (sf=%g), K=3 (IBD, AoA, I), c=%d+1, %d probes" % (
        args.n, args.sf, args.ncov, args.probes)

    base_config = {"workload": workload, "l2": "inputs larger than L2 (factor panels ~4.5 GB, matrices 1.5 GB)"}
    if args.impl == "reference":
        if rank != 0:
            return
        A, _, cov, y, info = make_inputs(args.n, args.sf, args.ncov)
        from scilmm_b200 import pedigree as P
        mats = [A, P.epistasis(A), sp.eye(A.shape[0]).tocsr()]
        ys = y / y.std()
        vals = []
        t_begin = time.time()
        nwarm = min(1, args.warmup)          # one warm-up pass is enough on the CPU (no clocks / caches to settle)
        i = 0
        while True:
            dt, nll_c, grad_c = cpu_reml_full(mats, cov, ys, sig, True, args.probes, seed=100 + i)
            log("reference step %d: %.2f s  nll %.10e" % (i, dt, nll_c))
            if i >= nwarm:
                vals.append(dt)
            i += 1
            if len(vals) >= args.steps or (args.ref_budget is not None and len(vals) >= 1 and
                                           sum(vals) + dt > args.ref_budget):
                break
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"nll": nll_c, "grad": grad_c})
        v = float(np.mean(vals))
        sample = ("oracle port, nothing extrapolated: %d full evaluations (oracle.estimation.reml_evaluation = the "
                  "reference's bolt_gradient_estimation line by line: scipy assembly, METIS analysis + multifrontal "
                  "LAPACK factorization repeated per call, logdet, fixed-effect solves, factor.L().dot(Z) and the "
                  "solve for all %d probe columns, scipy SpMM reductions) after %d warm-up; %d steps were requested"
                  % (len(vals), args.probes, nwarm, args.steps))
        if args.ref_budget is not None:
            sample += ", the time budget (--ref-budget %g s) allowed %d" % (args.ref_budget, len(vals))
        emit({"impl": "reference", "metric": "reml_iter_time", "value": v, "unit": "s",
              "n_gpus": args.gpus, "steps": len(vals), "warmup": nwarm, "steps_requested": args.steps,
              "warmup_requested": args.warmup, "ms_per_step": v * 1e3, "higher_is_better": False,
              "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
              "config": {**base_config, **info},
              "step_seconds": [round(x, 2) for x in vals], "wall_s": round(time.time() - t_begin, 1),
              "cpu_baseline": {"value": v, "unit": "s", "cores": os.cpu_count(), "kind": "port", "sample": sample},
              "e2e": {"value": v, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
              "nll": float(nll_c)})
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from scilmm_b200 import engine as E
    from scilmm_b200 import pedigree as P
    import scilmm_b200.SparseCholesky  # noqa: F401
    S = sys.modules["scilmm_b200.SparseCholesky"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    A, _, cov, y, info = make_inputs(args.n, args.sf, args.ncov)
    log("inputs", info)
    n = A.shape[0]
    mats = [A, P.epistasis(A), sp.eye(n).tocsr()]
    ys = y / y.std()
    K = len(mats)
    s = args.probes

    E.UPLOAD_THREADS = max(1, min(8, (os.cpu_count() or 4) // max(1, world)))
    chol = S.SparseCholesky(rng="device", seed=12345)     # counter-based device probes: same values for any N
    t0 = time.time()
    ses = chol._session(mats, cov, ys)
    torch.cuda.synchronize()
    setup_s = time.time() - t0
    st = ses.eng.stats()
    setup_parts = {k: round(v, 2) for k, v in ses.timings.items()}
    log("session %.1fs" % setup_s, ses.timings, {k: st[k] for k in ("nsuper", "nlevels", "nnzL", "lsize", "flops",
                                                                    "max_front_rows", "launches", "device_bytes")})

    # ---------------- device-resident steps
    sampler = ClockSampler(local_rank)
    sampler.start()                       # started before the warm-up so its start-up cost stays outside the timed region
    for _ in range(args.warmup):
        ses.evaluate(sig, True, s)
    barrier()
    sampler.lines = []
    E.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        nll, grad = ses.evaluate(sig, True, s)
    e1.record()
    barrier()
    launches = E.launch_count()
    clocks = sampler.stop()
    step_ms = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    if args.dump_outputs and rank == 0:
        # what evaluate() returns and keeps in ses.last; with N ranks W holds rank 0's probe columns
        last = ses.last
        dump_outputs(args.dump_outputs, {"nll": nll, "grad": grad, "logdet": last["logdet"], "beta": last["beta"]},
                     {k: last[k] for k in ("Viy", "Vir", "ViC", "W")}, n)

    # factorization alone (Cholesky GFLOP/s of the metric) and solve / reduction phases
    def ev(fn, reps=2):
        fn()
        best = 1e30
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b))
        return best

    def assemble():
        for k in range(K):
            ses.eng.add_values(ses.map_ids[k], ses.matset.values_ptr(k), float(sig[k]), k == 0)

    def assemble_factor():
        assemble()
        ses.eng.factorize()

    t_asm = ev(assemble)
    t_fac = ev(assemble_factor) - t_asm
    Bs = torch.randn(n, s, dtype=torch.float64, device="cuda")
    t_clone = ev(lambda: Bs.clone())
    t_solve = ev(lambda: ses.eng.solve_(Bs.clone())) - t_clone
    t_lmul = ev(lambda: ses.eng.lmul(Bs))
    Bn = torch.randn(n, cov.shape[1] + 1, dtype=torch.float64, device="cuda")
    t_solve_narrow = ev(lambda: ses.eng.solve_(Bn.clone()))
    Xq = torch.randn(n, s + 1, dtype=torch.float64, device="cuda")
    groups = ses.matset.pattern_groups(2)
    nbq = cov.shape[1] + 1
    Bq = torch.randn(n, nbq, dtype=torch.float64, device="cuda")

    def quadforms(W):
        """the quadratic-form / Gram pass of one evaluation: tiled kernel where the session built tiles"""
        out = []
        for ks in groups:
            if ses.use_tiles and ses.matset.has_tiles(ks) and nbq + W.shape[1] <= 160:
                out.append(ses.matset.quadform_tiled(ks, torch.cat([Bq, W], dim=1), nbq))
            else:
                out.append(ses.matset.quadform_gram_multi(ks, W, Bq))
        return out
    t_quad = ev(lambda: quadforms(Bs))
    t_quad_rowwise = ev(lambda: [ses.matset.quadform_multi(ks, Xq) for ks in groups])
    # the C3 "AI-REML iteration" of SURVEY 8d = one evaluation + compute_hess (reference :147-168)
    t_hess = ev(lambda: S._hess_device(ses, ses.eng), reps=1)
    # the phase that shards across ranks: this rank's probe columns through L*Z, the solve and the quadratic forms;
    # and the same for ALL columns, which gives the Amdahl bound of the step at this N
    lo_c, hi_c = S._shard.column_block(s, rank, world)
    Bloc = Bs[:, lo_c:hi_c].contiguous()

    def probe_pipeline(Bp):
        return quadforms(ses.eng.solve_(ses.eng.lmul(Bp)))
    t_shard_local = max_over_ranks(ev(lambda: probe_pipeline(Bloc)))
    t_shard_full = ev(lambda: probe_pipeline(Bs)) if world > 1 else t_shard_local
    # profiled pass: per-kernel-kind device time with events around every launch
    assemble()
    ses.eng.set_profiling(True)
    ses.eng.factorize()
    prof = ses.eng.profile()
    ses.eng.set_profiling(False)
    tma_dominant = prof.get("gemm_tma", {"ms": 0.0})["ms"] >= prof["gemm_big"]["ms"]
    gb = prof["gemm_tma"] if tma_dominant else prof["gemm_big"]
    gemm_all = {k: prof[k] for k in ("gemm_tma", "gemm_big") if k in prof and prof[k]["launches"]}
    # FP64 tensor peak: cuBLAS DGEMM measured in this run (MEASURED_PEAKS.json has no FP64 figure)
    Mg = 8192
    ga = torch.randn(Mg, Mg, dtype=torch.float64, device="cuda")
    gbm = torch.randn(Mg, Mg, dtype=torch.float64, device="cuda")
    t_dgemm = ev(lambda: torch.matmul(ga, gbm), reps=3)
    dgemm_tflops = 2.0 * Mg ** 3 / t_dgemm / 1e9
    del ga, gbm
    achieved = gb["flops"] / gb["ms"] / 1e9 if gb["ms"] > 0 else 0.0
    roofline = {"bound": "tensor",
                "kernel": ("gemm_tiles_tma_kernel (FP64 DMMA 128x128 tiles, TMA-staged operands)" if tma_dominant
                           else "gemm_tiles_kernel<128,128> (FP64 DMMA)"), "achieved": round(achieved, 3),
                "peak": round(dgemm_tflops, 3), "unit": "TFLOP/s", "frac": round(achieved / dgemm_tflops, 4),
                "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry)",
                **gemm_traffic_record(),
                "launches": gb["launches"], "kernel_ms_per_factorization": round(gb["ms"], 2),
                "all_128x128_tile_kernels": {k: {"ms": round(v["ms"], 2), "tflops": round(v["flops"] / max(v["ms"], 1e-9) / 1e9, 2),
                                                 "launches": v["launches"]} for k, v in gemm_all.items()},
                "share_of_factorization": round(gb["ms"] / max(1e-9, sum(v["ms"] for v in prof.values())), 3)}
    peaks = measured_peaks()
    hbm = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback"
    nnzs = ses.matset.nnz
    solve_bytes = 2.0 * (8.0 * st["lsize"]) + 2 * 2 * 8.0 * n * s
    # symmetric half traversal: (4 + 8) bytes per visited entry of A, 8 more for AoA on the shared pattern, the
    # gathered X rows are the real traffic (8 (s+1) bytes per visited entry, through L2) and are reported apart
    half = [(z + n) / 2.0 for z in nnzs]
    quad_bytes = 12.0 * half[0] + 4 * (n + 1) + 8.0 * half[1] + 12.0 * half[2] + 4 * (n + 1) + 2 * 8.0 * n * (s + 1)
    quad_gather_bytes = (half[0] + half[2]) * 8.0 * (s + 1)
    # SURVEY 8d figure for the pass: 12 nnz + 4(n+1) per pattern, 8 nnz for a matrix sharing a pattern, the dense
    # block [narrow | probes] read once per pattern group
    quad_bytes_survey = 12.0 * nnzs[0] + 8.0 * nnzs[1] + 12.0 * nnzs[2] + 2 * 4 * (n + 1) + 2 * 8.0 * n * (s + nbq)
    solve_flops = 4.0 * st["nnzL"] * s
    phases = {
        "assemble_ms": round(t_asm, 3), "factorize_ms": round(t_fac, 2), "solve128_ms": round(t_solve, 2),
        "lmul128_ms": round(t_lmul, 2), "quadforms_ms": round(t_quad, 2), "quadforms_rowwise_kernel_ms": round(t_quad_rowwise, 2),
        "solve_narrow_ms": round(t_solve_narrow, 2), "solve_narrow_cols": int(cov.shape[1] + 1),
        "solve_narrow_gbs": round((2.0 * 8.0 * st["lsize"]) / t_solve_narrow / 1e6, 1),
        "solve128_tflops": round(solve_flops / t_solve / 1e9, 2),
        "compute_hess_ms": round(t_hess, 2), "ai_reml_iter_ms": round(step_ms + t_hess, 2),
        "sharded_phase_ms": round(t_shard_local, 2), "sharded_phase_all_columns_ms": round(t_shard_full, 2),
        # Amdahl bound of the step at this N: the replicated assembly + factorization + 1/N of the probe pipeline
        # (the fixed-effect solve runs beside the pipeline on the auxiliary stream)
        "replicated_ms": round(t_asm + t_fac, 2),
        "amdahl_bound_ms": round(t_asm + t_fac + t_shard_full / world, 2),
        "cholesky_gflops": round(st["flops"] / t_fac / 1e6, 1),
        "cholesky_issued_gflops": round(st["issued_flops"] / t_fac / 1e6, 1),
        "solve_gbs": round(solve_bytes / t_solve / 1e6, 1), "quadforms_gbs": round(quad_bytes / t_quad / 1e6, 1),
        "quadforms_gather_gbs": round(quad_gather_bytes / t_quad / 1e6, 1),
        "quadforms_survey_bytes_gbs": round(quad_bytes_survey / t_quad / 1e6, 1),
        "quadforms_frac_of_hbm": round(quad_bytes_survey / t_quad / 1e6 / hbm, 3),
        "hbm_peak_gbs": hbm, "hbm_peak_source": hbm_src,
        "profile_ms": {k: round(v["ms"], 2) for k, v in prof.items() if v["launches"]},
    }

    # ---------------- size-independent parity properties at the full BASELINE size (SURVEY 8c): the factor is
    # bit-reproducible (no atomics, fixed summation order), V x = b holds for the solves, L*Z followed by the solve
    # round-trips, and (below, when the CPU arm runs) nll agrees with the oracle on the same inputs
    def factor_logdet():
        assemble()
        ses.eng.factorize()
        return ses.eng.logdet()
    ld1, ld2 = factor_logdet(), factor_logdet()
    Bchk = torch.randn(n, 8, dtype=torch.float64, device="cuda")
    Xchk = ses.eng.solve_(Bchk.clone())
    VX = sum(float(sig[k]) * ses.matset.spmm(k, Xchk) for k in range(K))
    solve_res = float((VX - Bchk).abs().max() / Bchk.abs().max())
    parity = {"logdet": ld1, "logdet_bitwise_repeatable": bool(ld1 == ld2), "solve_residual_rel": solve_res,
              "solve_residual_ok": bool(solve_res < 1e-10)}
    if not (parity["logdet_bitwise_repeatable"] and parity["solve_residual_ok"]):
        raise RuntimeError("parity check failed at full size: %r" % (parity,))

    # ---------------- e2e through the public API with host buffers
    chol_h = S.SparseCholesky(rng="host_buffer")
    chol_h._engines = chol._engines                      # same analysis; the session re-registers patterns
    Zhost = torch.from_numpy(np.random.default_rng(5).standard_normal((n, s))).pin_memory()
    chol_h.probe_source = lambda nn, ss: Zhost
    log_sig = np.log(sig)
    for _ in range(2):
        S.bolt_gradient_estimation(log_sig, chol_h, mats, cov, ys, True, s, False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        nll_h, grad_h = S.bolt_gradient_estimation(log_sig, chol_h, mats, cov, ys, True, s, False)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / args.steps)
    lo_e, hi_e = S._shard.column_block(s, rank, world)
    e2e = {"value": round(e2e_s, 4), "unit": "s", "h2d_bytes_per_step": int(n * (hi_e - lo_e) * 8 + K * 8),
           "d2h_bytes_per_step": int((K + 1) * 8 + (K * (cov.shape[1] ** 2 + 2) + 2 * cov.shape[1] ** 2) * 8),
           "api": "scilmm_b200.bolt_gradient_estimation(log_sig, SparseCholesky(), mats, cov, y, True, 128, False)"}

    # ---------------- a whole REML() fit through the public API, setup included (fresh functor: upload, analysis,
    # scatter maps, HE start, L-BFGS-B evaluations, final factorization, fixed effects, compute_hess)
    full_fit = None
    if not args.skip_fit:
        del ses
        chol._sessions.clear()
        chol._engines.clear()
        chol_h._sessions.clear()
        chol_h._engines.clear()
        release_host_caches(torch)
        chol_f = S.SparseCholesky(rng="device", seed=777)
        barrier()
        t0 = time.perf_counter()
        fit = S.REML(chol_f, mats[:-1], cov, y, reml=True, sim_num=s, verbose=False)
        torch.cuda.synchronize()
        fit_s = max_over_ranks(time.perf_counter() - t0)
        ses_f = next(iter(chol_f._sessions.values()))
        full_fit = {"wall_s": round(fit_s, 2), "setup_s": round(ses_f.setup_s, 2),
                    "setup_parts_s": {k: round(v, 2) for k, v in ses_f.timings.items()},
                    "evaluations": int(ses_f.n_eval), "sigma2": [float(v) for v in fit["covariance coefficients"]],
                    "se": [float(v) for v in fit["covariance std"]], "nll": float(fit["nll"]),
                    "api": "scilmm_b200.REML(SparseCholesky(rng='device'), [A, AoA], cov, y, sim_num=128)"}
        log("full fit", full_fit)
        del ses_f, chol_f
        # the same fit with ordering_method='nesdis_fast' (one METIS separator per bisection): shorter analysis, ~2 % more
        # factorization flops - the better trade for a single fit; estimates must agree with the default ordering
        release_host_caches(torch)
        chol_q = S.SparseCholesky(ordering_method="nesdis_fast", rng="device", seed=777)
        barrier()
        t0 = time.perf_counter()
        fit_q = S.REML(chol_q, mats[:-1], cov, y, reml=True, sim_num=s, verbose=False)
        torch.cuda.synchronize()
        fit_q_s = max_over_ranks(time.perf_counter() - t0)
        ses_q = next(iter(chol_q._sessions.values()))
        st_q = ses_q.eng.stats()
        full_fit["nesdis_fast"] = {
            "wall_s": round(fit_q_s, 2), "setup_s": round(ses_q.setup_s, 2), "evaluations": int(ses_q.n_eval),
            "factor_flops": st_q["flops"], "sigma2": [float(v) for v in fit_q["covariance coefficients"]],
            # another permutation gives another probe block (L Z)[P^-1] (reference :49-52): the two fits differ by
            # Monte-Carlo noise of the trace estimate, measured here in units of the reported standard errors
            "max_abs_diff_vs_default_over_se": float(np.max(np.abs(np.asarray(fit_q["covariance coefficients"]) -
                                                                   np.asarray(fit["covariance coefficients"])) /
                                                            np.asarray(fit["covariance std"])))}
        log("full fit, fast ordering", full_fit["nesdis_fast"])
        del ses_q, chol_q, fit_q, fit
        ses = None

    # ---------------- HE (config 4) secondary result
    he = None
    log("before HE:", host_mem())
    del ses, chol, chol_h, Zhost, Bs, Bn, Bloc, Xq, Bchk, Xchk, VX
    release_host_caches(torch)
    if not args.skip_he:
        try:
            he = bench_he(args, E, P, S, torch, hbm, barrier, max_over_ranks)
        except Exception as ex:   # keep the headline line even if the secondary workload cannot be generated
            he = {"error": repr(ex)}

    # ---------------- CPU baseline (rank 0, N=1)
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        r = cpu_reml_sample(mats, cov, ys, sig, True, s, args.cpu_cols)
        log("cpu parts", r["parts"])
        if abs(r["nll"] - nll_h) > 1e-10 * abs(r["nll"]) or abs(r["logdet"] - parity["logdet"]) > 1e-10 * abs(r["logdet"]):
            raise RuntimeError("GPU result differs from the CPU oracle beyond 1e-10: nll %r vs %r, logdet %r vs %r"
                               % (nll_h, r["nll"], parity["logdet"], r["logdet"]))
        cpu = {"value": round(r["scaled_s"], 2), "unit": "s", "cores": os.cpu_count(), "kind": "port",
               "measured_s": round(r["measured_s"], 2),
               "value_note": "value = measured_s with the probe-pipeline part scaled from %d to %d columns; the "
                             "--impl reference arm runs every column and extrapolates nothing" % (args.cpu_cols, s),
               "parts_s": {k: round(v, 2) for k, v in r["parts"].items()},
               "cholesky_gflops": round(r["flops"] / r["parts"]["factor"] / 1e9, 1),
               "nll_rel_diff_vs_gpu": abs(r["nll"] - nll_h) / abs(r["nll"]),
               "logdet_rel_diff_vs_gpu": abs(r["logdet"] - parity["logdet"]) / abs(r["logdet"]),
               "sample": "oracle port (CHOLMOD is not installed): full assembly, METIS analysis, supernodal LAPACK "
                         "factorization on all cores, logdet, deterministic solves; probe pipeline (BLAS L*Z, solve, "
                         "scipy SpMM reductions) on %d of %d columns; includes the per-evaluation re-analysis the "
                         "reference performs" % (args.cpu_cols, s)}

    if rank == 0:
        out = {"metric": "reml_iter_time", "value": round(step_ms / 1e3, 5), "unit": "s", "n_gpus": world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(step_ms, 3),
               "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
               "data": "synthetic",
               "config": {**base_config, **info},
               "stats": {"nnzL": st["nnzL"], "factor_flops": st["flops"], "panel_gb": round(st["lsize"] * 8 / 1e9, 2),
                         "nsuper": st["nsuper"], "levels": st["nlevels"], "max_front": st["max_front_rows"],
                         "symbolic_s": round(st["t_order"] + st["t_symbolic"], 2), "session_setup_s": round(setup_s, 1),
                         "session_setup_parts_s": setup_parts, "device_bytes": st["device_bytes"],
                         "parallelism": "probe columns sharded x%d, factor replicated" % world,
                         "probe_stream": "device Philox4x32-10 keyed by (seed, evaluation, row, column): identical "
                                         "values for any number of GPUs"},
               "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
               "phases": phases, "parity": parity, "cpu_baseline": cpu, "full_fit": full_fit, "he": he,
               "nll": float(nll), "grad": [float(g) for g in grad]}
        emit(out)
    if world > 1:
        dist.destroy_process_group()


def bench_he(args, E, P, S, torch, hbm, barrier, max_over_ranks):
    """Haseman-Elston fit, K=3 (IBD, AoA, household), BASELINE config 4.  With N ranks every rank uploads and holds
    only its row block of every matrix (blocks balanced by the entries on/below the diagonal)."""
    from scilmm_b200 import sharding
    rank, world = sharding.rank_world()
    A, H, cov, y, info = make_inputs(args.he_n, args.he_sf, 2, seed=0, with_household=True)
    n = A.shape[0]
    mats = [A, P.epistasis(A), H]
    log("HE inputs", info, "nnz(H)", H.nnz, "|", host_mem())
    bounds = sharding.row_blocks_by_lower_nnz(A, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    ms = E.MatSet(mats, row_range=(lo, hi))
    ms.resolve_symmetry_sharded(sharding.allreduce_sum_)
    yd = E.to_device(y)

    def run():
        part = ms.he_moments_device(yd)
        return sharding.allreduce_sum_(part)

    for _ in range(3):
        run()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    barrier()
    dev_ms = max_over_ranks(e0.elapsed_time(e1) / reps)
    alg_bytes = (12.0 * A.nnz + 4 * (n + 1)) + 8.0 * A.nnz + (12.0 * H.nnz + 4 * (n + 1)) + 3 * 8.0 * n
    # bytes the symmetric half traversal really has to move (entries on/below the diagonal): the honest denominator
    half = lambda z: (z + n) / 2.0
    real_bytes = (12.0 * half(A.nnz) + 8.0 * half(A.nnz) + 12.0 * half(H.nnz)) + 3 * 4 * (n + 1) + 3 * 8.0 * n
    h2d_local = int(ms.h2d_bytes + 8 * n)
    del ms
    e2e_s = 1e30
    for _ in range(2):          # best of two public calls (host page-locking / allocator noise on a shared box)
        barrier()
        S.HE_TIMINGS = {}
        t0 = time.perf_counter()
        est = S.HE(list(mats), cov, y.copy())
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        if dt < e2e_s:
            e2e_s, e2e_parts = dt, {k: round(v, 4) for k, v in S.HE_TIMINGS.items()}
        S.HE_TIMINGS = None
    out = {"workload": "HE fit, simulated pedigree %d (sf=%g), K=3 (IBD, AoA, household)" % (args.he_n, args.he_sf),
           **info, "nnz_household": int(H.nnz), "n_gpus": world, "device_ms": round(dev_ms, 4),
           "e2e_s": round(e2e_s, 3), "e2e_parts_s": e2e_parts, "h2d_bytes_per_rank": h2d_local, "rows_this_rank": [lo, hi],
           "estimates": [float(v) for v in est],
           "roofline": {"bound": "hbm", "kernel": "he_group_kernel<2> (IBD + AoA, lower triangle) + he_short_kernel (household) + "
                                  "he_cross_mapped_kernel<1,2> + reduce_all_kernel",
                        "bytes_formula": "SURVEY 8d: sum_k 12 nnz_k + 4(n+1) per pattern (8 nnz for a matrix sharing a "
                                         "pattern) + 3*8n; frac_real_bytes counts only the entries on/below the "
                                         "diagonal, which is what the symmetric traversal moves",
                        "achieved": round(alg_bytes / dev_ms / 1e6, 1), "peak": hbm * world, "unit": "GB/s",
                        "frac": round(alg_bytes / dev_ms / 1e6 / (hbm * world), 4), "algorithmic_bytes": alg_bytes,
                        "achieved_real_bytes": round(real_bytes / dev_ms / 1e6, 1),
                        "frac_real_bytes": round(real_bytes / dev_ms / 1e6 / (hbm * world), 4)}}
    if not args.skip_cpu and rank == 0 and world == 1:
        t_cpu, est_cpu = cpu_he(mats, cov, y)
        out["cpu_baseline"] = {"value": round(t_cpu, 2), "unit": "s", "cores": 1, "kind": "port",
                               "sample": "full oracle HE fit (scipy single-threaded kernels, as the reference)",
                               "rel_diff_vs_gpu": float(np.max(np.abs(est - est_cpu)) / np.max(np.abs(est_cpu)))}
    return out


if __name__ == "__main__":
    main()
