"""Developer probe: stage-by-stage device time of RemlSession.evaluate on the 250K config (sync after each stage)."""
import os, sys, time
import numpy as np, scipy.sparse as sp, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import bench
from scilmm_b200 import pedigree as P
import scilmm_b200.SparseCholesky
S = sys.modules["scilmm_b200.SparseCholesky"]
n = int(sys.argv[1]) if len(sys.argv) > 1 else 250000
A, _, cov, y, info = bench.make_inputs(n, 1e-3, 10)
mats = [A, P.epistasis(A), sp.eye(A.shape[0]).tocsr()]
ys = y / y.std()
chol = S.SparseCholesky(rng="device"); ses = chol._session(mats, cov, ys); sig = np.array([0.3, 0.15, 0.55])
for _ in range(2): ses.evaluate(sig, True, 128)
torch.cuda.synchronize()
def T(tag, fn, reps=3):
    fn(); torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(reps): r = fn()
    torch.cuda.synchronize(); print("%-28s %8.2f ms" % (tag, (time.perf_counter() - t0) / reps * 1e3), flush=True); return r
T("evaluate", lambda: ses.evaluate(sig, True, 128))
T("factor_at", lambda: ses.factor_at(sig))
T("logdet", lambda: ses.eng.logdet())
T("fixed_effects (12 rhs)", lambda: ses.fixed_effects())
Z = torch.randn(ses.n, 128, dtype=torch.float64, device="cuda")
T("randn n x 128", lambda: torch.randn(ses.n, 128, dtype=torch.float64, device="cuda"))
T("lmul", lambda: ses.eng.lmul(Z))
U = ses.eng.lmul(Z)
T("solve_ 128", lambda: ses.eng.solve_(U.clone()))
W = ses.eng.solve_(U.clone())
ViC, chol_, beta, Viy, _ = ses.fixed_effects()
X = torch.cat([W, Viy.unsqueeze(1)], dim=1).contiguous()
T("cat X", lambda: torch.cat([W, Viy.unsqueeze(1)], dim=1).contiguous())
groups = ses.matset.pattern_groups(2)
for ks in groups:
    T("quadform_multi %s" % ks, lambda: ses.matset.quadform_multi(ks, X))
    T("coldot_multi ViC %s" % ks, lambda: ses.matset.coldot_multi(ks, ViC, 0))
    T("quadform_multi W128 %s" % ks, lambda: ses.matset.quadform_multi(ks, W))
    T("quadform_gram_multi %s" % ks, lambda: ses.matset.quadform_gram_multi(ks, W, ses._ViCy))
B12 = torch.randn(ses.n, 12, dtype=torch.float64, device="cuda")
T("solve_ 12", lambda: ses.eng.solve_(B12.clone()))
T("solve_ 1", lambda: ses.eng.solve_(B12[:, 0].contiguous()))
Xt = torch.cat([ses._ViCy, W], dim=1).contiguous()
for ks in groups:
    if ses.matset.has_tiles(ks):
        print("tiles", ks, ses.matset.tile_stats(ks[0]), "setup", ses.timings)
        T("quadform_tiled [B|W] %s" % ks, lambda: ses.matset.quadform_tiled(ks, Xt, ses._ViCy.shape[1]))
        T("quadform_tiled W only %s" % ks, lambda: ses.matset.quadform_tiled(ks, W, 0))
        X16 = Xt[:, :28].contiguous()
        T("quadform_tiled 12+16 cols %s" % ks, lambda: ses.matset.quadform_tiled(ks, X16, 12))
B16 = torch.randn(ses.n, 16, dtype=torch.float64, device="cuda")
T("solve_ 16", lambda: ses.eng.solve_(B16.clone()))
T("lmul 16", lambda: ses.eng.lmul(B16))
T("hess", lambda: S._hess_device(ses, ses.eng), reps=1)
