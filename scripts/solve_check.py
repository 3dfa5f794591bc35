"""V x = b residuals and the L*Z -> solve round trip at the bench size for every RHS-width class (streaming kernels
up to 32 columns, DMMA tiles above), then solve / L*Z times.  usage: python scripts/solve_check.py [n_sim]"""
import os, sys, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import bench
from scilmm_b200 import engine as E, pedigree as P
import scilmm_b200.SparseCholesky
S = sys.modules["scilmm_b200.SparseCholesky"]
n_sim = int(sys.argv[1]) if len(sys.argv) > 1 else 250000
A, _, cov, y, info = bench.make_inputs(n_sim, 1e-3, 10)
n = A.shape[0]
import scipy.sparse as sp
mats = [A, P.epistasis(A), sp.eye(n).tocsr()]
sig = np.array([0.3, 0.15, 0.55])
chol = S.SparseCholesky(rng="device")
ses = chol._session(mats, cov, y / y.std())
ses.factor_at(sig)
print("logdet", ses.eng.logdet())
torch.manual_seed(0)
for k in (1, 2, 3, 4, 5, 8, 9, 12, 16, 17, 24, 32, 48, 64, 128):
    B = torch.randn(n, k, dtype=torch.float64, device="cuda")
    X = ses.eng.solve_(B.clone())
    VX = sum(float(sig[j]) * ses.matset.spmm(j, X) for j in range(3))
    res = float((VX - B).abs().max() / B.abs().max())
    LZ = ses.eng.lmul(B.clone())
    Y = ses.eng.solve_(LZ.clone(), mode=1)
    # forward half sweep of L Z returns Z with its rows permuted: compare permutation-invariant column moments
    rt = float(((Y * Y).sum(0) - (B * B).sum(0)).abs().max() / (B * B).sum(0).max()) + float((Y.sum(0) - B.sum(0)).abs().max()) / n
    print("nrhs %3d  residual %.3e  lmul->forward round trip %.3e" % (k, res, rt), flush=True)

def tm(fn, reps=5):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps
for k in (16, 32, 64, 128):
    B = torch.randn(n, k, dtype=torch.float64, device="cuda")
    print("nrhs %3d  solve %.2f ms  lmul %.2f ms" % (k, tm(lambda: ses.eng.solve_(B.clone())), tm(lambda: ses.eng.lmul(B))), flush=True)
