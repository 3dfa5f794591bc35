"""Drop-in for the reference module scilmm/SparseCholesky.py on a B200.

Same names, argument meaning and return values as the reference:
    SparseCholesky (the `cholesky_func` functor, reference :16-26)  ->  Factor with __call__/logdet/L/P
    HE (:192-281), REML (:177-189), bolt_gradient_estimation (:77-117), estimate_var_comps (:120-144),
    compute_hess (:147-168), compute_varcomp_stderr (:171-174), matrices_weighted_sum (:55-59),
    estimate_fixed_effects (:29-34), negative_log_likelihood (:37-46), simulate_vector (:49-52),
    compute_gradients (:62-74), MINQUE (:284-347), run_estimates (:350-395).

All sparse / factorization arithmetic runs in libscilmm_b200.so on the GPU.  The symbolic analysis
(ordering, elimination tree, supernodes, schedules) is cached per sparsity pattern inside the functor,
which is the structural change against the reference (it re-analyses on every call, :22-26 from :92).
There is no CPU fallback: without the CUDA library these functions raise.
"""
import functools
import hashlib
import time

import numpy as np
import scipy.linalg as la
import scipy.optimize as optimize
import scipy.sparse as sparse
import scipy.special as special
import scipy.stats as stats

from . import engine as _eng
from . import sharding as _shard
from ._lib import NotPositiveDefiniteError, SlmmError  # noqa: F401  (re-exported)

LOG_2PI = np.log(2 * np.pi)


def _pattern_key(m):
    h = hashlib.blake2b(digest_size=16)
    h.update(np.ascontiguousarray(m.indptr).view(np.uint8))
    h.update(np.ascontiguousarray(m.indices).view(np.uint8))
    return (m.shape[0], int(m.nnz), h.hexdigest())


def _fingerprint(a, max_samples=1 << 12, with_sum=False):
    """Cheap content fingerprint of a host array: shape + a hash of <= max_samples evenly strided elements
    (+ the full sum for the small dense inputs).  It is what makes the session cache notice in-place edits
    (`A.data *= 2`, a permuted phenotype) without hashing 10^8 values on every likelihood evaluation; an edit that
    touches none of the sampled elements and keeps the sum needs SparseCholesky.invalidate()."""
    a = np.asarray(a)
    flat = a.reshape(-1)
    step = max(1, flat.size // max_samples)
    h = hashlib.blake2b(np.ascontiguousarray(flat[::step]).view(np.uint8), digest_size=8).hexdigest()
    return (a.shape, h, float(flat.sum()) if with_sum else 0.0)


class B200Factor(object):
    """The Factor protocol of sksparse.cholmod (the four members the reference uses)."""

    def __init__(self, chol):
        self._chol = chol
        self._serial = chol.factorizations

    def _check(self):
        if self._chol.factorizations != self._serial:
            raise RuntimeError("this Factor was invalidated by a later factorization with the same pattern "
                               "(the device storage is reused across REML iterations)")

    # factor(b)  -- reference call sites :30,32,52,100,149,153
    def __call__(self, b):
        self._check()
        torch = _eng.require_cuda()
        if torch.is_tensor(b):
            x = b.to(device="cuda", dtype=torch.float64).contiguous().clone()
            return self._chol.solve_(x)
        b = np.asarray(b, dtype=np.float64)
        x = _eng.to_device(b, torch).contiguous()
        self._chol.solve_(x)
        return x.cpu().numpy()

    solve_A = __call__

    def logdet(self):
        self._check()
        return self._chol.logdet()

    def L(self):
        self._check()
        return self._chol.export_L()

    def P(self):
        return self._chol.perm().copy()

    # device-side extras used by the fused path
    def lmul(self, Z):
        self._check()
        return self._chol.lmul(Z)

    def stats(self):
        return self._chol.stats()


class SparseCholesky(object):
    """cholesky_func functor, reference scilmm/SparseCholesky.py:16-26.

    use_long / mode are accepted for signature compatibility (the engine is always supernodal LL' with
    32-bit row indices and 64-bit pointers).  ordering_method: 'nesdis' / 'metis' (nested dissection),
    'nesdis_fast' (one separator per bisection: ~30 % shorter analysis, ~2 % more factorization flops),
    'natural', or pass `perm` (perm[new] = old) to force a permutation (parity mode: L is unique given P).
    rng: 'numpy' draws probe vectors from the global numpy stream exactly like the reference (:50);
         'device' draws them on the GPU (distribution-equivalent, not stream-identical);
         'host_buffer' takes them from `probe_source(n, sim_num)` (a host array / pinned tensor).
    """

    def __init__(self, use_long=False, mode='supernodal', ordering_method='nesdis', perm=None, rng='numpy', seed=0):
        self._use_long = use_long
        self._mode = mode
        self._ordering_method = ordering_method
        self._perm = perm
        self.rng = rng
        self.seed = int(seed)         # key of the counter-based device probe stream (rng == 'device')
        self.probe_source = None      # callable(n, sim_num) -> host block, used when rng == 'host_buffer'
        self._engines = {}
        self._sessions = {}
        self._glmm = None             # the PQL session of glmm(): its device y and W^-1 change, so it is kept apart
        self.timings = {}

    def _engine_for(self, pattern, key=None):
        key = key or _pattern_key(pattern)
        eng = self._engines.get(key)
        if eng is None:
            t0 = time.time()
            eng = _eng.CholEngine(pattern, ordering=self._ordering_method, perm=self._perm)
            eng._self_map = None
            eng._dev_pattern = None
            self.timings['analyze_s'] = time.time() - t0
            if len(self._engines) >= 4:
                self._engines.pop(next(iter(self._engines)))
            self._engines[key] = eng
        return eng

    def __call__(self, sparse_mat):
        """Factor V.  Like sksparse.cholmod.cholesky (reference :23-26) only the LOWER triangle of the CSC matrix
        defines V: an input whose two triangles differ (or that stores one triangle only) is symmetrised from its
        lower triangle first (device check per call; symmetric input - the reference's case - takes no extra
        pass)."""
        torch = _eng.require_cuda()
        if not sparse.issparse(sparse_mat):
            raise TypeError("SparseCholesky expects a scipy.sparse matrix")
        m = sparse_mat
        if not sparse.isspmatrix_csc(m):
            m = m.tocsc()
        if m.shape[0] != m.shape[1]:
            raise ValueError("matrix must be square")
        if not m.has_sorted_indices:
            m = m.sorted_indices()
        pat = _eng.canonical_csr(sparse.csr_matrix((m.data, m.indices, m.indptr), shape=m.shape))   # = V' as CSR
        key = _pattern_key(pat)
        eng = self._engines.get(key)
        vals = _eng.to_device(pat.data, torch)
        dev = eng._dev_pattern if eng is not None and eng._dev_pattern is not None else \
            (_eng.to_device(pat.indptr, torch), _eng.to_device(pat.indices, torch))
        if not _eng.device_csr_is_symmetric(dev[0], dev[1], vals, pat.shape[0]):
            low = sparse.tril(m, format='csc')
            full = (low + sparse.tril(low, -1, format='csc').T).tocsc()
            full.sort_indices()
            return self.__call__(full)
        if eng is None:
            eng = self._engine_for(pat, key)
        if eng._dev_pattern is None:
            eng._dev_pattern = dev
            eng._self_map = eng.register_pattern_device(dev[0], dev[1], pat.nnz, 0)
        eng.add_values(eng._self_map, vals.data_ptr(), 1.0, True)
        eng.factorize()
        return B200Factor(eng)

    def invalidate(self):
        """Forget the cached REML sessions (device copies of mats / covariates / y).  The cache notices in-place
        edits through a sampled content fingerprint; call this after an edit it could miss."""
        self._sessions.clear()
        self._glmm = None

    # ---- fused session for the REML objective: matrices resident, patterns registered once
    def _session(self, mats, covariates, y):
        key = (tuple((id(m), int(m.nnz), _fingerprint(m.data)) for m in mats),
               (id(covariates), _fingerprint(covariates, with_sum=True)), (id(y), _fingerprint(y, with_sum=True)))
        ses = self._sessions.get(key)
        if ses is None:
            self._sessions.clear()
            ses = RemlSession(self, mats, covariates, y)
            self._sessions[key] = ses
        return ses


class RemlSession(object):
    """Device-resident state of one REML problem: K matrices, covariates, phenotype, one symbolic analysis."""

    def __init__(self, functor, mats, covariates, y):
        torch = _eng.require_cuda()
        self.torch = torch
        self.functor = functor
        self._refs = (list(mats), covariates, y)     # keeps the ids used as the cache key alive
        self.mats_host = [_eng.canonical_csr(m) for m in mats]
        self.K = K = len(mats)
        self.n = self.mats_host[0].shape[0]
        t0 = time.time()
        self.timings = {}
        # matrices go to HBM first: pattern sharing, CSR sanity, symmetry and the union pattern are all decided by
        # kernels on the resident arrays - the host never adds or scans the 10^8-entry patterns
        self.matset = _eng.MatSet(self.mats_host)
        self._groups = self.matset.pattern_groups(2)
        self._sym = [self.matset.is_symmetric(k) for k in range(K)]
        self._ident = [self._is_identity(k) for k in range(K)]
        self.timings['upload_s'] = time.time() - t0
        t1 = time.time()
        leaders = sorted(set(self.matset.pattern_id(k) for k in range(K)))
        big = max(leaders, key=lambda k: self.matset.nnz[k])
        if all(self.matset.pattern_is_subset(k, big) for k in leaders):
            union = self.mats_host[big]                 # every pattern is contained in the largest one
        else:
            union = None
            for k in leaders:       # pattern union (values are irrelevant; ones avoid cancellation)
                m = self.mats_host[k]
                ones = sparse.csr_matrix((np.ones(m.nnz), m.indices, m.indptr), shape=m.shape)
                union = ones if union is None else union + ones
            union = _eng.canonical_csr(union)
        if not all(self._sym):
            # V is defined by the lower triangles (CHOLMOD reads only the lower triangle of the CSC sum, reference
            # :23-26 after :59); the analysis needs the structurally symmetric pattern
            ones = sparse.csr_matrix((np.ones(union.nnz), union.indices, union.indptr), shape=union.shape)
            union = _eng.canonical_csr(ones + ones.T)
        self.union = union
        self.timings['union_s'] = time.time() - t1
        t1 = time.time()
        self.eng = functor._engine_for(union)
        self.timings['analyze_s'] = time.time() - t1
        t1 = time.time()
        self.map_ids = []
        cache = {}
        for k in range(K):
            tri = 0 if self._sym[k] else -1
            ck = (self.matset.pattern_id(k), tri)
            if ck not in cache:
                ptr_t, idx_t, _ = self.matset.device_arrays(k)
                cache[ck] = self.eng.register_pattern_device(ptr_t, idx_t, self.matset.nnz[k], tri)
            self.map_ids.append(cache[ck])
        self.timings['maps_s'] = time.time() - t1
        # tiled copies (fill-reducing order, 64 rows x 64 distinct columns) of the symmetric matrices for the
        # quadratic-form / Gram pass of compute_gradients; tiny matrices (the identity) keep the row-per-warp kernel
        t1 = time.time()
        self.use_tiles = True
        for ks in self._groups:
            if all(self._sym[k] for k in ks) and self.matset.nnz[ks[0]] >= 8 * self.n:
                for k in ks:
                    self.matset.build_tiles(k, self.eng)
        self.timings['tiles_s'] = time.time() - t1
        self.C = _eng.to_device(np.asarray(covariates, dtype=np.float64), torch)
        self.y = _eng.to_device(np.asarray(y, dtype=np.float64), torch)
        self.C_host = np.asarray(covariates, dtype=np.float64)
        self.y_host = np.asarray(y, dtype=np.float64)
        self.setup_s = time.time() - t0
        self.n_eval = 0               # evaluations so far: the `stream` index of the device probe generator
        self.overlap = True           # fixed-effect solve on the auxiliary stream beside the probe pipeline
        self.last = {}

    # K1 + K2
    def factor_at(self, sigmas):
        k = 0
        while k < self.K:      # consecutive matrices with one pattern (A, A o A) are scattered in one pass
            if k + 1 < self.K and self.map_ids[k + 1] == self.map_ids[k]:
                self.eng.add_values2(self.map_ids[k], self.matset.values_ptr(k), float(sigmas[k]),
                                     self.matset.values_ptr(k + 1), float(sigmas[k + 1]), k == 0)
                k += 2
            else:
                self.eng.add_values(self.map_ids[k], self.matset.values_ptr(k), float(sigmas[k]), k == 0)
                k += 1
        self.eng.factorize()
        return B200Factor(self.eng)

    def fixed_effects(self):
        """V^-1 C, chol(C'V^-1C), beta, V^-1 y, V^-1 (y - C beta)   (reference :29-34, one multi-RHS solve)."""
        return self._fixed_effects_finish(self._fixed_effects_start(overlap=False))

    def _fixed_effects_start(self, overlap=True):
        """Queues the (c+1)-column solve.  With overlap=True it goes to the engine's auxiliary stream: the narrow
        solve is a launch-latency-bound chain that leaves the SMs idle, so it runs beside the probe pipeline the
        caller issues on stream 0 next; _fixed_effects_finish joins the two."""
        torch = self.torch
        B = torch.cat([self.C, self.y.unsqueeze(1)], dim=1).contiguous()
        if overlap:
            self.eng.aux_begin()
            try:
                self.eng.solve_(B)
            finally:
                self.eng.aux_end()
        else:
            self.eng.solve_(B)
        return B, overlap

    def _fixed_effects_finish(self, pending):
        B, overlap = pending
        if overlap:
            self.eng.aux_join()
        c = self.C.shape[1]
        self._ViCy = B                                  # [V^-1 C | V^-1 y], kept for the Gram pass
        ViC = B[:, :c].contiguous()
        Viy = B[:, c].contiguous()
        CtViC = (self.C.t() @ ViC).cpu().numpy()
        CtViy = (self.C.t() @ Viy).cpu().numpy()
        chol = la.cho_factor(CtViC)
        beta = la.cho_solve(chol, CtViy)
        Vir = Viy - ViC @ self.torch.from_numpy(beta).to("cuda")       # V^-1 (y - C beta) by linearity
        return ViC, chol, beta, Viy, Vir

    def nll(self, logdet, beta, Vir, chol, reml):
        """Negative log-likelihood (reference :37-46) at the factored V from what fixed_effects() returned."""
        r = self.y - self.C @ self.torch.from_numpy(beta).to("cuda")
        nll = 0.5 * (float(r @ Vir) + self.n * LOG_2PI + logdet)
        if reml:
            nll += 0.5 * 2 * np.sum(np.log(np.diag(chol[0])))
        return nll

    @functools.cached_property
    def copy_stream(self):
        """CUDA stream of the host -> device copies that run under device work: probe and genotype blocks."""
        return self.torch.cuda.Stream()

    def draw_probes(self, sim_num):
        """The n x sim_num probe block of the next evaluation by functor.rng, as (Z, stream): Z drawn from the
        reference's global numpy stream (rng='numpy') or returned by probe_source (rng='host_buffer'), stream None;
        for rng='device' Z is None and stream is the evaluation index, the device stream that probes() draws only the
        local columns from."""
        if self.functor.rng == 'numpy':
            return np.random.randn(self.n, sim_num), None
        if self.functor.rng == 'host_buffer':
            return self.functor.probe_source(self.n, sim_num), None
        return None, self.n_eval

    def prefetch_probes(self, sim_num, Z, col_begin, col_end):
        """The local columns [col_begin, col_end) of the probe block Z (or of draw_probes() when Z is None) on the
        device: (device block, event to wait for or None), or (None, None) when the block is drawn on the device.
        Called BEFORE the factorization is queued: a whole contiguous float64 host tensor (pinned) goes up on the copy
        stream, so its DMA (207 MB at 128 columns and 250K individuals) runs under the factorization instead of after
        it; a host slice goes up by one pitched DMA; a CUDA block is copied, as the probe solve works in place."""
        torch = self.torch
        if Z is None:
            Z, _ = self.draw_probes(sim_num)
        if Z is None:
            return None, None
        if torch.is_tensor(Z) and Z.is_cuda:
            return Z[:, col_begin:col_end].clone(memory_format=torch.contiguous_format), None
        if not torch.is_tensor(Z):
            Z = np.ascontiguousarray(Z, dtype=np.float64)
        sliced = bool(col_begin or col_end != Z.shape[1])
        if torch.is_tensor(Z) and not (Z.dtype == torch.float64 and Z.is_contiguous()):
            return (Z[:, col_begin:col_end] if sliced else Z).contiguous().to("cuda", non_blocking=True), None
        if sliced:                                     # no packing of the slice on the host
            return _eng.upload_columns(Z, col_begin, col_end, torch), None
        if not torch.is_tensor(Z):
            return _eng.to_device(Z, torch), None
        with torch.cuda.stream(self.copy_stream):
            Zd = Z.to("cuda", non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        Zd.record_stream(torch.cuda.current_stream())
        return Zd, ev

    def probes(self, sim_num, Z=None, col_begin=0, col_end=None, pre=None, probe_stream=None):
        """W = V^-1 (L Z)[argsort P]   (reference :49-52) for the probe columns [col_begin, col_end) of the
        n x sim_num block Z, computed as P' L^-T Z: with P V P' = L L', V^-1 P' L Z = P' L^-T L^-1 L Z, so one
        backward half-sweep on Z (solve mode 3) replaces L Z and the full solve.  rng == 'device' draws ONLY those
        columns, from the counter-based stream keyed by (functor.seed, evaluation index or probe_stream, row, global
        column): the same values for any number of GPUs.  pre: what prefetch_probes returned for the same arguments."""
        col_end = sim_num if col_end is None else col_end
        Zd, ev = self.prefetch_probes(sim_num, Z, col_begin, col_end) if pre is None else pre
        if Zd is None:
            stream = self.n_eval if probe_stream is None else probe_stream
            Zd = self.eng.probe_normals(self.n, col_end - col_begin, col_begin, self.functor.seed, stream)
        elif ev is not None:
            self.torch.cuda.current_stream().wait_event(ev)
        return self.eng.solve_(Zd, mode=3)

    def _scan_blocks(self, sigmas, G, spans, red_len, reduce, finish, timing=None):
        """The genotype block pipeline of the association scan and the region tests.  For each column span (j0, j1) of
        the host (n, m) int8 matrix G, in order: int8 upload on a copy stream (span i + 1 goes up while span i is
        swept), one decode / centre / project kernel, one forward half-sweep F = L^-1 P x~ (solve mode 1), then
        reduce(i, F, buf), which queues the device reduction of span i's F into the float64 buffer buf of red_len(i)
        entries.  While the device sweeps span i, the host calls finish(i - 1, chol, q, t, nobs, gsum, red) with the
        host copies of span i - 1's projections q = (V^-1 C)' x~ (c x w) and t = (V^-1 r)' x~ (w), its non-missing
        counts and allele sums, and its reduction; chol is the Cholesky factor of C'V^-1 C (scipy.linalg.cho_factor).
        timing: a list that receives, per span, five timing events recorded on the compute stream around the upload
        wait, the genotype kernel, the sweep and the reduction (scripts/assoc_scan.py, scripts/region_scan.py)."""
        torch = self.torch
        n = self.n
        self.factor_at(sigmas)
        ViC, chol, _, _, Vir = self.fixed_effects()
        P = torch.cat([ViC, Vir.unsqueeze(1)], dim=1).contiguous()       # n x (c + 1)
        c1 = P.shape[1]
        block = max(j1 - j0 for j0, j1 in spans)
        nred = max(red_len(i) for i in range(len(spans)))
        # one int8 buffer: the upload of span i + 1 is issued after assoc_genotypes has returned for span i, and that
        # call waits for its kernels (device-side input check), so nothing still reads the buffer
        g8 = torch.empty(n * block, dtype=torch.int8, device="cuda")
        X = torch.empty(n * block, dtype=torch.float64, device="cuda")
        small = [dict(proj=torch.empty(c1 * block, dtype=torch.float64, device="cuda"),
                      nobs=torch.empty(block, dtype=torch.int64, device="cuda"),
                      gsum=torch.empty(block, dtype=torch.int64, device="cuda"),
                      red=torch.empty(nred, dtype=torch.float64, device="cuda")) for _ in range(2)]
        copy, main = self.copy_stream, torch.cuda.current_stream()
        uploaded = torch.cuda.Event()
        strides = [None]
        finish_s = self.last["finish_s"] = []          # host seconds per span: copies back + finish

        def upload(i):
            strides[0] = _eng.upload_genotype_block(G, spans[i][0], spans[i][1], g8, copy)
            uploaded.record(copy)

        def collect(i):
            """Host copies of span i's small outputs, whose kernels have completed.  They come back on the copy
            stream, so the host does not wait behind the sweep of span i + 1 queued on the compute stream."""
            w = spans[i][1] - spans[i][0]
            s = small[i % 2]
            t0 = time.perf_counter()
            with torch.cuda.stream(copy):
                proj = s["proj"][:c1 * w].view(c1, w).cpu().numpy()
                red = s["red"][:red_len(i)].cpu().numpy()
                nobs, gsum = s["nobs"][:w].cpu().numpy(), s["gsum"][:w].cpu().numpy()
            finish(i, chol, proj[:c1 - 1], proj[c1 - 1], nobs, gsum, red)
            finish_s.append(time.perf_counter() - t0)

        def mark(marks):
            if marks is not None:
                marks.append(torch.cuda.Event(enable_timing=True))
                marks[-1].record(main)

        upload(0)
        try:
            for i, (j0, j1) in enumerate(spans):
                w = j1 - j0
                s = small[i % 2]
                Xb = X[:n * w].view(n, w)
                marks = None if timing is None else []
                mark(marks)
                main.wait_event(uploaded)
                mark(marks)
                # returns once the kernels are done (device-side input check): span i - 1 is swept and reduced by then
                _eng.assoc_genotypes(g8, n, w, strides[0], P, Xb, s["proj"], s["nobs"], s["gsum"])
                mark(marks)
                self.eng.solve_(Xb, mode=1)
                mark(marks)
                reduce(i, Xb, s["red"])
                mark(marks)
                if timing is not None:
                    timing.append(marks)
                # while the device sweeps span i: statistics of span i - 1, then the host stages span i + 1
                if i > 0:
                    collect(i - 1)
                if i + 1 < len(spans):
                    upload(i + 1)
            main.synchronize()
            collect(len(spans) - 1)
        finally:
            torch.cuda.synchronize()                   # no copy may still target the buffers when they are freed

    def association(self, sigmas, G, block, col_begin=0, col_end=None, timing=None):
        """Mixed-model association test of the variants (columns) [col_begin, col_end) of the host (n, m) int8 genotype
        matrix G at the variance components `sigmas` (see association() for the statistic), in blocks of `block`
        variants through _scan_blocks, with a column sum of squares as the reduction and the c x c finalisation on the
        host.  Returns a dict of arrays of length col_end - col_begin in the units of the standardised y: beta, se,
        chi2, p, af, n_obs, and the score t with its variance xPx (score, var).  timing: as for _scan_blocks."""
        _check_scan_covariates(self.C.shape[1])
        col_end = G.shape[1] if col_end is None else int(col_end)
        m_loc = max(col_end - col_begin, 0)
        out = {k: np.full(m_loc, np.nan) for k in ("beta", "se", "chi2", "p", "af", "score", "var")}
        out["n_obs"] = np.zeros(m_loc, dtype=np.int64)
        if m_loc == 0:
            return out
        block = max(1, min(int(block), m_loc))
        spans = [(j0, min(j0 + block, col_end)) for j0 in range(col_begin, col_end, block)]

        def finish(i, chol, q, t, nobs, gsum, ss):
            j0, j1 = spans[i]
            xPx = ss - np.sum(q * la.cho_solve(chol, q), axis=0)
            ok = xPx > 1e-10 * ss                      # monomorphic (ss = 0) or in the span of C: NaN
            sl = slice(j0 - col_begin, j1 - col_begin)
            with np.errstate(invalid="ignore", divide="ignore"):
                xPx = np.where(ok, xPx, np.nan)
                out["beta"][sl] = t / xPx
                out["se"][sl] = 1.0 / np.sqrt(xPx)
                out["chi2"][sl] = t * t / xPx
                out["p"][sl] = special.chdtrc(1, out["chi2"][sl])
                out["af"][sl] = gsum / nobs / 2.0
                out["score"][sl] = np.where(ok, t, np.nan)
                out["var"][sl] = xPx
            out["n_obs"][sl] = nobs

        self._scan_blocks(sigmas, G, spans, lambda i: spans[i][1] - spans[i][0],
                          lambda i, F, buf: _eng.assoc_colsumsq(F, buf), finish, timing)
        return out

    def region_test(self, sigmas, G, bounds, weights, block, reg_begin=0, reg_end=None, timing=None):
        """Burden and SKAT tests of the regions [reg_begin, reg_end) of the host (n, m) int8 genotype matrix G (region r
        is the columns [bounds[r], bounds[r+1])) at the variance components `sigmas`; see region_test() for the
        statistics.  Consecutive whole regions are packed greedily into spans of `block` columns (no region straddles
        two), and each span goes through _scan_blocks with the region Gram (slmm_assoc_region_gram) as the
        reduction.  weights: length-m per-variant weights, or None for the default beta(maf; 1, 25).  Returns a dict of
        arrays of length reg_end - reg_begin in the units of the standardised y.  timing: as for _scan_blocks."""
        _check_scan_covariates(self.C.shape[1])
        bounds = np.asarray(bounds, dtype=np.int64)
        reg_end = len(bounds) - 1 if reg_end is None else int(reg_end)
        R = max(reg_end - reg_begin, 0)
        out = {k: np.full(R, np.nan) for k in REGION_FLOAT_KEYS}
        out["n_variants"] = (bounds[reg_begin + 1:reg_end + 1] - bounds[reg_begin:reg_end]).astype(np.int64)
        out["n_poly"] = np.zeros(R, dtype=np.int64)
        if R == 0:
            return out
        if int(out["n_variants"].max()) > block:
            raise ValueError("a region of %d variants does not fit a block of %d" % (out["n_variants"].max(), block))
        groups = []                                    # per span: its region indices [r0, r1)
        r0 = reg_begin
        for r in range(reg_begin, reg_end):
            if bounds[r + 1] - bounds[r0] > block:
                groups.append((r0, r))
                r0 = r
        groups.append((r0, reg_end))
        # every span is `block` columns wide (short only at the end of G): the sweep keeps one solve plan instead of
        # building one per width.  The columns after a span's last region are swept too and go to the Gram as regions
        # of at most 64 columns, cut at the 64-column strips, whose squares are ignored.
        m = G.shape[1]
        spans, rel = [], []
        for a, b in groups:
            j0 = int(bounds[a])
            width = min(block, m - j0)
            used = int(bounds[b]) - j0
            pad = list(range((used // 64 + 1) * 64, width, 64)) + [width] if used < width else []
            spans.append((j0, j0 + width))
            rel.append(np.concatenate([bounds[a:b + 1] - j0, pad]).astype(np.int32))

        def finish(i, chol, q, t, nobs, gsum, red):
            j0, j1 = spans[i]
            if weights is None:
                with np.errstate(invalid="ignore", divide="ignore"):
                    wts = skat_weights(gsum / nobs / 2.0)
            else:
                wts = weights[j0:j1]
            off = 0
            for k in range(groups[i][1] - groups[i][0]):
                a, b = int(rel[i][k]), int(rel[i][k + 1])
                FtF = red[off:off + (b - a) ** 2].reshape(b - a, b - a)
                off += (b - a) ** 2
                qr = q[:, a:b]
                Phi = FtF - qr.T @ la.cho_solve(chol, qr)
                r = groups[i][0] + k - reg_begin
                for key, v in region_statistics(t[a:b], Phi, FtF, wts[a:b]).items():
                    out[key][r] = v

        self._scan_blocks(sigmas, G, spans, lambda i: int(np.sum(np.diff(rel[i]).astype(np.int64) ** 2)),
                          lambda i, F, buf: _eng.assoc_region_gram(F, rel[i], buf), finish, timing)
        return out

    def blup(self, sigmas, matset, groups, colmap=None, probes=0, block_begin=0, block_end=None):
        """Device side of blup(): the predicted random effects of the K matrices of `matset` (over all N individuals;
        `groups`: their pattern groups of <= 2) from this session's fit on the observed individuals, at `sigmas` (this
        session's components, the residual last).  colmap: device int32 map of the N columns to this session's rows
        (-1 = no phenotype) or None when the matset is this session's own.  In the units of the standardised y.

        Returns a dict: U (N x K, sigma_k A_k[:, obs] u with u = V^-1 (y_s - C beta)), u (n), beta, corr (N x K, the
        fixed-effect term diag(sigma_k A_k V^-1 C M^-1 C'V^-1 A_k sigma_k) of the PEV, M = C'V^-1 C) and, with
        probes > 0, parts: one [nblocks, 2, N, G] CUDA tensor per group holding sum_j t_ij^2 and sum_j t_ij^4 of
        t = sigma_k A_k[:, obs] W for the probe blocks [block_begin, block_end) of BLUP_BLOCK columns (other slots 0).
        W = P' L^-T Z with Z from the device Philox stream (functor.seed, BLUP_PROBE_STREAM) whatever functor.rng is,
        one block of columns at a time (the draw and backward half-sweep of probes() for rng='device')."""
        torch = self.torch
        c = self.C.shape[1]
        if c + 1 > BLUP_MAX_COLUMNS:
            raise ValueError("blup takes at most %d covariates, got %d" % (BLUP_MAX_COLUMNS - 1, c))
        self.factor_at(sigmas)
        ViC, chol, beta, _, u = self.fixed_effects()
        X = torch.cat([u.unsqueeze(1), ViC], dim=1).contiguous()          # [u | V^-1 C], c + 1 <= 32 columns
        Minv = torch.from_numpy(la.cho_solve(chol, np.eye(c))).to("cuda")
        N, K = matset.n, len(sigmas) - 1
        U = torch.empty(N, K, dtype=torch.float64, device="cuda")
        corr = torch.empty(N, K, dtype=torch.float64, device="cuda")
        for ks in groups:
            Y = matset.blup_spmm(ks, [sigmas[k] for k in ks], X, colmap)
            for g, k in enumerate(ks):
                U[:, k] = Y[g, :, 0]
                Yc = Y[g, :, 1:]
                corr[:, k] = ((Yc @ Minv) * Yc).sum(dim=1)
        out = {"U": U, "u": u, "beta": beta, "corr": corr}
        if probes <= 0:
            return out
        nblocks = -(-int(probes) // BLUP_BLOCK)
        block_end = nblocks if block_end is None else block_end
        parts = [torch.zeros(nblocks, 2, N, len(ks), dtype=torch.float64, device="cuda") for ks in groups]
        for b in range(block_begin, block_end):
            c0 = b * BLUP_BLOCK
            w = min(int(probes), c0 + BLUP_BLOCK) - c0
            Z = self.eng.probe_normals(self.n, w, c0, self.functor.seed, BLUP_PROBE_STREAM)
            W = self.eng.solve_(Z, mode=3)
            for ks, part in zip(groups, parts):
                matset.blup_rowsumsq(ks, [sigmas[k] for k in ks], W, part[b, 0], part[b, 1], colmap)
            del Z, W
        out["parts"] = parts
        return out

    def spa(self, G, cols, score, var, mu, w, block, timing=None):
        """Saddlepoint p-values (slmm_assoc_spa) of the columns `cols` of the host (n, m) int8 genotype matrix G, given
        their scores U (`score`) and Var(U) (`var`) and the fitted means `mu` and weights `w` (host, length n).  The
        columns are gathered on the host in order and go up `block` at a time; slmm_assoc_genotypes with P = W C decodes
        and centres them and gives (W C)' x~.  Returns (p, status, iters) of length len(cols); see glmm_association().
        timing: a list that receives two timing events per block around the saddlepoint kernel."""
        torch = self.torch
        n, c, m = self.n, self.C.shape[1], len(cols)
        p, status, iters = np.full(m, np.nan), np.zeros(m, dtype=np.int8), np.zeros(m, dtype=np.int32)
        if m == 0:
            return p, status, iters
        CtWC = self.C_host.T @ (w[:, None] * self.C_host)
        Minv = _eng.to_device(la.cho_solve(la.cho_factor(CtWC), np.eye(c)), torch)
        mu_d, w_d = _eng.to_device(mu, torch), _eng.to_device(w, torch)
        WC = (w_d[:, None] * self.C).contiguous()
        block = max(1, min(int(block), m))
        f64 = dict(dtype=torch.float64, device="cuda")
        g8 = torch.empty(n * block, dtype=torch.int8, device="cuda")
        X = torch.empty(n * block, **f64)
        work = torch.empty(n * block, **f64)
        proj, sc, vr, pd = (torch.empty(k, **f64) for k in (c * block, block, block, block))
        nobs, gsum = (torch.empty(block, dtype=torch.int64, device="cuda") for _ in range(2))
        st, it = (torch.empty(block, dtype=torch.int32, device="cuda") for _ in range(2))
        for j0 in range(0, m, block):
            j1 = min(j0 + block, m)
            wd = j1 - j0
            Gb = G[:, cols[j0:j1]]
            if not (Gb.flags.c_contiguous or Gb.flags.f_contiguous):
                Gb = np.ascontiguousarray(Gb)
            strides = _eng.upload_genotype_block(Gb, 0, wd, g8)
            Xb = X[:n * wd].view(n, wd)
            _eng.assoc_genotypes(g8, n, wd, strides, WC, Xb, proj, nobs, gsum)
            sc[:wd].copy_(torch.from_numpy(np.ascontiguousarray(score[j0:j1], dtype=np.float64)))
            vr[:wd].copy_(torch.from_numpy(np.ascontiguousarray(var[j0:j1], dtype=np.float64)))
            if timing is not None:
                timing.append([torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)])
                timing[-1][0].record()
            _eng.assoc_spa(Xb, proj, Minv, self.C, mu_d, w_d, sc, vr, work, pd, st, it)
            if timing is not None:
                timing[-1][1].record()
            p[j0:j1] = pd[:wd].cpu().numpy()
            status[j0:j1] = st[:wd].cpu().numpy()
            iters[j0:j1] = it[:wd].cpu().numpy()
        return p, status, iters

    def _is_identity(self, k):
        m = self.mats_host[k]
        return m.nnz == self.n and np.array_equal(m.indices, np.arange(self.n)) and np.all(m.data == 1.0)

    def _ai_start(self, u, ViC):
        """First half of the average-information matrix at u = P y = V^-1 r: B = [A_1 u | ... | A_K u] (one
        store-enabled pass of the group SpMM per pattern group; the identity's column is u itself), the c x K
        projection block ViC' B, and the K-column FORWARD half-sweep F = L^-1 P B queued on the auxiliary stream so
        that it runs beside the quadratic-form pass the caller issues next.  _ai_finish joins the two."""
        torch = self.torch
        u1 = u.unsqueeze(1).contiguous()
        B = torch.empty(self.n, self.K, dtype=torch.float64, device="cuda")
        for ks in self._groups:
            rest = [k for k in ks if not self._ident[k]]
            for k in ks:
                if self._ident[k]:
                    B[:, k] = u
            if rest:
                _, stored = self.matset.coldot_multi(rest, u1, 0)
                for g, k in enumerate(rest):
                    B[:, k] = stored[g, :, 0]
        CtB = ViC.t() @ B                              # read before the in-place solve below
        self.eng.aux_begin()
        try:
            self.eng.solve_(B, mode=1)
        finally:
            self.eng.aux_end()
        return B, CtB

    def _ai_finish(self, pending, chol, reml):
        """AI_ij = 1/2 b_i' P b_j = 1/2 [F_i'F_j - (ViC'b_i)' (C'V^-1C)^-1 (ViC'b_j)]: b'V^-1 b' = (L^-1 P b)'(L^-1 P b'),
        and a Gram matrix does not depend on the row order.  ML (reml=False) drops the projection term."""
        F, CtB = pending
        self.eng.aux_join()
        AI = (F.t() @ F).cpu().numpy()
        if reml:
            CtB = CtB.cpu().numpy()
            AI -= CtB.T @ la.cho_solve(chol, CtB)
        AI = 0.5 * AI
        return 0.5 * (AI + AI.T)

    def evaluate(self, sigmas, reml, sim_num, Z=None, ai=False, probe_stream=None):
        """One REML evaluation: nll and d nll / d sigma  (reference :77-117 without the exp chain rule).
        ai=True also returns the average-information matrix AI = -compute_hess (symmetric components only):
        (nll, grad, AI).  probe_stream: index of the device probe stream (rng='device') to draw from instead of the
        evaluation counter; an AI-REML fit keeps one for all its iterations."""
        torch = self.torch
        # probe columns are sharded across ranks when torch.distributed is initialised
        rank, world = _shard.rank_world()
        lo, hi = _shard.column_block(sim_num, rank, world)
        pre = self.prefetch_probes(sim_num, Z, lo, hi)      # a host block goes up under the factorization
        self.factor_at(sigmas)
        logdet = self.eng.logdet()
        pending = self._fixed_effects_start(self.overlap)   # narrow solve on the auxiliary stream ...
        # ... beside the probe pipeline
        W = self.probes(sim_num, Z, lo, hi, pre=pre, probe_stream=probe_stream)
        self.n_eval += 1
        ViC, chol, beta, Viy, Vir = self._fixed_effects_finish(pending)
        if ai:
            if not all(self._sym):
                raise ValueError("the average-information matrix needs symmetric components")
            ai_pending = self._ai_start(Vir, ViC)      # forward sweep on the auxiliary stream ...
        nll = self.nll(logdet, beta, Vir, chol, reml)
        c = self.C.shape[1]
        K = self.K
        comp1 = torch.zeros(K, dtype=torch.float64, device="cuda")
        comp2 = torch.zeros(K, dtype=torch.float64, device="cuda")
        gram = torch.zeros(K, c, c, dtype=torch.float64, device="cuda")
        # Per pattern group ONE pass over the matrices: column quadratic forms of the probes W (symmetric matrices
        # are traversed on/below the diagonal only) and, riding along, the Gram matrix of the narrow block
        # B = [V^-1 C | V^-1 r]: its last diagonal entry is r'V^-1 A_k V^-1 r (:66), its leading c x c block feeds
        # the REML trace term (:70).
        s_loc = W.shape[1]
        Bq = self._ViCy
        Bq[:, c] = Vir                                 # Viy was copied out above; the block becomes [V^-1 C | V^-1 r]
        nbq = Bq.shape[1]
        for ks in self._groups:
            if self.use_tiles and self.matset.has_tiles(ks) and nbq <= 16 and nbq + s_loc <= 160:
                # tiled pass: X = [narrow block | probes], gathered rows staged in shared memory once per tile
                dots, G = self.matset.quadform_tiled(ks, torch.cat([Bq, W], dim=1), nbq)
                for g, k in enumerate(ks):
                    comp1[k] = dots[g, nbq:].sum()
                    comp2[k] = G[g][c, c]
                    gram[k] = G[g][:c, :c]
            elif all(self._sym[k] for k in ks) and Bq.shape[1] <= 16 and s_loc <= 160:
                dots, G = self.matset.quadform_gram_multi(ks, W, Bq)
                for g, k in enumerate(ks):
                    comp1[k] = dots[g].sum()
                    comp2[k] = G[g][c, c]
                    gram[k] = G[g][:c, :c]
            else:                                      # general matrices / very wide blocks: separate passes
                X = torch.cat([W, Vir.unsqueeze(1)], dim=1).contiguous()
                dots = self.matset.quadform_multi(ks, X)
                if reml:
                    _, stored = self.matset.coldot_multi(ks, ViC, 0)
                for g, k in enumerate(ks):
                    comp1[k] = dots[g, :s_loc].sum()
                    comp2[k] = dots[g, s_loc]
                    if reml:
                        gram[k] = ViC.t() @ stored[g]
        _shard.allreduce_sum_(comp1)                   # the only collective of an evaluation: K doubles
        comp1 = (comp1 / sim_num).cpu().numpy()
        comp2 = comp2.cpu().numpy()
        grad = 0.5 * (comp1 - comp2)
        if reml:
            gram_h = gram.cpu().numpy()
            for k in range(K):
                grad[k] -= 0.5 * np.trace(la.cho_solve(chol, gram_h[k]))
        self.last = dict(logdet=logdet, beta=beta, ViC=ViC, Vir=Vir, Viy=Viy, W=W, chol=chol)
        if ai:                                         # ... joined here; every rank computes it in full
            return nll, grad, self._ai_finish(ai_pending, chol, reml)
        return nll, grad


def _need_functor(cholesky_func):
    if not isinstance(cholesky_func, SparseCholesky):
        raise TypeError("scilmm_b200 needs its own SparseCholesky() functor as cholesky_func "
                        "(the engine has no CPU / CHOLMOD path)")
    return cholesky_func


# ------------------------------------------------------------------------------------------- reference API
def matrices_weighted_sum(mats, sig2g_array):
    """reference :55-59.  Host scipy assembly for callers that want V itself; the fused path never forms it."""
    V = sig2g_array[0] * mats[0]
    for i in range(1, len(sig2g_array)):
        V = V + sig2g_array[i] * mats[i]
    return V.tocsc()


def estimate_fixed_effects(factor, y, covariates):
    """reference :29-34."""
    invV_C = factor(covariates)
    L_CT_invV_C = la.cho_factor(covariates.T.dot(invV_C))
    fixed_effects = la.cho_solve(L_CT_invV_C, covariates.T.dot(factor(y)))
    mu = covariates.dot(fixed_effects)
    return invV_C, L_CT_invV_C, mu, fixed_effects


def negative_log_likelihood(factor, y, invV_y, mu, L_CT_invV_C, reml):
    """reference :37-46."""
    n = y.size
    nll = 0.5 * ((y - mu).dot(invV_y) + n * LOG_2PI + factor.logdet())
    if reml:
        nll += 0.5 * 2 * np.sum(np.log(np.diag(L_CT_invV_C[0])))
    return nll


def simulate_vector(factor, n, sim_num, p_inv=None):
    """reference :49-52: V^-1 (L Z)[argsort P] with Z from the global numpy stream, computed as P' L^-T Z by one
    backward half-sweep (RemlSession.probes); stays on the device until the final copy.  p_inv is accepted for
    signature compatibility (the engine applies P itself)."""
    torch = _eng.require_cuda()
    factor._check()
    Z = _eng.to_device(np.random.randn(n, sim_num), torch)
    return factor._chol.solve_(Z, mode=3).cpu().numpy()


def compute_gradients(sig2g_array, mats, sim_vec, invV_y, reml, invV_C, L_CT_invV_C):
    """reference :62-74 on the GPU kernels (fused SpMM + column reductions)."""
    torch = _eng.require_cuda()
    ms = _eng.MatSet(mats)
    W = _eng.to_device(np.asarray(sim_vec, dtype=np.float64), torch)
    r = _eng.to_device(np.asarray(invV_y, dtype=np.float64), torch)
    X = torch.cat([W, r.unsqueeze(1)], dim=1).contiguous()
    ViC = _eng.to_device(np.asarray(invV_C, dtype=np.float64), torch)
    grad = np.zeros(len(sig2g_array))
    for k in range(len(sig2g_array)):
        d = ms.quadform_multi([k], X)[0].cpu().numpy()
        grad[k] = 0.5 * (np.mean(d[:-1]) - d[-1])
        if reml:
            vec = (ViC.t() @ ms.spmm(k, ViC)).cpu().numpy()
            grad[k] -= 0.5 * np.trace(la.cho_solve(L_CT_invV_C, vec))
    return grad


def bolt_gradient_estimation(log_sig2g_array, cholesky_func, mats, covariates, y, reml, sim_num, verbose,
                             take_exp=True):
    """One REML evaluation (nll, gradient), reference :77-117."""
    functor = _need_functor(cholesky_func)
    sig2g_array = np.exp(log_sig2g_array) if take_exp else np.asarray(log_sig2g_array, dtype=float)
    if verbose:
        t0 = time.time()
        print('estimating nll and its gradient at:', sig2g_array)
    ses = functor._session(mats, covariates, y)
    nll, grad = ses.evaluate(sig2g_array, reml, sim_num)
    if take_exp:
        grad = grad * sig2g_array
    if verbose:
        print("grad : ", grad)
        print('nll: %0.8e   computation time: %0.2f seconds' % (nll, time.time() - t0))
    return nll, grad


def _he_start(mats, covariates, y):
    """reference :123-128: HE estimates of the first K-1 components, the rest to the identity, normalised."""
    he_est = HE(mats[:-1], covariates, y, compute_stderr=False)
    he_est = np.concatenate((he_est, [1 - he_est.sum()]))
    x0 = he_est
    if np.any(x0 < 0):
        x0 = np.ones((len(mats)))
    return x0 / x0.sum()


# AI-REML (Gilmour, Thompson & Cullis 1995; with Monte-Carlo traces and one probe block per fit as in BOLT-REML,
# Loh et al. 2015).  y is standardised by REML(), so an absolute floor is meaningful.
AIREML_FLOOR = 1e-6       # smallest variance component
AIREML_TOL = 1e-4         # stop when max |delta log sigma| < AIREML_TOL
AIREML_MAX_ITER = 30


def _aireml_step(sig, grad, AI):
    """Fisher scoring in theta = log sigma: g_t = sigma o grad, H_t = D AI D, delta = -H_t^-1 g_t.
    Boundary: a component on the floor whose score still points down (grad > 0) is fixed; a free component whose
    linearised step is delta_k <= -1 (sigma_k (1 + delta_k) <= 0) goes to the floor in this step and is fixed, and the
    others take the step of the reduced system with that move included.  The step is scaled to max |delta| <= 1.
    Returns (new sigma, size of the step: max |delta| before the scaling, jumps to the floor included)."""
    sig, grad = np.asarray(sig, dtype=float), np.asarray(grad, dtype=float)
    K = sig.size
    gt = sig * grad
    Ht = sig[:, None] * AI * sig[None, :]
    fixed = (sig <= AIREML_FLOOR) & (grad > 0)
    while True:
        free = np.flatnonzero(~fixed)
        lin = np.where(fixed, (AIREML_FLOOR - sig) / sig, 0.0)     # linearised move of the fixed components
        delta = np.zeros(K)
        if free.size:
            delta[free] = -np.linalg.solve(Ht[np.ix_(free, free)], gt[free] + Ht[free] @ lin)
        hit = ~fixed & (delta <= -1.0)
        if not hit.any():
            break
        fixed |= hit
    size = float(np.max(np.abs(delta[free]))) if free.size else 0.0
    if size > 1.0:
        delta = delta / size
    new = np.where(fixed, np.minimum(sig, AIREML_FLOOR), np.maximum(sig * np.exp(delta), AIREML_FLOOR))
    if fixed.any():
        size = max(size, float(np.max(np.log(sig[fixed] / new[fixed]))))
    return new, size


def _aireml_fit(functor, mats, covariates, y, reml, sim_num, verbose):
    """HE start + AI-REML on the session.  Every iteration uses the SAME probe block (one numpy draw, one
    probe_source call or one device stream index), so the fit is a deterministic root-finding problem.  Every rank
    computes the AI matrix in full and takes the same step.  Returns (sigma, {'iterations', 'converged'})."""
    sig = _he_start(mats, covariates, y)
    ses = functor._session(mats, covariates, y)
    if not all(ses._sym):
        raise ValueError("aireml=True needs symmetric components (AI = -hess holds only for symmetric A_k); "
                         "asymmetric: %s" % [k for k in range(ses.K) if not ses._sym[k]])
    Z, stream = ses.draw_probes(sim_num)
    converged, it = False, 0
    while it < AIREML_MAX_ITER:
        it += 1
        if verbose:
            t0 = time.time()
        nll, grad, AI = ses.evaluate(sig, reml, sim_num, Z=Z, ai=True, probe_stream=stream)
        sig, size = _aireml_step(sig, grad, AI)
        if verbose:
            print('AI-REML iteration %d: nll %0.8e, sigma %s, max |step| %.3e, %.2f seconds'
                  % (it, nll, sig, size, time.time() - t0))
        if size < AIREML_TOL:
            converged = True
            break
    if not converged:
        print('optimization failed with message: AI-REML did not converge in %d iterations' % AIREML_MAX_ITER)
    return sig, {"iterations": it, "converged": converged}


def estimate_var_comps(cholesky_func, mats, covariates, y, reml=True, sim_num=100, verbose=True, aireml=False):
    """reference :120-144.  aireml=True: average-information REML (_aireml_fit) instead of L-BFGS-B."""
    if aireml:
        return _aireml_fit(_need_functor(cholesky_func), mats, covariates, y, reml, sim_num, verbose)[0]
    x0 = _he_start(mats, covariates, y)
    optObj = optimize.minimize(bolt_gradient_estimation, np.log(x0),
                               args=(cholesky_func, mats, covariates, y, reml, sim_num, verbose, True),
                               jac=True, method='L-BFGS-B', options={'eps': 1e-5, 'ftol': 1e-7})
    if not optObj.success:
        print('optimization failed with message: %s' % optObj.message)
    return np.exp(optObj.x)


def _hess_device(ses, factor_eng, pre=None):
    """-0.5 y' P A_i P A_j P y on the device (reference :147-168) in THREE multi-RHS solves instead of the
    reference's 1 + K + K(K+1)/2 single-column ones: [C | y] (c+1 columns; reused from the caller when `pre` =
    (ViC, chol, Viy) is given), the K columns A_j P y, and the K(K+1)/2 columns A_i P A_j P y."""
    torch = ses.torch
    K = ses.K
    C, y = ses.C, ses.y
    c = C.shape[1]
    if pre is None:
        B = torch.cat([C, y.unsqueeze(1)], dim=1).contiguous()
        factor_eng.solve_(B)
        ViC, Viy = B[:, :c].contiguous(), B[:, c].contiguous()
        chol = la.cho_factor((C.t() @ ViC).cpu().numpy())
    else:
        ViC, chol, Viy = pre
    Minv = torch.from_numpy(la.cho_solve(chol, np.eye(c))).to("cuda")

    def project_solved(Viz):  # Viz = V^-1 z  ->  P z
        return Viz - ViC @ (Minv @ (C.t() @ Viz))

    def project(Zb):          # Zb: n x k block
        return project_solved(factor_eng.solve_(Zb.clone().contiguous()))

    Py = project_solved(Viy.unsqueeze(1))
    AjPy = torch.cat([ses.matset.spmm(j, Py) for j in range(K)], dim=1)       # n x K
    PAjPy = project(AjPy)
    pairs = [(i, j) for i in range(K) for j in range(i, K)]
    # A_i (P A_j P y) for all j >= i in ONE pass over A_i (a block of K - i columns)
    cols = torch.cat([ses.matset.spmm(i, PAjPy[:, i:].contiguous()) for i in range(K)], dim=1)
    vals = (-0.5 * (y @ project(cols))).cpu().numpy()
    hess = np.empty((K, K))
    for q, (i, j) in enumerate(pairs):
        hess[i, j] = hess[j, i] = vals[q]
    return hess


def compute_hess(mats, covariates, factor, y):
    """reference :147-168.  `factor` must be a B200Factor; solves are batched per stage."""
    if not isinstance(factor, B200Factor):
        raise TypeError("compute_hess needs a B200Factor")
    factor._check()
    ses = _AdHocSession(mats, covariates, y)
    return _hess_device(ses, factor._chol)


class _AdHocSession(object):
    def __init__(self, mats, covariates, y):
        torch = _eng.require_cuda()
        self.torch = torch
        self.K = len(mats)
        self.matset = _eng.MatSet(mats)
        self.C = _eng.to_device(np.asarray(covariates, dtype=np.float64), torch)
        self.y = _eng.to_device(np.asarray(y, dtype=np.float64), torch)


def compute_varcomp_stderr(mats, covariates, factor, y, sim_num):
    """reference :171-174."""
    hess = compute_hess(mats, covariates, factor, y)
    inv_neg_hess = la.inv(-hess)
    return np.sqrt(np.diag(inv_neg_hess) * (1 + 1.0 / sim_num))


def REML(cholesky_func, mats, covariates, y, reml=True, sim_num=100, verbose=False, aireml=False):
    """reference :177-189.  Returns the reference's three keys plus 'nll' (the log-likelihood the reference
    computes at :103 but drops) and 'engine' statistics.  aireml=True fits the variance components by AI-REML
    (see _aireml_fit) and adds the key 'aireml': {'iterations', 'converged'}."""
    functor = _need_functor(cholesky_func)
    y = y / y.std()
    mats = mats + [sparse.eye(y.shape[0]).tocsr()]
    if aireml:
        varcomp_estimates, ai_info = _aireml_fit(functor, mats, covariates, y, reml, sim_num, verbose)
    else:
        varcomp_estimates = estimate_var_comps(functor, mats, covariates, y, reml, sim_num, verbose)
    ses = functor._session(mats, covariates, y)
    factor = ses.factor_at(varcomp_estimates)
    ViC, chol, fixed_effects, Viy, Vir = ses.fixed_effects()
    nll = ses.nll(factor.logdet(), fixed_effects, Vir, chol, reml)
    hess = _hess_device(ses, ses.eng, pre=(ViC, chol, Viy))
    sigmas_sigmas = np.sqrt(np.diag(la.inv(-hess)) * (1 + 1.0 / sim_num))
    out = {"covariance coefficients": varcomp_estimates,
           "covariates coefficients": fixed_effects,
           "covariance std": sigmas_sigmas,
           "nll": nll,
           "engine": ses.eng.stats()}
    if aireml:
        out["aireml"] = ai_info
    return out


# ------------------------------------------------------------------------------------------- association scan
ASSOC_BLOCK = 512         # variants per block of the public scan: the fastest width measured (DESIGN.md 6c)
ASSOC_MAX_COVARIATES = 31   # [V^-1 C | V^-1 r] is projected in registers, c + 1 <= 32 (csrc/assoc.cu)
# device bytes a block holds per (individual, variant): x~, the solve plan of its width, int8 and small buffers.  Measured
# 40.7 / 41.9 / 49.3 at widths 512 / 256 / 128 (profiles/r05_assoc_scan.json).  The width is chosen so that these fit
# in half the free memory; the other half covers the plan of a narrower tail block, which is no larger.
ASSOC_BYTES_PER_ENTRY = 50


def _check_genotypes(G, n):
    """G as a C- or Fortran-ordered (n, m) int8 ndarray (a copy in C order when it is neither); ValueError otherwise."""
    G = np.asarray(G)
    if G.ndim != 2 or G.dtype != np.int8:
        raise ValueError("G must be a 2-D int8 array of allele counts (negative = missing)")
    if G.shape[0] != n:
        raise ValueError("G has %d rows for %d individuals" % (G.shape[0], n))
    if not (G.flags.c_contiguous or G.flags.f_contiguous):
        G = np.ascontiguousarray(G)
    return G


def _check_sigmas(sigmas, K):
    """sigmas as a float array of K + 1 variance components (the residual last); ValueError otherwise."""
    sigmas = np.asarray(sigmas, dtype=float)
    if sigmas.shape != (K + 1,):
        raise ValueError("need %d variance components (the residual last), got %d" % (K + 1, sigmas.size))
    return sigmas


def _check_scan_covariates(c):
    if c > ASSOC_MAX_COVARIATES:
        raise ValueError("the association scan takes at most %d covariates, got %d" % (ASSOC_MAX_COVARIATES, c))


def _scan_width(n, bytes_per_entry, floor):
    """Columns per genotype block: ASSOC_BLOCK, or as many as fit bytes_per_entry per (individual, column) into half
    the free device memory, and at least `floor`."""
    free = _eng.require_cuda().cuda.mem_get_info()[0]
    return int(max(floor, min(ASSOC_BLOCK, free // 2 // (bytes_per_entry * n))))


def _scan_session(functor, mats, covariates, y):
    """The session REML() left for the same inputs, or a new one.  REML() appends its own identity and divides y by
    its std into a new array, so those two are matched by content; the caller's matrices and covariates by the
    session key (object and content fingerprint)."""
    for ses in list(functor._sessions.values()):
        m_s, _, y_s = ses._refs
        if len(m_s) == len(mats) + 1 and ses._ident[-1] and m_s[-1].shape[0] == y.shape[0] \
                and np.array_equal(y_s, y):
            return functor._session(list(mats) + [m_s[-1]], covariates, y_s)
    return functor._session(list(mats) + [sparse.eye(y.shape[0]).tocsr()], covariates, y)


def association(cholesky_func, mats, covariates, y, sigmas, G):
    """Mixed-model association scan (GCTA --mlma, EMMAX) of the variants in G at the variance components `sigmas`.

    Arguments as for REML(): `mats` without the identity, `sigmas` = REML()['covariance coefficients'] (K + 1 values,
    the residual last); V = sum_k sigma_k A_k + sigma_e I on y / y.std().  At most 31 covariates (columns of C).  A call after REML() on the same functor
    reuses its device session.  G: (n, m) int8 ndarray in C or Fortran order, rows in y's order, entries 0 / 1 / 2
    allele counts and negative values for missing (any other value raises SlmmError).

    Per variant x: mean imputation and centring (x~), q = (V^-1 C)' x~, t = (V^-1 r)' x~ with r = y - C beta,
    xPx = x~'V^-1 x~ - q' (C'V^-1 C)^-1 q, beta = t / xPx, se = xPx^-1/2, chi2 = t^2 / xPx, p its chi^2_1 survival
    function: the coefficient of x~ and its standard error in the GLS fit of [C | x~] under the same V.  beta and se
    are in the units of y.  Monomorphic variants and those in the span of C (xPx <= 1e-10 x~'V^-1 x~) get NaN.

    Returns a dict of length-m arrays: beta, se, chi2, p, af (allele frequency of the non-missing entries), n_obs.
    With torch.distributed initialised every rank scans a contiguous slice of the variants and one all-reduce gives
    every rank the whole result."""
    functor = _need_functor(cholesky_func)
    G = _check_genotypes(G, y.shape[0])
    _check_scan_covariates(np.shape(covariates)[1])
    sigmas = _check_sigmas(sigmas, len(mats))
    scale = y.std()
    ses = _scan_session(functor, mats, covariates, y / scale)
    n, m = G.shape
    block = _scan_width(n, ASSOC_BYTES_PER_ENTRY, 8)
    rank, world = _shard.rank_world()
    lo, hi = _shard.column_block(m, rank, world)
    keys = ("beta", "se", "chi2", "p", "af", "n_obs")
    part = _shard.gather_slices(ses.association(sigmas, G, block, lo, hi), keys, m, lo, hi, "cuda")
    part["beta"] = part["beta"] * scale
    part["se"] = part["se"] * scale
    return {k: part[k] for k in keys}


# ------------------------------------------------------------------------------------------- region tests
REGION_MAX = 512            # widest region: the region Gram gathers its square from at most 8 x 8 64-column tiles
REGION_FLOAT_KEYS = ("burden_beta", "burden_se", "burden_chi2", "burden_p", "skat_q", "skat_p")
REGION_KEYS = ("n_variants", "n_poly") + REGION_FLOAT_KEYS


def skat_weights(af):
    """Default SKAT weights beta.pdf(maf; 1, 25), maf = min(af, 1 - af); 0 where af is undefined (no genotype)."""
    af = np.asarray(af, dtype=np.float64)
    maf = np.minimum(af, 1.0 - af)
    return np.where(np.isnan(af), 0.0, stats.beta.pdf(np.nan_to_num(maf), 1, 25))


def chi2_mixture_sf(q, lam):
    """P(sum_i lam_i chi2_1 > q) for positive weights lam (independent chi2_1 terms).

    All weights equal (within 1e-9 relative): the exact chi2_r survival function.  Otherwise the Lugannani-Rice
    saddlepoint approximation (Kuonen 1999), with its limit 1/2 - K3(0) / (6 sqrt(2 pi) K2(0)^3/2) (K2, K3: second and
    third derivatives of the cumulant generating function) where the signed root w is within 1e-3 of 0 (q near
    sum lam, where the formula is 0/0).  Against the closed form for lam = (a, a, b, b), a/b from 1.5 to 1000, the
    relative error stays within 0.63 % for p > 0.5, 4.0 % for 1e-6 < p <= 0.5 and 7.3 % down to 1e-300.  One dominant
    weight with tiny others nears the single chi2_1 case, where the saddlepoint is about 15 % off in the far tail
    (DESIGN.md 6e).  q <= 0 gives 1."""
    lam = np.asarray(lam, dtype=np.float64).ravel()
    r = lam.size
    if q <= 0:
        return 1.0
    lmax = lam.max()
    if lmax - lam.min() <= 1e-9 * lmax:
        return float(stats.chi2.sf(q / lam.mean(), r))
    lam, q = lam / lmax, q / lmax                  # scale-free: the root lies in (lo, 1/2)

    def K1(z):
        return np.sum(lam / (1.0 - 2.0 * z * lam))

    lo = -r / (2.0 * q) - 1.0                      # K'(lo) < q
    hi = 0.5 * (1.0 - 1.0 / (q + lam.sum()))       # K'(hi) > 1 / (1 - 2 hi) = q + sum lam > q
    z = optimize.brentq(lambda z: K1(z) - q, lo, hi, xtol=1e-15, rtol=4 * np.finfo(float).eps, maxiter=500)
    d = 1.0 - 2.0 * z * lam
    K = -0.5 * np.sum(np.log(d))
    w = np.sign(z) * np.sqrt(max(2.0 * (z * q - K), 0.0))
    if abs(w) < 1e-3:
        k2, k3 = 2.0 * np.sum(lam ** 2), 8.0 * np.sum(lam ** 3)
        return float(0.5 - k3 / (6.0 * np.sqrt(2.0 * np.pi) * k2 ** 1.5))
    v = z * np.sqrt(2.0 * np.sum(lam ** 2 / d ** 2))
    p = stats.norm.sf(w) + stats.norm.pdf(w) * (1.0 / v - 1.0 / w)
    return float(min(max(p, 0.0), 1.0))


def region_statistics(t, Phi, FtF, w):
    """Burden and SKAT statistics of one region from t = (V^-1 r)' X~ (length w_r), Phi = X~' P_V X~ and
    FtF = X~' V^-1 X~ (w_r x w_r) and the weights w, in the units of the standardised y (see region_test()).  Returns a
    dict with n_poly and the finite entries of REGION_FLOAT_KEYS; the others are NaN."""
    out = {"n_poly": int(np.sum(np.diag(FtF) > 0))}
    s, v, vF = w @ t, w @ Phi @ w, w @ FtF @ w
    if v > 1e-10 * vF:                             # not monomorphic, not in the span of C
        chi2 = s * s / v
        out.update(burden_beta=s / v, burden_se=1.0 / np.sqrt(v), burden_chi2=chi2, burden_p=special.chdtrc(1, chi2))
    lam = np.linalg.eigvalsh(w[:, None] * Phi * w[None, :])
    if lam[-1] > 1e-10 * np.sum(w * w * np.diag(FtF)):     # trace(W F'F W) >= its largest eigenvalue
        lam = lam[lam > 1e-10 * lam[-1]]
        Q = float(np.sum((w * t) ** 2))
        out.update(skat_q=Q, skat_p=chi2_mixture_sf(Q, lam))
    return out


def check_regions(bounds, weights, m):
    """(bounds as int64, weights as float64 or None) after the input rules of region_test(); ValueError otherwise."""
    bounds = np.asarray(bounds)
    if bounds.ndim != 1 or bounds.size < 2 or not np.issubdtype(bounds.dtype, np.integer):
        raise ValueError("bounds must be a 1-D int array of at least 2 region offsets")
    bounds = bounds.astype(np.int64)
    if bounds[0] != 0 or bounds[-1] != m:
        raise ValueError("bounds must start at 0 and end at m = %d, got %d and %d" % (m, bounds[0], bounds[-1]))
    widths = np.diff(bounds)
    if np.any(widths <= 0):
        raise ValueError("bounds must strictly increase")
    if widths.max() > REGION_MAX:
        raise ValueError("a region has %d variants; at most %d are supported" % (widths.max(), REGION_MAX))
    if weights is not None:
        weights = np.asarray(weights, dtype=np.float64)
        if weights.shape != (m,):
            raise ValueError("weights must have one entry per variant (%d), got shape %s" % (m, weights.shape))
        if not np.all(np.isfinite(weights)) or np.any(weights < 0):
            raise ValueError("weights must be finite and >= 0")
    return bounds, weights


def region_test(cholesky_func, mats, covariates, y, sigmas, G, bounds, weights=None):
    """Region-based rare-variant tests (burden and SKAT against the kinship-aware null, as famSKAT) of the variants in G
    at the variance components `sigmas`.

    cholesky_func, mats, covariates, y, sigmas and G as for association() (int8 allele counts, C or Fortran order, at
    most 31 covariates, a call after REML() reuses its device session).  bounds: int array like an indptr; region r is
    the columns [bounds[r], bounds[r+1]) of G, with bounds[0] = 0, bounds[-1] = m, strictly increasing, 1 to
    REGION_MAX = 512 variants per region.  weights: one finite weight >= 0 per variant; by default beta.pdf(maf; 1, 25)
    with maf = min(af, 1 - af) from the allele frequency of the non-missing entries (0 for a variant without any).

    Per region, in the units of y_s = y / y.std(): t = (V^-1 r)' X~, Phi = X~' P_V X~ = F'F - q' M^-1 q (F = L^-1 P X~,
    q = (V^-1 C)' X~, M = C'V^-1 C) and W = diag(w).
      burden: s = w't, v = w'Phi w, beta = s / v, se = v^-1/2, chi2 = s^2 / v and p its chi^2_1 survival function: the
        coefficient of the burden score X~ w and its standard error in the GLS fit of [C | X~ w] under the same V.
        beta and se are in the units of y per unit of the burden score.  NaN when v <= 1e-10 w'F'F w (no polymorphic
        variant, or the burden score in the span of C).
      SKAT: Q = sum_j w_j^2 t_j^2.  Under the null t ~ N(0, Phi), so Q ~ sum_i lam_i chi2_1 with lam = eig(W Phi W);
        eigenvalues <= 1e-10 lam_max are dropped and p = chi2_mixture_sf(Q, lam).  Q is left in the standardised units
        (the p-value is scale-free).  NaN when lam_max <= 1e-10 trace(W F'F W): the region carries no variation
        beyond C (for one variant this is association()'s rule).

    Returns a dict of length-R arrays: n_variants, n_poly (variants with F_j'F_j > 0), burden_beta, burden_se,
    burden_chi2, burden_p, skat_q, skat_p.  With torch.distributed initialised every rank tests a contiguous slice of
    the regions and one all-reduce gives every rank the whole result."""
    functor = _need_functor(cholesky_func)
    G = _check_genotypes(G, y.shape[0])
    _check_scan_covariates(np.shape(covariates)[1])
    sigmas = _check_sigmas(sigmas, len(mats))
    n, m = G.shape
    bounds, weights = check_regions(bounds, weights, m)
    block = _scan_width(n, ASSOC_BYTES_PER_ENTRY, 8)
    if np.diff(bounds).max() > block:
        raise ValueError("the widest region (%d variants) does not fit the %d columns that device memory allows"
                         % (np.diff(bounds).max(), block))
    scale = y.std()
    ses = _scan_session(functor, mats, covariates, y / scale)
    R = bounds.size - 1
    rank, world = _shard.rank_world()
    lo, hi = _shard.column_block(R, rank, world)
    part = _shard.gather_slices(ses.region_test(sigmas, G, bounds, weights, block, lo, hi), REGION_KEYS, R, lo, hi,
                                "cuda")
    part["burden_beta"] = part["burden_beta"] * scale
    part["burden_se"] = part["burden_se"] * scale
    return {k: part[k] for k in REGION_KEYS}


# ------------------------------------------------------------------------------------------- predicted random effects
BLUP_MAX_COLUMNS = 32       # [u | V^-1 C] goes through slmm_blup_spmm in one pass, one column per lane (csrc/blup.cu)
BLUP_BLOCK = 128            # probe columns per block of the PEV estimate (one mode-3 sweep, one rowsumsq pass)
BLUP_PROBE_STREAM = 2 ** 62   # Philox stream of the PEV probes: REML evaluations count their streams up from 0


def blup(cholesky_func, mats, covariates, y, sigmas, pev_probes=0):
    """Predicted random effects (BLUP) of every individual, phenotyped or not, at the variance components `sigmas`.

    mats: the K relationship matrices over all N individuals, without the identity (as for REML()).  covariates: N x c,
    finite on every row (the unphenotyped rows give their fixed part); c + 1 <= 32.  y: length N, NaN for an individual
    without a phenotype.  sigmas: REML()['covariance coefficients'] (K + 1 values, the residual last) of the fit on the
    phenotyped individuals:

        obs = ~np.isnan(y)
        sigmas = REML(chol, [A[obs][:, obs] for A in mats], covariates[obs], y[obs])['covariance coefficients']

    The model is REML's: s = y[obs].std(), y_s = y[obs] / s, V = sum_k sigma_k A_k[obs, obs] + sigma_e I,
    u = V^-1 (y_s - C beta) with the GLS beta.  Returns a dict:
      u: N x K, u_k = s sigma_k A_k[:, obs] u (the usual BLUP on the phenotyped rows, E[u_k | y] on the others);
      residual: length N, s sigma_e u on the phenotyped rows, NaN elsewhere;
      fixed: length N, s C beta;  beta: s beta;  yhat: fixed + u.sum(1).
    With pev_probes = p >= 2, also N x K arrays (units of y^2 for the first two):
      pev: prediction error variance sigma_k A_k,ii - sigma_k^2 (A_k P A_k)_ii, P = V^-1 - V^-1 C M^-1 C'V^-1,
        M = C'V^-1 C.  The fixed-effect term is exact; diag(A_k V^-1 A_k) is a Monte Carlo estimate from p probe
        columns W = P' L^-T Z (E[W W'] = V^-1), about sqrt(2 / p) relative error per entry (12 % at 128, 4 % at 1024);
      pev_se: its Monte Carlo standard error;
      reliability: 1 - pev / (sigma_k A_k,ii), NaN where that is 0.
    The probes always come from the device Philox stream keyed by the functor's `seed` (stream BLUP_PROBE_STREAM,
    which no REML evaluation uses), whatever its `rng` setting: the same seed gives the same bits.

    Without a NaN in y this is the in-sample prediction and a call after REML() on the same functor and inputs reuses
    its device session.  With NaN the phenotyped blocks A_k[obs][:, obs] are cut on the host and a session is set up on
    them (the cached analysis is reused when their pattern is the one REML() fitted); like any new session on the
    functor, it replaces the one REML() left, so a later call on the full inputs sets its session up again.  With
    torch.distributed initialised every rank sweeps a slice of the probe blocks; the PEV is the same bits for any
    number of ranks."""
    functor = _need_functor(cholesky_func)
    y = np.asarray(y, dtype=np.float64)
    C = np.asarray(covariates, dtype=np.float64)
    K = len(mats)
    N = y.shape[0]
    if y.ndim != 1:
        raise ValueError("y must be a vector")
    if K == 0 or any(m.shape != (N, N) for m in mats):
        raise ValueError("every matrix must be N x N with N = len(y) = %d" % N)
    sigmas = _check_sigmas(sigmas, K)
    if C.ndim != 2 or C.shape[0] != N:
        raise ValueError("covariates must be N x c with N = %d" % N)
    if not np.all(np.isfinite(C)):
        raise ValueError("covariates must be finite on every row, the unphenotyped ones included")
    if C.shape[1] + 1 > BLUP_MAX_COLUMNS:
        raise ValueError("blup takes at most %d covariates, got %d" % (BLUP_MAX_COLUMNS - 1, C.shape[1]))
    if np.any(np.isinf(y)):
        raise ValueError("y must be finite or NaN (no phenotype)")
    obs = ~np.isnan(y)
    n = int(obs.sum())
    if n < C.shape[1] + 1:
        raise ValueError("need at least c + 1 = %d phenotyped individuals, got %d" % (C.shape[1] + 1, n))
    p = int(pev_probes)
    if p < 0 or p == 1:
        raise ValueError("pev_probes must be 0 or at least 2")
    torch = _eng.require_cuda()
    scale = y[obs].std()
    if n == N:
        ses = _scan_session(functor, mats, covariates, y / scale)
        matset = ses.matset
        groups = [[k for k in ks if k < K] for ks in ses._groups]
        groups = [ks for ks in groups if ks]
        colmap = None
    else:
        idx = np.flatnonzero(obs)
        sub = [_eng.canonical_csr(m)[idx][:, idx] for m in mats]
        ses = _scan_session(functor, sub, C[idx], y[idx] / scale)
        matset = _eng.MatSet(mats)
        groups = matset.pattern_groups(2)
        colmap = np.full(N, -1, dtype=np.int32)
        colmap[idx] = np.arange(n, dtype=np.int32)
        colmap = _eng.to_device(colmap, torch)
    rank, world = _shard.rank_world()
    nblocks = -(-p // BLUP_BLOCK)
    lo, hi = _shard.column_block(nblocks, rank, world)
    res = ses.blup(sigmas, matset, groups, colmap, p, lo, hi)
    U = res["U"].cpu().numpy()
    resid = np.full(N, np.nan)
    resid[obs] = sigmas[-1] * res["u"].cpu().numpy()
    fixed = C @ res["beta"]
    out = {"u": scale * U, "residual": scale * resid, "fixed": scale * fixed, "yhat": scale * (fixed + U.sum(axis=1)),
           "beta": scale * res["beta"]}
    if p == 0:
        return out
    # every rank filled its own blocks' slots and zeros elsewhere: the sum over ranks adds exact zeros, and the
    # blocks are then added in one fixed order, so the estimate is the same bits for any number of ranks
    flat = torch.cat([part.reshape(-1) for part in res["parts"]])
    _shard.allreduce_sum_(flat)
    s2 = torch.empty(N, K, dtype=torch.float64, device="cuda")
    s4 = torch.empty(N, K, dtype=torch.float64, device="cuda")
    off = 0
    for ks, part in zip(groups, res["parts"]):
        part = flat[off:off + part.numel()].view(part.shape)
        off += part.numel()
        acc = part[0].clone()
        for b in range(1, nblocks):
            acc += part[b]
        for g, k in enumerate(ks):
            s2[:, k], s4[:, k] = acc[0, :, g], acc[1, :, g]
    diag = np.stack([sigmas[k] * _eng.canonical_csr(m).diagonal() for k, m in enumerate(mats)], axis=1)
    s2, s4, corr = s2.cpu().numpy(), s4.cpu().numpy(), res["corr"].cpu().numpy()
    pev = diag - s2 / p + corr
    se = np.sqrt(np.maximum(s4 - s2 * s2 / p, 0.0) / (p * (p - 1.0)))
    with np.errstate(invalid="ignore", divide="ignore"):
        out["reliability"] = np.where(diag != 0, 1.0 - pev / np.where(diag != 0, diag, 1.0), np.nan)
    out["pev"] = scale * scale * pev
    out["pev_se"] = scale * scale * se
    return out


# ------------------------------------------------------------------------------------------- binary traits
GLMM_TOL = 1e-5             # GMMAT's stopping rule on the relative changes of alpha and tau
GLMM_MAX_ITER = 50
GLMM_MU_EPS = 2.220446049250313e-16   # mu is clamped to [eps, 1 - eps], as R's binomial() (csrc/glmm.cu)
IRLS_TOL = 1e-10            # GLM start: stop when max |delta alpha| < IRLS_TOL (1 + max |alpha|)
IRLS_MAX_ITER = 100
# device bytes a saddlepoint block holds per (individual, variant): x~ and g~ in float64 and the int8 block
SPA_BYTES_PER_ENTRY = 20
GLMM_ASSOC_KEYS = ("beta", "se", "score", "chi2", "p", "p_normal", "spa", "af", "n_obs")


def _logit_working(eta, y):
    """(mu, w, Y~) of the logit link at eta, the formulas of slmm_glmm_working."""
    mu = np.clip(special.expit(eta), GLMM_MU_EPS, 1.0 - GLMM_MU_EPS)
    w = mu * (1.0 - mu)
    return mu, w, eta + (y - mu) / w


def _irls(C, y):
    """Logistic GLM (no random effects) by iteratively reweighted least squares from mu = (y + 1/2) / 2.  Returns alpha."""
    mu = (y + 0.5) / 2.0
    eta = np.log(mu / (1.0 - mu))
    alpha = np.zeros(C.shape[1])
    for _ in range(IRLS_MAX_ITER):
        _, w, z = _logit_working(eta, y)
        new = la.solve(C.T @ (w[:, None] * C), C.T @ (w * z), assume_a="pos")
        step = np.max(np.abs(new - alpha))
        alpha = new
        eta = C @ alpha
        if step < IRLS_TOL * (1.0 + np.max(np.abs(alpha))):
            break
    return alpha


def _check_binary(mats, covariates, y):
    """(C, y) as float64 after the input rules of glmm(); ValueError otherwise."""
    y = np.asarray(y, dtype=np.float64)
    if y.ndim != 1:
        raise ValueError("y must be a vector")
    n = y.shape[0]
    if len(mats) == 0 or any(m.shape != (n, n) for m in mats):
        raise ValueError("every matrix must be n x n with n = len(y) = %d" % n)
    C = np.asarray(covariates, dtype=np.float64)
    if C.ndim != 2 or C.shape[0] != n:
        raise ValueError("covariates must be n x c with n = %d" % n)
    if not np.all(np.isfinite(C)):
        raise ValueError("covariates must be finite")
    if np.any(np.isnan(y)):
        raise ValueError("y must not contain NaN")
    if not np.all((y == 0.0) | (y == 1.0)):
        raise ValueError("y must be 0 (control) or 1 (case)")
    if y.min() == y.max():
        raise ValueError("y needs both cases and controls")
    return C, y


def _glmm_session(functor, mats, covariates, Yt, w):
    """The functor's PQL session over mats + [W^-1] (W^-1 a diagonal CSR) with its device phenotype set to the working
    vector Yt and its diagonal values to 1 / w.  The session of an earlier call on the same mats and covariates (content
    fingerprint) is reused: only the two device vectors are rewritten, and not even those when they
    already hold Yt and 1 / w.  The session is never in the content-keyed cache (SparseCholesky._session): its host
    copies of y and W^-1 stop describing its device state after the first iteration."""
    torch = _eng.require_cuda()
    key = (tuple((m.shape, int(m.nnz), _fingerprint(m.data)) for m in mats),
           _fingerprint(covariates, with_sum=True))
    ses = functor._glmm
    D = 1.0 / w
    if ses is None or ses.glmm_key != key:
        functor._glmm = None                       # the old session's device memory goes before the new one is set up
        n = Yt.shape[0]
        Dm = sparse.csr_matrix((D, np.arange(n, dtype=np.int32), np.arange(n + 1, dtype=np.int32)), shape=(n, n))
        ses = RemlSession(functor, list(mats) + [Dm], covariates, Yt)
        ses.glmm_key = key
        functor._glmm = ses
    elif not (np.array_equal(ses.glmm_state[0], Yt) and np.array_equal(ses.glmm_state[1], w)):
        ses.y.copy_(torch.from_numpy(np.ascontiguousarray(Yt)))
        ses.matset.device_arrays(ses.K - 1)[2].copy_(torch.from_numpy(D))
    ses.glmm_state = (np.array(Yt, dtype=np.float64), np.array(w, dtype=np.float64))
    return ses


def glmm(cholesky_func, mats, covariates, y, sim_num=100, verbose=False):
    """Logistic mixed model of a 0/1 trait, fitted by penalised quasi-likelihood (PQL; Breslow & Clayton 1993) with
    GMMAT's average-information scheme (glmmkin, Chen et al. 2016): logit P(y_i = 1) = (C alpha)_i + b_i with random
    effects b ~ N(0, sum_k tau_k A_k) and the dispersion fixed at 1.

    mats: the K relationship matrices (n x n) without an identity; covariates: n x c, finite, with the intercept
    column; y: length n, 0 (control) or 1 (case), both present.  Anything else raises ValueError before any device work.

    Start: a logistic GLM by IRLS on the host gives alpha and eta = C alpha; tau_k = var(Y~) / (K + 1).  Per iteration:
    mu = logistic(eta) clamped to [eps, 1 - eps] (eps = 2.22e-16), w = mu (1 - mu), the working vector
    Y~ = eta + (y - mu) / w and Sigma = W^-1 + sum_k tau_k A_k; one REML evaluation with the average-information matrix
    on (Sigma, Y~) (RemlSession.evaluate), then an EM step tau_k <- max(floor, tau_k - 2 tau_k^2 grad_k / n) in the
    first iteration and the AI-REML step of REML(aireml=True) restricted to the K components after; alpha = the GLS
    coefficients of the evaluation and eta = Y~ - W^-1 Sigma^-1 (Y~ - C alpha) (the BLUP identity: no product with the
    A_k).  Stops when 2 max(|d alpha| / (|alpha| + |alpha_old| + tol), |d tau| / (|tau| + |tau_old| + tol)) < tol,
    tol = 1e-5, or after GLMM_MAX_ITER iterations (reported as REML() reports non-convergence).  Every iteration uses
    the same probe block (one numpy draw, one probe_source call or one device stream index), as REML(aireml=True) does,
    and under torch.distributed the probe columns are sharded the same way.  The working vector, W^-1 and eta stay on
    the device between iterations: slmm_glmm_working updates them in place.

    Returns a dict: 'covariance coefficients' (tau, logit scale) and 'covariance std' (sqrt(diag(AI^-1) (1 + 1/sim_num))
    from the last iteration's AI matrix); 'covariates coefficients' (alpha) and 'covariates std' (from (C'Sigma^-1 C)^-1
    of the last iteration); 'latent fractions' tau_k / (sum tau + pi^2 / 3), the liability-scale variance shares; 'mu',
    'eta', 'weights' (w) and 'working y' (Y~) of the returned alpha and random effects; 'glmm': {'iterations',
    'converged'}.  The fit's device session stays on the functor for glmm_association()."""
    functor = _need_functor(cholesky_func)
    C, y = _check_binary(mats, covariates, y)
    torch = _eng.require_cuda()
    n, K = y.shape[0], len(mats)
    alpha = _irls(C, y)
    eta = C @ alpha
    _, w, Yt = _logit_working(eta, y)
    tau = np.full(K, np.var(Yt, ddof=1) / (K + 1))
    ses = _glmm_session(functor, mats, covariates, Yt, w)
    if not all(ses._sym):
        raise ValueError("glmm needs symmetric relationship matrices; asymmetric: %s"
                         % [k for k in range(K) if not ses._sym[k]])
    Z, stream = ses.draw_probes(sim_num)
    y_d = _eng.to_device(y, torch)
    dvals = ses.matset.device_arrays(K)[2]
    eta_d = torch.empty(n, dtype=torch.float64, device="cuda")
    mu_d = torch.empty(n, dtype=torch.float64, device="cuda")
    converged, it = False, 0
    while it < GLMM_MAX_ITER:
        it += 1
        if verbose:
            t0 = time.time()
        nll, grad, AI = ses.evaluate(np.concatenate([tau, [1.0]]), True, sim_num, Z=Z, ai=True, probe_stream=stream)
        grad, AI = grad[:K], AI[:K, :K]
        tau_old, alpha_old = tau, alpha
        if it == 1:
            tau = np.maximum(AIREML_FLOOR, tau - 2.0 * tau * tau * grad / n)
        else:
            tau = _aireml_step(tau, grad, AI)[0]
        alpha = ses.last["beta"]
        _eng.glmm_working(ses.y, ses.last["Vir"], dvals, y_d, eta_d, mu_d)
        change = 2.0 * max(np.max(np.abs(alpha - alpha_old) / (np.abs(alpha) + np.abs(alpha_old) + GLMM_TOL)),
                           np.max(np.abs(tau - tau_old) / (np.abs(tau) + np.abs(tau_old) + GLMM_TOL)))
        if verbose:
            print('PQL iteration %d: nll %0.8e, tau %s, alpha %s, change %.3e, %.2f seconds'
                  % (it, nll, tau, alpha, change, time.time() - t0))
        if change < GLMM_TOL:
            converged = True
            break
    if not converged:
        print('optimization failed with message: PQL did not converge in %d iterations' % GLMM_MAX_ITER)
    mu = mu_d.cpu().numpy()
    w = mu * (1.0 - mu)                            # the kernel's w, bit for bit
    Yt = ses.y.cpu().numpy()
    ses.glmm_state = (Yt.copy(), w.copy())
    var_alpha = la.cho_solve(ses.last["chol"], np.eye(C.shape[1]))
    return {"covariance coefficients": tau,
            "covariance std": np.sqrt(np.diag(la.inv(AI)) * (1 + 1.0 / sim_num)),
            "covariates coefficients": alpha,
            "covariates std": np.sqrt(np.diag(var_alpha)),
            "latent fractions": tau / (tau.sum() + np.pi ** 2 / 3),
            "mu": mu, "eta": eta_d.cpu().numpy(), "weights": w, "working y": Yt,
            "glmm": {"iterations": it, "converged": converged}}


def glmm_association(cholesky_func, mats, covariates, y, fit, G, spa_cutoff=2.0):
    """Score test of each variant (column) of G against the logistic mixed model `fit` = glmm(...) of the same
    cholesky_func, mats, covariates and y, with saddlepoint-calibrated p-values (SAIGE, Zhou et al. 2018).

    G: (n, m) int8 ndarray in C or Fortran order, 0 / 1 / 2 allele counts and negative values for missing (any other
    value raises SlmmError), at most 31 covariates.  Phase 1 is the association scan (RemlSession.association) on the
    fit's session (Sigma = W^-1 + sum_k tau_k A_k, Y~; reused after glmm() on the same functor, otherwise set up from
    the fit's arrays without refitting): the score U = x~' P Y~ = x~' (y - mu) at the fixed point, Var(U) = x~' P x~,
    z = U / sqrt(Var(U)) and its normal p.  Phase 2 takes the variants with finite |z| > spa_cutoff: per variant
    g~ = x~ - C (C'WC)^-1 C'W x~, q = U sqrt(g~'W g~ / Var(U)) (the variance ratio of this variant, exactly), and the
    two-sided saddlepoint p-value of q under the cumulant generating function
    K(t) = sum_i log(1 - mu_i + mu_i e^{g~_i t}) - t sum_i g~_i mu_i: the roots of K'(zeta) = +-|q| and the
    Lugannani-Rice tail of each side, on the device (slmm_assoc_spa).  A variant whose |q| is outside the range of K',
    whose root is not bracketed, or whose signed root w is within 1e-3 of 0 keeps its normal p.

    Returns a dict of length-m arrays: beta = U / Var(U) (the one-step logit-scale effect) and se = Var(U)^-1/2, score
    (U), chi2 = z^2, p (the saddlepoint p where it was applied, the normal p otherwise), p_normal, spa (int8: 1 applied,
    0 below the cutoff, -1 fell back), af, n_obs.  Monomorphic variants and those in the span of C get NaN as in
    association().  With torch.distributed initialised every rank tests a contiguous slice of the variants in both
    phases and one all-reduce gives every rank the whole result."""
    functor = _need_functor(cholesky_func)
    C, y = _check_binary(mats, covariates, y)
    n, K = y.shape[0], len(mats)
    G = _check_genotypes(G, n)
    _check_scan_covariates(C.shape[1])
    spa_cutoff = float(spa_cutoff)
    if not spa_cutoff >= 0.0:
        raise ValueError("spa_cutoff must be >= 0")
    tau = np.asarray(fit["covariance coefficients"], dtype=np.float64)
    if tau.shape != (K,) or not np.all(np.isfinite(tau)) or np.any(tau < 0):
        raise ValueError("fit has %s covariance coefficients for %d matrices" % (tau.shape, K))
    mu, w, Yt = (np.asarray(fit[k], dtype=np.float64) for k in ("mu", "weights", "working y"))
    if any(a.shape != (n,) or not np.all(np.isfinite(a)) for a in (mu, w, Yt)) or not np.all(w > 0):
        raise ValueError("fit's mu, weights and working y must be finite vectors of length n = %d (weights > 0)" % n)
    ses = _glmm_session(functor, mats, covariates, Yt, w)
    m = G.shape[1]
    rank, world = _shard.rank_world()
    lo, hi = _shard.column_block(m, rank, world)
    part = ses.association(np.concatenate([tau, [1.0]]), G, _scan_width(n, ASSOC_BYTES_PER_ENTRY, 8), lo, hi)
    U, V = part["score"], part["var"]
    with np.errstate(invalid="ignore", divide="ignore"):
        z = U / np.sqrt(V)
    part["p_normal"] = part["p"].copy()
    part["spa"] = np.zeros(hi - lo, dtype=np.int8)
    flag = np.flatnonzero(np.isfinite(z) & (np.abs(np.nan_to_num(z)) > spa_cutoff))
    ps, status, iters = ses.spa(G, lo + flag, U[flag], V[flag], mu, w, _scan_width(n, SPA_BYTES_PER_ENTRY, 1))
    ses.last["spa_iters"] = iters
    part["spa"][flag] = status
    ok = status == 1
    part["p"][flag[ok]] = ps[ok]
    part = _shard.gather_slices(part, GLMM_ASSOC_KEYS, m, lo, hi, "cuda")
    return {k: part[k] for k in GLMM_ASSOC_KEYS}


# ------------------------------------------------------------------------------------------- Haseman-Elston
HE_TIMINGS = None      # set to a dict to collect the phases of the next he_moments call (upload / kernels)


def he_moments(mat_list, y, MQS=False, matset=None):
    """q and S of the HE normal equations on the GPU (reference :213-243).

    With torch.distributed initialised (world > 1) the rows are sharded: every rank uploads and holds ONLY its row
    block of every matrix (blocks balanced by the entries on/below the diagonal, which is what the kernels read),
    computes its partial moments, and one all-reduce of 2K + 2K^2 doubles combines them."""
    torch = _eng.require_cuda()
    rank, world = _shard.rank_world()
    t0 = time.time()
    if matset is not None:
        ms = matset
    elif world == 1:
        ms = _eng.MatSet(mat_list)
    else:
        big = max(range(len(mat_list)), key=lambda k: mat_list[k].nnz)
        bounds = _shard.row_blocks_by_lower_nnz(sparse.csr_matrix(mat_list[big]), world)
        ms = _eng.MatSet(mat_list, row_range=(int(bounds[rank]), int(bounds[rank + 1])))
    K, n = ms.K, ms.n
    y_dev = _eng.to_device(np.asarray(y, dtype=np.float64), torch)
    if HE_TIMINGS is not None:
        torch.cuda.synchronize()
        HE_TIMINGS["upload_s"] = time.time() - t0
        t0 = time.time()
    if ms.row_range == (0, n) and world == 1:
        out = ms.he_moments_device(y_dev).cpu().numpy()
    elif ms.row_range == (0, n):      # whole matrices on every rank (caller-supplied set): shard the rows only
        big = max(range(K), key=lambda k: ms.nnz[k])
        bounds = _shard.row_blocks_by_nnz(_eng._csr_arrays(mat_list[big])[0], world)
        part = ms.he_moments_device(y_dev, int(bounds[rank]), int(bounds[rank + 1])).clone()
        out = _shard.allreduce_sum_(part).cpu().numpy()
    else:
        ms.resolve_symmetry_sharded(_shard.allreduce_sum_)
        part = ms.he_moments_device(y_dev).clone()
        out = _shard.allreduce_sum_(part).cpu().numpy()
    if HE_TIMINGS is not None:
        HE_TIMINGS["moments_s"] = time.time() - t0
    q_off, q_diag, S_off, S_diag = _eng.MatSet.split_moments(out, K)
    if MQS:
        yy = float(np.dot(y, y))
        q = (q_off + q_diag) - yy
        S = (S_off + S_diag) - (n - 1)
    else:
        q, S = q_off, S_off
    return q, S, ms


def HE(mat_list, cov, y, MQS=False, verbose=False, sim_num=100, compute_stderr=False, y2=None, fix_indices=False):
    """Haseman-Elston regression, reference :192-281 (same outputs, including the bivariate mode's in-place
    mutation of mat_list / y2).

    Dense (ndarray) matrices - the reference's `else` branches at :224-231 - are converted to CSR and take the same
    kernels (explicit zeros contribute nothing to any moment).  sim_num=None is the reference's exact sampling
    variance (:260-268): <H A_i - H, H A_j - H>_F accumulated over blocks of unit vectors with SpMM kernels instead of
    sparse x sparse products (O(n/128) passes: small problems only, like the reference's).

    fix_indices=False reproduces the reference's K>1 indexing slips in the sampling-variance branch bit for bit
    (:254 weights every matrix after the first by he_est[K-1]; :262 rebinds mat_i to mat_list[j]; :267,:272 read the
    stale mat_j = mat_list[K-1]); they are harmless for K = 1.  fix_indices=True evaluates what the code intends:
    H = sum_k he_k A_k + (1 - sum he) I and V_q[i,j] = 2 tr(H (A_i - I) H (A_j - I))."""
    CTC = cov.T.dot(cov)
    y = y - cov.dot(np.linalg.solve(CTC, cov.T.dot(y)))
    y /= y.std()
    if y2 is not None:
        y2 -= cov.dot(np.linalg.solve(CTC, cov.T.dot(y2)))
        y2 /= y2.std()
        y = np.concatenate((y, y2))
        for m_i, m in enumerate(mat_list):
            m = m if sparse.issparse(m) else sparse.csr_matrix(np.asarray(m, dtype=np.float64))
            z = sparse.csr_matrix((m.shape[0], m.shape[0]))
            mat_list[m_i] = sparse.vstack([sparse.hstack([z, m]), sparse.hstack([m, z])]).tocsr()
    mats = [m if sparse.issparse(m) else sparse.csr_matrix(np.asarray(m, dtype=np.float64)) for m in mat_list]
    K = len(mats)
    n = y.shape[0]
    q, S, ms = he_moments(mats, y, MQS)
    he_est = np.linalg.solve(S, q)
    if not compute_stderr:
        return he_est

    torch = _eng.require_cuda()
    if ms.row_range != (0, ms.n):
        ms = _eng.MatSet(mats)          # the sampling-variance products need whole matrices on every rank
    stale = K - 1                       # reference :254 / :267,:272: loop variables left over from :216-232
    w = np.array([he_est[k if (fix_indices or k == 0) else stale] for k in range(K)])
    w_eye = 1.0 - he_est.sum()

    def Hdot(X):
        out = w_eye * X
        for k in range(K):
            if w[k] != 0.0:
                out = out + w[k] * ms.spmm(k, X)
        return out

    def minus_identity(k, X):           # (A_k - I) X
        return ms.spmm(k, X) - X

    V_q = np.empty((K, K))
    for i in range(K):
        for j in range(i + 1):
            if fix_indices:
                right, left = j, i
            else:
                right, left = stale, j  # the inner loop rebinds mat_i to mat_list[j] (:262); mat_j is stale
            if sim_num is None:
                # exact branch (:260-268): 2 <H A_i - H, H A_j - H>_F, column block by column block
                a_idx = i
                b_idx = i if j == i else (j if fix_indices else stale)
                acc = torch.zeros((), dtype=torch.float64, device="cuda")
                for c0 in range(0, n, 128):
                    c1 = min(n, c0 + 128)
                    E = torch.zeros(n, c1 - c0, dtype=torch.float64, device="cuda")
                    E[torch.arange(c0, c1, device="cuda"), torch.arange(c1 - c0, device="cuda")] = 1.0
                    Ua = Hdot(minus_identity(a_idx, E))
                    Ub = Ua if b_idx == a_idx else Hdot(minus_identity(b_idx, E))
                    acc += (Ua * Ub).sum()
                V_q[i, j] = 2 * float(acc)
            else:
                Zs = _eng.to_device(np.random.randn(n, sim_num), torch)
                t2 = Hdot(minus_identity(right, Zs))
                t4 = Hdot(minus_identity(left, t2))
                V_q[i, j] = 2 * float((Zs * t4).sum(dim=0).mean())
            V_q[j, i] = V_q[i, j]
    var_he_est = np.linalg.solve(S, np.linalg.solve(S, V_q).T).T
    return he_est, np.sqrt(np.diag(var_he_est))


def MINQUE(cholesky_func, mat_list, cov, y, compute_stderr=False, verbose=False, num_iter=100, sim_num=100):
    """Iterated MINQUE, reference :284-347 (same update rule, including the stale index at :335)."""
    functor = _need_functor(cholesky_func)
    torch = _eng.require_cuda()
    CTC = cov.T.dot(cov)
    y = y - cov.dot(np.linalg.solve(CTC, cov.T.dot(y)))
    y /= y.std()
    K = len(mat_list)
    n = y.shape[0]
    ms = _eng.MatSet(mat_list)
    y_dev = _eng.to_device(y, torch)
    yy = float(y.dot(y))
    H = None
    q = np.zeros(K)
    S = np.zeros((K, K))
    for iter_num in range(num_iter):
        q = np.zeros(K)
        S = np.zeros((K, K))
        if H is None:
            q0, S0, _ = he_moments(mat_list, y, MQS=True, matset=ms)
            q, S = q0, S0
        else:
            factor = functor(H)
            Z = _eng.to_device(np.random.randn(n, sim_num), torch)
            invH_simy = factor._chol.solve_(Z, mode=3)       # H^-1 (L Z)[argsort P] = P' L^-T Z
            invH_y = factor._chol.solve_(y_dev.clone())
            for i in range(K):
                q[i] = float(invH_y @ ms.spmm(i, invH_y)) - yy
                t = factor._chol.solve_(ms.spmm(i, invH_simy).contiguous())
                for j in range(i + 1):
                    S[i, j] = float((invH_simy * ms.spmm(j, t)).sum(dim=0).mean()) - (n - 1)
                    S[j, i] = S[i, j]
        minque_est = np.linalg.solve(S, q)
        if verbose:
            print(iter_num + 1, minque_est)
        stale_i = K - 1
        H = mat_list[0] * minque_est[0]
        for m in mat_list[1:]:
            H = H + m * minque_est[stale_i]
        H = H + sparse.eye(n, format='csr') * (1.0 - minque_est.sum())
    minque_est = np.linalg.solve(S, q)
    if not compute_stderr:
        return minque_est
    return minque_est, np.sqrt(0)


def run_estimates(A, df_phe, df_cov, reml=False, ignore_indices=False, df_phe2=None):
    """reference :350-395: align by IID, drop individuals without relatives, standardise covariates, fit.
    Differences: np.float -> float (:384) and the REML branch returns the dict instead of raising at :390."""
    import pandas as pd
    if not ignore_indices:
        indices = list(set(df_cov.index) & set(df_phe.index) & set(A.indices))
        df_cov = df_cov.loc[indices]
        df_phe = df_phe.loc[indices]
        if df_phe2 is not None:
            df_phe2 = df_phe2.loc[indices]
        A = A[indices][:, indices]
    has_relatives = np.asarray(A.sum(axis=1))[:, 0] > 1
    if any(~has_relatives):
        A = A[has_relatives][:, has_relatives]
        df_cov = df_cov.loc[has_relatives]
        df_phe = df_phe.loc[has_relatives]
        if df_phe2 is not None:
            df_phe2 = df_phe2.loc[has_relatives]
    A.eliminate_zeros()
    y = np.asarray(df_phe.values, dtype=float).reshape(-1)
    if df_phe2 is not None:
        y2 = np.asarray(df_phe2.values, dtype=float).reshape(-1)
        assert not reml
    else:
        y2 = None
    if isinstance(df_cov, pd.Series):
        df_cov = df_cov.to_frame()
    df_cov = df_cov.copy()
    df_cov['intercept'] = 1
    cov = df_cov.values.copy().astype(float)
    cov[:, :-1] -= cov[:, :-1].mean(axis=0)
    cov[:, :-1] /= cov[:, :-1].std(axis=0)
    if reml:
        reml_d = REML(SparseCholesky(), [A], cov, y, verbose=True)
        print("reml d are %s and %s" % (reml_d["covariance coefficients"], reml_d["covariance std"]))
        return reml_d
    he_est = HE([A], cov, y, compute_stderr=True, y2=y2)
    print("HE estimates are %s and %s" % (he_est[0], he_est[1]))
    return he_est


def run_estimates_from_paths(A, phe, cov, reml=False, ignore_indices=False):
    """reference :398-403."""
    import pandas as pd
    from scipy.io import mmread
    A = mmread(A).tocsr()
    index_col = None if ignore_indices else 0
    df_cov = pd.read_csv(cov, index_col=index_col)
    df_phe = pd.read_csv(phe, header=None, index_col=index_col)
    return run_estimates(A, df_phe, df_cov, reml=reml, ignore_indices=ignore_indices)
