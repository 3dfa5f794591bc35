"""Thin Python objects over the C-ABI handles.  torch is used only to own device memory and for the
tiny dense c x c / n x c algebra around the kernels; every sparse / factorization kernel is in
libscilmm_b200.so.  Nothing here computes on the CPU in place of a kernel."""
import ctypes as C

import numpy as np
import scipy.sparse as sp

from . import _lib
from ._lib import check, lib, np_ptr

ORDERINGS = {"natural": 0, "given": 1, "metis": 2, "nesdis": 2, "default": 2, "amd": 3, "mindeg": 3,
             "nesdis_fast": 4, "metis_fast": 4}


def _torch():
    import torch
    return torch


def require_cuda():
    torch = _torch()
    if not torch.cuda.is_available():
        raise RuntimeError("scilmm_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def device_count():
    c = C.c_int(0)
    check(lib().slmm_device_count(C.byref(c)))
    return c.value


def _as_i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def canonical_csr(m):
    """scipy CSR with sorted int32 indices and float64 data (the layout the reference hands scipy)."""
    m = sp.csr_matrix(m)
    if not m.has_sorted_indices:
        m = m.sorted_indices()
    if m.indices.dtype != np.int32 or m.indptr.dtype != np.int32:
        m = sp.csr_matrix((m.data, m.indices.astype(np.int32), m.indptr.astype(np.int32)), shape=m.shape)
    if m.data.dtype != np.float64:
        m = m.astype(np.float64)
    return m


UPLOAD_THREADS = 4          # worker threads of the staged upload (lowered when several ranks share the host's cores)


def to_device(a, torch=None):
    """Host ndarray -> CUDA tensor.  Large pageable arrays go through the library's ring of persistent pinned
    buffers (slmm_upload_h2d: no per-call page-locking, host copy overlapped with the DMA)."""
    torch = torch or require_cuda()
    a = np.ascontiguousarray(a)
    if a.nbytes < (4 << 20):
        return torch.from_numpy(a).to("cuda", non_blocking=False)
    out = torch.empty(a.shape, dtype=torch.from_numpy(a[:0].reshape(-1)).dtype, device="cuda")
    check(lib().slmm_upload_h2d(out.data_ptr(), np_ptr(a), int(a.nbytes), int(UPLOAD_THREADS)))
    return out


def upload_columns(Z, col_begin, col_end, torch=None, out=None, stream=None):
    """Columns [col_begin, col_end) of a C-ordered host float64 block (ndarray or CPU tensor, pinned or not) or int8
    genotype ndarray as a contiguous CUDA tensor: one pitched DMA, no host-side packing of the slice
    (slmm_upload_h2d_2d).  out: a device buffer of at least n * width elements of that dtype to fill instead of a new
    tensor; stream: a torch CUDA stream to issue the copy on instead of the default stream."""
    torch = torch or require_cuda()
    n, s = int(Z.shape[0]), int(Z.shape[1])
    if torch.is_tensor(Z):
        if Z.dtype != torch.float64 or not Z.is_contiguous() or Z.is_cuda:
            raise ValueError("upload_columns needs a contiguous float64 host block")
        src, itemsize, dtype = Z.data_ptr(), 8, torch.float64
    else:
        if Z.dtype not in (np.float64, np.int8) or not Z.flags.c_contiguous:
            raise ValueError("upload_columns needs a C-ordered float64 or int8 host block")
        src, itemsize = Z.ctypes.data, Z.itemsize
        dtype = torch.float64 if Z.dtype == np.float64 else torch.int8
    w = int(col_end) - int(col_begin)
    out = torch.empty(n, w, dtype=dtype, device="cuda") if out is None else out[:n * max(w, 0)].view(n, max(w, 0))
    if n == 0 or w <= 0:
        return out
    check(lib().slmm_upload_h2d_2d_on(out.data_ptr(), w * itemsize, src + int(col_begin) * itemsize, s * itemsize,
                                      w * itemsize, n, None if stream is None else stream.cuda_stream))
    return out


def upload_genotype_block(G, col_begin, col_end, out, stream=None):
    """Columns [col_begin, col_end) of a host (n, m) int8 genotype matrix into the flat device int8 buffer `out` (at
    least n * width entries) on `stream`.  Returns (row_stride, col_stride) of the block in `out`: a C-ordered matrix
    goes up as n rows of width bytes by one pitched DMA (strides (width, 1)); in a Fortran-ordered one the columns are
    one contiguous span, staged through the ring of pinned buffers (strides (1, n))."""
    n, w = int(G.shape[0]), int(col_end) - int(col_begin)
    if G.flags.c_contiguous:
        upload_columns(G, col_begin, col_end, out=out, stream=stream)
        return w, 1
    if not G.flags.f_contiguous or G.dtype != np.int8:
        raise ValueError("upload_genotype_block needs a C- or Fortran-ordered int8 host matrix")
    check(lib().slmm_upload_h2d_on(out.data_ptr(), G.ctypes.data + int(col_begin) * n, n * w, int(UPLOAD_THREADS),
                                   None if stream is None else stream.cuda_stream))
    return 1, n


def assoc_genotypes(Gd, n, width, strides, P, X, proj, nobs, gsum):
    """Association scan, device side of one genotype block (slmm_assoc_genotypes): decodes the int8 block Gd (element
    (i, j) at i * strides[0] + j * strides[1]) into X = centred allele counts (n x width, missing = 0), nobs / gsum =
    per-variant non-missing counts and allele sums (int64), proj = P' X for P = [V^-1 C | V^-1 r] (np x width).  An
    entry outside {0, 1, 2, negative} raises SlmmError."""
    check(lib().slmm_assoc_genotypes(Gd.data_ptr(), int(n), int(width), int(strides[0]), int(strides[1]), P.data_ptr(),
                                     int(P.shape[1]), X.data_ptr(), proj.data_ptr(), nobs.data_ptr(), gsum.data_ptr()))


def assoc_colsumsq(F, out):
    """out[j] = sum_i F[i, j]^2 of a contiguous n x width CUDA float64 block (slmm_assoc_colsumsq)."""
    check(lib().slmm_assoc_colsumsq(F.data_ptr(), int(F.shape[0]), int(F.shape[1]), out.data_ptr()))
    return out


# ------------------------------------------------------------------------------------------------ symbolic
class SymbolicView(object):
    """Host-only symbolic analysis (no GPU needed)."""

    def __init__(self, pattern, ordering="metis", perm=None):
        pattern = canonical_csr(pattern)
        n = pattern.shape[0]
        h = C.c_void_p()
        self._perm_in = None if perm is None else _as_i32(perm)
        code = ORDERINGS[ordering] if perm is None else 1
        check(lib().slmm_symbolic_create(n, np_ptr(pattern.indptr), np_ptr(pattern.indices), code,
                                         None if perm is None else np_ptr(self._perm_in), C.byref(h)))
        self._h = h
        self.n = n
        i = np.zeros(16, dtype=np.int64)
        d = np.zeros(8, dtype=np.float64)
        check(lib().slmm_symbolic_stats(h, np_ptr(i), np_ptr(d)))
        self.nsuper, self.nlevels, self.nnzL, self.lsize = int(i[1]), int(i[2]), int(i[3]), int(i[4])
        self.exported_nnz, self.max_front_rows, self.max_super_cols = int(i[5]), int(i[6]), int(i[7])
        self.ncomponents, self.total_rows = int(i[8]), int(i[9])
        self.flops, self.t_order, self.t_symbolic = float(d[0]), float(d[1]), float(d[2])

    def arrays(self):
        n, ns = self.n, self.nsuper
        out = dict(perm=np.zeros(n, np.int32), parent=np.zeros(n, np.int32), colcount=np.zeros(n, np.int32),
                   sn_first=np.zeros(ns + 1, np.int32), sn_nrow=np.zeros(ns, np.int32),
                   sn_parent=np.zeros(ns, np.int32), sn_rowptr=np.zeros(ns + 1, np.int64),
                   sn_lptr=np.zeros(ns + 1, np.int64), rows=np.zeros(self.total_rows, np.int32),
                   rel=np.zeros(self.total_rows, np.int32), level_ptr=np.zeros(self.nlevels + 1, np.int32),
                   level_sn=np.zeros(ns, np.int32))
        order = ["perm", "parent", "colcount", "sn_first", "sn_nrow", "sn_parent", "sn_rowptr", "sn_lptr", "rows",
                 "rel", "level_ptr", "level_sn"]
        check(lib().slmm_symbolic_arrays(self._h, *[np_ptr(out[k]) for k in order]))
        # leading dimension of every panel: rows rounded up to even (csrc/symbolic.h panel_ld: 16-byte aligned columns)
        out["sn_ld"] = ((out["sn_nrow"].astype(np.int64) + 1) & ~np.int64(1)).astype(np.int64)
        return out

    def entry_map(self, pattern):
        pattern = canonical_csr(pattern)
        tgt = np.zeros(pattern.nnz, dtype=np.int64)
        check(lib().slmm_symbolic_entry_map(self._h, np_ptr(pattern.indptr), np_ptr(pattern.indices), np_ptr(tgt)))
        return tgt

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().slmm_symbolic_destroy(self._h)
                self._h = None
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------ matrices
def _csr_arrays(m, row_range=None):
    """(indptr, indices, data, nnz) of a scipy CSR matrix as int32/int32/float64 contiguous arrays WITHOUT scanning
    them on the host (sortedness and ranges are verified on the device after the upload).  row_range = (r0, r1)
    takes the slices of a row block: indptr counted from 0, views of indices / data (no copy)."""
    if not sp.isspmatrix_csr(m):
        m = sp.csr_matrix(m)
    ip, ix, dt = m.indptr, m.indices, m.data
    if row_range is not None and tuple(row_range) != (0, m.shape[0]):
        r0, r1 = row_range
        a, b = int(ip[r0]), int(ip[r1])
        ip = (ip[r0:r1 + 1] - ip[r0]).astype(np.int32)
        ix, dt = ix[a:b], dt[a:b]
    if ip.dtype != np.int32:
        ip = ip.astype(np.int32)
    if ix.dtype != np.int32:
        ix = ix.astype(np.int32)
    if dt.dtype != np.float64:
        dt = dt.astype(np.float64)
    return np.ascontiguousarray(ip), np.ascontiguousarray(ix), np.ascontiguousarray(dt), int(ix.size)


class MatSet(object):
    """K CSR relationship matrices resident in HBM (slmm_matset_t).

    The host never scans the index arrays: uploads go through pinned staging, pattern sharing (IBD and its
    Hadamard square) is decided by an exact comparison ON THE DEVICE, and so is the CSR sanity check (sorted rows,
    indices in range); a matrix that fails it is canonicalised by scipy and uploaded again."""

    def __init__(self, mats, row_range=None):
        """row_range = (r0, r1): a ROW-BLOCK SHARD of the HE path - only rows [r0, r1) of every matrix are uploaded
        and held (SURVEY 8e); such a set serves he_moments_device only."""
        torch = require_cuda()
        self.n = mats[0].shape[0]
        self.K = len(mats)
        self.row_range = (0, self.n) if row_range is None else (int(row_range[0]), int(row_range[1]))
        h = C.c_void_p()
        check(lib().slmm_matset_create(self.n, self.K, C.byref(h)))
        self._h = h
        if self.row_range != (0, self.n):
            check(lib().slmm_matset_set_row_range(h, self.row_range[0], self.row_range[1]))
        self._sym_known = self.row_range == (0, self.n)
        self._keep = []
        self.nnz = []
        self.h2d_bytes = 0
        patterns = []                     # (k, indptr_host, nnz, ptr_t, idx_t)
        for k, m in enumerate(mats):
            if m.shape != (self.n, self.n):
                raise ValueError("all matrices must be n x n")
            self._bind(k, m, patterns, torch, verified=False)
        self._out = torch.zeros(2 * self.K + 2 * self.K * self.K, dtype=torch.float64, device="cuda")

    def _bind(self, k, m, patterns, torch, verified):
        ip, ix, dt, nnz = _csr_arrays(m, self.row_range)
        dat_t = to_device(dt, torch)
        self.h2d_bytes += dt.nbytes
        same = -1
        ptr_t = idx_t = None
        for (j, ipj, nnzj, ptr_j, idx_j) in patterns:
            if nnzj != nnz or not (ipj is ip or np.array_equal(ipj, ip)):       # row pointers: 4(n+1) bytes, cheap
                continue
            if idx_t is None:
                idx_t = to_device(ix, torch)
                self.h2d_bytes += ix.nbytes
            eq = C.c_int32(0)
            check(lib().slmm_device_arrays_equal_i32(idx_j.data_ptr(), idx_t.data_ptr(), nnz, C.byref(eq)))
            if eq.value:
                same, ptr_t, idx_t = j, ptr_j, idx_j
                break
        if same < 0:
            ptr_t = to_device(ip, torch)
            if idx_t is None:
                idx_t = to_device(ix, torch)
                self.h2d_bytes += ix.nbytes
            self.h2d_bytes += ip.nbytes
        check(lib().slmm_matset_bind_device(self._h, k, ptr_t.data_ptr(), idx_t.data_ptr(), dat_t.data_ptr(), nnz, same))
        if same < 0 and not verified:
            flags = C.c_int32(0)
            check(lib().slmm_matset_validate(self._h, k, C.byref(flags)))
            if flags.value & 2:
                raise ValueError("matrix %d: CSR indices / row pointers out of range" % k)
            if flags.value & 1:       # unsorted rows or duplicates: let scipy canonicalise, upload again
                if self.row_range != (0, self.n):
                    raise ValueError("matrix %d: row-block shards need canonical CSR (sorted rows, no duplicates)" % k)
                mc = sp.csr_matrix(m).copy()
                mc.sum_duplicates()
                return self._bind(k, canonical_csr(mc), patterns, torch, verified=True)
        if same < 0:
            patterns.append((k, ip, nnz, ptr_t, idx_t))
        if len(self._keep) > k:
            self._keep[k] = (ptr_t, idx_t, dat_t)
            self.nnz[k] = nnz
        else:
            self._keep.append((ptr_t, idx_t, dat_t))
            self.nnz.append(nnz)

    def values_ptr(self, k):
        return self._keep[k][2].data_ptr()

    def device_arrays(self, k):
        """(indptr, indices, data) torch tensors of matrix k in HBM."""
        return self._keep[k]

    def pattern_is_subset(self, k_small, k_big):
        """True when every stored entry of matrix k_small is also stored in matrix k_big (device check)."""
        a, b = self._keep[k_small], self._keep[k_big]
        if a[1].data_ptr() == b[1].data_ptr():
            return True
        return device_pattern_subset(a[0], a[1], b[0], b[1], self.n)

    def resolve_symmetry_sharded(self, allreduce_sum_):
        """Row-block shards cannot see the mirror image of their entries: every rank hashes its entries above / below
        the diagonal (slmm_matset_symmetry_hash), the two 64-bit sums are added over ranks (wrapping) and compared.
        COLLECTIVE: every rank of the group must call it.  Without it the shard reads full rows (still correct)."""
        if self._sym_known:
            return
        torch = _torch()
        h = np.zeros(2 * self.K, dtype=np.uint64)
        for k in range(self.K):
            check(lib().slmm_matset_symmetry_hash(self._h, k, np_ptr(h[2 * k:2 * k + 2])))
        t = torch.from_numpy(h.view(np.int64).copy()).to("cuda")
        allreduce_sum_(t)
        tot = t.cpu().numpy()
        for k in range(self.K):
            check(lib().slmm_matset_set_symmetric(self._h, k, 1 if tot[2 * k] == tot[2 * k + 1] else 0))
        self._sym_known = True

    def he_moments_device(self, y_dev, row_begin=None, row_end=None):
        """Partial moments of rows [row_begin,row_end) as a device tensor (layout: include/scilmm_b200.h)."""
        row_begin = self.row_range[0] if row_begin is None else row_begin
        row_end = self.row_range[1] if row_end is None else row_end
        check(lib().slmm_he_moments(self._h, y_dev.data_ptr(), int(row_begin), int(row_end), self._out.data_ptr()))
        return self._out

    @staticmethod
    def split_moments(out, K):
        out = np.asarray(out)
        q_off, q_diag = out[:K], out[K:2 * K]
        S_off = out[2 * K:2 * K + K * K].reshape(K, K)
        S_diag = out[2 * K + K * K:].reshape(K, K)
        S_off = np.tril(S_off) + np.tril(S_off, -1).T
        S_diag = np.tril(S_diag) + np.tril(S_diag, -1).T
        return q_off, q_diag, S_off, S_diag

    def spmm(self, k, X, out=None):
        torch = _torch()
        X2 = X if X.dim() == 2 else X.unsqueeze(1)
        X2 = X2.contiguous()
        ncols = X2.shape[1]
        if out is None:
            out = torch.empty_like(X2)
        for c0 in range(0, ncols, 256):
            c1 = min(ncols, c0 + 256)
            if c0 == 0 and c1 == ncols:
                check(lib().slmm_spmm(self._h, k, X2.data_ptr(), ncols, out.data_ptr()))
            else:
                blk = X2[:, c0:c1].contiguous()
                o = torch.empty_like(blk)
                check(lib().slmm_spmm(self._h, k, blk.data_ptr(), c1 - c0, o.data_ptr()))
                out[:, c0:c1] = o
        return out if X.dim() == 2 else out[:, 0]

    def coldot(self, k, X, row_begin=0, row_end=None):
        """d[c] = sum_i X[i,c] (A_k X)[i,c]  (device tensor of ncols doubles)."""
        torch = _torch()
        X2 = (X if X.dim() == 2 else X.unsqueeze(1)).contiguous()
        ncols = X2.shape[1]
        row_end = self.n if row_end is None else row_end
        out = torch.empty(ncols, dtype=torch.float64, device="cuda")
        for c0 in range(0, ncols, 256):
            c1 = min(ncols, c0 + 256)
            blk = X2 if (c0 == 0 and c1 == ncols) else X2[:, c0:c1].contiguous()
            o = out if (c0 == 0 and c1 == ncols) else torch.empty(c1 - c0, dtype=torch.float64, device="cuda")
            check(lib().slmm_spmm_coldot(self._h, k, blk.data_ptr(), c1 - c0, int(row_begin), int(row_end),
                                         o.data_ptr()))
            if o is not out:
                out[c0:c1] = o
        return out

    def pattern_id(self, k):
        v = C.c_int32(-1)
        check(lib().slmm_matset_pattern_id(self._h, int(k), C.byref(v)))
        return v.value

    def pattern_groups(self, max_group=2):
        """Lists of matrix indices sharing one pattern (at most max_group per list)."""
        groups, out = {}, []
        for k in range(self.K):
            groups.setdefault(self.pattern_id(k), []).append(k)
        for ks in groups.values():
            for i in range(0, len(ks), max_group):
                out.append(ks[i:i + max_group])
        return out

    def coldot_multi(self, ks, X, store_from=None, row_begin=0, row_end=None):
        """Fused pass over matrices `ks` (same pattern): returns (dots [len(ks), ncols], stored [len(ks), n, ncols -
        store_from] or None)."""
        torch = _torch()
        X2 = X.contiguous()
        n, ncols = X2.shape
        row_end = self.n if row_end is None else row_end
        store_from = ncols if store_from is None else store_from
        ks_arr = np.asarray(ks, dtype=np.int32)
        dots = torch.empty(len(ks), ncols, dtype=torch.float64, device="cuda")
        store = None
        if store_from < ncols:
            store = torch.zeros(len(ks), n, ncols - store_from, dtype=torch.float64, device="cuda")
        check(lib().slmm_spmm_coldot_multi(self._h, len(ks), np_ptr(ks_arr), X2.data_ptr(), int(ncols), int(store_from),
                                           store.data_ptr() if store is not None else None, int(row_begin),
                                           int(row_end), dots.data_ptr()))
        return dots, store

    def quadform_gram_multi(self, ks, X, XB, row_begin=0, row_end=None):
        """One pass over symmetric matrices `ks` (one pattern): (dots[g, c] = X[:,c]' A X[:,c],
        gram[g] = XB' A XB) for a wide block X (<= 160 columns) and a narrow one XB (<= 16 columns)."""
        torch = _torch()
        X2, B2 = X.contiguous(), XB.contiguous()
        ncols, nb = X2.shape[1], B2.shape[1]
        row_end = self.n if row_end is None else row_end
        ks_arr = np.asarray(ks, dtype=np.int32)
        dots = torch.empty(len(ks), ncols, dtype=torch.float64, device="cuda")
        half = torch.empty(len(ks), nb, nb, dtype=torch.float64, device="cuda")
        check(lib().slmm_quadform_gram_multi(self._h, len(ks), np_ptr(ks_arr), X2.data_ptr(), int(ncols),
                                             B2.data_ptr(), int(nb), int(row_begin), int(row_end),
                                             dots.data_ptr(), half.data_ptr()))
        return dots, half + half.transpose(1, 2)

    def build_tiles(self, k, chol_engine):
        """Tile matrix k (symmetric) in the fill-reducing order of `chol_engine` for quadform_tiled."""
        dp, di = chol_engine.device_perm()
        check(lib().slmm_matset_build_tiles(self._h, int(k), dp, di))
        self._tiled = getattr(self, "_tiled", set()) | {int(k)}

    def tile_stats(self, k):
        out = np.zeros(4, dtype=np.int64)
        check(lib().slmm_matset_tile_stats(self._h, int(k), np_ptr(out)))
        return dict(tiles=int(out[0]), entries=int(out[1]), distinct=int(out[2]), ctas=int(out[3]))

    def tile_cta_profile(self, k):
        """(ncta, 4) int64: tiles, non-empty rows, entries and clock64 span of every CTA in the last tiled pass."""
        ncta = self.tile_stats(k)["ctas"]
        out = np.zeros((ncta, 4), dtype=np.int64)
        check(lib().slmm_matset_tile_cta_profile(self._h, int(k), np_ptr(out), int(ncta)))
        return out

    def has_tiles(self, ks):
        t = getattr(self, "_tiled", set())
        return all(int(k) in t for k in ks)

    def quadform_tiled(self, ks, X, nb):
        """One pass over the tiled symmetric matrices `ks` (one pattern): X = [XB (nb columns) | W], <= 160 columns.
        Returns (dots[g, c] = X[:,c]' A X[:,c] for ALL columns, gram[g] = XB' A XB)."""
        torch = _torch()
        X2 = X.contiguous()
        ncols = X2.shape[1]
        ks_arr = np.asarray(ks, dtype=np.int32)
        dots = torch.empty(len(ks), ncols, dtype=torch.float64, device="cuda")
        half = torch.empty(len(ks), max(nb, 1), max(nb, 1), dtype=torch.float64, device="cuda")
        check(lib().slmm_quadform_tiled(self._h, len(ks), np_ptr(ks_arr), X2.data_ptr(), int(ncols), int(nb),
                                        dots.data_ptr(), half.data_ptr() if nb > 0 else None))
        return dots, (half + half.transpose(1, 2)) if nb > 0 else None

    def is_symmetric(self, k):
        v = C.c_int32(0)
        check(lib().slmm_matset_is_symmetric(self._h, int(k), C.byref(v)))
        return bool(v.value)

    def quadform_multi(self, ks, X, row_begin=0, row_end=None):
        """dots[g, c] = X[:,c]' A_ks[g] X[:,c] for matrices `ks` sharing one pattern (symmetric matrices are
        traversed on and below the diagonal only).  Any number of columns (processed 160 at a time)."""
        torch = _torch()
        X2 = (X if X.dim() == 2 else X.unsqueeze(1)).contiguous()
        ncols = X2.shape[1]
        row_end = self.n if row_end is None else row_end
        ks_arr = np.asarray(ks, dtype=np.int32)
        dots = torch.empty(len(ks), ncols, dtype=torch.float64, device="cuda")
        for c0 in range(0, ncols, 160):
            c1 = min(ncols, c0 + 160)
            whole = c0 == 0 and c1 == ncols
            blk = X2 if whole else X2[:, c0:c1].contiguous()
            o = dots if whole else torch.empty(len(ks), c1 - c0, dtype=torch.float64, device="cuda")
            check(lib().slmm_quadform_multi(self._h, len(ks), np_ptr(ks_arr), blk.data_ptr(), int(c1 - c0),
                                            int(row_begin), int(row_end), o.data_ptr()))
            if not whole:
                dots[:, c0:c1] = o
        return dots

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().slmm_matset_destroy(self._h)
                self._h = None
        except Exception:
            pass


def device_csr_is_symmetric(ptr_t, idx_t, dat_t, n):
    v = C.c_int32(0)
    check(lib().slmm_device_csr_is_symmetric(ptr_t.data_ptr(), idx_t.data_ptr(), dat_t.data_ptr(), int(n), C.byref(v)))
    return bool(v.value)


def device_pattern_subset(ap_t, ai_t, bp_t, bi_t, n):
    v = C.c_int32(0)
    check(lib().slmm_device_pattern_subset(ap_t.data_ptr(), ai_t.data_ptr(), bp_t.data_ptr(), bi_t.data_ptr(), int(n),
                                           C.byref(v)))
    return bool(v.value)


# ------------------------------------------------------------------------------------------------ factor
class CholEngine(object):
    """Symbolic analysis + device-resident supernodal factor (slmm_chol_t)."""

    def __init__(self, pattern, ordering="metis", perm=None):
        require_cuda()
        pattern = canonical_csr(pattern)
        self.n = pattern.shape[0]
        h = C.c_void_p()
        self._perm_in = None if perm is None else _as_i32(perm)
        code = ORDERINGS[ordering] if perm is None else 1
        check(lib().slmm_chol_analyze(self.n, np_ptr(pattern.indptr), np_ptr(pattern.indices), code,
                                      None if perm is None else np_ptr(self._perm_in), C.byref(h)))
        self._h = h
        self._perm = None
        self.factorizations = 0

    def stats(self):
        i = np.zeros(16, dtype=np.int64)
        d = np.zeros(8, dtype=np.float64)
        check(lib().slmm_chol_stats(self._h, np_ptr(i), np_ptr(d)))
        return dict(n=int(i[0]), nsuper=int(i[1]), nlevels=int(i[2]), nnzL=int(i[3]), lsize=int(i[4]),
                    exported_nnz=int(i[5]), max_front_rows=int(i[6]), max_super_cols=int(i[7]),
                    ncomponents=int(i[8]), launches=int(i[9]), device_bytes=int(i[10]), flops=float(d[0]),
                    t_order=float(d[1]), t_symbolic=float(d[2]), issued_flops=float(d[3]))

    def perm(self):
        if self._perm is None:
            p = np.zeros(self.n, dtype=np.int32)
            check(lib().slmm_chol_perm(self._h, np_ptr(p)))
            self._perm = p
        return self._perm

    def device_perm(self):
        """(d_perm, d_iperm) raw device pointers of the permutation (owned by the engine)."""
        a, b = C.c_void_p(), C.c_void_p()
        check(lib().slmm_chol_device_perm(self._h, C.byref(a), C.byref(b)))
        return a, b

    def register_pattern(self, pattern, tri=0):
        """Scatter map of a host pattern.  tri: 0 = both triangles stored with equal values (verified by the
        caller); +1 / -1 = CHOLMOD's rule, only the lower triangle of the CSC / CSR arrays defines the matrix."""
        pattern = canonical_csr(pattern)
        mid = C.c_int32(-1)
        check(lib().slmm_chol_register_pattern_tri(self._h, np_ptr(pattern.indptr), np_ptr(pattern.indices),
                                                   int(tri), C.byref(mid)))
        return mid.value

    def register_pattern_device(self, ptr_t, idx_t, nnz, tri=0):
        """Same from device-resident CSR arrays (torch int32 tensors): the map is built by a kernel."""
        mid = C.c_int32(-1)
        check(lib().slmm_chol_register_pattern_device(self._h, ptr_t.data_ptr(), idx_t.data_ptr(), int(nnz),
                                                      int(tri), C.byref(mid)))
        return mid.value

    def add_values(self, map_id, values_ptr, sigma, first):
        check(lib().slmm_chol_add_values(self._h, int(map_id), values_ptr, float(sigma), 1 if first else 0))

    def add_values2(self, map_id, values_ptr0, sigma0, values_ptr1, sigma1, first):
        check(lib().slmm_chol_add_values2(self._h, int(map_id), values_ptr0, float(sigma0), values_ptr1, float(sigma1),
                                          1 if first else 0))

    def factorize(self):
        col = C.c_int32(-1)
        code = lib().slmm_chol_factorize(self._h, C.byref(col))
        check(code, col.value)
        self.factorizations += 1

    def logdet(self):
        v = C.c_double(0.0)
        check(lib().slmm_chol_logdet(self._h, C.byref(v)))
        return v.value

    def solve_(self, B, mode=0):
        """In-place V^-1 B on a contiguous CUDA float64 tensor of shape (n,) or (n, k).
        mode 0: V^-1 B;  1: forward half only, L^-1 P B (result in the factor's row order);  2: backward half only,
        P' L^-T P B;  3: backward half from the factor's row order, P' L^-T B.  Mode 3 on Z equals mode 0 on lmul(Z)
        up to rounding (V^-1 P' L Z = P' L^-T Z), so it gives the probe block without L Z or the forward sweep."""
        if not B.is_contiguous():
            raise ValueError("solve_ needs a contiguous tensor")
        nrhs = 1 if B.dim() == 1 else B.shape[1]
        check(lib().slmm_chol_solve(self._h, B.data_ptr(), int(nrhs), int(mode)))
        return B

    def lmul(self, Z):
        torch = _torch()
        Z2 = (Z if Z.dim() == 2 else Z.unsqueeze(1)).contiguous()
        out = torch.empty_like(Z2)
        check(lib().slmm_chol_lmul(self._h, Z2.data_ptr(), out.data_ptr(), int(Z2.shape[1])))
        return out if Z.dim() == 2 else out[:, 0]

    def probe_normals(self, n, ncols, col_begin, seed, stream):
        """Columns [col_begin, col_begin+ncols) of the N(0,1) probe block of evaluation `stream` (device tensor)."""
        torch = _torch()
        out = torch.empty(int(n), int(ncols), dtype=torch.float64, device="cuda")
        check(lib().slmm_probe_normals(out.data_ptr(), int(n), int(ncols), int(col_begin), int(seed) & (2 ** 64 - 1),
                                       int(stream) & (2 ** 64 - 1)))
        return out

    def aux_begin(self):
        check(lib().slmm_chol_aux_begin(self._h))

    def aux_end(self):
        check(lib().slmm_chol_aux_end(self._h))

    def aux_join(self):
        check(lib().slmm_chol_aux_join(self._h))

    def panels(self):
        """Raw supernodal panels as one host array (layout: SymbolicView.arrays() sn_lptr / sn_ld / sn_nrow)."""
        out = np.zeros(self.stats()["lsize"], dtype=np.float64)
        check(lib().slmm_chol_copy_panels(self._h, np_ptr(out)))
        return out

    def set_profiling(self, on):
        check(lib().slmm_chol_set_profiling(self._h, 1 if on else 0))

    def timeline(self):
        """Factorize once in timeline mode; returns (ms since the fork, recording stream) per schedule event."""
        check(lib().slmm_chol_set_timeline(self._h, 1))
        try:
            self.factorize()
        finally:
            check(lib().slmm_chol_set_timeline(self._h, 0))
        n = C.c_int32(0)
        check(lib().slmm_chol_get_timeline(self._h, 0, C.byref(n), None, None))
        ms, st = np.zeros(n.value, np.float32), np.zeros(n.value, np.int32)
        check(lib().slmm_chol_get_timeline(self._h, n.value, C.byref(n), np_ptr(ms), np_ptr(st)))
        return ms, st

    def launch_timeline(self):
        """Per kernel launch of the last timeline-mode factorization: (end ms, stream, kind, grid, flops)."""
        n = C.c_int32(0)
        check(lib().slmm_chol_get_launch_timeline(self._h, 0, C.byref(n), None, None, None, None, None))
        end, fl = np.zeros(n.value, np.float32), np.zeros(n.value)
        st, kind, grid = (np.zeros(n.value, np.int32) for _ in range(3))
        check(lib().slmm_chol_get_launch_timeline(self._h, n.value, C.byref(n), np_ptr(end), np_ptr(st), np_ptr(kind),
                                                  np_ptr(grid), np_ptr(fl)))
        return end, st, kind, grid, fl

    def profile(self):
        """Per-kernel-kind device time (ms), issued flops and launch counts since set_profiling(True)."""
        ms, fl, n = np.zeros(13), np.zeros(13), np.zeros(13, dtype=np.int64)
        check(lib().slmm_chol_get_profile_ex(self._h, 13, np_ptr(ms), np_ptr(fl), np_ptr(n)))
        names = ["potrf_inv", "gemm_big", "gemm_small", "extend_add", "rhs_pull", "extend_add_big", "init_w",
                 "splitk_reduce", "_ev_record", "_ev_wait", "skinny_f1", "skinny_f2", "gemm_tma"]
        return {names[k]: dict(ms=float(ms[k]), flops=float(fl[k]), launches=int(n[k])) for k in range(13)
                if not names[k].startswith("_")}

    def launch_profile(self):
        """(ms, flops, kind, grid) arrays, one entry per launch of the profiled schedule runs."""
        n = C.c_int64(0)
        check(lib().slmm_chol_get_launch_profile(self._h, 0, C.byref(n), None, None, None, None))
        ms, fl = np.zeros(n.value, np.float32), np.zeros(n.value)
        kind, grid = np.zeros(n.value, np.int32), np.zeros(n.value, np.int32)
        check(lib().slmm_chol_get_launch_profile(self._h, n.value, C.byref(n), np_ptr(ms), np_ptr(fl), np_ptr(kind),
                                                 np_ptr(grid)))
        return ms, fl, kind, grid

    def export_L(self):
        st = self.stats()
        nnz = st["exported_nnz"]
        colptr = np.zeros(self.n + 1, dtype=np.int64)
        rowidx = np.zeros(nnz, dtype=np.int32)
        vals = np.zeros(nnz, dtype=np.float64)
        check(lib().slmm_chol_export_L(self._h, np_ptr(colptr), np_ptr(rowidx), np_ptr(vals)))
        return sp.csc_matrix((vals, rowidx, colptr), shape=(self.n, self.n))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().slmm_chol_destroy(self._h)
                self._h = None
        except Exception:
            pass


def launch_count(reset=False):
    v = C.c_int64(0)
    check(lib().slmm_launch_count(C.byref(v), 1 if reset else 0))
    return v.value


def gemm_selftest(M, N, K, lower=False, reps=5, seed=0):
    """C = A B^T through the DMMA tile kernel; returns (max abs error vs torch fp64, ms, TFLOP/s)."""
    torch = require_cuda()
    g = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn(K, M, generator=g, dtype=torch.float64, device="cuda")   # column-major M x K
    B = torch.randn(K, N, generator=g, dtype=torch.float64, device="cuda")   # column-major N x K
    Cm = torch.zeros(N, M, dtype=torch.float64, device="cuda")               # column-major M x N
    ms = C.c_float(0)
    check(lib().slmm_gemm_selftest(M, N, K, A.data_ptr(), B.data_ptr(), Cm.data_ptr(), 1 if lower else 0, reps,
                                   C.byref(ms)))
    ref = (A.t() @ B).t()          # (N x M) row-major == column-major M x N
    got = Cm
    if lower:
        mask = torch.tril(torch.ones(M, N, dtype=torch.bool, device="cuda")).t()
        err = ((got - ref) * mask).abs().max().item()
        flops = M * N * K
    else:
        err = (got - ref).abs().max().item()
        flops = 2.0 * M * N * K
    return err, ms.value, flops / (ms.value * 1e-3) / 1e12 if ms.value > 0 else 0.0
