// IBD (numerator relationship) matrix construction on the device: the step immediately before the hot path
// (SURVEY.md 8f-1).  Restates the reference's scilmm/Matrices/Numerator.py:
//   LD()               :5-34   row-recursive L (here T), Henderson/Quaas D and inbreeding F  - a per-individual Python
//                               loop on a lil_matrix there (12 s at n = 10,000);
//   create_numerator() :37-38   A = L D L'  (two scipy CSR x CSR products).
// The arithmetic follows the reference operation by operation so that the result is BIT-IDENTICAL to it:
//   * L: path weights are dyadic rationals with short mantissas, every partial sum is exact in binary64, so any
//     summation order gives the reference's values; rows are built level by level (depth of the ancestor chain) by
//     merging the parents' rows;
//   * D[i] = 1 - 0.25 * (#parents + F[p1] + F[p2])                       (:17)
//   * F[i] = ( sum over j in {i} u ancestors(i), DESCENDING j, of (L[i,j]^2) * D[j] ) - 1   (:21-26: j = max(ANC));
//     square, product and sum are separately rounded (no FMA), like the Python floats;
//   * A[i,k] = sum over common ancestors j, ASCENDING j, of (L[i,j] * D[j]) * L[k,j]: the order and the two rounded
//     products of scipy's csr_matmat applied to (L D) and then to (L D) L' (both operands with sorted rows).
// Only individuals with at most two parents that precede them are accepted (what Relationship.topo_sort :8-35
// guarantees downstream of the reference's loaders).
#include <algorithm>
#include <cstring>
#include <memory>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "common.h"

namespace slmm {

__global__ void __launch_bounds__(256) ibd_check_kernel(const int32_t* __restrict__ rp, const int32_t* __restrict__ ri,
                                                        int n, int* __restrict__ bad) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int b = rp[i], e = rp[i + 1];
    if (e - b > 2 || e < b) { *bad = 1; continue; }
    for (int p = b; p < e; p++)
      if (ri[p] < 0 || ri[p] >= i) *bad = 2;
    if (e - b == 2 && ri[b] == ri[b + 1]) *bad = 3;
  }
}

// depth[i] = 1 + max depth of the parents (0 for founders): relaxed until nothing changes (<= generations sweeps)
__global__ void __launch_bounds__(256) ibd_depth_kernel(const int32_t* __restrict__ rp, const int32_t* __restrict__ ri,
                                                        int n, int32_t* __restrict__ depth, int* __restrict__ changed) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int d = 0;
    for (int p = rp[i]; p < rp[i + 1]; p++) d = max(d, depth[ri[p]] + 1);
    if (d != depth[i]) { depth[i] = d; *changed = 1; }
  }
}

// Row of T for individual i: e_i + 1/2 (row p1 + row p2), sorted merge of the parents' rows (already built: they
// sit on a lower level).  COUNT pass (vals == nullptr) and FILL pass share the walk.
__global__ void __launch_bounds__(128) ibd_trow_kernel(const int32_t* __restrict__ rows_of_level, int nrows,
                                                       const int32_t* __restrict__ rp, const int32_t* __restrict__ ri,
                                                       const int64_t* __restrict__ tptr, const int32_t* __restrict__ tlen,
                                                       int32_t* __restrict__ tidx, double* __restrict__ tval,
                                                       int32_t* __restrict__ len_out, bool fill) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nrows) return;
  const int i = rows_of_level[q];
  const int b = rp[i], np = rp[i + 1] - b;
  const int32_t *ia = nullptr, *ib = nullptr;
  const double *va = nullptr, *vb = nullptr;
  int la = 0, lb = 0;
  if (np >= 1) { const int p = ri[b]; ia = tidx + tptr[p]; va = tval + tptr[p]; la = tlen[p]; }
  if (np >= 2) { const int p = ri[b + 1]; ib = tidx + tptr[p]; vb = tval + tptr[p]; lb = tlen[p]; }
  int32_t* oi = fill ? tidx + tptr[i] : nullptr;
  double* ov = fill ? tval + tptr[i] : nullptr;
  int a = 0, c = 0, out = 0;
  while (a < la || c < lb) {
    const int ja = a < la ? ia[a] : 0x7fffffff, jb = c < lb ? ib[c] : 0x7fffffff;
    const int j = min(ja, jb);
    if (fill) {
      double v = 0.0;
      if (ja == j) v += 0.5 * va[a];          // exact: dyadic path weights
      if (jb == j) v += 0.5 * vb[c];
      oi[out] = j;
      ov[out] = v;
    }
    a += (ja == j);
    c += (jb == j);
    out++;
  }
  if (fill) { oi[out] = i; ov[out] = 1.0; }
  else len_out[i] = out + 1;
}

// D and F for the rows of one level (reference :17 and :21-27), thread per row, strictly sequential arithmetic
__global__ void __launch_bounds__(128) ibd_df_kernel(const int32_t* __restrict__ rows_of_level, int nrows,
                                                     const int32_t* __restrict__ rp, const int32_t* __restrict__ ri,
                                                     const int64_t* __restrict__ tptr, const int32_t* __restrict__ tlen,
                                                     const int32_t* __restrict__ tidx, const double* __restrict__ tval,
                                                     double* __restrict__ D, double* __restrict__ F) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nrows) return;
  const int i = rows_of_level[q];
  const int b = rp[i], np = rp[i + 1] - b;
  double fsum = 0.0;
  if (np == 1) fsum = F[ri[b]];
  if (np == 2) fsum = __dadd_rn(F[ri[b]], F[ri[b + 1]]);
  const double di = __dsub_rn(1.0, __dmul_rn(0.25, __dadd_rn((double)np, fsum)));
  D[i] = di;
  const int32_t* idx = tidx + tptr[i];
  const double* val = tval + tptr[i];
  double f = 0.0;
  for (int t = tlen[i] - 1; t >= 0; t--) {            // j descending, starting with j = i
    const int j = idx[t];
    const double l = val[t];
    const double dj = (j == i) ? di : D[j];
    f = __dadd_rn(f, __dmul_rn(__dmul_rn(l, l), dj));
  }
  F[i] = __dsub_rn(f, 1.0);
}

__global__ void __launch_bounds__(256) ibd_compact_kernel(int n, const int64_t* __restrict__ tptr,
                                                          const int32_t* __restrict__ tlen,
                                                          const int32_t* __restrict__ tidx, const double* __restrict__ tval,
                                                          const int64_t* __restrict__ lptr, int32_t* __restrict__ lidx,
                                                          double* __restrict__ lval, uint64_t* __restrict__ keys) {
  // level-ordered pool -> row-ordered CSR; also emits the (column, row) sort keys of the transpose
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
    const int64_t src = tptr[i], dst = lptr[i];
    for (int t = lane; t < tlen[i]; t += 32) {
      const int j = tidx[src + t];
      lidx[dst + t] = j;
      lval[dst + t] = tval[src + t];
      keys[dst + t] = ((uint64_t)(uint32_t)j << 32) | (uint32_t)i;
    }
  }
}

__global__ void __launch_bounds__(256) ibd_colcount_kernel(const uint64_t* __restrict__ keys, int64_t nnz,
                                                           int32_t* __restrict__ count) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x)
    atomicAdd(count + (int)(keys[q] >> 32), 1);
}

// A = (L D) L'.  Warp per row i.  The warp owns a bitmap (n bits) and a dense accumulator (n doubles) in global
// scratch.  For j ascending over row i of L:  v = L[i,j] * D[j];  for k over column j of L (lanes):
// acc[k] = acc[k] + v * L[k,j].  Different k of one j are independent, the j loop is sequential (a __syncwarp between
// iterations), so every entry sums its terms in ascending j like scipy's csr_matmat.  The bitmap yields the sorted
// pattern; COUNT pass and NUMERIC pass share the marking.
__global__ void __launch_bounds__(256) ibd_numerator_kernel(int n, const int64_t* __restrict__ lptr,
                                                            const int32_t* __restrict__ lidx, const double* __restrict__ lval,
                                                            const int64_t* __restrict__ cptr, const uint64_t* __restrict__ ckeys,
                                                            const double* __restrict__ cval, const double* __restrict__ D,
                                                            uint32_t* __restrict__ bitmaps, double* __restrict__ accs,
                                                            int words, const int64_t* __restrict__ aptr,
                                                            int32_t* __restrict__ aidx, double* __restrict__ aval,
                                                            int32_t* __restrict__ alen, bool numeric) {
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  uint32_t* bm = bitmaps + (int64_t)w * words;
  double* acc = accs ? accs + (int64_t)w * n : nullptr;
  for (int i = w; i < n; i += warps) {
    int wmin = words, wmax = -1;
    for (int64_t t = lptr[i]; t < lptr[i + 1]; t++) {
      const int j = lidx[t];
      const double v = numeric ? __dmul_rn(lval[t], D[j]) : 0.0;
      for (int64_t c = cptr[j] + lane; c < cptr[j + 1]; c += 32) {
        const int k = (int)(uint32_t)ckeys[c];
        atomicOr(bm + (k >> 5), 1u << (k & 31));
        if (numeric) acc[k] = __dadd_rn(acc[k], __dmul_rn(v, cval[c]));
      }
      // column j of L holds j and its descendants: rows >= j; the last entry of the column bounds the range
      const int kfirst = j, klast = (int)(uint32_t)ckeys[cptr[j + 1] - 1];
      wmin = min(wmin, kfirst >> 5);
      wmax = max(wmax, klast >> 5);
      __syncwarp();
    }
    // scan the touched word range: count, or emit the sorted row and clear
    int64_t out = numeric ? aptr[i] : 0;
    int total = 0;
    for (int w0 = wmin; w0 <= wmax; w0 += 32) {
      const int wi = w0 + lane;
      uint32_t bits = wi <= wmax ? bm[wi] : 0u;
      const int cnt = __popc(bits);
      int pre = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, pre, o);
        if (lane >= o) pre += up;
      }
      const int tot = __shfl_sync(0xffffffffu, pre, 31);
      if (numeric) {
        int64_t pos = out + pre - cnt;
        while (bits) {
          const int bit = __ffs(bits) - 1;
          bits &= bits - 1;
          const int k = (wi << 5) + bit;
          aidx[pos] = k;
          aval[pos] = acc[k];
          acc[k] = 0.0;
          pos++;
        }
      }
      if (wi <= wmax) bm[wi] = 0u;
      out += tot;
      total += tot;
    }
    if (!numeric && lane == 0) alen[i] = total;
    __syncwarp();
  }
}

}  // namespace slmm

using namespace slmm;

struct slmm_ibd {
  int n = 0;
  int64_t nnzL = 0, nnzA = 0;
  int nlevels = 0;
  DevPtr<int64_t> d_lptr, d_aptr;
  DevPtr<int32_t> d_lidx, d_aidx;
  DevPtr<double> d_lval, d_aval, d_D, d_F;
  std::vector<int64_t> lptr, aptr;
};

namespace {
template <typename T>
std::vector<T> to_host(const T* d, size_t count) {
  std::vector<T> h(count);
  if (count) CUDA_OK(cudaMemcpy(h.data(), d, count * sizeof(T), cudaMemcpyDeviceToHost));
  return h;
}
}  // namespace

extern "C" {

int slmm_ibd_build(int32_t n, const int32_t* h_rel_indptr, const int32_t* h_rel_indices, slmm_ibd_t** out) {
  SLMM_TRY
  if (n <= 0 || !h_rel_indptr || !h_rel_indices || !out) throw std::invalid_argument("slmm_ibd_build: bad arguments");
  std::unique_ptr<slmm_ibd> h(new slmm_ibd());
  h->n = n;
  const int64_t nrel = h_rel_indptr[n];
  DevPtr<int32_t> rp_own = dev_upload(h_rel_indptr, (size_t)n + 1), ri_own = dev_upload(h_rel_indices, (size_t)nrel);
  const int32_t *rp = rp_own.get(), *ri = ri_own.get();
  DevPtr<int> d_flag = dev_alloc<int>(1);
  const int g1 = std::max(1, std::min(148 * 8, (n + 255) / 256));
  CUDA_OK(cudaMemset(d_flag.get(), 0, sizeof(int)));
  ibd_check_kernel<<<g1, 256>>>(rp, ri, n, d_flag.get());
  int flag = 0;
  CUDA_OK(cudaMemcpy(&flag, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost));
  if (flag) {
    throw std::invalid_argument(flag == 1 ? "an individual has more than two parents"
                                          : flag == 2 ? "parents must precede their children (topological order)"
                                                      : "duplicate parent");
  }
  // ---- levels
  DevPtr<int32_t> d_depth = dev_alloc<int32_t>(n);
  CUDA_OK(cudaMemset(d_depth.get(), 0, sizeof(int32_t) * n));
  for (int sweep = 0; sweep < n + 1; sweep++) {
    CUDA_OK(cudaMemset(d_flag.get(), 0, sizeof(int)));
    ibd_depth_kernel<<<g1, 256>>>(rp, ri, n, d_depth.get(), d_flag.get());
    CUDA_OK(cudaMemcpy(&flag, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost));
    if (!flag) break;
  }
  std::vector<int32_t> depth = to_host(d_depth.get(), n);
  int maxd = 0;
  for (int i = 0; i < n; i++) maxd = std::max(maxd, depth[i]);
  h->nlevels = maxd + 1;
  std::vector<int32_t> level_ptr(maxd + 2, 0), level_rows(n);
  for (int i = 0; i < n; i++) level_ptr[depth[i] + 1]++;
  for (int d = 0; d <= maxd; d++) level_ptr[d + 1] += level_ptr[d];
  {
    std::vector<int32_t> fill(level_ptr.begin(), level_ptr.end() - 1);
    for (int i = 0; i < n; i++) level_rows[fill[depth[i]]++] = i;
  }
  DevPtr<int32_t> d_level_rows = dev_upload(level_rows.data(), (size_t)n);
  // ---- T (the reference's L), level by level into a level-ordered pool
  DevPtr<int32_t> d_tlen = dev_alloc<int32_t>(n);
  DevPtr<int64_t> d_tptr = dev_alloc<int64_t>(n);
  std::vector<int64_t> tptr(n, 0);
  std::vector<int32_t> tlen(n, 0);
  int64_t pool = 0, cap = std::max<int64_t>(1024, 8LL * n);
  DevPtr<int32_t> d_tidx = dev_alloc<int32_t>((size_t)cap);
  DevPtr<double> d_tval = dev_alloc<double>((size_t)cap);
  h->d_D = dev_alloc<double>(n);
  h->d_F = dev_alloc<double>(n);
  for (int d = 0; d <= maxd; d++) {
    const int r0 = level_ptr[d], nr = level_ptr[d + 1] - r0;
    if (nr == 0) continue;
    const int grid = (nr + 127) / 128;
    ibd_trow_kernel<<<grid, 128>>>(d_level_rows.get() + r0, nr, rp, ri, d_tptr.get(), d_tlen.get(), d_tidx.get(), d_tval.get(),
                                   d_tlen.get(), false);
    std::vector<int32_t> len_all = to_host(d_tlen.get(), n);          // small: 4n bytes per level
    for (int q = 0; q < nr; q++) {
      const int i = level_rows[r0 + q];
      tlen[i] = len_all[i];
      tptr[i] = pool;
      pool += tlen[i];
    }
    if (pool > cap) {                                           // grow the pool (contents copied device to device)
      int64_t ncap = std::max(pool, cap * 2);
      DevPtr<int32_t> ni = dev_alloc<int32_t>((size_t)ncap);
      DevPtr<double> nv = dev_alloc<double>((size_t)ncap);
      const int64_t used = tptr[level_rows[r0]];
      CUDA_OK(cudaMemcpy(ni.get(), d_tidx.get(), used * sizeof(int32_t), cudaMemcpyDeviceToDevice));
      CUDA_OK(cudaMemcpy(nv.get(), d_tval.get(), used * sizeof(double), cudaMemcpyDeviceToDevice));
      d_tidx = std::move(ni); d_tval = std::move(nv); cap = ncap;
    }
    CUDA_OK(cudaMemcpy(d_tptr.get(), tptr.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice));
    ibd_trow_kernel<<<grid, 128>>>(d_level_rows.get() + r0, nr, rp, ri, d_tptr.get(), d_tlen.get(), d_tidx.get(), d_tval.get(),
                                   nullptr, true);
    ibd_df_kernel<<<grid, 128>>>(d_level_rows.get() + r0, nr, rp, ri, d_tptr.get(), d_tlen.get(), d_tidx.get(), d_tval.get(),
                                 h->d_D.get(), h->d_F.get());
    g_launch_count += 3;
  }
  CUDA_OK(cudaGetLastError());
  h->nnzL = pool;
  // ---- row-ordered CSR of L + sort keys of its transpose
  h->lptr.assign((size_t)n + 1, 0);
  for (int i = 0; i < n; i++) h->lptr[i + 1] = h->lptr[i] + tlen[i];
  h->d_lptr = dev_upload(h->lptr.data(), (size_t)n + 1);
  h->d_lidx = dev_alloc<int32_t>((size_t)pool);
  h->d_lval = dev_alloc<double>((size_t)pool);
  DevPtr<uint64_t> d_keys = dev_alloc<uint64_t>((size_t)pool);
  ibd_compact_kernel<<<std::max(1, std::min(148 * 8, (n + 7) / 8)), 256>>>(n, d_tptr.get(), d_tlen.get(), d_tidx.get(), d_tval.get(),
                                                                         h->d_lptr.get(), h->d_lidx.get(), h->d_lval.get(), d_keys.get());
  g_launch_count++;
  CUDA_OK(cudaDeviceSynchronize());
  d_tidx.reset(); d_tval.reset(); d_tptr.reset(); d_tlen.reset(); d_level_rows.reset(); d_depth.reset();
  // ---- L' as CSR (columns of L with ascending rows): stable radix sort of (column, row) keys
  DevPtr<uint64_t> d_keys2 = dev_alloc<uint64_t>((size_t)pool);
  DevPtr<double> d_cval = dev_alloc<double>((size_t)pool);
  {
    size_t tmp_bytes = 0;
    int bits = 32;
    while ((1LL << (bits - 32)) < n && bits < 64) bits++;
    CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys.get(), d_keys2.get(), h->d_lval.get(), d_cval.get(),
                                            (int64_t)pool, 0, bits));
    DevPtr<char> tmp = dev_alloc<char>(tmp_bytes);
    CUDA_OK(cub::DeviceRadixSort::SortPairs(tmp.get(), tmp_bytes, d_keys.get(), d_keys2.get(), h->d_lval.get(), d_cval.get(),
                                            (int64_t)pool, 0, bits));
    CUDA_OK(cudaDeviceSynchronize());
  }
  d_keys.reset();
  DevPtr<int32_t> d_ccount = dev_alloc<int32_t>(n);
  CUDA_OK(cudaMemset(d_ccount.get(), 0, sizeof(int32_t) * n));
  ibd_colcount_kernel<<<(int)std::min<int64_t>((pool + 255) / 256, 148 * 16), 256>>>(d_keys2.get(), pool, d_ccount.get());
  std::vector<int32_t> ccount = to_host(d_ccount.get(), n);
  d_ccount.reset();
  std::vector<int64_t> cptr((size_t)n + 1, 0);
  for (int j = 0; j < n; j++) cptr[j + 1] = cptr[j] + ccount[j];
  DevPtr<int64_t> d_cptr = dev_upload(cptr.data(), (size_t)n + 1);
  // ---- A = (L D) L'
  const int words = (n + 31) / 32;
  int warps = 148 * 8;
  const int64_t scratch_cap = (int64_t)6 << 30;                  // at most 6 GB of dense accumulators
  warps = (int)std::max<int64_t>(8, std::min<int64_t>(warps, scratch_cap / (8LL * n)));
  warps = (warps / 8) * 8;
  DevPtr<uint32_t> d_bm = dev_alloc<uint32_t>((size_t)warps * words);
  CUDA_OK(cudaMemset(d_bm.get(), 0, sizeof(uint32_t) * (size_t)warps * words));
  DevPtr<int32_t> d_alen = dev_alloc<int32_t>(n);
  ibd_numerator_kernel<<<warps / 8, 256>>>(n, h->d_lptr.get(), h->d_lidx.get(), h->d_lval.get(), d_cptr.get(), d_keys2.get(),
                                           d_cval.get(), h->d_D.get(), d_bm.get(), nullptr, words, nullptr, nullptr, nullptr,
                                           d_alen.get(), false);
  std::vector<int32_t> alen = to_host(d_alen.get(), n);
  d_alen.reset();
  h->aptr.assign((size_t)n + 1, 0);
  for (int i = 0; i < n; i++) h->aptr[i + 1] = h->aptr[i] + alen[i];
  h->nnzA = h->aptr[n];
  if (h->nnzA > 0x7fffffffLL) throw std::invalid_argument("IBD matrix has more than 2^31-1 entries (int32 CSR, as scipy)");
  h->d_aptr = dev_upload(h->aptr.data(), (size_t)n + 1);
  h->d_aidx = dev_alloc<int32_t>((size_t)h->nnzA);
  h->d_aval = dev_alloc<double>((size_t)h->nnzA);
  DevPtr<double> d_acc = dev_alloc<double>((size_t)warps * n);
  CUDA_OK(cudaMemset(d_acc.get(), 0, sizeof(double) * (size_t)warps * n));
  ibd_numerator_kernel<<<warps / 8, 256>>>(n, h->d_lptr.get(), h->d_lidx.get(), h->d_lval.get(), d_cptr.get(), d_keys2.get(),
                                           d_cval.get(), h->d_D.get(), d_bm.get(), d_acc.get(), words, h->d_aptr.get(),
                                           h->d_aidx.get(), h->d_aval.get(), nullptr, true);
  g_launch_count += 3;
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaGetLastError());
  *out = h.release();
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_ibd_sizes(const slmm_ibd_t* h, int64_t* nnz_L, int64_t* nnz_A, int32_t* nlevels) {
  if (!h) return SLMM_ERR_INVALID;
  if (nnz_L) *nnz_L = h->nnzL;
  if (nnz_A) *nnz_A = h->nnzA;
  if (nlevels) *nlevels = h->nlevels;
  return SLMM_OK;
}

static void copy_csr(int n, const std::vector<int64_t>& ptr, const int32_t* d_idx, const double* d_val, int32_t* h_indptr,
                     int32_t* h_indices, double* h_data) {
  for (int i = 0; i <= n; i++) h_indptr[i] = (int32_t)ptr[i];
  CUDA_OK(cudaMemcpy(h_indices, d_idx, sizeof(int32_t) * (size_t)ptr[n], cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(h_data, d_val, sizeof(double) * (size_t)ptr[n], cudaMemcpyDeviceToHost));
}

int slmm_ibd_copy_L(const slmm_ibd_t* h, int32_t* h_indptr, int32_t* h_indices, double* h_data) {
  SLMM_TRY
  if (!h || !h_indptr || !h_indices || !h_data) throw std::invalid_argument("null argument");
  if (h->nnzL > 0x7fffffffLL) throw std::invalid_argument("L has more than 2^31-1 entries");
  copy_csr(h->n, h->lptr, h->d_lidx.get(), h->d_lval.get(), h_indptr, h_indices, h_data);
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_ibd_copy_A(const slmm_ibd_t* h, int32_t* h_indptr, int32_t* h_indices, double* h_data) {
  SLMM_TRY
  if (!h || !h_indptr || !h_indices || !h_data) throw std::invalid_argument("null argument");
  copy_csr(h->n, h->aptr, h->d_aidx.get(), h->d_aval.get(), h_indptr, h_indices, h_data);
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_ibd_copy_DF(const slmm_ibd_t* h, double* h_D, double* h_F) {
  SLMM_TRY
  if (!h) throw std::invalid_argument("null argument");
  if (h_D) CUDA_OK(cudaMemcpy(h_D, h->d_D.get(), sizeof(double) * h->n, cudaMemcpyDeviceToHost));
  if (h_F) CUDA_OK(cudaMemcpy(h_F, h->d_F.get(), sizeof(double) * h->n, cudaMemcpyDeviceToHost));
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_ibd_destroy(slmm_ibd_t* h) {
  delete h;
  return SLMM_OK;
}

}  // extern "C"
