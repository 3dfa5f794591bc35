// HBM-bound CSR kernels of the path: Haseman-Elston moments (SpMV-dot + sparse Hadamard dot-reductions),
// SpMM, and SpMM fused with the column-wise quadratic-form reduction.
// Replaces scipy's csr_matvec / csr_matvecs / csr_elmult_csr on the call sites
// reference scilmm/SparseCholesky.py:65,66,70 (compute_gradients), :157,:161 (compute_hess), :223,:229 (HE).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <thread>
#include <vector>

#include "common.h"
#include "matset.h"

namespace slmm {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------------------
// One pass over a group of G matrices sharing one sparsity pattern: warp per row, lanes stride the row
// (coalesced index/value streams, y gathered through L2).  Per-lane partial sums live in registers across all
// rows of the warp; a single shuffle reduction per warp at the end, then per-CTA partials (deterministic).
//   q_off[g]  += a_g(i,j) y_i y_j      (i != j)        q_diag[g]  += a_g(i,i) y_i^2
//   S_off[g,h]+= a_g(i,j) a_h(i,j)     (i != j)        S_diag[g,h]+= a_g(i,i) a_h(i,i)
template <int G>
struct GroupArgs {
  const int32_t* indptr;
  const int32_t* indices;
  const double* data[G];
};

template <int G>
__global__ void __launch_bounds__(256) he_group_kernel(GroupArgs<G> a, const double* __restrict__ y, int row_begin,
                                                       int row_end, double* __restrict__ partial,
                                                       const int32_t* __restrict__ rend, double off_scale) {
  // rend != nullptr: symmetric matrices, only the entries with col <= row are read (rend[row] = one past the last
  // of them) and the off-diagonal sums are doubled at the end (off_scale = 2): half the index / value traffic.
  constexpr int UN = 4;
  constexpr int NP = G * (G + 1) / 2;
  constexpr int NV = 2 * G + 2 * NP;
  double qo[G], qd[G], so[NP], sd[NP];
#pragma unroll
  for (int g = 0; g < G; g++) qo[g] = qd[g] = 0.0;
#pragma unroll
  for (int p = 0; p < NP; p++) so[p] = sd[p] = 0.0;
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  int row = row_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  int nb = 0, ne = 0;
  double nyi = 0.0;
  if (row < row_end) { nb = a.indptr[row]; ne = rend ? rend[row] : a.indptr[row + 1]; nyi = y[row]; }
  for (; row < row_end; row += warps) {
    const int b = nb, e = ne;
    const double yi = nyi;
    if (row + warps < row_end) {         // row pointers of the next row are fetched under this row's loads
      nb = a.indptr[row + warps]; ne = rend ? rend[row + warps] : a.indptr[row + warps + 1]; nyi = y[row + warps];
    }
    double rowacc[G];
#pragma unroll
    for (int g = 0; g < G; g++) rowacc[g] = 0.0;
    // UN independent 32-entry chunks per trip: all index / value loads are issued before the dependent y gathers
    // (memory-level parallelism; a single chunk in flight per warp leaves the HBM pipe three quarters empty)
    for (int p0 = b + lane; p0 < e; p0 += 32 * UN) {
      int col[UN];
      double v[UN][G], yj[UN];
#pragma unroll
      for (int u = 0; u < UN; u++) {
        const int p = p0 + 32 * u;
        col[u] = p < e ? __ldcs(a.indices + p) : -1;
#pragma unroll
        for (int g = 0; g < G; g++) v[u][g] = p < e ? __ldcs(a.data[g] + p) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < UN; u++) yj[u] = col[u] >= 0 ? y[col[u]] : 0.0;
#pragma unroll
      for (int u = 0; u < UN; u++) {
        if (col[u] < 0) continue;
        if (col[u] != row) {
#pragma unroll
          for (int g = 0; g < G; g++) rowacc[g] += v[u][g] * yj[u];
          int q = 0;
#pragma unroll
          for (int g = 0; g < G; g++)
#pragma unroll
            for (int h = 0; h <= g; h++) so[q++] += v[u][g] * v[u][h];
        } else {
          int q = 0;
#pragma unroll
          for (int g = 0; g < G; g++) {
            qd[g] += v[u][g] * yi * yi;
#pragma unroll
            for (int h = 0; h <= g; h++) sd[q++] += v[u][g] * v[u][h];
          }
        }
      }
    }
#pragma unroll
    for (int g = 0; g < G; g++) qo[g] += rowacc[g] * yi;
  }
  __shared__ double sh[8][NV];
  const int warp = threadIdx.x >> 5;
  double vals[NV];
#pragma unroll
  for (int g = 0; g < G; g++) { vals[g] = qo[g] * off_scale; vals[G + g] = qd[g]; }
#pragma unroll
  for (int p = 0; p < NP; p++) { vals[2 * G + p] = so[p] * off_scale; vals[2 * G + NP + p] = sd[p]; }
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const double s = warp_sum(vals[k]);
    if (lane == 0) sh[warp][k] = s;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s = 0.0;
    for (int w = 0; w < 8; w++) s += sh[w][threadIdx.x];
    partial[(int64_t)blockIdx.x * NV + threadIdx.x] = s;
  }
}

// Hadamard dot of two matrices with different patterns: warp per row, lanes walk the shorter row and binary
// search the longer one (sorted indices).  out: [off, diag] partials per CTA.
__global__ void __launch_bounds__(256) he_cross_kernel(const int32_t* __restrict__ ap, const int32_t* __restrict__ ai,
                                                       const double* __restrict__ ax, const int32_t* __restrict__ bp,
                                                       const int32_t* __restrict__ bi, const double* __restrict__ bx,
                                                       int row_begin, int row_end, double* __restrict__ partial) {
  double off = 0.0, dg = 0.0;
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int row = row_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < row_end; row += warps) {
    int sb = ap[row], se = ap[row + 1], lb = bp[row], le = bp[row + 1];
    const int32_t *si = ai, *li = bi;
    const double *sx = ax, *lx = bx;
    if (se - sb > le - lb) {
      int t = sb; sb = lb; lb = t; t = se; se = le; le = t;
      si = bi; li = ai; sx = bx; lx = ax;
    }
    for (int p = sb + lane; p < se; p += 32) {
      const int col = si[p];
      int lo = lb, hi = le;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (li[mid] < col) lo = mid + 1; else hi = mid; }
      if (lo < le && li[lo] == col) {
        const double v = sx[p] * lx[lo];
        if (col == row) dg += v; else off += v;
      }
    }
  }
  __shared__ double sh[8][2];
  const int warp = threadIdx.x >> 5;
  off = warp_sum(off);
  dg = warp_sum(dg);
  if (lane == 0) { sh[warp][0] = off; sh[warp][1] = dg; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double s = 0.0;
    for (int w = 0; w < 8; w++) s += sh[w][threadIdx.x];
    partial[(int64_t)blockIdx.x * 2 + threadIdx.x] = s;
  }
}

// Short-row matrices (household indicator: ~2 entries per row): a warp per row would idle 30 lanes and put one
// memory latency per row on every warp.  Thread per row instead; same outputs as he_group_kernel<1>.
__global__ void __launch_bounds__(256) he_short_kernel(const int32_t* __restrict__ indptr,
                                                       const int32_t* __restrict__ indices,
                                                       const double* __restrict__ data, const double* __restrict__ y,
                                                       int row_begin, int row_end, double* __restrict__ partial,
                                                       const int32_t* __restrict__ rend, double off_scale) {
  double qo = 0.0, qd = 0.0, so = 0.0, sd = 0.0;
  for (int row = row_begin + blockIdx.x * blockDim.x + threadIdx.x; row < row_end; row += gridDim.x * blockDim.x) {
    const int b = indptr[row], e = rend ? rend[row] : indptr[row + 1];
    const double yi = y[row];
    double acc = 0.0;
    for (int p = b; p < e; p++) {
      const int col = indices[p];
      const double v = data[p];
      if (col != row) { acc += v * y[col]; so += v * v; } else { qd += v * yi * yi; sd += v * v; }
    }
    qo += acc * yi;
  }
  __shared__ double sh[8][4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  qo = warp_sum(qo) * off_scale; qd = warp_sum(qd); so = warp_sum(so) * off_scale; sd = warp_sum(sd);
  if (lane == 0) { sh[warp][0] = qo; sh[warp][1] = qd; sh[warp][2] = so; sh[warp][3] = sd; }
  __syncthreads();
  if (threadIdx.x < 4) {
    double s2 = 0.0;
    for (int w = 0; w < 8; w++) s2 += sh[w][threadIdx.x];
    partial[(int64_t)blockIdx.x * 4 + threadIdx.x] = s2;
  }
}

// Position map of one pattern inside another (built once per pattern pair and cached: patterns do not change
// between HE calls): map[p] = 2 * (position of probe entry p in the target's arrays) + (1 if diagonal), or -1
// when the target has no such entry (or, for symmetric sets, when the entry lies above the diagonal).
__global__ void __launch_bounds__(256) cross_map_kernel(const int32_t* __restrict__ pp, const int32_t* __restrict__ pi,
                                                        const int32_t* __restrict__ tp, const int32_t* __restrict__ ti,
                                                        int r0, int n, int lower_only, int64_t* __restrict__ map) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int row = r0 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < n; row += warps) {
    const int sb = pp[row], se = pp[row + 1], lb = tp[row], le = tp[row + 1];
    for (int p = sb + lane; p < se; p += 32) {
      const int col = pi[p];
      int64_t out = -1;
      if (!(lower_only && col > row)) {
        int lo = lb, hi = le;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (ti[mid] < col) lo = mid + 1; else hi = mid; }
        if (lo < le && ti[lo] == col) out = 2 * (int64_t)lo + (col == row ? 1 : 0);
      }
      map[p] = out;
    }
  }
}

// Hadamard dots of GP probe matrices with GT target matrices through the cached position map: a flat, fully
// coalesced pass over the probe's entries of rows [row_begin,row_end) plus one gather per matched entry.
// partial: [GP*GT][off, diag] per CTA.
template <int GP, int GT>
__global__ void __launch_bounds__(256) he_cross_mapped_kernel(GroupArgs<GP> pr, GroupArgs<GT> tg,
                                                              const int64_t* __restrict__ map, int row_begin,
                                                              int row_end, double off_scale,
                                                              double* __restrict__ partial) {
  constexpr int NV = GP * GT * 2;
  double acc[NV];
#pragma unroll
  for (int k = 0; k < NV; k++) acc[k] = 0.0;
  const int64_t pb = pr.indptr[row_begin], pe = pr.indptr[row_end];
  for (int64_t p = pb + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < pe; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = map[p];
    if (m < 0) continue;
    const int64_t t = m >> 1;
    const int d = (int)(m & 1);
#pragma unroll
    for (int gp = 0; gp < GP; gp++)
#pragma unroll
      for (int gt = 0; gt < GT; gt++) acc[(gp * GT + gt) * 2 + d] += pr.data[gp][p] * tg.data[gt][t];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ double sh[8][NV];
#pragma unroll
  for (int k = 0; k < NV; k++) {
    const double v = warp_sum(acc[k]) * ((k & 1) ? 1.0 : off_scale);
    if (lane == 0) sh[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double s2 = 0.0;
    for (int w = 0; w < 8; w++) s2 += sh[w][threadIdx.x];
    partial[(int64_t)blockIdx.x * NV + threadIdx.x] = s2;
  }
}

// final deterministic reduction of per-CTA partials: dst[map[k]] (+)= sum_b partial[b*nv + k]
__global__ void reduce_partials_kernel(const double* __restrict__ partial, int nblocks, int nv,
                                       const int32_t* __restrict__ dst_index, double* __restrict__ dst) {
  const int k = blockIdx.x;
  __shared__ double sh[256];
  double s = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += 256) s += partial[(int64_t)b * nv + k];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int d = dst_index ? dst_index[k] : k;
    if (d >= 0) dst[d] = sh[0];
  }
}

// One final reduction for ALL moments of an HE call: value j sums partial[off_j + b * stride_j] over its pass's
// CTAs in fixed order and lands in dst[dst_j].  The descriptor table is cached on the device (it depends only on the
// set of matrices), so a call issues its passes and this one kernel - no per-pass reductions, no small H2D copies.
__global__ void reduce_all_kernel(const double* __restrict__ partial, const RedDesc* __restrict__ desc,
                                  double* __restrict__ dst) {
  const RedDesc d = desc[blockIdx.x];
  __shared__ double sh[256];
  double s = 0.0;
  for (int b = threadIdx.x; b < d.nblocks; b += 256) s += partial[d.off + (int64_t)b * d.stride];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0 && d.dst >= 0) dst[d.dst] = sh[0];
}

// ---------------------------------------------------------------------------------------------------------
// SpMM on C-ordered blocks: out[i,:] = sum_j A[i,j] X[j,:].  A warp owns a row; lanes own columns
// (each X row is contiguous, so every gathered row is a coalesced read).  CPL = columns per lane.
template <int CPL, bool DOT>
__global__ void __launch_bounds__(256) spmm_kernel(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                   const double* __restrict__ data, const double* __restrict__ X, int ncols,
                                                   int row_begin, int row_end, double* __restrict__ out,
                                                   double* __restrict__ partial) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  double dot[CPL];
#pragma unroll
  for (int c = 0; c < CPL; c++) dot[c] = 0.0;
  for (int row = row_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < row_end; row += warps) {
    const int b = indptr[row], e = indptr[row + 1];
    double acc[CPL];
#pragma unroll
    for (int c = 0; c < CPL; c++) acc[c] = 0.0;
    for (int p0 = b; p0 < e; p0 += 32) {
      // stage up to 32 (col, val) pairs in registers, then broadcast them one at a time
      const int pl = p0 + lane;
      const int mycol = pl < e ? indices[pl] : 0;
      const double myval = pl < e ? data[pl] : 0.0;
      const int cnt = min(32, e - p0);
      for (int k = 0; k < cnt; k++) {
        const int col = __shfl_sync(0xffffffffu, mycol, k);
        const double v = __shfl_sync(0xffffffffu, myval, k);
        const double* xr = X + (int64_t)col * ncols;
#pragma unroll
        for (int c = 0; c < CPL; c++) {
          const int j = lane + 32 * c;
          if (j < ncols) acc[c] += v * xr[j];
        }
      }
    }
    if (DOT) {
      const double* xi = X + (int64_t)row * ncols;
#pragma unroll
      for (int c = 0; c < CPL; c++) {
        const int j = lane + 32 * c;
        if (j < ncols) dot[c] += acc[c] * xi[j];
      }
    } else {
      double* orow = out + (int64_t)row * ncols;
#pragma unroll
      for (int c = 0; c < CPL; c++) {
        const int j = lane + 32 * c;
        if (j < ncols) orow[j] = acc[c];
      }
    }
  }
  if (DOT) {
    __shared__ double sh[8][32 * CPL];
#pragma unroll
    for (int c = 0; c < CPL; c++) sh[warp][lane + 32 * c] = dot[c];
    __syncthreads();
    for (int j = threadIdx.x; j < ncols; j += 256) {
      double s = 0.0;
      for (int w = 0; w < 8; w++) s += sh[w][j];
      partial[(int64_t)blockIdx.x * ncols + j] = s;
    }
  }
}

// Narrow blocks (ncols <= 4: the single vectors and K-column blocks of compute_hess, reference :157,:161): the
// lanes-own-columns mapping above would leave 28+ of 32 lanes idle.  Here the lanes stride the ENTRIES of the row
// (coalesced index / value streams, 4 independent chunks in flight) and one shuffle reduction per row finishes it.
template <int NC>
__global__ void __launch_bounds__(256) spmv_narrow_kernel(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                          const double* __restrict__ data, const double* __restrict__ X,
                                                          int row_begin, int row_end, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int row = row_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < row_end; row += warps) {
    const int b = indptr[row], e = indptr[row + 1];
    double acc[NC];
#pragma unroll
    for (int c = 0; c < NC; c++) acc[c] = 0.0;
    for (int p0 = b + lane; p0 < e; p0 += 128) {
      int col[4];
      double v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int p = p0 + 32 * u;
        col[u] = p < e ? __ldcs(indices + p) : -1;
        v[u] = p < e ? __ldcs(data + p) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if (col[u] < 0) continue;
        const double* xr = X + (int64_t)col[u] * NC;
#pragma unroll
        for (int c = 0; c < NC; c++) acc[c] += v[u] * xr[c];
      }
    }
#pragma unroll
    for (int c = 0; c < NC; c++) {
      const double s2 = warp_sum(acc[c]);
      if (lane == 0) out[(int64_t)row * NC + c] = s2;
    }
  }
}

// SpMM + column quadratic forms for G matrices that share ONE sparsity pattern (e.g. IBD and its Hadamard
// square): index stream and the gathered X rows - the dominant traffic, ncols*8 bytes per nonzero - are read
// once for all G.  dots[g][c] = sum_i X[i,c] (A_g X)[i,c]; optionally (A_g X)[:, store_from:] is written out
// (the few covariate columns whose full Gram matrix is needed, reference scilmm/SparseCholesky.py:70).
template <int CPL, int G>
__global__ void __launch_bounds__(256) spmm_group_kernel(const int32_t* __restrict__ indptr,
                                                         const int32_t* __restrict__ indices, GroupArgs<G> vals,
                                                         const double* __restrict__ X, int ncols, int row_begin,
                                                         int row_end, int store_from, double* __restrict__ store,
                                                         int64_t store_stride, double* __restrict__ partial) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  const int nstore = ncols - store_from;
  double dot[G][CPL];
#pragma unroll
  for (int g = 0; g < G; g++)
#pragma unroll
    for (int c = 0; c < CPL; c++) dot[g][c] = 0.0;
  for (int row = row_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < row_end; row += warps) {
    const int b = indptr[row], e = indptr[row + 1];
    double acc[G][CPL];
#pragma unroll
    for (int g = 0; g < G; g++)
#pragma unroll
      for (int c = 0; c < CPL; c++) acc[g][c] = 0.0;
    for (int p0 = b; p0 < e; p0 += 32) {
      const int pl = p0 + lane;
      const int mycol = pl < e ? indices[pl] : 0;
      double myval[G];
#pragma unroll
      for (int g = 0; g < G; g++) myval[g] = pl < e ? vals.data[g][pl] : 0.0;
      const int cnt = min(32, e - p0);
      for (int k = 0; k < cnt; k++) {
        const int col = __shfl_sync(0xffffffffu, mycol, k);
        double v[G];
#pragma unroll
        for (int g = 0; g < G; g++) v[g] = __shfl_sync(0xffffffffu, myval[g], k);
        const double* xr = X + (int64_t)col * ncols;
#pragma unroll
        for (int c = 0; c < CPL; c++) {
          const int j = lane + 32 * c;
          if (j < ncols) {
            const double x = xr[j];
#pragma unroll
            for (int g = 0; g < G; g++) acc[g][c] += v[g] * x;
          }
        }
      }
    }
    const double* xi = X + (int64_t)row * ncols;
#pragma unroll
    for (int c = 0; c < CPL; c++) {
      const int j = lane + 32 * c;
      if (j < ncols) {
        const double x = xi[j];
#pragma unroll
        for (int g = 0; g < G; g++) {
          dot[g][c] += acc[g][c] * x;
          if (j >= store_from) store[g * store_stride + (int64_t)row * nstore + (j - store_from)] = acc[g][c];
        }
      }
    }
  }
  __shared__ double sh[8][32 * CPL];
  for (int g = 0; g < G; g++) {
    __syncthreads();
#pragma unroll
    for (int c = 0; c < CPL; c++) sh[warp][lane + 32 * c] = dot[g][c];
    __syncthreads();
    for (int j = threadIdx.x; j < ncols; j += 256) {
      double s2 = 0.0;
      for (int w = 0; w < 8; w++) s2 += sh[w][j];
      partial[((int64_t)blockIdx.x * G + g) * ncols + j] = s2;
    }
  }
}

// Column quadratic forms x_c' A x_c for SYMMETRIC matrices sharing one pattern: only the entries on and below the
// diagonal are visited (indices are sorted, so they are a prefix of every row), off-diagonal entries weighted
// twice.  This halves the dominant traffic of the pass - the gathered rows of X, ncols*8 bytes per visited entry.
//   dots[g][c] = sum_i x[i,c] * ( a_g(i,i) x[i,c] + 2 sum_{j<i} a_g(i,j) x[j,c] )
// Replaces np.sum(mats[i].dot(sim_vec) * sim_vec, axis=0) and invV_y.dot(mats[i].dot(invV_y)),
// reference scilmm/SparseCholesky.py:65-66 (same value up to summation order).
constexpr int QF_NB = 16;   // widest narrow block [V^-1 C | V^-1 r] the Gram pass takes

template <int CPL, int G>
__global__ void __launch_bounds__(256) quadform_sym_kernel(const int32_t* __restrict__ indptr,
                                                           const int32_t* __restrict__ indices, GroupArgs<G> vals,
                                                           const double* __restrict__ X, int ncols, int row_begin,
                                                           int row_end, double* __restrict__ partial) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  double dot[G][CPL];
#pragma unroll
  for (int g = 0; g < G; g++)
#pragma unroll
    for (int c = 0; c < CPL; c++) dot[g][c] = 0.0;
  for (int row = row_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < row_end; row += warps) {
    const int b = indptr[row], e = indptr[row + 1];
    double acc[G][CPL];
#pragma unroll
    for (int g = 0; g < G; g++)
#pragma unroll
      for (int c = 0; c < CPL; c++) acc[g][c] = 0.0;
    for (int p0 = b; p0 < e; p0 += 32) {
      const int pl = p0 + lane;
      const int mycol = pl < e ? __ldg(indices + pl) : 0x7fffffff;
      const bool mine = mycol <= row;
      const int cnt = __popc(__ballot_sync(0xffffffffu, mine));   // sorted row: the lanes with col <= row are a prefix
      double myval[G];
      const double wgt = mycol == row ? 1.0 : 2.0;
#pragma unroll
      for (int g = 0; g < G; g++) myval[g] = mine ? wgt * __ldg(vals.data[g] + pl) : 0.0;
      for (int k = 0; k < cnt; k++) {
        const int col = __shfl_sync(0xffffffffu, mycol, k);
        double v[G];
#pragma unroll
        for (int g = 0; g < G; g++) v[g] = __shfl_sync(0xffffffffu, myval[g], k);
        const double* xr = X + (int64_t)col * ncols;
#pragma unroll
        for (int c = 0; c < CPL; c++) {
          const int j = lane + 32 * c;
          if (j < ncols) {
            const double x = xr[j];
#pragma unroll
            for (int g = 0; g < G; g++) acc[g][c] += v[g] * x;
          }
        }
      }
      if (cnt < 32) break;
    }
    const double* xi = X + (int64_t)row * ncols;
#pragma unroll
    for (int c = 0; c < CPL; c++) {
      const int j = lane + 32 * c;
      if (j < ncols) {
        const double x = xi[j];
#pragma unroll
        for (int g = 0; g < G; g++) dot[g][c] += acc[g][c] * x;
      }
    }
  }
  __shared__ double sh[8][32 * CPL];
  for (int g = 0; g < G; g++) {
    __syncthreads();
#pragma unroll
    for (int c = 0; c < CPL; c++) sh[warp][lane + 32 * c] = dot[g][c];
    __syncthreads();
    for (int j = threadIdx.x; j < ncols; j += 256) {
      double s2 = 0.0;
      for (int w = 0; w < 8; w++) s2 += sh[w][j];
      partial[((int64_t)blockIdx.x * G + g) * ncols + j] = s2;
    }
  }
}

// Gram matrix XB' A XB of a NARROW block (n x nb, nb <= 16, e.g. [V^-1 C | V^-1 r]) for symmetric matrices sharing
// one pattern, again on/below the diagonal only:
//   hb_i = a(i,i)/2 xb_i + sum_{j<i} a(i,j) xb_j,   Mh = sum_i xb_i hb_i',   XB' A XB = Mh + Mh'.
// A warp owns a row and works on two entries at a time: lane = (half, j), half = which entry, j = column of XB.
// Lane (half, j) accumulates Mh[8*half + a][j], a = 0..7, over all rows of the warp.
// Replaces invV_C.T.dot(mats[i].dot(invV_C)) and invV_y.dot(mats[i].dot(invV_y)), reference :66,:70.
template <int G>
__global__ void __launch_bounds__(256) gram_sym_kernel(const int32_t* __restrict__ indptr,
                                                       const int32_t* __restrict__ indices, GroupArgs<G> vals,
                                                       const double* __restrict__ XB, int nb, int row_begin,
                                                       int row_end, double* __restrict__ partial) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int half = lane >> 4, j = lane & 15;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  double mh[G][8];
#pragma unroll
  for (int g = 0; g < G; g++)
#pragma unroll
    for (int a = 0; a < 8; a++) mh[g][a] = 0.0;
  for (int row = row_begin + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < row_end; row += warps) {
    const int b = indptr[row], e = indptr[row + 1];
    double hb[G];
#pragma unroll
    for (int g = 0; g < G; g++) hb[g] = 0.0;
    for (int p0 = b; p0 < e; p0 += 32) {
      const int pl = p0 + lane;
      const int mycol = pl < e ? __ldg(indices + pl) : 0x7fffffff;
      const bool mine = mycol <= row;
      const int cnt = __popc(__ballot_sync(0xffffffffu, mine));
      double myval[G];
      const double wgt = mycol == row ? 0.5 : 1.0;
#pragma unroll
      for (int g = 0; g < G; g++) myval[g] = mine ? wgt * __ldg(vals.data[g] + pl) : 0.0;
#pragma unroll 4
      for (int k = 0; k < cnt; k += 2) {
        const int src = min(k + half, 31);
        const int col = __shfl_sync(0xffffffffu, mycol, src);
        double v[G];
#pragma unroll
        for (int g = 0; g < G; g++) v[g] = __shfl_sync(0xffffffffu, myval[g], src);   // 0 for entries past the prefix
        const double x = (j < nb && col <= row) ? XB[(int64_t)col * nb + j] : 0.0;
#pragma unroll
        for (int g = 0; g < G; g++) hb[g] += v[g] * x;
      }
      if (cnt < 32) break;
    }
    const double xbi = j < nb ? XB[(int64_t)row * nb + j] : 0.0;
#pragma unroll
    for (int g = 0; g < G; g++) hb[g] += __shfl_xor_sync(0xffffffffu, hb[g], 16);
#pragma unroll
    for (int a = 0; a < 8; a++) {
      const double xa = __shfl_sync(0xffffffffu, xbi, 8 * half + a);
#pragma unroll
      for (int g = 0; g < G; g++) mh[g][a] += xa * hb[g];
    }
  }
  __shared__ double sh[8][G][QF_NB][QF_NB];    // [warp][g][a][j]
#pragma unroll
  for (int g = 0; g < G; g++)
#pragma unroll
    for (int a = 0; a < 8; a++) sh[warp][g][8 * half + a][j] = mh[g][a];
  __syncthreads();
  for (int q = threadIdx.x; q < G * nb * nb; q += 256) {
    const int g = q / (nb * nb), a = (q / nb) % nb, jj = q % nb;
    double s2 = 0.0;
    for (int w = 0; w < 8; w++) s2 += sh[w][g][a][jj];
    partial[(int64_t)blockIdx.x * G * nb * nb + q] = s2;
  }
}

// Symmetry check (pattern and values, bitwise): every stored (i,j), j > i, must have a stored (j,i) with the same
// value.  flag is set to 1 on the first violation.
__global__ void __launch_bounds__(256) symmetry_check_kernel(const int32_t* __restrict__ indptr,
                                                             const int32_t* __restrict__ indices,
                                                             const double* __restrict__ data, int n,
                                                             int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n; row += warps) {
    const int b = indptr[row], e = indptr[row + 1];
    for (int p = b + lane; p < e; p += 32) {
      const int col = indices[p];
      if (col == row) continue;
      bool okv = false;
      if (col >= 0 && col < n) {
        int lo = indptr[col], hi = indptr[col + 1];
        const int end = hi;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (indices[mid] < row) lo = mid + 1; else hi = mid; }
        okv = lo < end && indices[lo] == row &&
              __double_as_longlong(data[lo]) == __double_as_longlong(data[p]);
      }
      if (!okv) *flag = 1;
    }
  }
}

// Symmetry check for ROW-BLOCK SHARDS, where the mirror image of an entry usually lives on another GPU: every stored
// off-diagonal entry (i, j, value bits) is hashed under the key (min, max, bits); entries above the diagonal are summed
// (mod 2^64) into out[0], entries below into out[1].  The matrix equals its transpose exactly when the two multisets of
// keys coincide, so after a sum over all shards out[0] == out[1] (a mismatch survives with probability ~2^-64).
// Integer sums are order independent: the result is deterministic.
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__global__ void __launch_bounds__(256) symmetry_hash_kernel(const int32_t* __restrict__ indptr,
                                                            const int32_t* __restrict__ indices,
                                                            const double* __restrict__ data, int r0, int r1,
                                                            unsigned long long* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  unsigned long long up = 0, lo = 0;
  for (int row = r0 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < r1; row += warps) {
    const int b = indptr[row], e = indptr[row + 1];
    for (int p = b + lane; p < e; p += 32) {
      const int col = indices[p];
      if (col == row) continue;
      const unsigned long long a = (unsigned long long)min(row, col), c = (unsigned long long)max(row, col);
      const unsigned long long h = mix64(mix64((a << 32) | c) ^ (unsigned long long)__double_as_longlong(data[p]));
      if (col > row) up += h; else lo += h;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    up += __shfl_xor_sync(0xffffffffu, up, o);
    lo += __shfl_xor_sync(0xffffffffu, lo, o);
  }
  if (lane == 0) { atomicAdd(out, up); atomicAdd(out + 1, lo); }
}

// rend[row] = one past the last entry of the (sorted) row with col <= row
__global__ void __launch_bounds__(256) row_end_kernel(const int32_t* __restrict__ indptr,
                                                      const int32_t* __restrict__ indices, int r0, int n,
                                                      int32_t* __restrict__ rend) {
  for (int row = r0 + blockIdx.x * blockDim.x + threadIdx.x; row < n; row += gridDim.x * blockDim.x) {
    int lo = indptr[row], hi = indptr[row + 1];
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (indices[mid] <= row) lo = mid + 1; else hi = mid; }
    rend[row] = lo;
  }
}

// CSR sanity on the device (the host never scans the 10^8-entry index arrays): rows strictly increasing (sorted, no
// duplicates), indices inside [0,n), row pointers monotone.  flag bits: 1 unsorted/duplicate, 2 out of range.
__global__ void __launch_bounds__(256) csr_validate_kernel(const int32_t* __restrict__ indptr,
                                                           const int32_t* __restrict__ indices, int r0, int r1, int n,
                                                           int64_t nnz, int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  int bad = 0;
  for (int row = r0 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); row < r1; row += warps) {
    const int b = indptr[row], e = indptr[row + 1];
    if (b > e || b < 0 || (int64_t)e > nnz) { bad |= 2; continue; }
    for (int p = b + lane; p < e; p += 32) {
      const int c = indices[p];
      if (c < 0 || c >= n) bad |= 2;
      if (p + 1 < e && indices[p + 1] <= c) bad |= 1;
    }
  }
  if (bad) atomicOr(flag, bad);
}

// exact comparison of two index arrays (pattern sharing between e.g. IBD and its Hadamard square)
__global__ void __launch_bounds__(256) arrays_differ_kernel(const int32_t* __restrict__ a, const int32_t* __restrict__ b,
                                                            int64_t count, int* __restrict__ flag) {
  int bad = 0;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < count; q += (int64_t)gridDim.x * blockDim.x)
    if (a[q] != b[q]) bad = 1;
  if (bad) *flag = 1;
}

// every entry of pattern A must be present in pattern B (sorted rows): flag = 1 otherwise
__global__ void __launch_bounds__(256) pattern_subset_kernel(const int32_t* __restrict__ ap, const int32_t* __restrict__ ai,
                                                             const int32_t* __restrict__ bp, const int32_t* __restrict__ bi,
                                                             int n, int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n; row += warps) {
    const int sb = ap[row], se = ap[row + 1], lb = bp[row], le = bp[row + 1];
    for (int p = sb + lane; p < se; p += 32) {
      const int col = ai[p];
      int lo = lb, hi = le;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (bi[mid] < col) lo = mid + 1; else hi = mid; }
      if (!(lo < le && bi[lo] == col)) *flag = 1;
    }
  }
}

}  // namespace slmm

using namespace slmm;

namespace slmm {

static uint64_t hash_bytes(const void* p, size_t nbytes) {
  const uint64_t* w = (const uint64_t*)p;
  uint64_t h = 1469598103934665603ull;
  size_t nw = nbytes / 8;
  for (size_t i = 0; i < nw; i++) { h ^= w[i]; h *= 1099511628211ull; h ^= h >> 29; }
  const unsigned char* b = (const unsigned char*)p + nw * 8;
  for (size_t i = 0; i < nbytes % 8; i++) { h ^= b[i]; h *= 1099511628211ull; }
  return h;
}

static int he_grid(int rows) {
  // warp-per-row kernels with <= 64 registers (4 resident CTAs of 256 threads per SM): two waves over 148 SMs
  const int warps_needed = std::max(1, rows);
  return std::max(1, std::min(148 * 8, (warps_needed + 7) / 8));
}

template <int G>
static void launch_group(slmm_matset* ms, const int* members, const double* d_y, int r0, int r1, double* d_out,
                         const int32_t* rend) {
  const int K = ms->K;
  constexpr int NP = G * (G + 1) / 2, NV = 2 * G + 2 * NP;
  GroupArgs<G> a;
  a.indptr = ms->m[members[0]].indptr;
  a.indices = ms->m[members[0]].indices;
  for (int g = 0; g < G; g++) a.data[g] = ms->m[members[g]].data;
  // exactly two waves of resident CTAs (occupancy is set by the register count): with any other count the last,
  // partial wave costs up to 20 % (measured: 6 CTAs per SM 0.53 ms, 7: 0.60, 8: 0.56, 4: 0.65 at the 1M config)
  static int occ = 0;
  if (occ == 0) {
    CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, he_group_kernel<G>, 256, 0));
    occ = std::max(1, occ);
  }
  const int grid = std::max(1, std::min(148 * occ * 2, (r1 - r0 + 7) / 8));
  double* part = ms->he_part((size_t)grid * NV);
  he_group_kernel<G><<<grid, 256>>>(a, d_y, r0, r1, part, rend, rend ? 2.0 : 1.0);
  // destination indices inside [q_off | q_diag | S_off | S_diag]
  std::vector<int32_t> dst(NV);
  for (int g = 0; g < G; g++) { dst[g] = members[g]; dst[G + g] = K + members[g]; }
  int q = 0;
  for (int g = 0; g < G; g++)
    for (int h = 0; h <= g; h++) {
      dst[2 * G + q] = 2 * K + members[g] * K + members[h];
      dst[2 * G + NP + q] = 2 * K + K * K + members[g] * K + members[h];
      q++;
    }
  ms->he_add(part, grid, NV, dst.data());
  g_launch_count += 1;
  // the copy above must not be overwritten by the next group before the kernel ran: d_dst is consumed in
  // stream order and the next memcpy is also stream-ordered (pageable source is staged synchronously).
}

}  // namespace slmm

namespace slmm {
template <int CPL, int G>
static void launch_spmm_group(slmm_matset* ms, const int32_t* ks, const double* d_X, int ncols, int store_from,
                              double* d_store, int r0, int r1, double* d_dots) {
  GroupArgs<G> v;
  v.indptr = ms->m[ks[0]].indptr;
  v.indices = ms->m[ks[0]].indices;
  for (int g = 0; g < G; g++) v.data[g] = ms->m[ks[g]].data;
  const int grid = he_grid(r1 - r0);
  double* part = ms->partial((size_t)grid * G * ncols);
  const int64_t stride = (int64_t)ms->n * (ncols - store_from);
  spmm_group_kernel<CPL, G><<<grid, 256>>>(v.indptr, v.indices, v, d_X, ncols, r0, r1, store_from, d_store, stride, part);
  reduce_partials_kernel<<<G * ncols, 256>>>(part, grid, G * ncols, nullptr, d_dots);
  g_launch_count += 2;
}

}  // namespace slmm

extern "C" {

int slmm_matset_create(int32_t n, int32_t K, slmm_matset_t** out) {
  SLMM_TRY
  if (n <= 0 || K <= 0 || K > MAXK || !out) throw std::invalid_argument("slmm_matset_create: need 0 < K <= 8, n > 0");
  std::unique_ptr<slmm_matset> ms(new slmm_matset());
  ms->n = n;
  ms->K = K;
  ms->r1 = n;
  ms->m.resize(K);
  ms->d_y = dev_alloc<double>(n);
  ms->d_out = dev_alloc<double>(2 * K + 2 * K * K);
  ms->d_dst = dev_alloc<int32_t>(64);
  *out = ms.release();
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_destroy(slmm_matset_t* ms) {
  delete ms;
  return SLMM_OK;
}

int slmm_matset_upload(slmm_matset_t* ms, int32_t k, const int32_t* indptr, const int32_t* indices, const double* data) {
  SLMM_TRY
  if (!ms || k < 0 || k >= ms->K || !indptr || !indices || !data) throw std::invalid_argument("bad arguments");
  CsrDev& c = ms->m[k];
  ms->cross_maps.clear();
  ms->tiles.clear();
  c = CsrDev();
  if (ms->sharded()) throw std::invalid_argument("slmm_matset_upload takes whole matrices (row-block shards bind device arrays)");
  const int n = ms->n;
  c.nnz = indptr[n];
  c.h_indptr.assign(indptr, indptr + n + 1);
  c.idx_hash = hash_bytes(indices, (size_t)c.nnz * 4);
  c.pattern = k;
  for (int j = 0; j < ms->K; j++) {
    const CsrDev& o = ms->m[j];
    if (j == k || o.pattern != j || o.nnz != c.nnz || o.h_indptr.empty() || o.idx_hash != c.idx_hash) continue;
    if (memcmp(o.h_indptr.data(), indptr, sizeof(int32_t) * (n + 1)) == 0) { c.pattern = j; break; }
  }
  if (c.pattern == k) {
    c.own_indptr = dev_upload(indptr, n + 1);
    c.own_indices = dev_upload(indices, c.nnz);
    c.indptr = c.own_indptr.get();
    c.indices = c.own_indices.get();
  } else {
    c.indptr = ms->m[c.pattern].indptr;
    c.indices = ms->m[c.pattern].indices;
  }
  c.own_data = dev_upload(data, c.nnz);
  c.data = c.own_data.get();
  CUDA_OK(cudaStreamSynchronize(0));
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_bind_device(slmm_matset_t* ms, int32_t k, const int32_t* d_indptr, const int32_t* d_indices,
                            const double* d_data, int64_t nnz, int32_t same_as) {
  SLMM_TRY
  if (!ms || k < 0 || k >= ms->K || !d_indptr || !d_indices || !d_data) throw std::invalid_argument("bad arguments");
  if (same_as >= ms->K || same_as == k) throw std::invalid_argument("bad same_as");
  CsrDev& c = ms->m[k];
  ms->cross_maps.clear();
  ms->tiles.clear();
  c = CsrDev();
  // row-block shards: d_indptr has r1 - r0 + 1 entries counting from 0; the kernels index rows globally
  c.indptr = d_indptr - ms->r0; c.indices = d_indices; c.data = d_data; c.nnz = nnz;
  c.pattern = same_as >= 0 ? ms->m[same_as].pattern : k;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_nnz(const slmm_matset_t* ms, int32_t k, int64_t* out) {
  if (!ms || k < 0 || k >= ms->K || !out) return SLMM_ERR_INVALID;
  *out = ms->m[k].nnz;
  return SLMM_OK;
}

int slmm_matset_values(const slmm_matset_t* ms, int32_t k, const double** out) {
  if (!ms || k < 0 || k >= ms->K || !out) return SLMM_ERR_INVALID;
  *out = ms->m[k].data;
  return SLMM_OK;
}

int slmm_he_moments(slmm_matset_t* ms, const double* d_y, int32_t r0, int32_t r1, double* d_out) {
  SLMM_TRY
  if (!ms || !d_y || !d_out) throw std::invalid_argument("null argument");
  const int K = ms->K;
  if (r0 < ms->r0 || r1 > ms->r1 || r0 > r1) throw std::invalid_argument("bad row range (outside the rows this set holds)");
  for (int k = 0; k < K; k++)
    if (!ms->m[k].data) throw std::invalid_argument("matrix not set");
  CUDA_OK(cudaMemsetAsync(d_out, 0, sizeof(double) * (2 * K + 2 * K * K), 0));
  ms->he_used = 0;
  ms->he_desc.clear();
  // Symmetric matrices (checked once per matrix on the device): every pass reads only the entries on and below
  // the diagonal and doubles the off-diagonal sums.
  bool sym_all = true;
  for (int k = 0; k < K && sym_all; k++) {
    int32_t f = 0;
    const int rc = slmm_matset_is_symmetric(ms, k, &f);
    if (rc != SLMM_OK) return rc;
    sym_all = f != 0;
  }
  auto row_ends = [&](int k) -> const int32_t* {
    if (!sym_all) return nullptr;
    CsrDev& lead = ms->m[ms->m[k].pattern];
    if (!lead.rend) {
      const int rows = ms->r1 - ms->r0;
      lead.rend_base = dev_alloc<int32_t>(rows);
      lead.rend = lead.rend_base.get() - ms->r0;
      row_end_kernel<<<std::max(1, std::min(148 * 8, (rows + 255) / 256)), 256>>>(lead.indptr, lead.indices, ms->r0, ms->r1, lead.rend);
      g_launch_count++;
    }
    return lead.rend;
  };
  const double off_scale = sym_all ? 2.0 : 1.0;
  // pattern groups
  std::vector<char> done(K, 0);
  for (int k = 0; k < K; k++) {
    if (done[k]) continue;
    int members[MAXK], G = 0;
    for (int j = k; j < K; j++)
      if (!done[j] && ms->m[j].pattern == ms->m[k].pattern) { members[G++] = j; done[j] = 1; }
    for (int g0 = 0; g0 < G; g0 += 4) {           // at most 4 matrices fused per pass
      const int gn = std::min(4, G - g0);
      const CsrDev& lead = ms->m[members[g0]];
      if (gn == 1 && lead.nnz < (int64_t)8 * ms->n) {      // short rows: thread per row
        const int rows = r1 - r0;
        const int grid = std::max(1, std::min(148 * 8, (rows + 255) / 256));
        double* part = ms->he_part((size_t)grid * 4);
        he_short_kernel<<<grid, 256>>>(lead.indptr, lead.indices, lead.data, d_y, r0, r1, part, row_ends(members[g0]), off_scale);
        const int k0 = members[g0];
        const int32_t dst[4] = {k0, K + k0, 2 * K + k0 * K + k0, 2 * K + K * K + k0 * K + k0};
        ms->he_add(part, grid, 4, dst);
        g_launch_count += 1;
        continue;
      }
      switch (gn) {
        case 1: launch_group<1>(ms, members + g0, d_y, r0, r1, d_out, row_ends(members[g0])); break;
        case 2: launch_group<2>(ms, members + g0, d_y, r0, r1, d_out, row_ends(members[g0])); break;
        case 3: launch_group<3>(ms, members + g0, d_y, r0, r1, d_out, row_ends(members[g0])); break;
        default: launch_group<4>(ms, members + g0, d_y, r0, r1, d_out, row_ends(members[g0])); break;
      }
    }
  }
  // pairs of different patterns: one fused pass per (group chunk, group chunk); chunks of <= 2 matrices
  {
    std::vector<std::vector<int>> chunks;
    std::vector<char> seen(K, 0);
    for (int k = 0; k < K; k++) {
      if (seen[k]) continue;
      std::vector<int> mem;
      for (int t = k; t < K; t++)
        if (!seen[t] && ms->m[t].pattern == ms->m[k].pattern) { mem.push_back(t); seen[t] = 1; }
      for (size_t q = 0; q < mem.size(); q += 2)
        chunks.push_back(std::vector<int>(mem.begin() + q, mem.begin() + std::min(mem.size(), q + 2)));
    }
    for (size_t a = 0; a < chunks.size(); a++)
      for (size_t b = 0; b < a; b++) {
        if (ms->m[chunks[a][0]].pattern == ms->m[chunks[b][0]].pattern) {
          // same pattern but different chunk (groups larger than the fused pass): fall back to pairwise kernel
          for (int i : chunks[a]) for (int j : chunks[b]) {
            const int grid = he_grid(r1 - r0);
            double* part = ms->he_part((size_t)grid * 2);
            he_cross_kernel<<<grid, 256>>>(ms->m[i].indptr, ms->m[i].indices, ms->m[i].data, ms->m[j].indptr,
                                           ms->m[j].indices, ms->m[j].data, r0, r1, part);
            const int hi2 = std::max(i, j), lo2 = std::min(i, j);
            const int32_t dst[2] = {2 * K + hi2 * K + lo2, 2 * K + K * K + hi2 * K + lo2};
            ms->he_add(part, grid, 2, dst);
            g_launch_count += 1;
          }
          continue;
        }
        // probe = the side with fewer nonzeros
        const std::vector<int>& P = ms->m[chunks[a][0]].nnz <= ms->m[chunks[b][0]].nnz ? chunks[a] : chunks[b];
        const std::vector<int>& T = (&P == &chunks[a]) ? chunks[b] : chunks[a];
        const int gp = (int)P.size(), gt = (int)T.size(), nv = gp * gt * 2;
        const int lp = ms->m[P[0]].pattern, lt = ms->m[T[0]].pattern;
        DevPtr<int64_t>& owned_map = ms->cross_maps[std::make_pair(lp, lt)];
        if (!owned_map) {       // once per pattern pair: where every probe entry sits in the target
          owned_map = dev_alloc<int64_t>(ms->m[lp].nnz);
          cross_map_kernel<<<he_grid(ms->r1 - ms->r0), 256>>>(ms->m[lp].indptr, ms->m[lp].indices, ms->m[lt].indptr,
                                                              ms->m[lt].indices, ms->r0, ms->r1, sym_all ? 1 : 0, owned_map.get());
          g_launch_count++;
        }
        const int64_t* map = owned_map.get();
        const int64_t pn = ms->m[lp].nnz;
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(148 * 8, (pn + 255) / 256));
        double* part = ms->he_part((size_t)grid * nv);
        GroupArgs<2> pa, ta;
        pa.indptr = ms->m[P[0]].indptr; pa.indices = ms->m[P[0]].indices;
        ta.indptr = ms->m[T[0]].indptr; ta.indices = ms->m[T[0]].indices;
        for (int q = 0; q < 2; q++) {
          pa.data[q] = ms->m[P[std::min(q, gp - 1)]].data;
          ta.data[q] = ms->m[T[std::min(q, gt - 1)]].data;
        }
        GroupArgs<1> p1, t1;
        p1.indptr = pa.indptr; p1.indices = pa.indices; p1.data[0] = pa.data[0];
        t1.indptr = ta.indptr; t1.indices = ta.indices; t1.data[0] = ta.data[0];
        if (gp == 1 && gt == 1) he_cross_mapped_kernel<1, 1><<<grid, 256>>>(p1, t1, map, r0, r1, off_scale, part);
        else if (gp == 1 && gt == 2) he_cross_mapped_kernel<1, 2><<<grid, 256>>>(p1, ta, map, r0, r1, off_scale, part);
        else if (gp == 2 && gt == 1) he_cross_mapped_kernel<2, 1><<<grid, 256>>>(pa, t1, map, r0, r1, off_scale, part);
        else he_cross_mapped_kernel<2, 2><<<grid, 256>>>(pa, ta, map, r0, r1, off_scale, part);
        std::vector<int32_t> dst(nv);
        for (int x = 0; x < gp; x++)
          for (int z = 0; z < gt; z++) {
            const int hi2 = std::max(P[x], T[z]), lo2 = std::min(P[x], T[z]);
            dst[(x * gt + z) * 2] = 2 * K + hi2 * K + lo2;
            dst[(x * gt + z) * 2 + 1] = 2 * K + K * K + hi2 * K + lo2;
          }
        ms->he_add(part, grid, nv, dst.data());
        g_launch_count += 1;
      }
  }
  // one reduction for every moment of the call; the table is uploaded only when it changed (first call)
  if (!ms->he_desc.empty()) {
    const size_t nd = ms->he_desc.size();
    if (!ms->d_he_desc || ms->he_desc_cached.size() != nd ||
        memcmp(ms->he_desc_cached.data(), ms->he_desc.data(), nd * sizeof(RedDesc)) != 0) {
      ms->d_he_desc.reset();
      ms->d_he_desc = dev_upload(ms->he_desc.data(), nd);
      ms->he_desc_cached = ms->he_desc;
    }
    reduce_all_kernel<<<(int)nd, 256>>>(ms->he_arena.get(), ms->d_he_desc.get(), d_out);
    g_launch_count++;
  }
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_he_moments_host(slmm_matset_t* ms, const double* h_y, double* h_out) {
  SLMM_TRY
  if (!ms || !h_y || !h_out) throw std::invalid_argument("null argument");
  CUDA_OK(cudaMemcpyAsync(ms->d_y.get(), h_y, sizeof(double) * ms->n, cudaMemcpyHostToDevice, 0));
  int rc = slmm_he_moments(ms, ms->d_y.get(), 0, ms->n, ms->d_out.get());
  if (rc != SLMM_OK) return rc;
  CUDA_OK(cudaMemcpy(h_out, ms->d_out.get(), sizeof(double) * (2 * ms->K + 2 * ms->K * ms->K), cudaMemcpyDeviceToHost));
  return SLMM_OK;
  SLMM_CATCH
}

static int spmm_impl(slmm_matset_t* ms, int32_t k, const double* d_X, int32_t ncols, int32_t r0, int32_t r1,
                     double* d_out, bool dot) {
  if (!ms || k < 0 || k >= ms->K || !d_X || !d_out || ncols <= 0) throw std::invalid_argument("bad arguments");
  if (ms->sharded()) throw std::invalid_argument("row-block shards serve slmm_he_moments only");
  if (ncols > 256) throw std::invalid_argument("at most 256 columns per call");
  if (r0 < 0 || r1 > ms->n || r0 > r1) throw std::invalid_argument("bad row range");
  const CsrDev& c = ms->m[k];
  if (!c.data) throw std::invalid_argument("matrix not set");
  const int grid = he_grid(r1 - r0);
  if (!dot && ncols <= 4) {
    switch (ncols) {
      case 1: spmv_narrow_kernel<1><<<grid, 256>>>(c.indptr, c.indices, c.data, d_X, r0, r1, d_out); break;
      case 2: spmv_narrow_kernel<2><<<grid, 256>>>(c.indptr, c.indices, c.data, d_X, r0, r1, d_out); break;
      case 3: spmv_narrow_kernel<3><<<grid, 256>>>(c.indptr, c.indices, c.data, d_X, r0, r1, d_out); break;
      default: spmv_narrow_kernel<4><<<grid, 256>>>(c.indptr, c.indices, c.data, d_X, r0, r1, d_out); break;
    }
    g_launch_count++;
    CUDA_OK(cudaGetLastError());
    return SLMM_OK;
  }
  double* part = dot ? ms->partial((size_t)grid * ncols) : nullptr;
  const int cpl = (ncols + 31) / 32;
#define SPMM_CASE(C)                                                                                                  \
  if (dot) spmm_kernel<C, true><<<grid, 256>>>(c.indptr, c.indices, c.data, d_X, ncols, r0, r1, nullptr, part);       \
  else spmm_kernel<C, false><<<grid, 256>>>(c.indptr, c.indices, c.data, d_X, ncols, r0, r1, d_out, nullptr);
  if (cpl <= 1) { SPMM_CASE(1) }
  else if (cpl <= 2) { SPMM_CASE(2) }
  else if (cpl <= 4) { SPMM_CASE(4) }
  else { SPMM_CASE(8) }
#undef SPMM_CASE
  if (dot) reduce_partials_kernel<<<ncols, 256>>>(part, grid, ncols, nullptr, d_out);
  g_launch_count += dot ? 2 : 1;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
}

int slmm_spmm(slmm_matset_t* ms, int32_t k, const double* d_X, int32_t ncols, double* d_out) {
  SLMM_TRY
  return spmm_impl(ms, k, d_X, ncols, 0, ms ? ms->n : 0, d_out, false);
  SLMM_CATCH
}

int slmm_spmm_coldot(slmm_matset_t* ms, int32_t k, const double* d_X, int32_t ncols, int32_t r0, int32_t r1,
                     double* d_out) {
  SLMM_TRY
  return spmm_impl(ms, k, d_X, ncols, r0, r1, d_out, true);
  SLMM_CATCH
}

int slmm_spmm_coldot_multi(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* d_X, int32_t ncols,
                           int32_t store_from, double* d_store, int32_t r0, int32_t r1, double* d_dots) {
  SLMM_TRY
  if (!ms || !ks || !d_X || !d_dots || nk <= 0 || nk > 2 || ncols <= 0 || ncols > 160)
    throw std::invalid_argument("slmm_spmm_coldot_multi: need 1 <= nk <= 2, ncols <= 160");
  if (store_from < 0 || store_from > ncols || (store_from < ncols && !d_store)) throw std::invalid_argument("bad store range");
  if (ms->sharded()) throw std::invalid_argument("row-block shards serve slmm_he_moments only");
  if (r0 < 0 || r1 > ms->n || r0 > r1) throw std::invalid_argument("bad row range");
  for (int g = 0; g < nk; g++) {
    if (ks[g] < 0 || ks[g] >= ms->K || !ms->m[ks[g]].data) throw std::invalid_argument("matrix not set");
    if (ms->m[ks[g]].pattern != ms->m[ks[0]].pattern) throw std::invalid_argument("matrices must share one pattern");
  }
  const int cpl = (ncols + 31) / 32;
#define GROUP_CASE(C)                                                                                       \
  if (nk == 1) launch_spmm_group<C, 1>(ms, ks, d_X, ncols, store_from, d_store, r0, r1, d_dots);            \
  else launch_spmm_group<C, 2>(ms, ks, d_X, ncols, store_from, d_store, r0, r1, d_dots);
  if (cpl <= 1) { GROUP_CASE(1) } else if (cpl <= 2) { GROUP_CASE(2) } else if (cpl <= 3) { GROUP_CASE(3) }
  else if (cpl <= 4) { GROUP_CASE(4) } else { GROUP_CASE(5) }
#undef GROUP_CASE
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_validate(slmm_matset_t* ms, int32_t k, int32_t* flags_out) {
  SLMM_TRY
  if (!ms || k < 0 || k >= ms->K || !flags_out || !ms->m[k].data) throw std::invalid_argument("bad arguments");
  const CsrDev& c = ms->m[k];
  DevPtr<int> d_flag = dev_alloc<int>(1);
  CUDA_OK(cudaMemsetAsync(d_flag.get(), 0, sizeof(int), 0));
  csr_validate_kernel<<<he_grid(ms->r1 - ms->r0), 256>>>(c.indptr, c.indices, ms->r0, ms->r1, ms->n, c.nnz, d_flag.get());
  g_launch_count++;
  int flag = 0;
  CUDA_OK(cudaMemcpy(&flag, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost));
  *flags_out = flag;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_device_arrays_equal_i32(const int32_t* d_a, const int32_t* d_b, int64_t count, int32_t* out) {
  SLMM_TRY
  if (!d_a || !d_b || !out || count < 0) throw std::invalid_argument("bad arguments");
  DevPtr<int> d_flag = dev_alloc<int>(1);
  CUDA_OK(cudaMemsetAsync(d_flag.get(), 0, sizeof(int), 0));
  if (count > 0) {
    const int grid = (int)std::min<int64_t>((count + 255) / 256, 148 * 16);
    arrays_differ_kernel<<<grid, 256>>>(d_a, d_b, count, d_flag.get());
    g_launch_count++;
  }
  int flag = 1;
  CUDA_OK(cudaMemcpy(&flag, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost));
  *out = flag ? 0 : 1;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_is_symmetric(slmm_matset_t* ms, int32_t k, int32_t* out) {
  SLMM_TRY
  if (!ms || k < 0 || k >= ms->K || !out || !ms->m[k].data) throw std::invalid_argument("bad arguments");
  CsrDev& c = ms->m[k];
  if (c.symmetric < 0 && ms->sharded()) { *out = 0; return SLMM_OK; }   // unknown until slmm_matset_set_symmetric
  if (c.symmetric < 0) {
    // one streaming pass: hash sums of the entries above / below the diagonal (the test the row-block shards use; a
    // mismatch survives with probability ~2^-64).  The exact kernel (a binary search per entry: 9 ms per matrix at
    // 1M individuals, a quarter of HE()'s device-side time) is slmm_device_csr_is_symmetric.
    DevPtr<unsigned long long> d = dev_alloc<unsigned long long>(2);
    CUDA_OK(cudaMemsetAsync(d.get(), 0, 2 * sizeof(unsigned long long), 0));
    symmetry_hash_kernel<<<he_grid(ms->n), 256>>>(c.indptr, c.indices, c.data, 0, ms->n, d.get());
    g_launch_count++;
    unsigned long long h2[2] = {0, 1};
    CUDA_OK(cudaMemcpy(h2, d.get(), sizeof(h2), cudaMemcpyDeviceToHost));
    c.symmetric = h2[0] == h2[1] ? 1 : 0;
  }
  *out = c.symmetric;
  return SLMM_OK;
  SLMM_CATCH
}

}  // extern "C"

namespace slmm {
template <int CPL, int G>
static void launch_quadform_sym(slmm_matset* ms, const int32_t* ks, const double* d_X, int ncols, const double* d_XB,
                                int nb, int r0, int r1, double* d_dots, double* d_gram) {
  GroupArgs<G> v;
  v.indptr = ms->m[ks[0]].indptr;
  v.indices = ms->m[ks[0]].indices;
  for (int g = 0; g < G; g++) v.data[g] = ms->m[ks[g]].data;
  const int grid = he_grid(r1 - r0);
  const size_t np = (size_t)grid * G * ncols, ng = d_XB ? (size_t)grid * G * nb * nb : 0;
  double* part = ms->partial(np + ng);
  quadform_sym_kernel<CPL, G><<<grid, 256>>>(v.indptr, v.indices, v, d_X, ncols, r0, r1, part);
  reduce_partials_kernel<<<G * ncols, 256>>>(part, grid, G * ncols, nullptr, d_dots);
  g_launch_count += 2;
  if (d_XB) {
    gram_sym_kernel<G><<<grid, 256>>>(v.indptr, v.indices, v, d_XB, nb, r0, r1, part + np);
    reduce_partials_kernel<<<G * nb * nb, 256>>>(part + np, grid, G * nb * nb, nullptr, d_gram);
    g_launch_count += 2;
  }
}
}  // namespace slmm

extern "C" {

int slmm_quadform_multi(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* d_X, int32_t ncols,
                        int32_t r0, int32_t r1, double* d_dots) {
  return slmm_quadform_gram_multi(ms, nk, ks, d_X, ncols, nullptr, 0, r0, r1, d_dots, nullptr);
}

int slmm_quadform_gram_multi(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* d_X, int32_t ncols,
                             const double* d_XB, int32_t nb, int32_t r0, int32_t r1, double* d_dots,
                             double* d_gram_half) {
  SLMM_TRY
  if (!ms || !ks || !d_X || !d_dots || nk <= 0 || nk > 2 || ncols <= 0 || ncols > 160)
    throw std::invalid_argument("slmm_quadform_gram_multi: need 1 <= nk <= 2, ncols <= 160");
  if (d_XB && (nb <= 0 || nb > QF_NB || !d_gram_half)) throw std::invalid_argument("narrow block: 1 <= nb <= 16");
  if (ms->sharded()) throw std::invalid_argument("row-block shards serve slmm_he_moments only");
  if (r0 < 0 || r1 > ms->n || r0 > r1) throw std::invalid_argument("bad row range");
  bool sym = true;
  for (int g = 0; g < nk; g++) {
    if (ks[g] < 0 || ks[g] >= ms->K || !ms->m[ks[g]].data) throw std::invalid_argument("matrix not set");
    if (ms->m[ks[g]].pattern != ms->m[ks[0]].pattern) throw std::invalid_argument("matrices must share one pattern");
    int32_t f = 0;
    const int rc = slmm_matset_is_symmetric(ms, ks[g], &f);
    if (rc != SLMM_OK) return rc;
    sym = sym && f;
  }
  if (!sym) {
    if (d_XB) throw std::invalid_argument("the fused Gram path needs symmetric matrices (use slmm_spmm_coldot_multi)");
    return slmm_spmm_coldot_multi(ms, nk, ks, d_X, ncols, ncols, nullptr, r0, r1, d_dots);   // full rows
  }
  const int cpl = (ncols + 31) / 32;
#define QF_CASE(C)                                                                                   \
  if (nk == 1) launch_quadform_sym<C, 1>(ms, ks, d_X, ncols, d_XB, nb, r0, r1, d_dots, d_gram_half); \
  else launch_quadform_sym<C, 2>(ms, ks, d_X, ncols, d_XB, nb, r0, r1, d_dots, d_gram_half);
  if (cpl <= 1) { QF_CASE(1) } else if (cpl <= 2) { QF_CASE(2) } else if (cpl <= 3) { QF_CASE(3) }
  else if (cpl <= 4) { QF_CASE(4) } else { QF_CASE(5) }
#undef QF_CASE
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_device_csr_is_symmetric(const int32_t* d_indptr, const int32_t* d_indices, const double* d_data, int32_t n,
                                 int32_t* out) {
  SLMM_TRY
  if (!d_indptr || !d_indices || !d_data || !out || n <= 0) throw std::invalid_argument("bad arguments");
  DevPtr<int> d_flag = dev_alloc<int>(1);
  CUDA_OK(cudaMemsetAsync(d_flag.get(), 0, sizeof(int), 0));
  symmetry_check_kernel<<<he_grid(n), 256>>>(d_indptr, d_indices, d_data, n, d_flag.get());
  g_launch_count++;
  int flag = 1;
  CUDA_OK(cudaMemcpy(&flag, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost));
  *out = flag ? 0 : 1;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_device_pattern_subset(const int32_t* d_ap, const int32_t* d_ai, const int32_t* d_bp, const int32_t* d_bi,
                               int32_t n, int32_t* out) {
  SLMM_TRY
  if (!d_ap || !d_ai || !d_bp || !d_bi || !out || n <= 0) throw std::invalid_argument("bad arguments");
  DevPtr<int> d_flag = dev_alloc<int>(1);
  CUDA_OK(cudaMemsetAsync(d_flag.get(), 0, sizeof(int), 0));
  pattern_subset_kernel<<<he_grid(n), 256>>>(d_ap, d_ai, d_bp, d_bi, n, d_flag.get());
  g_launch_count++;
  int flag = 1;
  CUDA_OK(cudaMemcpy(&flag, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost));
  *out = flag ? 0 : 1;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_set_row_range(slmm_matset_t* ms, int32_t r0, int32_t r1) {
  SLMM_TRY
  if (!ms || r0 < 0 || r1 > ms->n || r0 > r1) throw std::invalid_argument("bad row range");
  for (const CsrDev& c : ms->m)
    if (c.data) throw std::invalid_argument("set the row range before binding matrices");
  ms->r0 = r0;
  ms->r1 = r1;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_symmetry_hash(slmm_matset_t* ms, int32_t k, uint64_t* h_out2) {
  SLMM_TRY
  if (!ms || k < 0 || k >= ms->K || !h_out2 || !ms->m[k].data) throw std::invalid_argument("bad arguments");
  const CsrDev& c = ms->m[k];
  DevPtr<unsigned long long> d = dev_alloc<unsigned long long>(2);
  CUDA_OK(cudaMemsetAsync(d.get(), 0, 2 * sizeof(unsigned long long), 0));
  symmetry_hash_kernel<<<he_grid(ms->r1 - ms->r0), 256>>>(c.indptr, c.indices, c.data, ms->r0, ms->r1, d.get());
  g_launch_count++;
  CUDA_OK(cudaMemcpy(h_out2, d.get(), 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_set_symmetric(slmm_matset_t* ms, int32_t k, int32_t flag) {
  if (!ms || k < 0 || k >= ms->K) return SLMM_ERR_INVALID;
  ms->m[k].symmetric = flag ? 1 : 0;
  return SLMM_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Host -> device copies of large PAGEABLE arrays (the scipy CSR arrays the reference API hands us).  cudaMemcpy from
// pageable memory runs at a fraction of the link rate and Tensor.pin_memory() first copies the whole array into a
// freshly page-locked allocation (page-locking is the slow part).  Here a few worker threads copy chunks into a
// small ring of PERSISTENT pinned buffers and queue the DMA of each chunk as soon as it is staged, so the host copy
// of chunk i+1 overlaps the transfer of chunk i and nothing is page-locked per call.
namespace {
struct Stager {
  static constexpr int MAXT = 8, RING = 2;
  static constexpr size_t CHUNK = (size_t)8 << 20;
  void* buf[MAXT][RING] = {};
  cudaEvent_t ev[MAXT][RING] = {};
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  cudaStream_t st = nullptr;
  int device = -1;
  void init(int T) {
    int dev = 0;
    CUDA_OK(cudaGetDevice(&dev));
    if (st == nullptr || dev != device) {
      device = dev;
      CUDA_OK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
      CUDA_OK(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
      CUDA_OK(cudaEventCreateWithFlags(&ev_out, cudaEventDisableTiming));
    }
    for (int t = 0; t < T; t++)          // page-locked once per process, only for the workers actually used
      for (int r = 0; r < RING; r++)
        if (buf[t][r] == nullptr) {
          CUDA_OK(cudaHostAlloc(&buf[t][r], CHUNK, cudaHostAllocDefault));
          CUDA_OK(cudaEventCreateWithFlags(&ev[t][r], cudaEventDisableTiming));
        }
  }
};
Stager g_stager;
}  // namespace

int slmm_upload_h2d(void* d_dst, const void* h_src, int64_t nbytes, int32_t threads) {
  return slmm_upload_h2d_on(d_dst, h_src, nbytes, threads, nullptr);
}

int slmm_upload_h2d_on(void* d_dst, const void* h_src, int64_t nbytes, int32_t threads, void* stream) {
  SLMM_TRY
  if (!d_dst || !h_src || nbytes < 0) throw std::invalid_argument("bad arguments");
  if (nbytes == 0) return SLMM_OK;
  cudaStream_t on = (cudaStream_t)stream;
  if (nbytes < (int64_t)(4 << 20)) {            // small arrays: the driver's own staging is as good
    CUDA_OK(cudaMemcpyAsync(d_dst, h_src, (size_t)nbytes, cudaMemcpyHostToDevice, on));
    return SLMM_OK;
  }
  Stager& S = g_stager;
  const int T = std::max(1, std::min<int>(Stager::MAXT, threads > 0 ? threads : 4));
  S.init(T);
  const int64_t nchunks = (nbytes + (int64_t)Stager::CHUNK - 1) / (int64_t)Stager::CHUNK;
  int dev = S.device;
  // the destination may be recycled memory with work still queued on the calling stream
  CUDA_OK(cudaEventRecord(S.ev_in, on));
  CUDA_OK(cudaStreamWaitEvent(S.st, S.ev_in, 0));
  std::vector<cudaError_t> err(T, cudaSuccess);
  auto work = [&](int t) {
    cudaError_t e = cudaSetDevice(dev);
    int use = 0;
    for (int64_t c = t; c < nchunks && e == cudaSuccess; c += T, use++) {
      const int r = use % Stager::RING;
      const size_t off = (size_t)c * Stager::CHUNK, sz = std::min<size_t>(Stager::CHUNK, (size_t)nbytes - off);
      if (use >= Stager::RING) e = cudaEventSynchronize(S.ev[t][r]);      // the DMA that last used this buffer is done
      if (e != cudaSuccess) break;
      memcpy(S.buf[t][r], (const char*)h_src + off, sz);
      e = cudaMemcpyAsync((char*)d_dst + off, S.buf[t][r], sz, cudaMemcpyHostToDevice, S.st);
      if (e == cudaSuccess) e = cudaEventRecord(S.ev[t][r], S.st);
    }
    err[t] = e;
  };
  std::vector<std::thread> pool;
  for (int t = 1; t < T; t++) pool.emplace_back(work, t);
  work(0);
  for (auto& th : pool) th.join();
  for (int t = 0; t < T; t++) CUDA_OK(err[t]);
  CUDA_OK(cudaEventRecord(S.ev_out, S.st));
  CUDA_OK(cudaStreamWaitEvent(on, S.ev_out, 0));
  // the staging buffers are reused by the next call: its first writes must not overtake this call's last DMAs
  CUDA_OK(cudaEventSynchronize(S.ev_out));
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_upload_h2d_2d(void* d_dst, int64_t dst_pitch, const void* h_src, int64_t src_pitch, int64_t width_bytes,
                       int64_t rows) {
  return slmm_upload_h2d_2d_on(d_dst, dst_pitch, h_src, src_pitch, width_bytes, rows, nullptr);
}

int slmm_upload_h2d_2d_on(void* d_dst, int64_t dst_pitch, const void* h_src, int64_t src_pitch, int64_t width_bytes,
                          int64_t rows, void* stream) {
  SLMM_TRY
  cudaStream_t on = (cudaStream_t)stream;
  if (!d_dst || !h_src || width_bytes < 0 || rows < 0 || dst_pitch < width_bytes || src_pitch < width_bytes)
    throw std::invalid_argument("bad arguments");
  if (width_bytes == 0 || rows == 0) return SLMM_OK;
  // the DMA engine walks the pitched source: no host-side packing of the column slice
  CUDA_OK(cudaMemcpy2DAsync(d_dst, (size_t)dst_pitch, h_src, (size_t)src_pitch, (size_t)width_bytes, (size_t)rows,
                            cudaMemcpyHostToDevice, on));
  CUDA_OK(cudaStreamSynchronize(on));           // the host block may be reused by the caller right away
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_pattern_id(const slmm_matset_t* ms, int32_t k, int32_t* out) {
  if (!ms || k < 0 || k >= ms->K || !out) return SLMM_ERR_INVALID;
  *out = ms->m[k].pattern;
  return SLMM_OK;
}

}  // extern "C"
