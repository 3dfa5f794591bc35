// Predicted random effects (BLUP) and their stochastic prediction error variances: the column-mapped products of the
// relationship matrices over ALL individuals with blocks that live on the observed ones.  The reference has no
// counterpart.
//
// A_k is held over all N individuals; the fit (and so every solved block X) covers the n observed ones.  colmap[N]
// sends a column of A_k to its row of X, or to -1 for an individual without a phenotype (the entry is skipped); a NULL
// map is the identity (n = N).  Both kernels give a warp one row of A_k, read the row's entries in stored order and
// use no atomics, so their output is the same bits on every run.
#include "common.h"
#include "matset.h"

namespace slmm {

constexpr int BL_MAXG = 2;        // matrices of one pattern group
constexpr int BL_SPMM_COLS = 32;  // columns of the product: one per lane
constexpr int BL_SUMSQ_COLS = 128;  // columns of a probe block: four per lane

template <int G>
struct BlupGroup {
  const int32_t* indptr;
  const int32_t* indices;
  const double* data[G];
  double sigma[G];
};

namespace {
__device__ __forceinline__ double bl_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
}  // namespace

// Y_g[i, :] = sigma_g A_g[i, obs] X for every row i of A: out[(g * N + i) * ncols + lane].  Up to 32 (column, value)
// pairs of the row are staged one per lane, the column already mapped, then broadcast one at a time; every lane adds
// the entry's product into its own column.
template <int G>
__global__ void __launch_bounds__(256) blup_spmm_kernel(BlupGroup<G> a, const int32_t* __restrict__ colmap,
                                                        const double* __restrict__ X, int ncols, int N,
                                                        double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= N) return;
  const int b = a.indptr[row], e = a.indptr[row + 1];
  double acc[G];
#pragma unroll
  for (int g = 0; g < G; g++) acc[g] = 0.0;
  for (int p0 = b; p0 < e; p0 += 32) {
    const int pl = p0 + lane;
    int mycol = -1;
    double myval[G];
#pragma unroll
    for (int g = 0; g < G; g++) myval[g] = 0.0;
    if (pl < e) {
      const int c = a.indices[pl];
      mycol = colmap ? colmap[c] : c;
#pragma unroll
      for (int g = 0; g < G; g++) myval[g] = a.data[g][pl];
    }
    const int cnt = min(32, e - p0);
    // unrolled with predicated loads: several gathered rows of X are in flight per lane (a skipped entry adds 0)
#pragma unroll 8
    for (int k = 0; k < cnt; k++) {
      const int col = __shfl_sync(0xffffffffu, mycol, k);
      double v[G];
#pragma unroll
      for (int g = 0; g < G; g++) v[g] = __shfl_sync(0xffffffffu, myval[g], k);
      const double x = (col >= 0 && lane < ncols) ? __ldg(X + (int64_t)col * ncols + lane) : 0.0;
#pragma unroll
      for (int g = 0; g < G; g++) acc[g] = fma(v[g], x, acc[g]);
    }
  }
  if (lane < ncols)
#pragma unroll
    for (int g = 0; g < G; g++) out[((int64_t)g * N + row) * ncols + lane] = a.sigma[g] * acc[g];
}

// Per row i and matrix g: sum2[i * G + g] = sum_j t_ij^2 and sum4[i * G + g] = sum_j t_ij^4 with
// t = sigma_g A_g[i, obs] W for a probe block W of <= 128 columns (CPL per lane).  t is never written out: each
// gathered W row (1 KB at 128 columns) is used for every matrix of the group and then dropped.
template <int CPL, int G>
__global__ void __launch_bounds__(256) blup_rowsumsq_kernel(BlupGroup<G> a, const int32_t* __restrict__ colmap,
                                                            const double* __restrict__ W, int ncols, int N,
                                                            double* __restrict__ sum2, double* __restrict__ sum4) {
  const int lane = threadIdx.x & 31;
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= N) return;
  const int b = a.indptr[row], e = a.indptr[row + 1];
  double acc[G][CPL];
#pragma unroll
  for (int g = 0; g < G; g++)
#pragma unroll
    for (int c = 0; c < CPL; c++) acc[g][c] = 0.0;
  for (int p0 = b; p0 < e; p0 += 32) {
    const int pl = p0 + lane;
    int mycol = -1;
    double myval[G];
#pragma unroll
    for (int g = 0; g < G; g++) myval[g] = 0.0;
    if (pl < e) {
      const int c = a.indices[pl];
      mycol = colmap ? colmap[c] : c;
#pragma unroll
      for (int g = 0; g < G; g++) myval[g] = a.data[g][pl];
    }
    const int cnt = min(32, e - p0);
    // not unrolled: each entry already puts CPL loads per lane in flight, and an unrolled, predicated loop measured
    // slower at 128 columns (7.4 against 6.6 ms per block at 250K, DESIGN.md 6d)
    for (int k = 0; k < cnt; k++) {
      const int col = __shfl_sync(0xffffffffu, mycol, k);
      double v[G];
#pragma unroll
      for (int g = 0; g < G; g++) v[g] = __shfl_sync(0xffffffffu, myval[g], k);
      if (col < 0) continue;
      const double* wr = W + (int64_t)col * ncols;
#pragma unroll
      for (int c = 0; c < CPL; c++) {
        const int j = lane + 32 * c;
        if (j < ncols) {
          const double x = wr[j];
#pragma unroll
          for (int g = 0; g < G; g++) acc[g][c] = fma(v[g], x, acc[g][c]);
        }
      }
    }
  }
#pragma unroll
  for (int g = 0; g < G; g++) {
    double s2 = 0.0, s4 = 0.0;
#pragma unroll
    for (int c = 0; c < CPL; c++) {
      const double t = a.sigma[g] * acc[g][c];
      const double t2 = t * t;
      s2 += t2;
      s4 = fma(t2, t2, s4);
    }
    s2 = bl_warp_sum(s2);
    s4 = bl_warp_sum(s4);
    if (lane == 0) {
      sum2[row * G + g] = s2;
      sum4[row * G + g] = s4;
    }
  }
}

// *bad = 1 if a map entry lies outside [-1, nobs): the kernels would read X / W out of range.
__global__ void blup_colmap_check_kernel(const int32_t* __restrict__ colmap, int N, int64_t nobs, int* __restrict__ bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N && (colmap[i] < -1 || colmap[i] >= nobs)) *bad = 1;
}

namespace {
// The map check's flag, one int per device, kept across calls (the PEV calls the rowsumsq pass once per probe block).
struct BlupFlag {
  DevPtr<int> buf;
  int device = -1;
  int* get() {
    int dev = 0;
    CUDA_OK(cudaGetDevice(&dev));
    if (dev != device) {
      buf.reset();
      buf = dev_alloc<int>(1);
      device = dev;
    }
    return buf.get();
  }
};
BlupFlag g_blup_flag;

template <int G>
BlupGroup<G> blup_group(const slmm_matset_t* ms, const int32_t* ks, const double* sigmas) {
  BlupGroup<G> a;
  const CsrDev& lead = ms->m[ks[0]];
  a.indptr = lead.indptr;
  a.indices = lead.indices;
  for (int g = 0; g < G; g++) {
    a.data[g] = ms->m[ks[g]].data;
    a.sigma[g] = sigmas[g];
  }
  return a;
}

void blup_check(const slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* sigmas, const int32_t* d_colmap,
                const double* d_X, int64_t nobs, int32_t ncols, int32_t max_cols, const char* who) {
  if (!ms || !ks || !sigmas || !d_X || nk <= 0 || nk > BL_MAXG || ncols <= 0 || ncols > max_cols)
    throw std::invalid_argument(std::string(who) + ": need 1 <= nk <= 2 and 1 <= ncols <= " + std::to_string(max_cols));
  if (ms->sharded()) throw std::invalid_argument("row-block shards serve slmm_he_moments only");
  if (nobs <= 0 || nobs > ms->n) throw std::invalid_argument(std::string(who) + ": need 0 < nobs <= n");
  if (!d_colmap && nobs != ms->n) throw std::invalid_argument(std::string(who) + ": without a column map nobs must be n");
  for (int g = 0; g < nk; g++) {
    if (ks[g] < 0 || ks[g] >= ms->K || !ms->m[ks[g]].data) throw std::invalid_argument("matrix not set");
    if (ms->m[ks[g]].pattern != ms->m[ks[0]].pattern) throw std::invalid_argument("matrices must share one pattern");
  }
  if (d_colmap) {             // checked on the device: the map is device data
    int* d_bad = g_blup_flag.get();
    CUDA_OK(cudaMemsetAsync(d_bad, 0, sizeof(int), 0));
    blup_colmap_check_kernel<<<(ms->n + 255) / 256, 256>>>(d_colmap, ms->n, nobs, d_bad);
    g_launch_count++;
    CUDA_OK(cudaGetLastError());
    int bad = 0;
    CUDA_OK(cudaMemcpy(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad) throw std::invalid_argument(std::string(who) + ": column map entries must lie in [-1, nobs)");
  }
}

inline unsigned blup_grid(int N) { return (unsigned)(((int64_t)N * 32 + 255) / 256); }
}  // namespace

}  // namespace slmm

using namespace slmm;

extern "C" {

int slmm_blup_spmm(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* sigmas, const int32_t* d_colmap,
                   const double* d_X, int64_t nobs, int32_t ncols, double* d_out) {
  SLMM_TRY
  blup_check(ms, nk, ks, sigmas, d_colmap, d_X, nobs, ncols, BL_SPMM_COLS, "slmm_blup_spmm");
  if (!d_out) throw std::invalid_argument("bad arguments");
  const int N = ms->n;
  if (nk == 1)
    blup_spmm_kernel<1><<<blup_grid(N), 256>>>(blup_group<1>(ms, ks, sigmas), d_colmap, d_X, ncols, N, d_out);
  else
    blup_spmm_kernel<2><<<blup_grid(N), 256>>>(blup_group<2>(ms, ks, sigmas), d_colmap, d_X, ncols, N, d_out);
  g_launch_count++;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_blup_rowsumsq(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* sigmas, const int32_t* d_colmap,
                       const double* d_W, int64_t nobs, int32_t ncols, double* d_sum2, double* d_sum4) {
  SLMM_TRY
  blup_check(ms, nk, ks, sigmas, d_colmap, d_W, nobs, ncols, BL_SUMSQ_COLS, "slmm_blup_rowsumsq");
  if (!d_sum2 || !d_sum4) throw std::invalid_argument("bad arguments");
  const int N = ms->n;
  const int cpl = (ncols + 31) / 32;
#define BL_SUMSQ(C, G)                                                                                             \
  blup_rowsumsq_kernel<C, G><<<blup_grid(N), 256>>>(blup_group<G>(ms, ks, sigmas), d_colmap, d_W, ncols, N, d_sum2, \
                                                     d_sum4)
#define BL_SUMSQ_G(C) \
  if (nk == 1) BL_SUMSQ(C, 1); else BL_SUMSQ(C, 2);
  if (cpl <= 1) { BL_SUMSQ_G(1) }
  else if (cpl <= 2) { BL_SUMSQ_G(2) }
  else { BL_SUMSQ_G(4) }
#undef BL_SUMSQ_G
#undef BL_SUMSQ
  g_launch_count++;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

}  // extern "C"
