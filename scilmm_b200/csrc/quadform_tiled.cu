// Column quadratic forms w_c' A w_c of the probe block and the Gram matrix of the narrow block [V^-1 C | V^-1 r]
// (reference scilmm/SparseCholesky.py:65-66,70: np.sum(mats[i].dot(sim_vec) * sim_vec, axis=0),
// invV_y.dot(mats[i].dot(invV_y)), invV_C.T.dot(mats[i].dot(invV_C))) on a TILED copy of the matrix.
//
// Why: the row-per-warp kernel (sparse_ops.cu quadform_sym_kernel) gathers one 8*ncols-byte row of the dense block
// per visited entry: 32 GB through L2 at the 250K config for 1.5 GB of algorithmic traffic - 2 % of the HBM roofline.
// In the factor's fill-reducing (nested dissection) order the entries of 64 consecutive rows share their columns
// (8.8 entries per distinct (row block, column) pair, measured on the 250K IBD matrix; 1.4 in the input order).  So the
// lower triangle is cut into tiles of 64 permuted rows x 64 DISTINCT columns; a CTA stages the 64 gathered rows of the
// dense block in shared memory once and every entry of the tile reads them from there:
//   dots[g][c] = sum_i x[i,c] * ( sum_j v_g(i,j) x[j,c] ),  v = a for the diagonal, 2a below it (symmetric matrix);
//   Mh[g]      = sum_i xb_i (sum_j v_g(i,j) xb_j)'  for the first nb columns (the narrow block), Gram = (Mh + Mh')/2:
//                the pass leaves the row products hb_i = sum_j v(i,j) xb_j per (CTA, row block) pair in global memory
//                and a small second kernel folds the outer products (a serial fold inside the pass cost 34 of 40 ms:
//                the tree's leaves give some CTAs hundreds of tiny row blocks).
// Everything is accumulated in a fixed order (tiles are assigned to CTAs by a static partition, rows to warps by
// index): results are bit-reproducible.  The tiling is built once per session on the device (two radix sorts).
#include <algorithm>
#include <cassert>
#ifdef SLMM_DEBUG_ASSERTS
#define QT_ASSERT(x) assert(x)
#else
#define QT_ASSERT(x) ((void)0)   // device-side checks of the tile structures: build with -DSLMM_DEBUG_ASSERTS
#endif
#include <cstring>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.h"
#include "matset.h"

namespace slmm {

constexpr int QT_RB = 64;     // permuted rows per row block
constexpr int QT_CH = 64;     // distinct columns per tile (rows of the dense block staged in shared memory)
constexpr int QT_NB = 16;     // widest narrow block
constexpr int QT_ECAP = 768;  // entries of a tile staged in shared memory (larger tiles read them from global memory)

// ---- build ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) qt_keys_kernel(const int32_t* __restrict__ ap, const int32_t* __restrict__ ai, int n,
                                                      const int32_t* __restrict__ iperm, uint64_t* __restrict__ keys,
                                                      uint32_t* __restrict__ pos, unsigned long long* __restrict__ nkeep) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  unsigned long long kept = 0;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
    const int pi = iperm[r];
    for (int p = ap[r] + lane; p < ap[r + 1]; p += 32) {
      const int pj = iperm[ai[p]];
      uint64_t key = ~0ull;
      if (pj <= pi) {                       // one of the two mirrored copies (+ the diagonal)
        key = ((((uint64_t)(pi / QT_RB)) << 28 | (uint64_t)pj) << 6) | (uint64_t)(pi % QT_RB);
        kept++;
      }
      keys[p] = key;
      pos[p] = (uint32_t)p;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
  if (lane == 0 && kept) atomicAdd(nkeep, kept);
}

__global__ void __launch_bounds__(256) qt_heads_kernel(const uint64_t* __restrict__ keys, int64_t m, int32_t* __restrict__ head) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < m; e += (int64_t)gridDim.x * blockDim.x)
    head[e] = (e == 0 || (keys[e] >> 6) != (keys[e - 1] >> 6)) ? 1 : 0;
}

// first entry of every row block in the sorted key array
__global__ void __launch_bounds__(256) qt_rbstart_kernel(const uint64_t* __restrict__ keys, int64_t m, int nrb,
                                                         int64_t* __restrict__ rbstart) {
  for (int rb = blockIdx.x * blockDim.x + threadIdx.x; rb <= nrb; rb += gridDim.x * blockDim.x) {
    const uint64_t want = (uint64_t)rb << 34;
    int64_t lo = 0, hi = m;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (keys[mid] < want) lo = mid + 1; else hi = mid; }
    rbstart[rb] = lo;
  }
}

__global__ void __launch_bounds__(256) qt_gather_kernel(const int32_t* __restrict__ src, const int64_t* __restrict__ idx, int count,
                                                        int32_t* __restrict__ out) {
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < count; q += gridDim.x * blockDim.x) out[q] = src[idx[q]];
}

__global__ void __launch_bounds__(256) qt_keys2_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ pos,
                                                       const int32_t* __restrict__ gidx, int64_t m,
                                                       const int32_t* __restrict__ dcol_base, const int32_t* __restrict__ tile_base,
                                                       const int32_t* __restrict__ ai, uint64_t* __restrict__ keys2,
                                                       int32_t* __restrict__ dcols) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < m; e += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t key = keys[e];
    const int rb = (int)(key >> 34), pj = (int)((key >> 6) & 0xfffffffull), lrow = (int)(key & 63);
    const int g = gidx[e] - 1;                       // global index of the (row block, column) pair
    const int dcol = g - dcol_base[rb];
    QT_ASSERT(dcol >= 0);
    const int tile = tile_base[rb] + dcol / QT_CH, lcol = dcol % QT_CH;
    const int diag = (rb * QT_RB + lrow) == pj ? 1 : 0;
    keys2[e] = ((uint64_t)tile << 13) | ((uint64_t)lrow << 7) | ((uint64_t)lcol << 1) | (uint64_t)diag;
    if (e == 0 || (keys[e - 1] >> 6) != (key >> 6)) dcols[g] = ai[pos[e]];      // ORIGINAL id of the gathered row
  }
}

__global__ void __launch_bounds__(256) qt_tileptr_kernel(const uint64_t* __restrict__ keys2, int64_t m, int ntiles,
                                                         int64_t* __restrict__ tile_ptr, uint16_t* __restrict__ rowptr) {
  // thread per (tile, local row): first entry with key >= (tile, lrow, 0)
  const int64_t total = (int64_t)ntiles * (QT_RB + 1) + 1;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t tile = q / (QT_RB + 1);
    const int lr = (int)(q % (QT_RB + 1));
    const uint64_t want = ((uint64_t)tile << 13) + ((uint64_t)lr << 7);       // lr == 64 carries into the tile bits
    int64_t lo = 0, hi = m;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (keys2[mid] < want) lo = mid + 1; else hi = mid; }
    if (tile < ntiles) {
      // row starts are relative to the tile's first entry: search the tile start as well (lr == 0 gives it)
      const uint64_t w0 = (uint64_t)tile << 13;
      int64_t l0 = 0, h0 = m;
      while (l0 < h0) { const int64_t mid = (l0 + h0) >> 1; if (keys2[mid] < w0) l0 = mid + 1; else h0 = mid; }
      rowptr[tile * (QT_RB + 1) + lr] = (uint16_t)(lo - l0);
      if (lr == 0) tile_ptr[tile] = l0;
    } else if (lr == 0) {
      tile_ptr[ntiles] = m;
    }
  }
}

__global__ void __launch_bounds__(256) qt_pack_kernel(const uint64_t* __restrict__ keys2, int64_t m, uint16_t* __restrict__ rc) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < m; e += (int64_t)gridDim.x * blockDim.x)
    rc[e] = (uint16_t)(keys2[e] & 0x7f);            // local column << 1 | diagonal flag
}

__global__ void __launch_bounds__(256) qt_values_kernel(const uint16_t* __restrict__ rc, const uint32_t* __restrict__ pos,
                                                        const double* __restrict__ data, int64_t m, int64_t nnz,
                                                        double* __restrict__ out) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < m; e += (int64_t)gridDim.x * blockDim.x) {
    QT_ASSERT((int64_t)pos[e] < nnz);
    out[e] = ((rc[e] & 1) ? 1.0 : 2.0) * data[pos[e]];          // off-diagonal entries stand for both triangles
  }
}

// ---- the pass ---------------------------------------------------------------------------------------------------
struct QtArgs {
  int64_t nentries, ndistinct;
  int32_t ntiles, nrb, n, pad;
  const int64_t* tile_ptr;
  const int32_t *tile_rb, *tile_dc0, *tile_nc, *dcols, *rowid, *cta_begin, *pair_base;
  double* hpairs;
  long long* cta_cycles;
  const uint16_t *rowptr, *rc;
  const uint8_t* roword;
  const double* vals[2];
};

__device__ __forceinline__ void qt_cp_async8(double* smem_dst, const double* gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(gsrc) : "memory");
}

template <int CPL, int G>
__global__ void __launch_bounds__(256, 2) quadform_tiled_kernel(QtArgs a, const double* __restrict__ X, int ncx, int nb,
                                                                double* __restrict__ part_dots, double* __restrict__ part_gram) {
  constexpr int LDX = CPL * 32;
  extern __shared__ double qsm[];
  double* Xs = qsm;                                   // [QT_CH][LDX]  gathered rows of the dense block
  double* hbS = Xs + QT_CH * LDX;                     // [QT_RB][G][QT_NB]  narrow-block row products of this row block
  double* vS = hbS + QT_RB * G * QT_NB;               // [G][QT_ECAP]  values of the tile's entries
  uint16_t* rcS = reinterpret_cast<uint16_t*>(vS + G * QT_ECAP);      // [QT_ECAP]  local column << 1 | diagonal flag
  __shared__ uint16_t rp_s[QT_RB + 1];
  __shared__ uint8_t ro_s[QT_RB];                     // row order of the tile: slot s of warp w at [s * 8 + w]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t_begin = a.cta_begin[blockIdx.x], t_end = a.cta_begin[blockIdx.x + 1];
  const long long clk0 = clock64();
  double dot[G][CPL];
#pragma unroll
  for (int g = 0; g < G; g++)
#pragma unroll
    for (int c = 0; c < CPL; c++) dot[g][c] = 0.0;
  for (int q = tid; q < QT_CH * LDX + QT_RB * G * QT_NB; q += 256) qsm[q] = 0.0;   // incl. the padding columns of Xs
  int pair = a.pair_base[blockIdx.x];
  __syncthreads();
  QT_ASSERT(t_begin >= 0 && t_begin <= t_end && t_end <= a.ntiles);
  // metadata of a tile is fetched one tile ahead; all independent loads of the staging phase are issued before any is
  // consumed (the per-CTA profile put the fixed cost of a tile at 16 000 cycles = 4-5 dependent global round trips)
  int rb_n = 0, nc_n = 0, dc0_n = 0;
  int64_t tb_n = 0, te_n = 0;
  if (t_begin < t_end) {
    rb_n = a.tile_rb[t_begin]; nc_n = a.tile_nc[t_begin]; dc0_n = a.tile_dc0[t_begin];
    tb_n = a.tile_ptr[t_begin]; te_n = a.tile_ptr[t_begin + 1];
  }
  for (int t = t_begin; t < t_end; t++) {
    const int rb = rb_n, nc = nc_n, dc0 = dc0_n;
    const int64_t tb = tb_n;
    const int ne = (int)(te_n - tb_n);
    if (t + 1 < t_end) {
      rb_n = a.tile_rb[t + 1]; nc_n = a.tile_nc[t + 1]; dc0_n = a.tile_dc0[t + 1];
      tb_n = te_n; te_n = a.tile_ptr[t + 2];
    }
    QT_ASSERT(rb >= 0 && rb < a.nrb && nc > 0 && nc <= QT_CH && dc0 >= 0 && (int64_t)dc0 + nc <= a.ndistinct);
    QT_ASSERT(tb >= 0 && ne >= 0 && tb + ne <= a.nentries);
    // stage the tile: row starts, entries (if they fit), the nc gathered rows of X
    const bool staged = ne <= QT_ECAP;
    const uint16_t v_rp = tid <= QT_RB ? a.rowptr[(int64_t)t * (QT_RB + 1) + tid] : (uint16_t)0;
    const uint8_t v_ro = tid < QT_RB ? a.roword[(int64_t)t * QT_RB + tid] : (uint8_t)0;
    int dcv[QT_CH / 8];
#pragma unroll
    for (int q = 0; q < QT_CH / 8; q++) dcv[q] = (warp + 8 * q < nc) ? a.dcols[dc0 + warp + 8 * q] : -1;
    uint16_t v_rc[QT_ECAP / 256];
#pragma unroll
    for (int q = 0; q < QT_ECAP / 256; q++) v_rc[q] = (staged && tid + 256 * q < ne) ? a.rc[tb + tid + 256 * q] : (uint16_t)0;
    if (staged) {
      for (int e = tid; e < ne; e += 256) {
#pragma unroll
        for (int g = 0; g < G; g++) qt_cp_async8(vS + g * QT_ECAP + e, a.vals[g] + tb + e);
      }
    }
    if (tid <= QT_RB) rp_s[tid] = v_rp;
    if (tid < QT_RB) ro_s[tid] = v_ro;
#pragma unroll
    for (int q = 0; q < QT_ECAP / 256; q++)
      if (staged && tid + 256 * q < ne) rcS[tid + 256 * q] = v_rc[q];
#pragma unroll
    for (int q = 0; q < QT_CH / 8; q++) {
      if (dcv[q] < 0) continue;
      QT_ASSERT(dcv[q] < a.n);
      const double* src = X + (int64_t)dcv[q] * ncx;
      double* dst = Xs + (warp + 8 * q) * LDX;
      for (int j = lane; j < ncx; j += 32) qt_cp_async8(dst + j, src + j);
    }
    asm volatile("cp.async.wait_all;\n" ::: "memory");
    __syncthreads();
    // first entry chunk of the warp's next row, fetched one row ahead (tiles too large for the staging buffer)
    int nx_rc = 0;
    double nx_v[G];
#pragma unroll
    for (int g = 0; g < G; g++) nx_v[g] = 0.0;
    if (!staged && ro_s[warp] != 0xFF) {
      const int r0 = ro_s[warp];
      const int pl = rp_s[r0] + lane;
      if (pl < rp_s[r0 + 1]) {
        nx_rc = (int)a.rc[tb + pl];
#pragma unroll
        for (int g = 0; g < G; g++) nx_v[g] = __ldcs(a.vals[g] + tb + pl);
      }
    }
    // rows by decreasing length, dealt to the warps in snake order at build time: the barrier at the end of the tile
    // cost 20 % of the warp samples when warp w simply took rows w, w + 8, ...
    for (int slot = 0; slot < QT_RB / 8; slot++) {
      const int lr = ro_s[slot * 8 + warp];
      if (lr == 0xFF) break;                               // the remaining slots of this warp are empty rows
      const int e0 = rp_s[lr], e1 = rp_s[lr + 1];
      QT_ASSERT(e0 < e1 && tb + e1 <= a.tile_ptr[t + 1]);
      const int cur_rc = nx_rc;
      double cur_v[G];
#pragma unroll
      for (int g = 0; g < G; g++) cur_v[g] = nx_v[g];
      if (!staged && slot + 1 < QT_RB / 8) {
        const int rn = ro_s[(slot + 1) * 8 + warp];
        const int pl = rn != 0xFF ? rp_s[rn] + lane : 0;
        const bool in = rn != 0xFF && pl < rp_s[rn + 1];
        nx_rc = in ? (int)a.rc[tb + pl] : 0;
#pragma unroll
        for (int g = 0; g < G; g++) nx_v[g] = in ? __ldcs(a.vals[g] + tb + pl) : 0.0;
      }
      if (e0 == e1) continue;
      double acc[G][CPL];
#pragma unroll
      for (int g = 0; g < G; g++)
#pragma unroll
        for (int c = 0; c < CPL; c++) acc[g][c] = 0.0;
      // the row's own x_i: issued before the entry loop so its latency hides behind it
      const int row = a.rowid[rb * QT_RB + lr];
      QT_ASSERT(row >= 0 && row < a.n);
      const double* xi = X + (int64_t)row * ncx + lane;
      double xrow[CPL];
#pragma unroll
      for (int c = 0; c < CPL; c++) xrow[c] = (lane + 32 * c < ncx) ? xi[32 * c] : 0.0;
      for (int p0 = e0; p0 < e1; p0 += 32) {
        const int pl = p0 + lane;
        const bool first = p0 == e0 && !staged;                 // already in registers
        const int myrc = pl < e1 ? (first ? cur_rc : (int)(staged ? rcS[pl] : a.rc[tb + pl])) : 0;
        double myv[G];
#pragma unroll
        for (int g = 0; g < G; g++)
          myv[g] = pl < e1 ? (first ? cur_v[g] : (staged ? vS[g * QT_ECAP + pl] : __ldcs(a.vals[g] + tb + pl))) : 0.0;
        const int cnt = min(32, e1 - p0);
        for (int k = 0; k < cnt; k++) {
          const int lcol = __shfl_sync(0xffffffffu, myrc, k) >> 1;
          QT_ASSERT(lcol >= 0 && lcol < nc);
          double v[G];
#pragma unroll
          for (int g = 0; g < G; g++) v[g] = __shfl_sync(0xffffffffu, myv[g], k);
          const double* xr = Xs + lcol * LDX + lane;
#pragma unroll
          for (int c = 0; c < CPL; c++) {
            const double x = xr[32 * c];
#pragma unroll
            for (int g = 0; g < G; g++) acc[g][c] += v[g] * x;
          }
        }
      }
#pragma unroll
      for (int c = 0; c < CPL; c++)
#pragma unroll
        for (int g = 0; g < G; g++) dot[g][c] += acc[g][c] * xrow[c];
      if (lane < nb) {                               // this warp owns the row: plain accumulation
#pragma unroll
        for (int g = 0; g < G; g++) hbS[(lr * G + g) * QT_NB + lane] += acc[g][0];
      }
    }
    __syncthreads();
    // end of the row block (or of this CTA's range): park the narrow-block row products of this (CTA, row block)
    // pair in global memory; qt_gram_finish_kernel folds them into the Gram matrix
    if (nb > 0 && (t + 1 == t_end || rb_n != rb)) {
      double* hp = a.hpairs + (int64_t)pair * (QT_RB * 2 * QT_NB);
      for (int q = tid; q < QT_RB * G * QT_NB; q += 256) { hp[q] = hbS[q]; hbS[q] = 0.0; }
      pair++;
      __syncthreads();
    }
  }
  // per-CTA partials: dots over the 8 warps (fixed order)
  double* red = Xs;                                    // [8][G][LDX]
  __syncthreads();
#pragma unroll
  for (int g = 0; g < G; g++)
#pragma unroll
    for (int c = 0; c < CPL; c++) red[(warp * G + g) * LDX + lane + 32 * c] = dot[g][c];
  __syncthreads();
  for (int q = tid; q < G * ncx; q += 256) {
    const int g = q / ncx, j = q - g * ncx;
    double s = 0.0;
    for (int w = 0; w < 8; w++) s += red[(w * G + g) * LDX + j];
    part_dots[(int64_t)blockIdx.x * G * ncx + q] = s;
  }
  if (tid == 0) a.cta_cycles[blockIdx.x] = clock64() - clk0;
}

// Gram fold: Mh[g] += xb_i hb_i' over the rows of every (CTA, row block) pair.  CTA c takes pairs c, c + gridDim, ...
// (a fixed assignment), warp w the rows w, w + 8, ...; lane q < nb owns column q of Mh in registers.
template <int G>
__global__ void __launch_bounds__(256) qt_gram_finish_kernel(const double* __restrict__ hpairs, const int32_t* __restrict__ pair_rb,
                                                             int npairs, const int32_t* __restrict__ rowid,
                                                             const double* __restrict__ X, int ncx, int nb,
                                                             double* __restrict__ part_gram) {
  __shared__ double red[8][G][QT_NB][QT_NB];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double mh[G][QT_NB];
#pragma unroll
  for (int g = 0; g < G; g++)
#pragma unroll
    for (int p = 0; p < QT_NB; p++) mh[g][p] = 0.0;
  for (int pr = blockIdx.x; pr < npairs; pr += gridDim.x) {
    const int rb = pair_rb[pr];
    const double* hp = hpairs + (int64_t)pr * (QT_RB * 2 * QT_NB);
    for (int lr = warp; lr < QT_RB; lr += 8) {
      const int row = rowid[rb * QT_RB + lr];
      if (row < 0) continue;
      const double bi = lane < nb ? X[(int64_t)row * ncx + lane] : 0.0;
      double hb[G];
#pragma unroll
      for (int g = 0; g < G; g++) hb[g] = lane < nb ? hp[(lr * G + g) * QT_NB + lane] : 0.0;
#pragma unroll
      for (int p = 0; p < QT_NB; p++) {
        const double bp = __shfl_sync(0xffffffffu, bi, p);      // 0 for p >= nb
#pragma unroll
        for (int g = 0; g < G; g++) mh[g][p] += bp * hb[g];
      }
    }
  }
  if (lane < QT_NB) {
#pragma unroll
    for (int g = 0; g < G; g++)
#pragma unroll
      for (int p = 0; p < QT_NB; p++) red[warp][g][p][lane] = mh[g][p];
  }
  __syncthreads();
  for (int q = threadIdx.x; q < G * nb * nb; q += 256) {
    const int g = q / (nb * nb), p = (q / nb) % nb, j = q % nb;
    double s2 = 0.0;
    for (int w = 0; w < 8; w++) s2 += red[w][g][p][j];
    part_gram[(int64_t)blockIdx.x * G * nb * nb + q] = 0.5 * s2;        // Gram = half + half'
  }
}

__global__ void qt_reduce_kernel(const double* __restrict__ partial, int nblocks, int nv, double* __restrict__ dst) {
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
  if (threadIdx.x == 0) dst[k] = sh[0];
}

template <int CPL, int G>
static void qt_launch(const QuadTiles& T, const QtArgs& a, const double* d_X, int ncx, int nb, double* part_dots,
                      double* part_gram, double* d_dots, double* d_gram) {
  const size_t smem = ((size_t)QT_CH * CPL * 32 + (size_t)QT_RB * G * QT_NB + (size_t)G * QT_ECAP) * sizeof(double) + QT_ECAP * sizeof(uint16_t);
  static bool attr_done = false;
  if (!attr_done) {
    CUDA_OK(cudaFuncSetAttribute(quadform_tiled_kernel<CPL, G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_done = true;
  }
  quadform_tiled_kernel<CPL, G><<<T.ncta, 256, smem>>>(a, d_X, ncx, nb, part_dots, part_gram);
  qt_reduce_kernel<<<G * ncx, 256>>>(part_dots, T.ncta, G * ncx, d_dots);
  g_launch_count += 2;
  if (nb > 0) {
    const int gf = std::max(1, std::min(T.npairs, 148 * 4));
    qt_gram_finish_kernel<G><<<gf, 256>>>(T.hpairs.get(), T.pair_rb.get(), T.npairs, T.rowid.get(), d_X, ncx, nb, part_gram);
    qt_reduce_kernel<<<G * nb * nb, 256>>>(part_gram, gf, G * nb * nb, d_gram);
    g_launch_count += 2;
  }
}

template <typename T>
static std::vector<T> qt_to_host(const T* d, size_t count) {
  std::vector<T> h(count);
  if (count) CUDA_OK(cudaMemcpy(h.data(), d, count * sizeof(T), cudaMemcpyDeviceToHost));
  return h;
}

}  // namespace slmm

using namespace slmm;

extern "C" {

int slmm_matset_build_tiles(slmm_matset_t* ms, int32_t k, const int32_t* d_perm, const int32_t* d_iperm) {
  SLMM_TRY
  if (!ms || k < 0 || k >= ms->K || !d_perm || !d_iperm || !ms->m[k].data) throw std::invalid_argument("bad arguments");
  if (ms->sharded()) throw std::invalid_argument("row-block shards serve slmm_he_moments only");
  const int lead = ms->m[k].pattern;
  const CsrDev& c = ms->m[lead];
  const int n = ms->n;
  if ((int64_t)n > (1 << 28) - 1) throw std::invalid_argument("n too large for the tile keys");
  QuadTiles& T = ms->tiles[lead];
  if (T.ntiles == 0) {
    const int64_t nnz = c.nnz;
    const int nrb = (n + QT_RB - 1) / QT_RB;
    DevPtr<uint64_t> keys = dev_alloc<uint64_t>(nnz), keys_s = dev_alloc<uint64_t>(nnz);
    DevPtr<uint32_t> pos = dev_alloc<uint32_t>(nnz), pos_s = dev_alloc<uint32_t>(nnz);
    DevPtr<unsigned long long> d_cnt = dev_alloc<unsigned long long>(1);
    CUDA_OK(cudaMemset(d_cnt.get(), 0, sizeof(unsigned long long)));
    const int gw = std::max(1, std::min(148 * 8, (n + 7) / 8));
    qt_keys_kernel<<<gw, 256>>>(c.indptr, c.indices, n, d_iperm, keys.get(), pos.get(), d_cnt.get());
    unsigned long long cnt = 0;
    CUDA_OK(cudaMemcpy(&cnt, d_cnt.get(), sizeof(cnt), cudaMemcpyDeviceToHost));
    const int64_t m = (int64_t)cnt;
    if (m <= 0 || m >= (int64_t)0x7fffffff) throw std::invalid_argument("tile build: empty matrix or too many entries");
    size_t tmp_bytes = 0, tb2 = 0;
    CUDA_OK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys.get(), keys_s.get(), pos.get(), pos_s.get(), nnz, 0, 64));
    DevPtr<int32_t> head = dev_alloc<int32_t>(m), gidx = dev_alloc<int32_t>(m);
    CUDA_OK(cub::DeviceScan::InclusiveSum(nullptr, tb2, head.get(), gidx.get(), m));
    DevPtr<char> tmp = dev_alloc<char>(std::max(tmp_bytes, tb2));
    CUDA_OK(cub::DeviceRadixSort::SortPairs(tmp.get(), tmp_bytes, keys.get(), keys_s.get(), pos.get(), pos_s.get(), nnz, 0, 64));
    const int ge = (int)std::min<int64_t>((m + 255) / 256, 148 * 16);
    qt_heads_kernel<<<ge, 256>>>(keys_s.get(), m, head.get());
    CUDA_OK(cub::DeviceScan::InclusiveSum(tmp.get(), tb2, head.get(), gidx.get(), m));
    DevPtr<int64_t> d_rbstart = dev_alloc<int64_t>(nrb + 1);
    qt_rbstart_kernel<<<(nrb + 256) / 256, 256>>>(keys_s.get(), m, nrb, d_rbstart.get());
    std::vector<int64_t> rbstart = qt_to_host(d_rbstart.get(), (size_t)nrb + 1);
    head.reset();
    // distinct columns per row block -> tiles
    std::vector<int32_t> gfirst(nrb, 0), glast(nrb, 0);
    {
      // g at the first / last entry of every non-empty row block (two gathers through a small index list)
      std::vector<int64_t> want;
      for (int rb = 0; rb < nrb; rb++)
        if (rbstart[rb + 1] > rbstart[rb]) { want.push_back(rbstart[rb]); want.push_back(rbstart[rb + 1] - 1); }
      DevPtr<int64_t> d_want = dev_upload(want.data(), want.size());
      DevPtr<int32_t> d_got = dev_alloc<int32_t>(want.size());
      qt_gather_kernel<<<std::max<int>(1, (int)((want.size() + 255) / 256)), 256>>>(gidx.get(), d_want.get(), (int)want.size(), d_got.get());
      std::vector<int32_t> got = qt_to_host(d_got.get(), want.size());
      size_t q = 0;
      for (int rb = 0; rb < nrb; rb++)
        if (rbstart[rb + 1] > rbstart[rb]) { gfirst[rb] = got[q++]; glast[rb] = got[q++]; }
    }
    std::vector<int32_t> dcol_base(nrb, 0), tile_base(nrb, 0), tile_rb, tile_dc0, tile_nc;
    int64_t ndist = 0;
    for (int rb = 0; rb < nrb; rb++) {
      tile_base[rb] = (int32_t)tile_rb.size();
      if (rbstart[rb + 1] == rbstart[rb]) { dcol_base[rb] = (int32_t)ndist; continue; }
      const int D = glast[rb] - gfirst[rb] + 1;
      dcol_base[rb] = gfirst[rb] - 1;
      for (int c0 = 0; c0 < D; c0 += QT_CH) {
        tile_rb.push_back(rb);
        tile_dc0.push_back(dcol_base[rb] + c0);
        tile_nc.push_back(std::min(QT_CH, D - c0));
      }
      ndist = glast[rb];
    }
    const int ntiles = (int)tile_rb.size();
    DevPtr<int32_t> d_dcol_base = dev_upload(dcol_base.data(), dcol_base.size()), d_tile_base = dev_upload(tile_base.data(), tile_base.size());
    T.dcols = dev_alloc<int32_t>((size_t)ndist);
    uint64_t* keys2 = keys.get();                     // reuse the unsorted key buffer
    qt_keys2_kernel<<<ge, 256>>>(keys_s.get(), pos_s.get(), gidx.get(), m, d_dcol_base.get(), d_tile_base.get(), c.indices, keys2, T.dcols.get());
    gidx.reset();
    int bits = 13;
    while ((1LL << (bits - 13)) < ntiles + 1 && bits < 64) bits++;
    T.pos = dev_alloc<uint32_t>((size_t)m);
    CUDA_OK(cub::DeviceRadixSort::SortPairs(tmp.get(), tmp_bytes, keys2, keys_s.get(), pos_s.get(), T.pos.get(), m, 0, bits));
    T.tile_ptr = dev_alloc<int64_t>((size_t)ntiles + 1);
    T.rowptr = dev_alloc<uint16_t>((size_t)ntiles * (QT_RB + 1));
    const int64_t tot = (int64_t)ntiles * (QT_RB + 1) + 1;
    qt_tileptr_kernel<<<(int)std::min<int64_t>((tot + 255) / 256, 148 * 32), 256>>>(keys_s.get(), m, ntiles, T.tile_ptr.get(), T.rowptr.get());
    T.rc = dev_alloc<uint16_t>((size_t)m);
    qt_pack_kernel<<<ge, 256>>>(keys_s.get(), m, T.rc.get());
    g_launch_count += 7;
    CUDA_OK(cudaDeviceSynchronize());
    tmp.reset(); keys.reset(); keys_s.reset(); pos.reset(); pos_s.reset();
    T.tile_rb = dev_upload(tile_rb.data(), tile_rb.size());
    T.tile_dc0 = dev_upload(tile_dc0.data(), tile_dc0.size());
    T.tile_nc = dev_upload(tile_nc.data(), tile_nc.size());
    // original row ids of the permuted rows (padding rows of the last block: -1)
    std::vector<int32_t> perm = qt_to_host(d_perm, (size_t)n), rowid((size_t)nrb * QT_RB, -1);
    for (int i = 0; i < n; i++) rowid[i] = perm[i];
    T.rowid = dev_upload(rowid.data(), rowid.size());
    // static partition of the tiles over the CTAs (two resident per SM) by a cost model in units of one entry:
    // entries + 6 per non-empty row
    // + 430 per tile (staging round trips, barriers).  Entries alone left one CTA with
    // 25 646 row segments against a mean of 4 632 (the pass took as long as that CTA: 5 of the 6 ms).
    std::vector<int64_t> tptr = qt_to_host(T.tile_ptr.get(), (size_t)ntiles + 1);
    std::vector<uint16_t> rptr = qt_to_host(T.rowptr.get(), (size_t)ntiles * (QT_RB + 1));
    const int ncta = std::max(1, std::min(148 * 2, ntiles));
    std::vector<int32_t> cta_begin(ncta + 1, ntiles);
    {
      const double per_tile = 430.0, per_row = 6.0;      // least-squares fit of per-CTA cycle counts (scripts/tile_profile.py)
      std::vector<double> cost((size_t)ntiles);
      double total = 0;
      for (int t = 0; t < ntiles; t++) {
        int rows = 0;
        const uint16_t* rp = rptr.data() + (size_t)t * (QT_RB + 1);
        for (int r = 0; r < QT_RB; r++) rows += rp[r + 1] > rp[r];
        cost[t] = (double)(tptr[t + 1] - tptr[t]) + per_row * rows + per_tile;
        total += cost[t];
      }
      double acc = 0;
      int cta = 0;
      cta_begin[0] = 0;
      for (int t = 0; t < ntiles; t++) {
        acc += cost[t];
        while (cta + 1 < ncta && acc >= total * (cta + 1) / ncta) cta_begin[++cta] = t + 1;
      }
      for (int q = cta + 1; q <= ncta; q++) cta_begin[q] = ntiles;
      // row order of every tile
      std::vector<uint8_t> roword((size_t)ntiles * QT_RB, 0xFF);
      for (int t = 0; t < ntiles; t++) {
        const uint16_t* rp = rptr.data() + (size_t)t * (QT_RB + 1);
        int idx[QT_RB], cnt = 0;
        for (int r = 0; r < QT_RB; r++)
          if (rp[r + 1] > rp[r]) idx[cnt++] = r;
        std::stable_sort(idx, idx + cnt, [&](int x, int y) { return (rp[x + 1] - rp[x]) > (rp[y + 1] - rp[y]); });
        for (int p2 = 0; p2 < cnt; p2++) {
          const int slot = p2 / 8, w = (slot & 1) ? 7 - (p2 % 8) : (p2 % 8);
          roword[(size_t)t * QT_RB + slot * 8 + w] = (uint8_t)idx[p2];
        }
      }
      T.roword = dev_upload(roword.data(), roword.size());
      T.cta_stats.assign((size_t)ncta * 3, 0);
      for (int c2 = 0; c2 < ncta; c2++)
        for (int t = cta_begin[c2]; t < cta_begin[c2 + 1]; t++) {
          const uint16_t* rp = rptr.data() + (size_t)t * (QT_RB + 1);
          int rows = 0;
          for (int r = 0; r < QT_RB; r++) rows += rp[r + 1] > rp[r];
          T.cta_stats[(size_t)c2 * 3] += 1;
          T.cta_stats[(size_t)c2 * 3 + 1] += rows;
          T.cta_stats[(size_t)c2 * 3 + 2] += tptr[t + 1] - tptr[t];
        }
    }
    T.cta_begin = dev_upload(cta_begin.data(), cta_begin.size());
    T.cta_cycles = dev_alloc<long long>((size_t)ncta);
    CUDA_OK(cudaMemset(T.cta_cycles.get(), 0, (size_t)ncta * sizeof(long long)));
    // (CTA, row block) pairs: where each CTA parks the narrow-block row products of the row blocks it touches
    std::vector<int32_t> pair_base(ncta + 1, 0), pair_rb;
    for (int c2 = 0; c2 < ncta; c2++) {
      pair_base[c2] = (int32_t)pair_rb.size();
      for (int t = cta_begin[c2]; t < cta_begin[c2 + 1]; t++)
        if (t == cta_begin[c2] || tile_rb[t] != tile_rb[t - 1]) pair_rb.push_back(tile_rb[t]);
    }
    pair_base[ncta] = (int32_t)pair_rb.size();
    T.npairs = (int)pair_rb.size();
    T.pair_base = dev_upload(pair_base.data(), pair_base.size());
    T.pair_rb = dev_upload(pair_rb.data(), pair_rb.size());
    T.hpairs = dev_alloc<double>((size_t)T.npairs * QT_RB * 2 * QT_NB);
    T.ntiles = ntiles; T.nrb = nrb; T.ncta = ncta; T.nentries = m; T.ndistinct = ndist;
    CUDA_OK(cudaDeviceSynchronize());
  }
  // weighted values of matrix k in tile order
  bool have = false;
  for (int q : T.vals_of) have = have || q == k;
  if (!have) {
    DevPtr<double> v = dev_alloc<double>((size_t)T.nentries);
    qt_values_kernel<<<(int)std::min<int64_t>((T.nentries + 255) / 256, 148 * 16), 256>>>(T.rc.get(), T.pos.get(), ms->m[k].data, T.nentries, ms->m[k].nnz, v.get());
    CUDA_OK(cudaDeviceSynchronize());
    g_launch_count++;
    T.vals.push_back(std::move(v));
    T.vals_of.push_back(k);
  }
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_matset_tile_stats(const slmm_matset_t* ms, int32_t k, int64_t* out4) {
  if (!ms || k < 0 || k >= ms->K || !out4) return SLMM_ERR_INVALID;
  auto it = ms->tiles.find(ms->m[k].pattern);
  if (it == ms->tiles.end()) { out4[0] = out4[1] = out4[2] = out4[3] = 0; return SLMM_OK; }
  out4[0] = it->second.ntiles; out4[1] = it->second.nentries; out4[2] = it->second.ndistinct; out4[3] = it->second.ncta;
  return SLMM_OK;
}

int slmm_matset_tile_cta_profile(const slmm_matset_t* ms, int32_t k, int64_t* out, int32_t ncta) {
  SLMM_TRY
  if (!ms || k < 0 || k >= ms->K || !out) throw std::invalid_argument("bad arguments");
  auto it = ms->tiles.find(ms->m[k].pattern);
  if (it == ms->tiles.end() || ncta != it->second.ncta) throw std::invalid_argument("no tiles / wrong CTA count");
  const QuadTiles& T = it->second;
  CUDA_OK(cudaDeviceSynchronize());
  std::vector<long long> cyc = qt_to_host(T.cta_cycles.get(), (size_t)ncta);
  for (int c = 0; c < ncta; c++) {
    for (int q = 0; q < 3; q++) out[(size_t)c * 4 + q] = T.cta_stats[(size_t)c * 3 + q];
    out[(size_t)c * 4 + 3] = cyc[c];
  }
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_quadform_tiled(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* d_X, int32_t ncols, int32_t nb,
                        double* d_dots, double* d_gram_half) {
  SLMM_TRY
  if (!ms || !ks || !d_X || !d_dots || nk <= 0 || nk > 2 || ncols <= 0 || ncols > 160 || nb < 0 || nb > QT_NB || nb > ncols)
    throw std::invalid_argument("slmm_quadform_tiled: need 1 <= nk <= 2, ncols <= 160, nb <= 16");
  if (nb > 0 && !d_gram_half) throw std::invalid_argument("narrow block without a Gram output");
  auto it = ms->tiles.find(ms->m[ks[0]].pattern);
  if (it == ms->tiles.end() || it->second.ntiles == 0) throw std::invalid_argument("build the tiles first (slmm_matset_build_tiles)");
  QuadTiles& T = it->second;
  QtArgs a;
  a.nentries = T.nentries; a.ndistinct = T.ndistinct; a.ntiles = T.ntiles; a.nrb = T.nrb; a.n = ms->n; a.pad = 0;
  a.tile_ptr = T.tile_ptr.get(); a.tile_rb = T.tile_rb.get(); a.tile_dc0 = T.tile_dc0.get(); a.tile_nc = T.tile_nc.get();
  a.dcols = T.dcols.get(); a.rowid = T.rowid.get(); a.cta_begin = T.cta_begin.get(); a.rowptr = T.rowptr.get(); a.rc = T.rc.get();
  a.roword = T.roword.get(); a.pair_base = T.pair_base.get(); a.hpairs = T.hpairs.get(); a.cta_cycles = T.cta_cycles.get();
  for (int g = 0; g < nk; g++) {
    a.vals[g] = nullptr;
    for (size_t q = 0; q < T.vals_of.size(); q++)
      if (T.vals_of[q] == ks[g]) a.vals[g] = T.vals[q].get();
    if (!a.vals[g]) throw std::invalid_argument("matrix has no tiled values (slmm_matset_build_tiles per matrix)");
  }
  if (nk == 1) a.vals[1] = a.vals[0];
  const size_t np = (size_t)T.ncta * nk * ncols, ng = (size_t)std::max(1, std::min(T.npairs, 148 * 4)) * nk * nb * nb;
  double* part = ms->partial(np + ng);
  const int cpl = (ncols + 31) / 32;
#define QT_CASE(C)                                                                                             \
  if (nk == 1) qt_launch<C, 1>(T, a, d_X, ncols, nb, part, part + np, d_dots, d_gram_half);                      \
  else qt_launch<C, 2>(T, a, d_X, ncols, nb, part, part + np, d_dots, d_gram_half);
  if (cpl <= 1) { QT_CASE(1) } else if (cpl <= 2) { QT_CASE(2) } else if (cpl <= 3) { QT_CASE(3) }
  else if (cpl <= 4) { QT_CASE(4) } else { QT_CASE(5) }
#undef QT_CASE
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

}  // extern "C"
