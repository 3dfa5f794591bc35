// Mixed-model association scan (GCTA --mlma / EMMAX statistic at fixed variance components): the device side of one
// block of b genotyped variants.  slmm_assoc_genotypes decodes the int8 block, centres it and projects it on
// [V^-1 C | V^-1 r] before the forward half-sweep overwrites it; slmm_assoc_colsumsq takes the column norms after the
// sweep.  The reference has no counterpart.
//
// Every column is reduced over fixed chunks of AS_CHUNK rows, in the same order whatever the block width or the
// memory order of the host matrix, so a variant's projection and norm do not depend on how the scan is blocked.
#include "common.h"

#include <algorithm>
#include <vector>

namespace slmm {

constexpr int AS_TR = 64;        // rows of one shared-memory tile
constexpr int AS_TC = 32;        // columns of a CTA (one per lane)
constexpr int AS_CHUNK = 1024;   // rows of a CTA
constexpr int AS_MAXP = 32;      // c + 1 projection rows held in registers

// Tile of AS_TR rows x AS_TC columns of the int8 block into shared memory, coalesced for either memory order: the
// thread index runs along the unit-stride dimension.  Entries outside {0, 1, 2, negative} raise *flag; rows / columns
// past the end read as missing.
__device__ __forceinline__ void as_load_tile(int8_t (*s)[AS_TC + 1], const int8_t* __restrict__ G, int64_t n, int b,
                                             int64_t rs, int64_t cs, int64_t row0, int col0, int* __restrict__ flag) {
  const bool col_fast = cs == 1;
  bool bad = false;
  for (int idx = threadIdx.x; idx < AS_TR * AS_TC; idx += blockDim.x) {
    const int r = col_fast ? idx / AS_TC : idx % AS_TR;
    const int c = col_fast ? idx % AS_TC : idx / AS_TR;
    const int64_t row = row0 + r;
    const int col = col0 + c;
    int8_t v = -1;
    if (row < n && col < b) {
      v = G[row * rs + (int64_t)col * cs];
      bad |= v > 2;
    }
    s[r][c] = v;
  }
  if (bad) *flag = 1;
}

// Pass 1: non-missing count and allele sum per column (integers: atomics are exact and order-free).
__global__ void __launch_bounds__(256) assoc_colstats_kernel(const int8_t* __restrict__ G, int64_t n, int b, int64_t rs,
                                                             int64_t cs, unsigned long long* __restrict__ nobs,
                                                             unsigned long long* __restrict__ sum,
                                                             int* __restrict__ flag) {
  __shared__ int8_t s[AS_TR][AS_TC + 1];
  __shared__ int red[2][8][AS_TC];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col0 = blockIdx.x * AS_TC;
  const int64_t r_begin = (int64_t)blockIdx.y * AS_CHUNK, r_end = min(n, r_begin + AS_CHUNK);
  int cnt = 0, acc = 0;
  for (int64_t row0 = r_begin; row0 < r_end; row0 += AS_TR) {
    as_load_tile(s, G, n, b, rs, cs, row0, col0, flag);
    __syncthreads();
    for (int r = warp; r < AS_TR; r += 8) {
      const int v = s[r][lane];
      if (v >= 0) { cnt++; acc += v; }
    }
    __syncthreads();
  }
  red[0][warp][lane] = cnt;
  red[1][warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && col0 + lane < b) {
    int tc = 0, ts = 0;
    for (int w = 0; w < 8; w++) { tc += red[0][w][lane]; ts += red[1][w][lane]; }
    atomicAdd(nobs + col0 + lane, (unsigned long long)tc);
    atomicAdd(sum + col0 + lane, (unsigned long long)ts);
  }
}

// Pass 2: x~ = g - mu (0 where missing) as a C-ordered n x b FP64 block in the original row order, and per-CTA partials
// of P' x~ for the n x np block P = [V^-1 C | V^-1 r]: part[(chunk * np + k) * b + col].  The P rows of a tile are one
// contiguous span, staged in shared memory next to the genotypes: the inner loop then reads them as broadcasts
// instead of waiting on an L2 round trip per row.  MAXP (>= np) sizes the register accumulators.
template <int MAXP>
__global__ void __launch_bounds__(256) assoc_center_project_kernel(
    const int8_t* __restrict__ G, int64_t n, int b, int64_t rs, int64_t cs, const unsigned long long* __restrict__ nobs,
    const unsigned long long* __restrict__ sum, const double* __restrict__ P, int np, double* __restrict__ X,
    double* __restrict__ part) {
  __shared__ int8_t s[AS_TR][AS_TC + 1];
  __shared__ double sp[AS_TR * MAXP];
  __shared__ double red[8][AS_TC];
  __shared__ int dummy_flag;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col0 = blockIdx.x * AS_TC, col = col0 + lane;
  const int64_t r_begin = (int64_t)blockIdx.y * AS_CHUNK, r_end = min(n, r_begin + AS_CHUNK);
  double mu = 0.0;
  if (col < b && nobs[col] > 0) mu = (double)sum[col] / (double)nobs[col];
  double acc[MAXP];
#pragma unroll
  for (int k = 0; k < MAXP; k++) acc[k] = 0.0;
  for (int64_t row0 = r_begin; row0 < r_end; row0 += AS_TR) {
    as_load_tile(s, G, n, b, rs, cs, row0, col0, &dummy_flag);     // validated by pass 1
    const int rows = r_end - row0 < AS_TR ? (int)(r_end - row0) : AS_TR;
    for (int i = threadIdx.x; i < rows * np; i += blockDim.x) sp[i] = P[row0 * np + i];
    __syncthreads();
    for (int r = warp; r < rows; r += 8) {
      const int v = s[r][lane];
      const double x = v < 0 ? 0.0 : (double)v - mu;
      if (col < b) X[(row0 + r) * b + col] = x;
      const double* p = sp + r * np;
#pragma unroll
      for (int k = 0; k < MAXP; k++)
        if (k < np) acc[k] = fma(p[k], x, acc[k]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < MAXP; k++) {
    if (k >= np) break;
    red[warp][lane] = acc[k];
    __syncthreads();
    if (warp == 0 && col < b) {
      double t = 0.0;
      for (int w = 0; w < 8; w++) t += red[w][lane];
      part[((int64_t)blockIdx.y * np + k) * b + col] = t;
    }
    __syncthreads();
  }
}

// Per-CTA partials of sum_i F[i, col]^2 over a C-ordered n x b block: part[chunk * b + col].
__global__ void __launch_bounds__(256) assoc_colsumsq_kernel(const double* __restrict__ F, int64_t n, int b,
                                                             double* __restrict__ part) {
  __shared__ double red[8][AS_TC];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col = blockIdx.x * AS_TC + lane;
  const int64_t r_begin = (int64_t)blockIdx.y * AS_CHUNK, r_end = min(n, r_begin + AS_CHUNK);
  double acc = 0.0;
  if (col < b)
    for (int64_t row = r_begin + warp; row < r_end; row += 8) {
      const double v = F[row * b + col];
      acc = fma(v, v, acc);
    }
  red[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && col < b) {
    double t = 0.0;
    for (int w = 0; w < 8; w++) t += red[w][lane];
    part[(int64_t)blockIdx.y * b + col] = t;
  }
}

// out[j] = sum over chunks of part[chunk * width + j], chunks in order.
__global__ void assoc_reduce_chunks_kernel(const double* __restrict__ part, int nchunks, int width,
                                           double* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= width) return;
  double t = 0.0;
  for (int c = 0; c < nchunks; c++) t += part[(int64_t)c * width + j];
  out[j] = t;
}

// Region Gram (region tests): the block's columns are cut into RG_S-wide strips and tile (I, J), I >= J, is the
// RG_S x RG_S product F[:, strip I]' F[:, strip J] over one chunk of RG_CHUNK rows.  Warp w owns output rows
// 8w..8w+7 of the tile and sums every row of the chunk in row order, 4 rows per DMMA, so an entry's value depends only
// on its two columns of F and not on where they sit in the block.  Diagonal tiles skip the 8 x 8 blocks above the
// diagonal; the scatter mirrors the lower triangle.
constexpr int RG_S = 64;         // strip width: a row segment of a strip is 512 contiguous bytes
constexpr int RG_CHUNK = 2048;   // rows of a CTA
constexpr int RG_KR = 32;        // rows staged in shared memory per step
constexpr int RG_LD = RG_S + 4;  // padded row: the 16 lanes of a half-warp fragment load hit distinct banks
constexpr int RG_MAXW = 512;     // widest region

// D = A B + D on the FP64 tensor pipe, m8n8k4 (as dense_tiles.cuh, which this file does not include): lane (g, t)
// holds A[g][t], B[t][g] and D[g][2t], D[g][2t + 1].
__device__ __forceinline__ void rg_dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(256) assoc_region_gram_kernel(const double* __restrict__ F, int64_t n, int b,
                                                                const int* __restrict__ tile_i,
                                                                const int* __restrict__ tile_j, int ntiles,
                                                                double* __restrict__ part) {
  __shared__ double sI[RG_KR][RG_LD];
  __shared__ double sJ[RG_KR][RG_LD];
  const int tile = blockIdx.x;
  const int ci0 = tile_i[tile] * RG_S, cj0 = tile_j[tile] * RG_S;
  const bool diag = ci0 == cj0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int64_t r_begin = (int64_t)blockIdx.y * RG_CHUNK, r_end = min(n, r_begin + RG_CHUNK);
  double (*sB)[RG_LD] = diag ? sI : sJ;
  double acc[8][2];
#pragma unroll
  for (int nj = 0; nj < 8; nj++) acc[nj][0] = acc[nj][1] = 0.0;
  const int c = threadIdx.x & (RG_S - 1);
  for (int64_t row0 = r_begin; row0 < r_end; row0 += RG_KR) {
    for (int r = threadIdx.x / RG_S; r < RG_KR; r += 256 / RG_S) {
      const int64_t row = row0 + r;
      const bool in = row < r_end;
      sI[r][c] = in && ci0 + c < b ? F[row * b + ci0 + c] : 0.0;
      if (!diag) sJ[r][c] = in && cj0 + c < b ? F[row * b + cj0 + c] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < RG_KR; k += 4) {
      const double a = sI[k + t][8 * warp + g];
#pragma unroll
      for (int nj = 0; nj < 8; nj++)
        if (!diag || nj <= warp) rg_dmma884(acc[nj][0], acc[nj][1], a, sB[k + t][8 * nj + g]);
    }
    __syncthreads();
  }
  double* out = part + ((int64_t)blockIdx.y * ntiles + tile) * (RG_S * RG_S) + (8 * warp + g) * RG_S + 2 * t;
#pragma unroll
  for (int nj = 0; nj < 8; nj++) {
    out[8 * nj] = acc[nj][0];
    out[8 * nj + 1] = acc[nj][1];
  }
}

// Region r's w x w square, packed at out_off[r], from the chunk-reduced tiles: entry (a, c) reads the lower-triangle
// entry of columns max(a, c), min(a, c), so the square is symmetric bit for bit.  Strip I's tiles are J = jmin[I]..I,
// stored from tile_base[I] on.
__global__ void assoc_region_scatter_kernel(const double* __restrict__ tiles, const int* __restrict__ bounds,
                                            const int64_t* __restrict__ out_off, const int* __restrict__ jmin,
                                            const int* __restrict__ tile_base, double* __restrict__ out) {
  const int r = blockIdx.x;
  const int c0 = bounds[r], w = bounds[r + 1] - c0;
  double* o = out + out_off[r];
  for (int e = blockIdx.y * blockDim.x + threadIdx.x; e < w * w; e += gridDim.y * blockDim.x) {
    const int a = e / w, c = e - a * w;
    const int hi = c0 + max(a, c), lo = c0 + min(a, c);
    const int I = hi / RG_S, J = lo / RG_S;
    o[e] = tiles[(int64_t)(tile_base[I] + J - jmin[I]) * (RG_S * RG_S) + (hi % RG_S) * RG_S + lo % RG_S];
  }
}

namespace {
// Grow-only work space of the scan (partials, integer column stats, error flag), kept per device across blocks.
struct AssocScratch {
  DevPtr<unsigned char> buf;
  size_t bytes = 0;
  int device = -1;
  unsigned char* get(size_t need) {
    int dev = 0;
    CUDA_OK(cudaGetDevice(&dev));
    if (dev != device || need > bytes) {
      buf.reset();
      buf = dev_alloc<unsigned char>(need);
      bytes = need;
      device = dev;
    }
    return buf.get();
  }
};
AssocScratch g_assoc_scratch;

// Pinned staging of the region plan: the copy to the device is queued behind the sweep, so the host does not wait
// for it; the next call waits on `copied` (long past by then) before it rewrites the buffer.
struct HostFree { void operator()(void* p) const noexcept { cudaFreeHost(p); } };
struct PinnedPlan {
  std::unique_ptr<unsigned char[], HostFree> buf;
  size_t bytes = 0;
  Event copied;
  unsigned char* get(size_t need) {
    if (copied) CUDA_OK(cudaEventSynchronize(copied.get()));
    if (need > bytes) {
      buf.reset();
      void* p = nullptr;
      CUDA_OK(cudaMallocHost(&p, need));
      buf.reset((unsigned char*)p);
      bytes = need;
    }
    if (!copied) copied = make_event(cudaEventDisableTiming);
    return buf.get();
  }
};
PinnedPlan g_region_plan;

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }
}  // namespace

}  // namespace slmm

using namespace slmm;

extern "C" {

int slmm_assoc_genotypes(const int8_t* d_G, int64_t n, int32_t b, int64_t row_stride, int64_t col_stride,
                         const double* d_P, int32_t np, double* d_X, double* d_proj, int64_t* d_nobs, int64_t* d_sum) {
  SLMM_TRY
  if (!d_G || !d_P || !d_X || !d_proj || !d_nobs || !d_sum || n <= 0 || b <= 0) throw std::invalid_argument("bad arguments");
  if (np <= 0 || np > AS_MAXP) throw std::invalid_argument("slmm_assoc_genotypes: need 1 <= c + 1 <= 32");
  if (!((row_stride == 1 && col_stride >= n) || (col_stride == 1 && row_stride >= b)))
    throw std::invalid_argument("slmm_assoc_genotypes: one of the strides must be 1 and the other span the block");
  const int nchunks = (int)((n + AS_CHUNK - 1) / AS_CHUNK);
  const size_t part_bytes = align256((size_t)nchunks * np * b * sizeof(double));
  unsigned char* w = g_assoc_scratch.get(part_bytes + 256);
  double* part = (double*)w;
  int* flag = (int*)(w + part_bytes);
  unsigned long long* nobs = (unsigned long long*)d_nobs;
  unsigned long long* sum = (unsigned long long*)d_sum;
  CUDA_OK(cudaMemsetAsync(flag, 0, sizeof(int), 0));
  CUDA_OK(cudaMemsetAsync(nobs, 0, (size_t)b * sizeof(int64_t), 0));
  CUDA_OK(cudaMemsetAsync(sum, 0, (size_t)b * sizeof(int64_t), 0));
  const dim3 grid((b + AS_TC - 1) / AS_TC, nchunks);
  assoc_colstats_kernel<<<grid, 256>>>(d_G, n, b, row_stride, col_stride, nobs, sum, flag);
#define AS_PROJECT(M) assoc_center_project_kernel<M><<<grid, 256>>>(d_G, n, b, row_stride, col_stride, nobs, sum, d_P, np, d_X, part)
  if (np <= 4) AS_PROJECT(4);
  else if (np <= 16) AS_PROJECT(16);
  else AS_PROJECT(32);
#undef AS_PROJECT
  assoc_reduce_chunks_kernel<<<(np * b + 255) / 256, 256>>>(part, nchunks, np * b, d_proj);
  g_launch_count += 3;
  CUDA_OK(cudaGetLastError());
  int bad = 0;
  CUDA_OK(cudaMemcpy(&bad, flag, sizeof(int), cudaMemcpyDeviceToHost));
  if (bad) throw std::invalid_argument("slmm_assoc_genotypes: genotype entries must be 0, 1, 2 or negative (missing)");
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_assoc_colsumsq(const double* d_F, int64_t n, int32_t b, double* d_out) {
  SLMM_TRY
  if (!d_F || !d_out || n <= 0 || b <= 0) throw std::invalid_argument("bad arguments");
  const int nchunks = (int)((n + AS_CHUNK - 1) / AS_CHUNK);
  double* part = (double*)g_assoc_scratch.get((size_t)nchunks * b * sizeof(double));
  const dim3 grid((b + AS_TC - 1) / AS_TC, nchunks);
  assoc_colsumsq_kernel<<<grid, 256>>>(d_F, n, b, part);
  assoc_reduce_chunks_kernel<<<(b + 255) / 256, 256>>>(part, nchunks, b, d_out);
  g_launch_count += 2;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_assoc_region_gram(const double* d_F, int64_t n, int32_t b, int32_t nregions, const int32_t* h_bounds,
                           double* d_out) {
  SLMM_TRY
  if (!d_F || !d_out || !h_bounds || n <= 0 || b <= 0 || nregions <= 0) throw std::invalid_argument("bad arguments");
  if (h_bounds[0] != 0 || h_bounds[nregions] != b)
    throw std::invalid_argument("slmm_assoc_region_gram: bounds must start at 0 and end at the block width");
  const int nstrips = (b + RG_S - 1) / RG_S;
  // strip I pairs with strips jmin[I]..I: the lowest strip of any region that reaches into strip I
  int wmax = 0;
  for (int r = 0; r < nregions; r++) {
    const int w = h_bounds[r + 1] - h_bounds[r];
    if (w <= 0 || w > RG_MAXW)
      throw std::invalid_argument("slmm_assoc_region_gram: bounds must increase, by at most 512 per region");
    wmax = std::max(wmax, w);
  }
  std::vector<int> jmin(nstrips);
  for (int s = 0; s < nstrips; s++) jmin[s] = s;
  for (int r = 0; r < nregions; r++)
    for (int s = h_bounds[r] / RG_S; s <= (h_bounds[r + 1] - 1) / RG_S; s++) jmin[s] = std::min(jmin[s], h_bounds[r] / RG_S);
  int ntiles = 0;
  for (int s = 0; s < nstrips; s++) ntiles += s - jmin[s] + 1;
  // plan: out_off[nregions] (int64), then int32 bounds[nregions + 1], tile_i[ntiles], tile_j[ntiles], jmin[nstrips],
  // tile_base[nstrips]
  const size_t plan_bytes = (size_t)nregions * 8 + ((size_t)nregions + 1 + 2 * (size_t)ntiles + 2 * (size_t)nstrips) * 4;
  unsigned char* h = g_region_plan.get(plan_bytes);
  int64_t* h_off = (int64_t*)h;
  int* h_b = (int*)(h_off + nregions);
  int *h_ti = h_b + nregions + 1, *h_tj = h_ti + ntiles, *h_jmin = h_tj + ntiles, *h_base = h_jmin + nstrips;
  int64_t off = 0;
  for (int r = 0; r < nregions; r++) {
    h_off[r] = off;
    off += (int64_t)(h_bounds[r + 1] - h_bounds[r]) * (h_bounds[r + 1] - h_bounds[r]);
  }
  std::copy(h_bounds, h_bounds + nregions + 1, h_b);
  for (int s = 0, k = 0; s < nstrips; s++) {
    h_jmin[s] = jmin[s];
    h_base[s] = k;
    for (int j = jmin[s]; j <= s; j++, k++) { h_ti[k] = s; h_tj[k] = j; }
  }
  const int nchunks = (int)((n + RG_CHUNK - 1) / RG_CHUNK);
  const size_t tile_elems = (size_t)ntiles * RG_S * RG_S;
  const size_t part_bytes = align256((size_t)nchunks * tile_elems * sizeof(double));
  const size_t tiles_bytes = align256(tile_elems * sizeof(double));
  unsigned char* w = g_assoc_scratch.get(part_bytes + tiles_bytes + plan_bytes);
  double* part = (double*)w;
  double* tiles = (double*)(w + part_bytes);
  unsigned char* d_plan = w + part_bytes + tiles_bytes;
  CUDA_OK(cudaMemcpyAsync(d_plan, h, plan_bytes, cudaMemcpyHostToDevice, 0));
  CUDA_OK(cudaEventRecord(g_region_plan.copied.get(), 0));
  const int64_t* d_off = (const int64_t*)d_plan;
  const int* d_b = (const int*)(d_off + nregions);
  const int *d_ti = d_b + nregions + 1, *d_tj = d_ti + ntiles, *d_jmin = d_tj + ntiles, *d_base = d_jmin + nstrips;
  assoc_region_gram_kernel<<<dim3(ntiles, nchunks), 256>>>(d_F, n, b, d_ti, d_tj, ntiles, part);
  const int64_t width = (int64_t)tile_elems;
  assoc_reduce_chunks_kernel<<<(unsigned)((width + 255) / 256), 256>>>(part, nchunks, (int)width, tiles);
  const int gy = std::min(64, (wmax * wmax + 255) / 256);
  assoc_region_scatter_kernel<<<dim3(nregions, gy), 256>>>(tiles, d_b, d_off, d_jmin, d_base, d_out);
  g_launch_count += 3;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

}  // extern "C"
