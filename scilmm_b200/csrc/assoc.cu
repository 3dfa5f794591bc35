// Mixed-model association scan (GCTA --mlma / EMMAX statistic at fixed variance components): the device side of one
// block of b genotyped variants.  slmm_assoc_genotypes decodes the int8 block, centres it and projects it on
// [V^-1 C | V^-1 r] before the forward half-sweep overwrites it; slmm_assoc_colsumsq takes the column norms after the
// sweep.  The reference has no counterpart.
//
// Every column is reduced over fixed chunks of AS_CHUNK rows, in the same order whatever the block width or the
// memory order of the host matrix, so a variant's projection and norm do not depend on how the scan is blocked.
#include "common.h"

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

}  // extern "C"
