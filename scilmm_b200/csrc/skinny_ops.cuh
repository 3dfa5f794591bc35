// Narrow right-hand sides (nrhs <= 32): the supernode-blocked triangular solves and L*Z as HBM-STREAMING kernels.
//
// factor(b) for the c+1 fixed-effect columns, a single phenotype vector, the K and K(K+1)/2 columns of compute_hess
// (reference scilmm/SparseCholesky.py:30,32,100,149,153), the K-column forward half-sweep of AI-REML and the per-GPU
// probe slice at 4 or more GPUs all have at most 32 columns.  There every GemmOp of the solve schedules is
// C(M x N) (+/-)= A(M x K) B(N x K)^T  with M = nrhs: 2*M flops per 8 bytes of L - far below the machine balance - so
// the bound is HBM (each sweep reads L once: 8*nnz(L) bytes), not the tensor pipe.  The DMMA tile kernel wastes a
// 64-row tile on <= 32 rows, pays a producer/consumer hand-off per 16-wide K slab and reached 1.2 TB/s on the 12-column
// solve of the 250K config; these kernels stage the small A operand in shared memory, stream B from global memory
// with many independent loads and keep the accumulators in registers.  Same GemmOp descriptors, same schedules, same
// deterministic split-K reduction.
//
// Two flavours, by the memory layout of B (the factor panel or an inverse block):
//   F1  B(j,k) = B[j + k*b_sk]   consecutive OUTPUT columns j are contiguous (forward sweep, L*Z)
//   F2  B(j,k) = B[j*b_sj + k]   consecutive k are contiguous (backward sweep: L' and gathered rows)
// 5..32 right-hand sides run on the FP64 tensor pipe (the *_dmma kernels): NMT = row tiles of 8, M <= 8 NMT, NMT in
// {1, 2, 4}; rows past M are zero-padded in shared memory.
#pragma once
#include "dense_tiles.cuh"

namespace slmm {

constexpr int SK_F1_COLS = 128;    // output columns per CTA, flavour 1
constexpr int SK_F1_KC = 256;      // register-blocked F1: k chunk staged in shared memory per pass
constexpr int SK_F2_COLS = 64;     // output columns per CTA, flavour 2 (8 warps x 8 columns)
constexpr int SK_F2_KMAX = 512;    // a register-blocked F2 work item holds its whole K range of A in shared memory

// 1..4 right-hand sides, register-blocked: the MT accumulators of one output column in registers, the small operand in
// shared memory, L streamed with many independent coalesced loads per thread.
//   F1: thread <-> output column, loop over k; a warp reads 32 consecutive doubles per k.
//   F2: warp <-> output column, lanes stride k; one shuffle reduction per column.
template <int MT>
__global__ void __launch_bounds__(SK_F1_COLS) skinny_f1_kernel(const GemmOp* __restrict__ ops,
                                                               const int32_t* __restrict__ tile_op) {
  __shared__ double As[SK_F1_KC * MT];                 // [k][i]
  const int tile = blockIdx.x;
  const GemmOp& op = ops[tile_op[tile]];
  const int j = (tile - op.tile_start) * SK_F1_COLS + threadIdx.x;
  const int M = op.M, N = op.N, K = op.K, flags = op.flags;
  const bool active = j < N;
  // lower-triangular B (L11 of L*Z): B(j,k) = 0 for k > j; op.pad = first k of this (split) part
  const int kend = (flags & GF_TRIL_B) ? min(K, max(0, min(N - 1, (tile - op.tile_start) * SK_F1_COLS + SK_F1_COLS - 1) + 1 - op.pad)) : K;
  const int kmine = (flags & GF_TRIL_B) ? min(K, max(0, j + 1 - op.pad)) : K;
  const double* __restrict__ Bj = op.B + j;
  const int64_t b_sk = op.b_sk;
  double acc[MT];
#pragma unroll
  for (int i = 0; i < MT; i++) acc[i] = 0.0;
  for (int k0 = 0; k0 < kend; k0 += SK_F1_KC) {
    const int kc = min(SK_F1_KC, kend - k0);
    __syncthreads();
    {
      // stage A(0..M, k0..k0+kc) as [k][MT]: coalesced along the M values of one k (contiguous in the RHS block), four
      // independent loads in flight per thread (a load-store loop per element cost ~1 us of latency per trip)
      const int total = kc * M;
      const double* __restrict__ Ab = op.A + (int64_t)k0 * op.a_sk;
      const int64_t a_sk = op.a_sk;
      for (int q0 = threadIdx.x; q0 < total; q0 += 4 * SK_F1_COLS) {
        double v[4];
        int dst[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int q = q0 + u * SK_F1_COLS;
          const int k = q / M, i = q - k * M;
          dst[u] = q < total ? k * MT + i : -1;
          v[u] = q < total ? Ab[(int64_t)k * a_sk + i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (dst[u] >= 0) As[dst[u]] = v[u];
      }
      if (M < MT)
        for (int q = threadIdx.x; q < kc * (MT - M); q += SK_F1_COLS) As[(q / (MT - M)) * MT + M + q % (MT - M)] = 0.0;
    }
    __syncthreads();
    if (!active) continue;
    const int kl = min(kc, kmine - k0);
    int k = 0;
    for (; k + 16 <= kl; k += 16) {                    // 16 independent loads in flight per thread: the kernel is bound
      double b[16];                                    // by rounds x memory latency, not by issue
#pragma unroll
      for (int u = 0; u < 16; u++) b[u] = __ldcs(Bj + (int64_t)(k0 + k + u) * b_sk);
#pragma unroll
      for (int u = 0; u < 16; u++)
#pragma unroll
        for (int i = 0; i < MT; i++) acc[i] += As[(k + u) * MT + i] * b[u];
    }
    for (; k + 4 <= kl; k += 4) {
      double b[4];
#pragma unroll
      for (int u = 0; u < 4; u++) b[u] = __ldcs(Bj + (int64_t)(k0 + k + u) * b_sk);
#pragma unroll
      for (int u = 0; u < 4; u++)
#pragma unroll
        for (int i = 0; i < MT; i++) acc[i] += As[(k + u) * MT + i] * b[u];
    }
    for (; k < kl; k++) {
      const double b = __ldcs(Bj + (int64_t)(k0 + k) * b_sk);
#pragma unroll
      for (int i = 0; i < MT; i++) acc[i] += As[k * MT + i] * b;
    }
  }
  if (!active) return;
  double* c = op.C + (int64_t)j * op.c_sj;
  const bool accum = flags & GF_ACCUM, neg = flags & GF_NEG;
#pragma unroll
  for (int i = 0; i < MT; i++)
    if (i < M) {
      const double v = neg ? -acc[i] : acc[i];
      c[i] = accum ? c[i] + v : v;
    }
}

template <int MT>
__global__ void __launch_bounds__(256, 2) skinny_f2_kernel(const GemmOp* __restrict__ ops,
                                                        const int32_t* __restrict__ tile_op) {
  extern __shared__ double As2[];                      // [i][K] (lanes read consecutive k: conflict free)
  const int tile = blockIdx.x;
  const GemmOp& op = ops[tile_op[tile]];
  const int j0 = (tile - op.tile_start) * SK_F2_COLS;
  const int M = op.M, N = op.N, K = op.K, flags = op.flags;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int32_t* __restrict__ kidx = op.a_kidx;
  {
    // stage A(0..M, 0..K) as [i][K] (lanes of the main loop read consecutive k): source walked with i fastest (the M
    // values of one gathered row are contiguous), four independent loads in flight per thread
    const int total = K * M;
    const int64_t a_sk = op.a_sk;
    for (int q0 = threadIdx.x; q0 < total; q0 += 4 * 256) {
      double v[4];
      int dst[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int q = q0 + u * 256;
        const int k = q / M, i = q - k * M;
        dst[u] = q < total ? i * K + k : -1;
        v[u] = q < total ? op.A[(int64_t)i + (int64_t)(kidx ? kidx[k] : k) * a_sk] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (dst[u] >= 0) As2[dst[u]] = v[u];
    }
    for (int q = threadIdx.x + M * K; q < MT * K; q += 256) As2[q] = 0.0;
  }
  __syncthreads();
  const bool accum = flags & GF_ACCUM, neg = flags & GF_NEG;
  // each warp owns columns warp, warp + 8, ...; two columns per trip with 4 + 4 independent coalesced loads in flight
  for (int jj = warp; jj < SK_F2_COLS; jj += 16) {
    const int j0c = j0 + jj, j1c = j0 + jj + 8;
    if (j0c >= N) break;
    const bool two = j1c < N && jj + 8 < SK_F2_COLS;
    const double* __restrict__ B0 = op.B + (int64_t)j0c * op.b_sj;
    const double* __restrict__ B1 = op.B + (int64_t)(two ? j1c : j0c) * op.b_sj;
    double acc0[MT], acc1[MT];
#pragma unroll
    for (int i = 0; i < MT; i++) acc0[i] = acc1[i] = 0.0;
    int k = lane;
    for (; k + 96 < K; k += 128) {
      double b0[4], b1[4];
#pragma unroll
      for (int u = 0; u < 4; u++) { b0[u] = __ldcs(B0 + k + 32 * u); b1[u] = __ldcs(B1 + k + 32 * u); }
#pragma unroll
      for (int u = 0; u < 4; u++)
#pragma unroll
        for (int i = 0; i < MT; i++) {
          const double a = As2[i * K + k + 32 * u];
          acc0[i] += a * b0[u];
          acc1[i] += a * b1[u];
        }
    }
    for (; k < K; k += 32) {
      const double b0 = __ldcs(B0 + k), b1 = __ldcs(B1 + k);
#pragma unroll
      for (int i = 0; i < MT; i++) {
        const double a = As2[i * K + k];
        acc0[i] += a * b0;
        acc1[i] += a * b1;
      }
    }
    // reduce the accumulators over the warp; lane i ends up with row i
    double m0 = 0.0, m1 = 0.0;
#pragma unroll
    for (int i = 0; i < MT; i++) {
      double v0 = acc0[i], v1 = acc1[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        v0 += __shfl_xor_sync(0xffffffffu, v0, o);
        v1 += __shfl_xor_sync(0xffffffffu, v1, o);
      }
      if (lane == i) { m0 = v0; m1 = v1; }
    }
    if (lane < M) {
      double* c0 = op.C + lane + (int64_t)j0c * op.c_sj;
      const double v0 = neg ? -m0 : m0;
      *c0 = accum ? *c0 + v0 : v0;
      if (two) {
        double* c1 = op.C + lane + (int64_t)j1c * op.c_sj;
        const double v1 = neg ? -m1 : m1;
        *c1 = accum ? *c1 + v1 : v1;
      }
    }
  }
}

template <int NMT> struct SkDmma {
  // k chunk of the staged operand: the copy of A (8 NMT rows) must leave room for 2-3 resident CTAs per SM
  static constexpr int KC = NMT <= 2 ? 512 : 256;    // F2
  static constexpr int KP = KC + 4;                  // leading dimension = 4 mod 16: conflict-free fragment reads
  static constexpr int SMEM = 8 * NMT * KP * (int)sizeof(double);
  static constexpr int F1_KC = 256, F1_KP = F1_KC + 4;
  static constexpr int F1_SMEM = 8 * NMT * F1_KP * (int)sizeof(double);
  static constexpr int OCC = NMT <= 2 ? 3 : 2;
};

// Backward-sweep flavour on the tensor pipe (A staged chunk by chunk along K, so unlike skinny_f2_kernel K is not
// limited): a warp owns 8 output columns, its B fragment b[k = t][n = g] = B(j0 + g, kk + t) comes
// STRAIGHT from global memory (each lane 8 bytes, a quad 32 contiguous bytes of one column of L: whole sectors, 256
// bytes per warp load like a coalesced load), the A fragments from shared memory (leading dimension = 4 mod 16:
// conflict free).  The register-blocked kernel would read 12..16 shared-memory values per pair of streamed values at
// these widths and be bound by that; here it is 2 per streamed value.
template <int NMT>
__global__ void __launch_bounds__(256, SkDmma<NMT>::OCC) skinny_f2_dmma_kernel(const GemmOp* __restrict__ ops,
                                                                              const int32_t* __restrict__ tile_op) {
  constexpr int KC = SkDmma<NMT>::KC, KP = SkDmma<NMT>::KP;
  extern __shared__ double Ad[];                       // [8 * NMT][KP], zero beyond (M, chunk)
  const int tile = blockIdx.x;
  const GemmOp& op = ops[tile_op[tile]];
  const int j0 = (tile - op.tile_start) * SK_F2_COLS;
  const int M = op.M, N = op.N, K = op.K, flags = op.flags;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int32_t* __restrict__ kidx = op.a_kidx;
  const int jb = j0 + 8 * warp;                        // this warp's 8 output columns
  const bool wactive = jb < N;
  const int jg = min(jb + g, N - 1);                   // clamped: columns past N are computed and dropped
  const double* __restrict__ Bg = op.B + (int64_t)jg * op.b_sj + t;
  const double* a0 = Ad + g * KP + t;
  double d[NMT][2];
#pragma unroll
  for (int m = 0; m < NMT; m++) d[m][0] = d[m][1] = 0.0;
  for (int k0 = 0; k0 < K; k0 += KC) {
    const int kc = min(KC, K - k0), kc4 = (kc + 3) & ~3;
    __syncthreads();
    {
      const int64_t a_sk = op.a_sk;
      const int total = kc * M;
      for (int q0 = threadIdx.x; q0 < total; q0 += 4 * 256) {
        double v[4];
        int dst[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int q = q0 + u * 256;
          const int k = q / M, i = q - k * M;
          dst[u] = q < total ? i * KP + k : -1;
          v[u] = q < total ? op.A[(int64_t)i + (int64_t)(kidx ? kidx[k0 + k] : k0 + k) * a_sk] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (dst[u] >= 0) Ad[dst[u]] = v[u];
      }
      // zero padding: rows M..8*NMT over [0, kc4) and the k tail [kc, kc4) of the live rows
      for (int q = threadIdx.x; q < (8 * NMT - M) * kc4; q += 256) Ad[(M + q / kc4) * KP + q % kc4] = 0.0;
      if (kc4 > kc)
        for (int q = threadIdx.x; q < M * (kc4 - kc); q += 256) Ad[(q / (kc4 - kc)) * KP + kc + q % (kc4 - kc)] = 0.0;
    }
    __syncthreads();
    if (!wactive) continue;
    const double* __restrict__ Bk = Bg + k0;
    int kk = 0;
    for (; kk + 32 <= kc; kk += 32) {                  // 8 independent 8-byte loads in flight per lane
      double b[8];
#pragma unroll
      for (int u = 0; u < 8; u++) b[u] = __ldcs(Bk + kk + 4 * u);
#pragma unroll
      for (int u = 0; u < 8; u++)
#pragma unroll
        for (int m = 0; m < NMT; m++) dmma884(d[m][0], d[m][1], a0[m * 8 * KP + kk + 4 * u], b[u]);
    }
    for (; kk < kc4; kk += 4) {
      const double b = (kk + t < kc) ? __ldcs(Bk + kk) : 0.0;
#pragma unroll
      for (int m = 0; m < NMT; m++) dmma884(d[m][0], d[m][1], a0[m * 8 * KP + kk], b);
    }
  }
  if (!wactive) return;
  const bool accum = flags & GF_ACCUM, neg = flags & GF_NEG;
#pragma unroll
  for (int m = 0; m < NMT; m++) {
    const int i = 8 * m + g;
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int j = jb + 2 * t + h;
      if (i < M && j < N) {
        double* c = op.C + (int64_t)i * op.c_si + (int64_t)j * op.c_sj;
        const double v = neg ? -d[m][h] : d[m][h];
        *c = accum ? *c + v : v;
      }
    }
  }
}

// Forward flavour: a warp owns 16 output columns (two 8-column DMMA tiles); its B fragment b[k = t][n = g] =
// B(jb + g, kk + t) comes straight from global memory - for a fixed k the 8 lanes of a g-group read 64 contiguous
// bytes, the 8 warps of a CTA 1 KB of that k-row.  A(M x K) is staged in K chunks of F1_KC as [i][F1_KP]
// (leading dimension = 4 mod 16: conflict-free fragment reads).

template <int NMT>
__global__ void __launch_bounds__(256, SkDmma<NMT>::OCC) skinny_f1_dmma_kernel(const GemmOp* __restrict__ ops,
                                                                              const int32_t* __restrict__ tile_op) {
  constexpr int SK_F1D_KC = SkDmma<NMT>::F1_KC, SK_F1D_KCP = SkDmma<NMT>::F1_KP;
  extern __shared__ double As[];                       // [8 * NMT][SK_F1D_KCP]
  const int tile = blockIdx.x;
  const GemmOp& op = ops[tile_op[tile]];
  const int jt0 = (tile - op.tile_start) * SK_F1_COLS;
  const int M = op.M, N = op.N, K = op.K, flags = op.flags;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const bool tril = flags & GF_TRIL_B;
  // lower-triangular B (L11 of L*Z): B(j,k) = 0 for k > j; op.pad = first k of this (split) part
  const int kend = tril ? min(K, max(0, min(N - 1, jt0 + SK_F1_COLS - 1) + 1 - op.pad)) : K;
  const int jb = jt0 + 16 * warp;
  const bool wactive = jb < N;
  const int jc0 = min(jb + g, N - 1), jc1 = min(jb + 8 + g, N - 1);      // clamped: columns past N are dropped
  const int64_t b_sk = op.b_sk;
  const double* __restrict__ B0 = op.B + jc0 + (int64_t)t * b_sk;
  const double* __restrict__ B1 = op.B + jc1 + (int64_t)t * b_sk;
  const int kw = tril ? min(kend, max(0, min(N - 1, jb + 15) + 1 - op.pad)) : kend;     // this warp's own k bound
  const int lim0 = tril ? jc0 - op.pad : K, lim1 = tril ? jc1 - op.pad : K;              // entries with k > lim are zero
  double d[NMT][2][2];
#pragma unroll
  for (int m = 0; m < NMT; m++) d[m][0][0] = d[m][0][1] = d[m][1][0] = d[m][1][1] = 0.0;
  const double* a0 = As + g * SK_F1D_KCP + t;
  for (int k0 = 0; k0 < kend; k0 += SK_F1D_KC) {
    const int kc = min(SK_F1D_KC, kend - k0), kc4 = (kc + 3) & ~3;
    __syncthreads();
    {
      const int total = kc * M;
      const double* __restrict__ Ab = op.A + (int64_t)k0 * op.a_sk;
      const int64_t a_sk = op.a_sk;
      for (int q0 = threadIdx.x; q0 < total; q0 += 4 * 256) {
        double v[4];
        int dst[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int q = q0 + u * 256;
          const int k = q / M, i = q - k * M;
          dst[u] = q < total ? i * SK_F1D_KCP + k : -1;
          v[u] = q < total ? Ab[(int64_t)k * a_sk + i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
          if (dst[u] >= 0) As[dst[u]] = v[u];
      }
      for (int q = threadIdx.x; q < (8 * NMT - M) * kc4; q += 256) As[(M + q / kc4) * SK_F1D_KCP + q % kc4] = 0.0;
      if (kc4 > kc)
        for (int q = threadIdx.x; q < M * (kc4 - kc); q += 256) As[(q / (kc4 - kc)) * SK_F1D_KCP + kc + q % (kc4 - kc)] = 0.0;
    }
    __syncthreads();
    if (!wactive) continue;
    const int kl = min(kc, kw - k0);                   // k range of this chunk this warp needs
    int kk = 0;
    for (; kk + 16 <= kl; kk += 16) {                  // 4 k-steps x 2 column tiles: 8 independent loads per lane
      double b0[4], b1[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int kg = k0 + kk + 4 * u + t;
        b0[u] = kg <= lim0 ? __ldcs(B0 + (int64_t)(k0 + kk + 4 * u) * b_sk) : 0.0;
        b1[u] = kg <= lim1 ? __ldcs(B1 + (int64_t)(k0 + kk + 4 * u) * b_sk) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 4; u++)
#pragma unroll
        for (int m = 0; m < NMT; m++) {
          const double a = a0[m * 8 * SK_F1D_KCP + kk + 4 * u];
          dmma884(d[m][0][0], d[m][0][1], a, b0[u]);
          dmma884(d[m][1][0], d[m][1][1], a, b1[u]);
        }
    }
    for (; kk < kl; kk += 4) {
      const int kg = k0 + kk + t;
      const bool in = kk + t < kc;
      const double b0 = (in && kg <= lim0) ? __ldcs(B0 + (int64_t)(k0 + kk) * b_sk) : 0.0;
      const double b1 = (in && kg <= lim1) ? __ldcs(B1 + (int64_t)(k0 + kk) * b_sk) : 0.0;
#pragma unroll
      for (int m = 0; m < NMT; m++) {
        const double a = a0[m * 8 * SK_F1D_KCP + kk];
        dmma884(d[m][0][0], d[m][0][1], a, b0);
        dmma884(d[m][1][0], d[m][1][1], a, b1);
      }
    }
  }
  if (!wactive) return;
  const bool accum = flags & GF_ACCUM, neg = flags & GF_NEG;
#pragma unroll
  for (int m = 0; m < NMT; m++) {
    const int i = 8 * m + g;
#pragma unroll
    for (int nt = 0; nt < 2; nt++)
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int j = jb + 8 * nt + 2 * t + h;
        if (i < M && j < N) {
          double* c = op.C + (int64_t)i * op.c_si + (int64_t)j * op.c_sj;
          const double v = neg ? -d[m][nt][h] : d[m][nt][h];
          *c = accum ? *c + v : v;
        }
      }
  }
}

}  // namespace slmm
