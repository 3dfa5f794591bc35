// Numeric supernodal LL' factorization, logdet, multi-RHS solves and L*Z on the device.
// Host code here only builds launch schedules (once per pattern / per RHS width) and walks them.
//
// Data layout in HBM
//   panels   : for supernode s the ms x ns column-major trapezoid (ld = ms rounded up to even, symbolic.h panel_ld)
//              at sn_lptr[s]; strict upper part of
//              the diagonal block stays zero.
//   inverses : one 64 x 64 column-major slot per diagonal block (TRSM and the triangular solves become GEMMs).
//   arena[2] : update (Schur complement) matrices rs x rs, ping-pong by depth parity, so a child's update lives
//              exactly until its parent's level has pulled it (parent-pull extend-add: atomics-free, fixed order).
//   RHS      : permuted n x nrhs row-major block + per-level contribution blocks rs x nrhs (same ping-pong).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <vector>

#include "common.h"
#include "dense_tiles.cuh"
#include "dense_tiles_tma.cuh"
#include "potrf_block.cuh"
#include "skinny_ops.cuh"
#include "symbolic.h"

namespace slmm {

static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }
const std::string& last_error() { return g_last_error; }
int64_t g_launch_count = 0;

constexpr int NBO = 1024;    // outer block: columns updated together with K = NBO

// One pull work item: target columns (rows, for RHS blocks) [c0,c1) of parent front p, and the range [e0,e1) of
// PullEntry records listing exactly the children that contribute to it (a parent can have > 1000 children, most
// of them touching only a few targets: walking all children per item was the dominant cost of the pulls).
struct PullItem { int32_t p, c0, c1, e0, e1; };
// rows [ta,tb) of the child's below-diagonal row list map into the item's target range
struct PullEntry { int64_t rel_off, src_off; int32_t rsc, ta, tb, pad; };

struct DevSym {
  const int32_t *sn_first, *sn_nrow, *rows, *rel, *child_ptr, *child_idx;
  const int64_t *sn_rowptr, *sn_lptr, *sn_uptr;
};

// ---------------------------------------------------------------------------------------------------------
// small kernels
__global__ void scatter_axpy_kernel(const int64_t* __restrict__ map, const double* __restrict__ vals, double sigma,
                                    double* __restrict__ Lx, int64_t nnz) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; e < nnz; e += stride) {
    const int64_t tgt = map[e];
    if (tgt >= 0) Lx[tgt] = __dadd_rn(Lx[tgt], __dmul_rn(sigma, vals[e]));   // no FMA: scipy rounds twice
  }
}

// two matrices that share one sparsity pattern (IBD and its Hadamard square) in one pass: the scatter map and the
// targets are read / read-modify-written once; the rounding sequence is the one of two consecutive passes
__global__ void scatter_axpy2_kernel(const int64_t* __restrict__ map, const double* __restrict__ v0, double s0,
                                     const double* __restrict__ v1, double s1, double* __restrict__ Lx, int64_t nnz) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; e < nnz; e += stride) {
    const int64_t tgt = map[e];
    if (tgt >= 0) Lx[tgt] = __dadd_rn(__dadd_rn(Lx[tgt], __dmul_rn(s0, v0[e])), __dmul_rn(s1, v1[e]));
  }
}

__device__ __forceinline__ int lower_bound_dev(const int32_t* a, int n, int v) {
  int lo = 0, hi = n;
  while (lo < hi) { int mid = (lo + hi) >> 1; if (a[mid] < v) lo = mid + 1; else hi = mid; }
  return lo;
}

// Parent-pull extend-add of the children's update matrices.  One group of TPI threads (a warp for small parents,
// a whole CTA for large ones) owns target columns [c0,c1) of one parent front and walks the children in fixed
// order, so no two groups ever write the same entry (atomics-free, deterministic).  Rows are processed four at a
// time per thread with all loads issued before the stores: rel[] is strictly increasing, so the four targets are
// distinct and the read-modify-write chains are independent.
template <int TPI>
__global__ void __launch_bounds__(TPI < 128 ? 128 : TPI) extend_add_kernel(const PullItem* __restrict__ items, int nitems,
                                                                         const PullEntry* __restrict__ entries,
                                                                         DevSym S, double* __restrict__ Lx,
                                                                         const double* __restrict__ arena_child,
                                                                         double* __restrict__ arena_parent) {
  constexpr int GROUPS = (TPI < 128 ? 128 : TPI) / TPI;
  const int w = blockIdx.x * GROUPS + threadIdx.x / TPI, lane = threadIdx.x % TPI;
  if (w >= nitems) return;
  const PullItem it = items[w];
  const int p = it.p;
  const int nsp = S.sn_first[p + 1] - S.sn_first[p], msp = S.sn_nrow[p], rsp = msp - nsp;
  double* panel = Lx + S.sn_lptr[p];
  double* Up = arena_parent + S.sn_uptr[p];
  for (int q = it.e0; q < it.e1; q++) {
    const PullEntry en = entries[q];
    const int rsc = en.rsc;
    const int32_t* __restrict__ relc = S.rel + en.rel_off;
    const double* Uc = arena_child + en.src_off;
    for (int tt = en.ta; tt < en.tb; tt++) {
      const int pc = relc[tt];
      const double* __restrict__ src = Uc + (int64_t)tt * rsc;
      double* dst = pc < nsp ? panel + (int64_t)pc * ((msp + 1) & ~1) : Up + (int64_t)(pc - nsp) * rsp - nsp;
      int u = tt + lane;
      for (; u + 3 * TPI < rsc; u += 4 * TPI) {
        const int r0 = relc[u], r1 = relc[u + TPI], r2 = relc[u + 2 * TPI], r3 = relc[u + 3 * TPI];
        const double v0 = src[u], v1 = src[u + TPI], v2 = src[u + 2 * TPI], v3 = src[u + 3 * TPI];
        const double d0 = dst[r0], d1 = dst[r1], d2 = dst[r2], d3 = dst[r3];
        dst[r0] = d0 + v0; dst[r1] = d1 + v1; dst[r2] = d2 + v2; dst[r3] = d3 + v3;
      }
      for (; u < rsc; u += TPI) dst[relc[u]] += src[u];
    }
    // Two children can hit the same parent entry, and the thread that owns an entry differs from child to child:
    // the group must finish one child's read-modify-writes before any of its threads starts the next child.
    if (TPI >= 128) __syncthreads(); else __syncwarp();
  }
}

// Same pull for RHS blocks: target rows [c0,c1) of the parent front; rows < ns land in the permuted solution
// block, the others in the parent's contribution block.  `sign` lets L*Z reuse it.
__global__ void vec_pull_kernel(const PullItem* __restrict__ items, int nitems, const PullEntry* __restrict__ entries,
                                DevSym S, double* __restrict__ X, const double* __restrict__ arena_child,
                                double* __restrict__ arena_parent, const int64_t* __restrict__ vptr, int nrhs) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= nitems) return;
  const PullItem it = items[w];
  const int p = it.p;
  const int fp = S.sn_first[p], nsp = S.sn_first[p + 1] - fp;
  double* Vp = arena_parent + vptr[p];
  for (int q = it.e0; q < it.e1; q++) {
    const PullEntry en = entries[q];
    const int32_t* relc = S.rel + en.rel_off;
    const double* Vc = arena_child + en.src_off;
    for (int tt = en.ta; tt < en.tb; tt++) {
      const int pr = relc[tt];
      const double* src = Vc + (int64_t)tt * nrhs;
      double* dst = pr < nsp ? X + (int64_t)(fp + pr) * nrhs : Vp + (int64_t)(pr - nsp) * nrhs;
      for (int j = lane; j < nrhs; j += 32) dst[j] += src[j];
    }
  }
}

__global__ void gather_rows_kernel(const double* __restrict__ src, double* __restrict__ dst,
                                   const int32_t* __restrict__ perm, int n, int nrhs, int scatter) {
  // gather: dst[i,:] = src[perm[i],:]   scatter: dst[perm[i],:] = src[i,:]
  const int64_t total = (int64_t)n * nrhs;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(q / nrhs), j = (int)(q % nrhs);
    const int64_t o = (int64_t)perm[i] * nrhs + j;
    if (scatter) dst[o] = src[q]; else dst[q] = src[o];
  }
}

// Scatter map of one input pattern into the panel storage, built ON THE DEVICE from the device-resident CSR arrays
// (the host version walks 10^8 entries with a binary search each and then uploads 8 bytes per entry).  Warp per row.
// tri: see symbolic.cpp entry_map.  *bad is set when an entry falls outside the analysed pattern.
__global__ void __launch_bounds__(256) entry_map_kernel(const int32_t* __restrict__ ap, const int32_t* __restrict__ ai,
                                                        int n, const int32_t* __restrict__ iperm,
                                                        const int32_t* __restrict__ col2sn, DevSym S, int tri,
                                                        int64_t* __restrict__ target, int* __restrict__ bad) {
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
    const int pr = iperm[r];
    const int b = ap[r], e = ap[r + 1];
    for (int p = b + lane; p < e; p += 32) {
      const int c = ai[p];
      const int pc = iperm[c];
      int ir = pr, ic = pc;
      int64_t out = -1;
      bool take = true;
      if (tri == 0) take = ic <= ir;
      else {
        take = !((tri > 0 && c < r) || (tri < 0 && c > r));
        if (ic > ir) { ir = pc; ic = pr; }
      }
      if (take) {
        const int s = col2sn[ic];
        const int ms = S.sn_nrow[s];
        const int32_t* rows = S.rows + S.sn_rowptr[s];
        const int pos = lower_bound_dev(rows, ms, ir);
        if (pos < ms && rows[pos] == ir) out = S.sn_lptr[s] + (int64_t)(ic - S.sn_first[s]) * ((ms + 1) & ~1) + pos;
        else *bad = 1;
      }
      target[p] = out;
    }
  }
}

// Hutchinson probe block Z ~ N(0,1) (np.random.randn(n, sim_num), reference scilmm/SparseCholesky.py:50) drawn on
// the device from a COUNTER-BASED stream: element (row i, global column c) of evaluation `stream` is a pure function
// of (seed, stream, i, c) - Philox4x32-10 keyed by the seed, counter (i, c, stream) - so a rank that owns columns
// [col_begin, col_begin + ncols) draws exactly the values the single-GPU run draws for them: results do not depend
// on the number of GPUs, and only the local columns are ever generated.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__global__ void __launch_bounds__(256) probe_normals_kernel(double* __restrict__ out, int64_t n, int ncols, int col_begin,
                                                            uint64_t seed, uint64_t stream) {
  const int64_t total = n * ncols;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = q / ncols;
    const int c = (int)(q - i * ncols) + col_begin;
    uint32_t x[4];
    philox4x32_10((uint32_t)i, (uint32_t)c, (uint32_t)stream, (uint32_t)(stream >> 32) ^ (uint32_t)(i >> 32),
                  (uint32_t)seed, (uint32_t)(seed >> 32), x);
    const uint64_t a = (((uint64_t)x[0] << 32) | x[1]) >> 11, b = (((uint64_t)x[2] << 32) | x[3]) >> 11;
    const double u1 = ((double)a + 0.5) * 0x1.0p-53, u2 = ((double)b + 0.5) * 0x1.0p-53;    // both in (0, 1)
    out[q] = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);                                       // Box-Muller
  }
}

struct WBlock { int64_t off; int32_t n, pad; };

// identity into every wide (outer-block) inverse slot, before the batched triangular inversion
__global__ void init_identity_kernel(const WBlock* __restrict__ blocks, double* __restrict__ W) {
  const WBlock b = blocks[blockIdx.x];
  double* w = W + b.off;
  const int64_t total = (int64_t)b.n * b.n;
  for (int64_t q = threadIdx.x; q < total; q += blockDim.x) w[q] = (q % b.n == q / b.n) ? 1.0 : 0.0;
}

__global__ void logdet_kernel(const double* __restrict__ Lx, const int32_t* __restrict__ col2sn,
                              const int32_t* __restrict__ sn_first, const int32_t* __restrict__ sn_nrow,
                              const int64_t* __restrict__ sn_lptr, int n, double* __restrict__ partial) {
  __shared__ double sh[256];
  double acc = 0.0;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const int s = col2sn[j], c = j - sn_first[s];
    acc += log(Lx[sn_lptr[s] + (int64_t)c * ((sn_nrow[s] + 1) & ~1) + c]);
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}

// ---------------------------------------------------------------------------------------------------------
struct Launch {
  // EV_RECORD / EV_WAIT carry no kernel: the launch's stream records / waits for event event()
  enum Kind { POTRF, GEMM_BIG, GEMM_SMALL, PULL_MAT, PULL_VEC, PULL_MAT_BIG, INIT_W, REDUCE, EV_RECORD, EV_WAIT,
              SKINNY_F1, SKINNY_F2 /* narrow-RHS streaming kernels */,
              GEMM_TMA /* 128 x 128 DMMA tiles with TMA-staged operands (dense_tiles_tma.cuh); aux_off = first tensor map */ } kind;
  int64_t off;      // offset into the matching op array
  int32_t count;    // ops / items; the event id of EV_RECORD / EV_WAIT
  int32_t grid;     // CTAs
  int32_t variant;  // PULL_*: parity of the children's arena;  SKINNY_*: row template MT
  double flops;     // dense flops issued by this launch (0 for pulls)
  int64_t tile_off; // GEMM launches: offset of this launch's tile -> op table
  int32_t stream;   // 0: main (high priority) stream   1: bulk stream (look-ahead trailing updates)
  int64_t aux_off = 0;
  int event() const { return count; }
  int child_parity() const { return variant; }
  int row_mt() const { return variant; }
};

// work size the profiles report per launch: tiles / blocks of the GEMM-type kernels, ops / items of the others
static int32_t work_size(const Launch& L) {
  return (L.kind <= Launch::GEMM_SMALL || L.kind >= Launch::SKINNY_F1) ? L.grid : L.count;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda: it must load
// on machines without a driver for the host-only analysis).  2-D FP64 tensor: dim 0 = rows (contiguous), dim 1 = k
// with a stride of `ld` elements; boxes of 16 x 16 elements, 128-byte swizzle.
static CUtensorMap encode_tmap(const double* base, uint64_t rows, uint64_t cols, uint64_t ld) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (!p || q != cudaDriverEntryPointSuccess) throw std::runtime_error("cuTensorMapEncodeTiled is not available");
    fn = (EncodeFn)p;
  }
  CUtensorMap m;
  const cuuint64_t gdim[2] = {rows, cols};
  const cuuint64_t gstride[1] = {ld * sizeof(double)};
  const cuuint32_t box[2] = {16, (cuuint32_t)TMA_KS};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult rc = fn(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled failed (" + std::to_string((int)rc) + ")");
  return m;
}

constexpr int BIG_STAGES = 4, SMALL_STAGES = 4;
constexpr int BIG_SMEM = BIG_STAGES * 16 * (128 + 4) * 2 * 8 + 2 * BIG_STAGES * 8;
constexpr int SMALL_SMEM = SMALL_STAGES * 16 * (64 + 4) * 2 * 8 + 2 * SMALL_STAGES * 8;
constexpr int BIG_THREADS = 32 * (2 * 4 + NPW), SMALL_THREADS = 32 * (2 * 2 + NPW);

struct Schedule {
  std::vector<Launch> launches;
  std::vector<GemmOp> gemm;
  std::vector<PotrfOp> potrf;
  std::vector<PullItem> pull;
  std::vector<PullEntry> pull_entries;
  DevPtr<PullEntry> d_pull_entries;
  std::vector<ReduceOp> reduce;
  std::vector<CUtensorMap> tmaps; // two per GEMM_TMA op (A, B), in op order
  DevPtr<CUtensorMap> d_tmaps;
  std::vector<int32_t> tile_op;   // per GEMM launch: op index (relative to the launch's first op) of every tile
  DevPtr<int32_t> d_tile_op;
  int nevents = 0;                // events used by EV_RECORD / EV_WAIT
  int64_t ws_size = 0;            // doubles of split-K workspace (max over phases)
  int64_t ws2_size = 0;           // second workspace: split-K of bulk-stream ops running beside the chain's
  DevPtr<double> d_ws;
  DevPtr<double> d_ws2;
  DevPtr<ReduceOp> d_reduce;
  DevPtr<GemmOp> d_gemm;
  DevPtr<PotrfOp> d_potrf;
  DevPtr<PullItem> d_pull;
  double flops = 0;
  // CUDA graph of the serial walk of this launch list (built lazily on first use; every kernel argument is fixed
  // per schedule)
  GraphExec gexec;
  bool graph_failed = false;
  Launch& add(Launch::Kind kind, int64_t off, int32_t count, int32_t grid, double flops, int stream) {
    launches.push_back(Launch{kind, off, count, grid, 0, flops, 0, stream});
    return launches.back();
  }
  int record(int stream) {
    const int ev = nevents++;
    add(Launch::EV_RECORD, 0, ev, 0, 0.0, stream);
    return ev;
  }
  void wait(int ev, int stream) { add(Launch::EV_WAIT, 0, ev, 0, 0.0, stream); }
  void upload() {
    if (ws_size > 0 || ws2_size > 0) {              // patch workspace offsets into pointers
      d_ws = dev_alloc<double>(ws_size);
      d_ws2 = dev_alloc<double>(ws2_size);
      for (GemmOp& op : gemm) {
        if (op.flags & GF_WS) { op.C = d_ws.get() + (int64_t)(intptr_t)op.C; op.flags &= ~GF_WS; }
        if (op.flags & GF_WS2) { op.C = d_ws2.get() + (int64_t)(intptr_t)op.C; op.flags &= ~GF_WS2; }
      }
      for (ReduceOp& r : reduce) {
        r.ws = ((r.flags & GF_WS2) ? d_ws2 : d_ws).get() + (int64_t)(intptr_t)r.ws;
        r.flags &= ~GF_WS2;
      }
    }
    d_reduce = dev_upload(reduce.data(), reduce.size());
    d_gemm = dev_upload(gemm.data(), gemm.size());
    d_potrf = dev_upload(potrf.data(), potrf.size());
    d_pull = dev_upload(pull.data(), pull.size());
    d_tile_op = dev_upload(tile_op.data(), tile_op.size());
    d_tmaps = dev_upload(tmaps.data(), tmaps.size());
    d_pull_entries = dev_upload(pull_entries.data(), pull_entries.size());
  }
  size_t device_bytes() const {
    return gemm.size() * sizeof(GemmOp) + potrf.size() * sizeof(PotrfOp) + pull.size() * sizeof(PullItem) +
           reduce.size() * sizeof(ReduceOp) + (size_t)(ws_size + ws2_size) * 8 + tile_op.size() * 4 + pull_entries.size() * sizeof(PullEntry);
  }
};

// collects the GEMM ops of one phase and splits them into the two tile configurations
struct PhaseBuilder {
  std::vector<GemmOp> big, small, sk1, sk2;   // sk1 / sk2: narrow-RHS streaming flavours (skinny_ops.cuh)
  std::vector<GemmOp> tma;                    // big-tile ops whose operands a tensor map can describe (dense_tiles_tma.cuh)
  int skinny_mt = 0;                          // > 0: ops with M <= skinny_mt take the streaming kernels (row template MT)
  int ws_id = 0;                              // which split-K workspace this builder's partial products use
  std::vector<PotrfOp> potrf;
  std::vector<ReduceOp> reduces;
  int64_t ws_used = 0;
  bool allow_split = true;    // builders whose launches run beside another builder's must not share the split-K workspace
  static bool tma_ok(const GemmOp& op) {
    return op.a_si == 1 && op.b_sj == 1 && op.a_kidx == nullptr && !(op.flags & GF_TRIL_B) &&
           (op.a_sk % 2) == 0 && (op.b_sk % 2) == 0 && op.a_sk > 0 && op.b_sk > 0 && op.K >= 64;
  }
  void push(const GemmOp& op, bool small_tiles) {
    // an in-place op (C == A: the triangular panel multiply) must stay inside ONE tile column; the TMA tile grid is
    // shifted by one column when B starts on an odd element, which would split N = 128 over two tile columns
    const bool tma_splits_inplace = op.C == op.A && op.N + (int)(((uintptr_t)op.B >> 3) & 1) > 128;
    if (small_tiles) small.push_back(op);
    else if (tma_ok(op) && !tma_splits_inplace) tma.push_back(op);
    else big.push_back(op);
  }
  // split op along K into S parts whose partial products land in the workspace, + the fixed-order reduction
  template <typename Push>
  void split_k(const GemmOp& op, int S, int kc, Push push) {
    const int64_t mn = (int64_t)op.M * op.N;
    ReduceOp r;
    memset(&r, 0, sizeof(r));
    r.C = op.C; r.c_si = op.c_si; r.c_sj = op.c_sj; r.M = op.M; r.N = op.N; r.S = S;
    r.flags = (op.flags & (GF_ACCUM | GF_NEG)) | (ws_id ? GF_WS2 : 0);
    r.ws = (const double*)(intptr_t)ws_used;
    reduces.push_back(r);
    for (int c = 0; c < S; c++) {
      GemmOp part = op;
      const int k0 = c * kc;
      part.K = std::min(kc, op.K - k0);
      if (op.a_kidx) part.a_kidx = op.a_kidx + k0; else part.A = op.A + (int64_t)k0 * op.a_sk;
      part.B = op.B + (int64_t)k0 * op.b_sk;
      part.C = (double*)(intptr_t)(ws_used + (int64_t)c * mn);
      part.c_si = 1; part.c_sj = op.M;
      part.flags = (ws_id ? GF_WS2 : GF_WS) | (op.flags & GF_TRIL_B);
      part.pad = k0;                          // triangular B: first k of the part
      push(part);
    }
    ws_used += (int64_t)S * mn;
  }
  bool add_skinny(const GemmOp& op) {
    if (skinny_mt <= 0 || op.M > skinny_mt || op.a_si != 1 || op.c_si != 1 || (op.flags & (GF_LOWER | GF_BIGTILE))) return false;
    const bool f1 = op.b_sj == 1 && op.a_kidx == nullptr;
    if (!f1 && op.b_sk != 1) return false;
    if (!f1 && (op.flags & GF_TRIL_B)) return false;
    std::vector<GemmOp>& dst = f1 ? sk1 : sk2;
    const int cols = f1 ? SK_F1_COLS : SK_F2_COLS, kmin = 64;
    const int64_t nj = (op.N + cols - 1) / cols;
    // enough CTAs to keep the HBM pipe full, K parts of >= kmin.  F1 is bound by (k rounds per thread) x (memory
    // latency): 8 resident 128-thread CTAs per SM with 16 loads in flight each cover the bandwidth-latency product
    int S = 1;
    const int64_t target = f1 ? 148 * 8 : 148 * 4;
    const bool can_split = allow_split && op.C != op.A;
    if (can_split && nj < target) S = (int)std::min<int64_t>((target + nj - 1) / nj, std::max(1, op.K / kmin));
    if (!f1 && skinny_mt < 8) S = std::max(S, (op.K + SK_F2_KMAX - 1) / SK_F2_KMAX);      // the register-blocked F2 stages its whole K range of A
    if (S > 1 && !can_split) return false;
    int kc = op.K;
    if (S > 1) {
      kc = (((op.K + S - 1) / S) + 15) / 16 * 16;
      if (!f1 && skinny_mt < 8) kc = std::min(kc, SK_F2_KMAX);
      S = (op.K + kc - 1) / kc;
    }
    if (S <= 1) { GemmOp o = op; o.pad = 0; dst.push_back(o); }
    else split_k(op, S, kc, [&](const GemmOp& part) { dst.push_back(part); });
    return true;
  }
  void add(GemmOp op) {
    if (op.M <= 0 || op.N <= 0 || op.K <= 0) return;
    if (add_skinny(op)) return;
    // Tile configuration: 128 x 128 tiles for large outputs; outputs that would leave most of the 148 SMs idle
    // (the diagonal-block steps of the solves: nrhs x NBO with K = NBO) take 64 x 64 tiles and, when K allows,
    // split K across CTAs into workspace partials that splitk_reduce_kernel adds in fixed order.
    const bool lower = op.flags & GF_LOWER;
    const int64_t tb = (int64_t)((op.M + 127) / 128) * ((op.N + 127) / 128);
    const int64_t ts = (int64_t)((op.M + 63) / 64) * ((op.N + 63) / 64);
    // GF_BIGTILE: in-place ops whose N must stay inside ONE tile column (another tile of the same rows would read
    // what this one overwrites)
    const bool force_big = op.flags & GF_BIGTILE;
    op.flags &= ~GF_BIGTILE;
    // lower-masked updates inside a wide front's diagonal block (K = 64 in-block steps, the K = 1024 update of the next
    // block's 1024 x 1024 diagonal part): at most 36 useful 128 x 128 tiles sit on the critical chain with one long K
    // loop each; 64 x 64 tiles put 4x the CTAs on it (0.152 -> ~0.05 ms for the K = 1024 step, 25 -> ~13 us for K = 64)
    const bool small_tiles = !force_big && (!(op.M > 64 && op.N > 64) || (!lower && tb < 40 && op.K >= 128) ||
                                            (lower && tb <= 64));
    const int64_t tiles = small_tiles ? ts : tb;
    if (allow_split && !lower && (op.flags & GF_TRIL_B) && op.K >= 4096 && op.C != op.A && !small_tiles) {
      // L11 * Z of a wide front: the tile of the last 128 columns would run the whole K = ns alone (one CTA, 2.7 ms at
      // the 250K root).  K parts of 2048: a part's tiles left of its first column only write zeros, the others are
      // equal pieces of work; the fixed-order reduction adds the parts.
      const int kc = 2048;
      const int S = (op.K + kc - 1) / kc;
      split_k(op, S, kc, [&](GemmOp part) { part.flags = (ws_id ? GF_WS2 : GF_WS) | GF_TRIL_B; push(part, false); });
      return;
    }
    if (allow_split && !lower && !(op.flags & GF_TRIL_B) && tiles <= 148 && op.K >= 256 && op.C != op.A) {
      int S = (int)std::min<int64_t>(std::min<int64_t>(64, op.K / 64), std::max<int64_t>(1, 148 / tiles));   // one wave of CTAs
      const int kc = S > 0 ? (((op.K + S - 1) / S) + 15) / 16 * 16 : op.K;
      S = (op.K + kc - 1) / kc;
      if (S >= 2) {
        op.flags &= ~GF_TRIL_B;
        split_k(op, S, kc, [&](GemmOp part) { part.pad = 0; part.flags = ws_id ? GF_WS2 : GF_WS; push(part, small_tiles); });
        return;
      }
    }
    push(op, small_tiles);
  }
  static double op_flops(const GemmOp& op) {
    if (op.flags & GF_LOWER) {       // entries on/below the diagonal of an M x N region (M >= N)
      const double nn = std::min(op.M, op.N);
      return 2.0 * op.K * ((double)op.M * op.N - nn * (nn - 1) / 2.0);
    }
    if (op.flags & GF_TRIL_B) return (double)op.M * op.N * op.K;      // about half of K per output column
    return 2.0 * op.M * op.N * op.K;
  }
  void flush(Schedule& sch, int stream = 0) {
    if (!potrf.empty()) {
      double pf = 0;
      for (const PotrfOp& o : potrf) pf += 2.0 * o.nb * o.nb * o.nb / 3.0;
      sch.add(Launch::POTRF, (int64_t)sch.potrf.size(), (int32_t)potrf.size(), (int32_t)potrf.size(), pf, stream);
      sch.potrf.insert(sch.potrf.end(), potrf.begin(), potrf.end());
    }
    // one launch per op list; a tile is tm x tn outputs.  The streaming kernels take all M <= skinny_mt rows of a block
    // of output columns in one CTA.
    const struct { std::vector<GemmOp>& ops; Launch::Kind kind; int tm, tn; } lists[] = {
        {tma, Launch::GEMM_TMA, 128, 128}, {big, Launch::GEMM_BIG, 128, 128}, {small, Launch::GEMM_SMALL, 64, 64},
        {sk1, Launch::SKINNY_F1, skinny_mt, SK_F1_COLS}, {sk2, Launch::SKINNY_F2, skinny_mt, SK_F2_COLS}};
    for (const auto& l : lists) {
      std::vector<GemmOp>& v = l.ops;
      if (v.empty()) continue;
      const bool is_tma = l.kind == Launch::GEMM_TMA;
      int64_t tiles = 0;
      double lf = 0;
      for (GemmOp& op : v) {
        int em = 0, en = 0;
        if (is_tma) {      // TMA operands that start on an odd element: map based one element early, tile grid shifted
          em = (int)(((uintptr_t)op.A >> 3) & 1);
          en = (int)(((uintptr_t)op.B >> 3) & 1);
          op.pad = em | (en << 1);
        }
        op.tiles_m = (op.M + em + l.tm - 1) / l.tm;
        op.tiles_n = (op.N + en + l.tn - 1) / l.tn;
        op.tile_start = (int32_t)tiles;
        tiles += (int64_t)op.tiles_m * op.tiles_n;
        const double f = op_flops(op);
        sch.flops += f;
        lf += f;
      }
      if (tiles > 2000000000LL) throw std::runtime_error("too many tiles in one phase");
      const int64_t tile_off = (int64_t)sch.tile_op.size();
      sch.tile_op.resize(tile_off + tiles);
      for (size_t q = 0; q < v.size(); q++)
        std::fill(sch.tile_op.begin() + tile_off + v[q].tile_start,
                  sch.tile_op.begin() + tile_off + v[q].tile_start + (int64_t)v[q].tiles_m * v[q].tiles_n, (int32_t)q);
      if (is_tma) {
        // tensor maps of the two operands: base rounded down to 16 bytes (op.pad bit 0 / 1 = the operand starts one
        // element after its map's base), extents = the op's own M / N x K so that ragged edges are zero-filled
        for (GemmOp& op : v) {
          const int sa = op.pad & 1, sb = (op.pad >> 1) & 1;
          sch.tmaps.push_back(encode_tmap(op.A - sa, (uint64_t)op.M + sa, (uint64_t)op.K, (uint64_t)op.a_sk));
          sch.tmaps.push_back(encode_tmap(op.B - sb, (uint64_t)op.N + sb, (uint64_t)op.K, (uint64_t)op.b_sk));
        }
      }
      Launch& L = sch.add(l.kind, (int64_t)sch.gemm.size(), (int32_t)v.size(), (int32_t)tiles, lf, stream);
      L.tile_off = tile_off;
      if (is_tma) L.aux_off = (int64_t)sch.tmaps.size() - 2 * (int64_t)v.size();
      if (l.kind == Launch::SKINNY_F1 || l.kind == Launch::SKINNY_F2) L.variant = skinny_mt;
      sch.gemm.insert(sch.gemm.end(), v.begin(), v.end());
    }
    if (!reduces.empty()) {
      int64_t blocks = 0;
      for (ReduceOp& r : reduces) {
        r.block_start = (int32_t)blocks;
        blocks += ((int64_t)r.M * r.N + 255) / 256;
      }
      sch.add(Launch::REDUCE, (int64_t)sch.reduce.size(), (int32_t)reduces.size(), (int32_t)blocks, 0.0, stream);
      sch.reduce.insert(sch.reduce.end(), reduces.begin(), reduces.end());
      if (ws_id) sch.ws2_size = std::max(sch.ws2_size, ws_used); else sch.ws_size = std::max(sch.ws_size, ws_used);
    }
    big.clear(); small.clear(); tma.clear(); sk1.clear(); sk2.clear(); potrf.clear(); reduces.clear();
    ws_used = 0;
  }
  bool empty() const { return big.empty() && small.empty() && tma.empty() && sk1.empty() && sk2.empty() && potrf.empty(); }
};

static GemmOp make_op(double* C, int64_t c_si, int64_t c_sj, const double* A, int64_t a_si, int64_t a_sk,
                      const double* B, int64_t b_sj, int64_t b_sk, int M, int N, int K, int flags,
                      const int32_t* kidx = nullptr) {
  GemmOp op;
  memset(&op, 0, sizeof(op));
  op.C = C; op.A = A; op.B = B; op.a_kidx = kidx;
  op.c_si = c_si; op.c_sj = c_sj; op.a_si = a_si; op.a_sk = a_sk; op.b_sj = b_sj; op.b_sk = b_sk;
  op.M = M; op.N = N; op.K = K; op.flags = flags;
  return op;
}

struct SolvePlan {
  int nrhs = 0;
  DevPtr<double> X, X2;
  DevPtr<double> arena[2];
  DevPtr<int64_t> d_vptr;
  Schedule fwd, bwd, lmul;
  size_t bytes = 0;
};

struct EntryMap { DevPtr<int64_t> d_map; int64_t nnz = 0; };

}  // namespace slmm

using namespace slmm;

struct slmm_chol {
  Symbolic S;
  // device copies of the symbolic structure
  DevPtr<int32_t> d_sn_first, d_sn_nrow, d_rows, d_rel, d_child_ptr, d_child_idx, d_col2sn, d_perm, d_iperm;
  DevPtr<int64_t> d_sn_rowptr, d_sn_lptr, d_sn_uptr;
  std::vector<int64_t> uptr, invptr;
  std::vector<int64_t> wptr;          // [nsuper+1] offsets of the wide inverse blocks of each supernode
  std::vector<WBlock> wblocks;
  DevPtr<WBlock> d_wblocks;
  DevPtr<double> Lx;
  DevPtr<double> inv;
  DevPtr<double> W;                   // inverses of the NBO-wide diagonal blocks (supernodes wider than NBI)
  DevPtr<double> wscratch;            // wide fronts: products of one recursive-doubling level
  std::vector<int64_t> wscratch_off;
  DevPtr<double> arena[2];
  int64_t arena_size[2] = {0, 0};
  DevPtr<int> d_info;
  DevPtr<double> d_partial;
  Schedule fact;
  std::vector<EntryMap> maps;
  std::map<int, std::unique_ptr<SolvePlan>> plans;
  Stream s_main, s_bulk;              // factorization streams (main: highest priority)
  Stream s_aux;                        // auxiliary stream: a second solve running beside the one on stream 0
  cudaStream_t cur = nullptr;          // stream the single-stream schedules (solves, L*Z) are issued on (0 or s_aux)
  Event ev_aux;
  Event ev_fork, ev_join;
  std::vector<Event> events;
  bool factored = false;
  bool profiling = false;
  bool timeline = false;               // events of the two-stream schedules carry timestamps (eager issue, no graphs)
  Event tl_fork, tl_join;              // timed twins of ev_fork / ev_join
  std::vector<Event> tl_events;        // timed twins of `events`
  std::vector<Event> tl_launch;        // one timed event after every kernel of the schedule
  int tl_count = 0;
  double prof_ms[16] = {};
  double prof_flops[16] = {};
  int64_t prof_n[16] = {};
  std::vector<float> prof_launch_ms;       // per launch of the last profiled schedule run
  std::vector<double> prof_launch_flops;
  std::vector<int32_t> prof_launch_kind, prof_launch_grid;
  size_t bytes = 0;
  int64_t exported_nnz = 0;

  // the graph execs, streams and events are destroyed only after the work queued on them has finished (errors
  // are ignored: teardown also runs at interpreter shutdown)
  ~slmm_chol() { cudaDeviceSynchronize(); }

  DevSym devsym() const {
    return DevSym{d_sn_first.get(), d_sn_nrow.get(), d_rows.get(), d_rel.get(), d_child_ptr.get(), d_child_idx.get(),
                  d_sn_rowptr.get(), d_sn_lptr.get(), d_sn_uptr.get()};
  }
};

namespace slmm {

static void init_kernel_attributes() {
  static bool done = false;
  if (done) return;
  CUDA_OK(cudaFuncSetAttribute(gemm_tiles_kernel<128, 128, 2, 4, BIG_STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, BIG_SMEM));
  CUDA_OK(cudaFuncSetAttribute(gemm_tiles_kernel<64, 64, 2, 2, SMALL_STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMALL_SMEM));
  CUDA_OK(cudaFuncSetAttribute(potrf_inv_kernel_v4, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF4_SMEM));
  CUDA_OK(cudaFuncSetAttribute(gemm_tiles_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_SMEM));
#define SKD_ATTR(NMT)                                                                                                         \
  CUDA_OK(cudaFuncSetAttribute(skinny_f2_dmma_kernel<NMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SkDmma<NMT>::SMEM));   \
  CUDA_OK(cudaFuncSetAttribute(skinny_f1_dmma_kernel<NMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SkDmma<NMT>::F1_SMEM));
  SKD_ATTR(1) SKD_ATTR(2) SKD_ATTR(4)
#undef SKD_ATTR
  done = true;
}

static void launch_one(slmm_chol* h, const Schedule& sch, const Launch& L, const DevSym& ds, double* X,
                       const DevPtr<double>* vec_arena, const int64_t* d_vptr, int nrhs, cudaStream_t st) {
  switch (L.kind) {
    case Launch::POTRF:
      potrf_inv_kernel_v4<<<L.grid, 256, POTRF4_SMEM, st>>>(sch.d_potrf.get() + L.off, h->d_info.get());
      break;
    case Launch::GEMM_BIG:
      gemm_tiles_kernel<128, 128, 2, 4, BIG_STAGES><<<L.grid, BIG_THREADS, BIG_SMEM, st>>>(sch.d_gemm.get() + L.off, sch.d_tile_op.get() + L.tile_off);
      break;
    case Launch::GEMM_TMA:
      gemm_tiles_tma_kernel<<<L.grid, TMA_THREADS, TMA_SMEM, st>>>(sch.d_gemm.get() + L.off, sch.d_tile_op.get() + L.tile_off, sch.d_tmaps.get() + L.aux_off);
      break;
    case Launch::GEMM_SMALL:
      gemm_tiles_kernel<64, 64, 2, 2, SMALL_STAGES><<<L.grid, SMALL_THREADS, SMALL_SMEM, st>>>(sch.d_gemm.get() + L.off, sch.d_tile_op.get() + L.tile_off);
      break;
    case Launch::PULL_MAT:
      extend_add_kernel<32><<<(L.count + 3) / 4, 128, 0, st>>>(sch.d_pull.get() + L.off, L.count, sch.d_pull_entries.get(), ds, h->Lx.get(),
                                                               h->arena[L.child_parity()].get(), h->arena[L.child_parity() ^ 1].get());
      break;
    case Launch::PULL_MAT_BIG:
      extend_add_kernel<256><<<L.count, 256, 0, st>>>(sch.d_pull.get() + L.off, L.count, sch.d_pull_entries.get(), ds, h->Lx.get(),
                                                      h->arena[L.child_parity()].get(), h->arena[L.child_parity() ^ 1].get());
      break;
    case Launch::PULL_VEC:
      vec_pull_kernel<<<(L.count + 3) / 4, 128, 0, st>>>(sch.d_pull.get() + L.off, L.count, sch.d_pull_entries.get(), ds, X,
                                                         vec_arena[L.child_parity()].get(),
                                                         vec_arena[L.child_parity() ^ 1].get(), d_vptr, nrhs);
      break;
    case Launch::REDUCE:
      splitk_reduce_kernel<<<L.grid, 256, 0, st>>>(sch.d_reduce.get() + L.off, L.count);
      break;
    case Launch::SKINNY_F1:
    case Launch::SKINNY_F2: {
      const GemmOp* ops = sch.d_gemm.get() + L.off;
      const int32_t* top = sch.d_tile_op.get() + L.tile_off;
      const bool f1 = L.kind == Launch::SKINNY_F1;
#define SKD_CASE(NMT)                                                                          \
  if (f1) skinny_f1_dmma_kernel<NMT><<<L.grid, 256, SkDmma<NMT>::F1_SMEM, st>>>(ops, top);  \
  else skinny_f2_dmma_kernel<NMT><<<L.grid, 256, SkDmma<NMT>::SMEM, st>>>(ops, top);
#define SK_CASE(MT)                                                                        \
  if (f1) skinny_f1_kernel<MT><<<L.grid, SK_F1_COLS, 0, st>>>(ops, top);                   \
  else skinny_f2_kernel<MT><<<L.grid, 256, SK_F2_KMAX * MT * sizeof(double), st>>>(ops, top);
      switch (L.row_mt()) {
        case 1: SK_CASE(1) break;
        case 2: SK_CASE(2) break;
        case 4: SK_CASE(4) break;
        case 8: SKD_CASE(1) break;
        case 16: SKD_CASE(2) break;
        default: SKD_CASE(4) break;
      }
#undef SK_CASE
#undef SKD_CASE
      break;
    }
    case Launch::INIT_W:
      init_identity_kernel<<<L.count, 256, 0, st>>>(h->d_wblocks.get(), h->W.get());
      break;
    default:
      break;
  }
}

static bool is_kernel(const Launch& L) { return L.kind != Launch::EV_RECORD && L.kind != Launch::EV_WAIT; }

// Issues a launch list.  With `two`, every launch goes to the stream it names, the priority stream (critical chain)
// or the bulk stream (look-ahead trailing updates), ordered through `events`; otherwise all of them go to `one` in
// list order, which is a valid topological order.  `per_launch` (optional) gets an event recorded after every kernel
// on that kernel's stream.
static void issue_schedule(slmm_chol* h, const Schedule& sch, double* X, const DevPtr<double>* vec_arena,
                           const int64_t* d_vptr, int nrhs, bool two, cudaStream_t one,
                           const std::vector<Event>& events, std::vector<Event>* per_launch = nullptr) {
  const DevSym ds = h->devsym();
  size_t nk = 0;
  for (const Launch& L : sch.launches) {
    cudaStream_t st = two ? (L.stream ? h->s_bulk.get() : h->s_main.get()) : one;
    if (L.kind == Launch::EV_RECORD) { if (two) CUDA_OK(cudaEventRecord(events[L.event()].get(), st)); continue; }
    if (L.kind == Launch::EV_WAIT) { if (two) CUDA_OK(cudaStreamWaitEvent(st, events[L.event()].get(), 0)); continue; }
    launch_one(h, sch, L, ds, X, vec_arena, d_vptr, nrhs, st);
    if (per_launch) {
      if (nk >= per_launch->size()) per_launch->push_back(make_event(cudaEventDefault));
      CUDA_OK(cudaEventRecord((*per_launch)[nk].get(), st));
    }
    nk++;
  }
}

// Runs `body` on the priority stream (with `two`, on the bulk stream too) between a fork from the legacy default
// stream (event `fork`) and a join back to it (event `join`), so that callers see plain stream-0 semantics.
template <typename Body>
static void forked(slmm_chol* h, bool two, cudaEvent_t fork, cudaEvent_t join, Body body) {
  CUDA_OK(cudaEventRecord(fork, 0));
  CUDA_OK(cudaStreamWaitEvent(h->s_main.get(), fork, 0));
  if (two) CUDA_OK(cudaStreamWaitEvent(h->s_bulk.get(), fork, 0));
  body();
  if (two) {
    CUDA_OK(cudaEventRecord(h->ev_join.get(), h->s_bulk.get()));
    CUDA_OK(cudaStreamWaitEvent(h->s_main.get(), h->ev_join.get(), 0));
  }
  CUDA_OK(cudaEventRecord(join, h->s_main.get()));
  CUDA_OK(cudaStreamWaitEvent(0, join, 0));
}

// Captures the serial walk of a launch list into a graph.  Capture happens on the (non-blocking) priority stream:
// the legacy default stream cannot be captured.
static GraphExec capture_schedule(slmm_chol* h, const Schedule& sch, double* X, const DevPtr<double>* vec_arena,
                                  const int64_t* d_vptr, int nrhs) {
  cudaStream_t origin = h->s_main.get();
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  CUDA_OK(cudaStreamBeginCapture(origin, cudaStreamCaptureModeRelaxed));
  try {
    issue_schedule(h, sch, X, vec_arena, d_vptr, nrhs, false, origin, h->events);
    CUDA_OK(cudaGetLastError());
  } catch (...) {
    cudaStreamEndCapture(origin, &graph);
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    throw;
  }
  CUDA_OK(cudaStreamEndCapture(origin, &graph));
  const cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  CUDA_OK(e);
  return GraphExec(exec);
}

// Walks a launch list.  Single-stream schedules (solves, L*Z) run on the legacy default stream like every other
// call of the library, or on the auxiliary stream inside an auxiliary section.  The factorization schedule names two
// streams: its critical chain (diagonal-block factorizations, panel solves, next-panel updates) runs on a
// highest-priority stream, the look-ahead trailing updates on a second one, ordered by events; both are forked from /
// joined to the default stream.
//
// The lists are static (every kernel argument is fixed once the schedule is uploaded), so each single-stream list is
// captured ONCE into a CUDA graph and replayed: a 12-column solve is a chain of ~1000 tiny launches whose cost was the
// host's launch rate, not the kernels.  Two-stream lists are issued launch by launch: replaying the look-ahead pair
// from a graph loses the stream priorities the chain relies on (measured: factorization 183 -> 190 ms at the 250K
// config).
//
// Profiling mode walks any list serially on the current stream with an event after every kernel, and sums the
// kernel times per kind.  Timeline mode issues a two-stream list with timed events, so the host can read when each
// panel / bulk update finished relative to the fork (where is the critical path: the chain or the bulk stream?).
static void run_schedule(slmm_chol* h, Schedule& sch, double* X, const DevPtr<double>* vec_arena, const int64_t* d_vptr,
                         int nrhs) {
  int64_t nk = 0;
  for (const Launch& L : sch.launches) nk += is_kernel(L) ? 1 : 0;
  if (nk == 0) return;
  if (h->profiling) {
    const Event start = make_event(cudaEventDefault);
    std::vector<Event> done;
    CUDA_OK(cudaEventRecord(start.get(), h->cur));
    issue_schedule(h, sch, X, vec_arena, d_vptr, nrhs, false, h->cur, h->events, &done);
    CUDA_OK(cudaEventSynchronize(done.back().get()));
    size_t i = 0;
    for (const Launch& L : sch.launches) {
      if (!is_kernel(L)) continue;
      float ms = 0;
      CUDA_OK(cudaEventElapsedTime(&ms, (i ? done[i - 1] : start).get(), done[i].get()));
      const int k = (int)L.kind;
      h->prof_ms[k] += ms;
      h->prof_flops[k] += L.flops;
      h->prof_n[k] += 1;
      h->prof_launch_ms.push_back(ms);
      h->prof_launch_flops.push_back(L.flops);
      h->prof_launch_kind.push_back(k);
      h->prof_launch_grid.push_back(work_size(L));
      i++;
    }
  } else {
    // schedules with events run on the priority + bulk stream pair; inside an auxiliary section (cur != 0) the
    // pair may already be in use by the solve on stream 0, so the list is walked serially (a valid order)
    const bool two = sch.nevents > 0 && h->s_main != nullptr && h->cur == nullptr;
    while ((int)h->events.size() < sch.nevents) h->events.push_back(make_event(cudaEventDisableTiming));
    if (two && h->timeline) {
      while ((int)h->tl_events.size() < sch.nevents) h->tl_events.push_back(make_event(cudaEventDefault));
      forked(h, true, h->tl_fork.get(), h->tl_join.get(), [&] {
        issue_schedule(h, sch, X, vec_arena, d_vptr, nrhs, true, nullptr, h->tl_events, &h->tl_launch);
      });
      CUDA_OK(cudaEventSynchronize(h->tl_join.get()));
      h->tl_count = sch.nevents + 2;
    } else if (two) {
      forked(h, true, h->ev_fork.get(), h->ev_join.get(),
             [&] { issue_schedule(h, sch, X, vec_arena, d_vptr, nrhs, true, nullptr, h->events); });
    } else {
      if (h->s_main != nullptr && sch.gexec == nullptr && !sch.graph_failed) {
        try {
          sch.gexec = capture_schedule(h, sch, X, vec_arena, d_vptr, nrhs);
        } catch (const std::exception&) {
          sch.graph_failed = true;      // fall back to launch-by-launch for this schedule
        }
      }
      cudaGraphExec_t exec = sch.gexec.get();
      if (exec == nullptr)
        issue_schedule(h, sch, X, vec_arena, d_vptr, nrhs, false, h->cur, h->events);
      else if (h->cur != nullptr)
        CUDA_OK(cudaGraphLaunch(exec, h->cur));            // auxiliary section: the whole list on the auxiliary stream
      else
        forked(h, false, h->ev_fork.get(), h->ev_join.get(), [&] { CUDA_OK(cudaGraphLaunch(exec, h->s_main.get())); });
    }
  }
  g_launch_count += nk;
  CUDA_OK(cudaGetLastError());
}

static void add_pull_items(Schedule& sch, const Symbolic& S, const std::vector<int64_t>& src_ptr, int level,
                           int lo_kind, Launch::Kind kind, int chunk, int min_rows = 0, int max_rows = 1 << 30) {
  // lo_kind: 0 -> targets [0, ns)   1 -> targets [ns, ms)   2 -> targets [0, ms)
  // only parents with min_rows <= ms < max_rows are listed (lets the caller pick a kernel per size class)
  // src_ptr[c]: offset of child c's update matrix / contribution block inside its level arena
  const int64_t off = (int64_t)sch.pull.size();
  std::vector<std::vector<PullEntry>> per_item;
  for (int q = S.level_ptr[level]; q < S.level_ptr[level + 1]; q++) {
    const int p = S.level_sn[q];
    if (S.child_ptr[p + 1] == S.child_ptr[p]) continue;
    const int ns = S.sn_first[p + 1] - S.sn_first[p], ms = S.sn_nrow[p];
    if (ms < min_rows || ms >= max_rows) continue;
    const int a = lo_kind == 1 ? ns : 0, b = lo_kind == 0 ? ns : ms;
    // do not cross the ns boundary inside one item (the kernels branch on it per target)
    std::vector<int> starts;
    for (int c0 = a; c0 < b;) {
      int c1 = std::min(b, c0 + chunk);
      if (c0 < ns && c1 > ns) c1 = ns;
      starts.push_back(c0);
      c0 = c1;
    }
    if (starts.empty()) continue;
    starts.push_back(b);
    const int nit = (int)starts.size() - 1;
    per_item.assign(nit, std::vector<PullEntry>());
    // children in fixed order; each child's sorted target list is cut at the item boundaries
    for (int cq = S.child_ptr[p]; cq < S.child_ptr[p + 1]; cq++) {
      const int c = S.child_idx[cq];
      const int nsc = S.sn_first[c + 1] - S.sn_first[c], rsc = S.sn_nrow[c] - nsc;
      if (rsc == 0) continue;
      const int64_t rel_off = S.sn_rowptr[c] + nsc;
      const int32_t* relc = S.rel.data() + rel_off;
      int t = (int)(std::lower_bound(relc, relc + rsc, a) - relc);
      int item = 0;
      while (t < rsc && relc[t] < b) {
        while (starts[item + 1] <= relc[t]) item++;
        int tb = t;
        while (tb < rsc && relc[tb] < starts[item + 1]) tb++;
        per_item[item].push_back({rel_off, src_ptr[c], rsc, t, tb, 0});
        t = tb;
      }
    }
    for (int i = 0; i < nit; i++) {
      if (per_item[i].empty()) continue;
      const int32_t e0 = (int32_t)sch.pull_entries.size();
      sch.pull_entries.insert(sch.pull_entries.end(), per_item[i].begin(), per_item[i].end());
      sch.pull.push_back({p, starts[i], starts[i + 1], e0, (int32_t)sch.pull_entries.size()});
    }
  }
  const int cnt = (int)(sch.pull.size() - off);
  if (cnt > 0) sch.add(kind, off, cnt, 0, 0.0, 0).variant = (level + 1) & 1;
}

// Supernode s as a dense front: first column f, ns columns, ms rows (rs below the diagonal block), and its panel P
// with leading dimension ld.
struct Front {
  int s, f, ns, ms, rs;
  int64_t ld;
  double* P;
};
static Front front(const slmm_chol* h, int s) {
  const Symbolic& S = h->S;
  const int f = S.sn_first[s], ns = S.sn_first[s + 1] - f, ms = S.sn_nrow[s];
  return Front{s, f, ns, ms, ms - ns, panel_ld(ms), h->Lx.get() + S.sn_lptr[s]};
}

// Outer (NBO-wide) diagonal block `ob` of a front: column range, and where its inverse lives.  A block made
// of a single NBI block reuses the POTRF kernel's 64 x 64 inverse slot; wider blocks get their own slot in W.
struct OuterBlock { int o0, nbo, ldw; double* winv; };
static int num_outer(int ns) { return (ns + NBO - 1) / NBO; }
static OuterBlock outer_block(const slmm_chol* h, const Front& F, int ob) {
  OuterBlock b;
  b.o0 = ob * NBO;
  b.nbo = std::min(F.ns, b.o0 + NBO) - b.o0;
  if (b.nbo <= NBI) {
    b.winv = h->inv.get() + h->invptr[F.s] + (int64_t)(b.o0 / NBI) * NBI * NBI;
    b.ldw = NBI;
  } else {
    int64_t off = h->wptr[F.s];
    for (int q = 0; q < ob; q++) off += (int64_t)NBO * NBO;      // every earlier block of s is a full one
    b.winv = h->W.get() + off;
    b.ldw = b.nbo;
  }
  return b;
}

// outer blocks of the widest front of level d
static int max_outer(const Symbolic& S, int d) {
  int m = 0;
  for (int q = S.level_ptr[d]; q < S.level_ptr[d + 1]; q++) {
    const int s = S.level_sn[q];
    m = std::max(m, num_outer(S.sn_first[s + 1] - S.sn_first[s]));
  }
  return m;
}

// Two-stream look-ahead of the wide fronts.  Each phase of a level puts its critical chain on the main stream and
// the look-ahead remainders on the bulk stream: `bulk` holds updates that the chain needs only in a later outer
// block, `below` (factorization only) the rows below the next diagonal block, which that block's triangular panel
// multiply reads.  The bulk work starts once the chain's launches of the phase have produced its operands; the
// chain waits for it before anything that touches the same entries again, and at the end of the level.
struct LookAhead {
  PhaseBuilder chain, below, bulk;
  int last_bulk_ev = -1, below_ev = -1;
  // updated: the chain's launches of this phase write entries the earlier bulk launches may still be writing
  // reads_below: they read rows `below` updated
  void flush_phase(Schedule& sch, bool updated, bool reads_below = false) {
    const bool side = !below.empty() || !bulk.empty();
    const int ev_chain = side ? sch.record(0) : -1;
    if (updated && last_bulk_ev >= 0) { sch.wait(last_bulk_ev, 0); last_bulk_ev = -1; }
    if (reads_below && below_ev >= 0) { sch.wait(below_ev, 0); below_ev = -1; }
    chain.flush(sch, 0);
    if (!side) return;
    sch.wait(ev_chain, 1);
    if (!below.empty()) {           // rows below the next block first, with their own event
      below.flush(sch, 1);
      below_ev = last_bulk_ev = sch.record(1);
    }
    if (!bulk.empty()) {
      bulk.flush(sch, 1);
      last_bulk_ev = sch.record(1);
    }
  }
  // level boundary: everything of this level is complete before the pulls
  void end_level(Schedule& sch) {
    if (last_bulk_ev >= 0) sch.wait(last_bulk_ev, 0);
    last_bulk_ev = below_ev = -1;
  }
};

// One step of a front's factorization program.  Phase p of a level executes step p of every front of the level.
struct FStep {
  enum Kind { POTRF, TRSM, UPD, WINV1, WINV2, CPANEL, OUTER, SCHUR } kind;
  int a, b;       // POTRF/TRSM/UPD: inner block index ib, -     WINV1/2: outer block, m     CPANEL: outer block, j
};

static void build_factor_schedule(slmm_chol* h) {
  const Symbolic& S = h->S;
  Schedule& sch = h->fact;
  LookAhead la;
  // bulk-stream ops run beside the chain: the split-K workspace has one user
  la.below.allow_split = la.bulk.allow_split = false;
  PhaseBuilder& pb = la.chain;
  std::vector<std::vector<FStep>> prog;
  for (int d = S.nlevels - 1; d >= 0; d--) {
    add_pull_items(sch, S, h->uptr, d, 0, Launch::PULL_MAT, 8, 0, 512);
    add_pull_items(sch, S, h->uptr, d, 0, Launch::PULL_MAT_BIG, 4, 512);
    // ---- programs
    const int nl = S.level_ptr[d + 1] - S.level_ptr[d];
    prog.assign(nl, std::vector<FStep>());
    size_t max_steps = 0;
    for (int q = 0; q < nl; q++) {
      const Front F = front(h, S.level_sn[S.level_ptr[d] + q]);
      std::vector<FStep>& pr = prog[q];
      if (F.ns <= NBO) {
        // narrow front: per 64 columns POTRF, panel solve of ALL rows below, in-block update; Schur complement last
        const int nib = (F.ns + NBI - 1) / NBI;
        for (int ib = 0; ib < nib; ib++) {
          pr.push_back({FStep::POTRF, ib, 0});
          pr.push_back({FStep::TRSM, ib, 0});
          if (ib + 1 < nib) pr.push_back({FStep::UPD, ib, 0});
        }
        if (F.rs > 0) pr.push_back({FStep::SCHUR, 0, 0});
      } else {
        // Wide front (a dense panel chain): the 64-column steps touch ONLY the w x w diagonal block of the current
        // outer block (tiny launches: they find free SMs at once even while bulk updates fill the machine), the
        // block inverse W = L_D^-1 is built by recursive doubling from the 64 x 64 inverses, and the rows below take
        // one triangular multiply L21 = A21 W' (128-column blocks, in place, last block first).
        for (int ob = 0; ob < num_outer(F.ns); ob++) {
          const int o0 = ob * NBO, o1 = std::min(F.ns, o0 + NBO), w = o1 - o0;
          for (int c0 = o0; c0 < o1; c0 += NBI) {
            const int ib = c0 / NBI;
            pr.push_back({FStep::POTRF, ib, 0});
            if (std::min(o1, c0 + NBI) < o1) { pr.push_back({FStep::TRSM, ib, 0}); pr.push_back({FStep::UPD, ib, 0}); }
          }
          for (int m = NBI; m < w; m *= 2) { pr.push_back({FStep::WINV1, ob, m}); pr.push_back({FStep::WINV2, ob, m}); }
          if (F.ms > o1)
            for (int j = (w + 127) / 128 - 1; j >= 0; j--) pr.push_back({FStep::CPANEL, ob, j});
          if (o1 < F.ns) pr.push_back({FStep::OUTER, ob, 0});
          else if (F.rs > 0) pr.push_back({FStep::SCHUR, 0, 0});
        }
      }
      max_steps = std::max(max_steps, pr.size());
    }
    // ---- phases
    for (size_t ph = 0; ph < max_steps; ph++) {
      bool outer_done = false, needs_below = false;
      for (int q = 0; q < nl; q++) {
        if (ph >= prog[q].size()) continue;
        const FStep st = prog[q][ph];
        if (st.kind == FStep::CPANEL || st.kind == FStep::SCHUR) needs_below = true;
        const Front F = front(h, S.level_sn[S.level_ptr[d] + q]);
        const bool wide = F.ns > NBO;
        if (st.kind == FStep::POTRF || st.kind == FStep::TRSM || st.kind == FStep::UPD) {
          const int ib = st.a, c0 = ib * NBI, c1 = std::min(F.ns, c0 + NBI), nb = c1 - c0;
          const int ob = c0 / NBO, ob0 = ob * NBO, ob_end = std::min(F.ns, ob0 + NBO);
          // where the inverse of this 64 x 64 block lives: its private slot, or (wide fronts) the diagonal of W
          double* inv = h->inv.get() + h->invptr[F.s] + (int64_t)ib * NBI * NBI;
          int64_t inv_ld = NBI;
          if (wide) {
            const OuterBlock wb = outer_block(h, F, ob);
            if (wb.nbo > NBI) { inv = wb.winv + (c0 - ob0) + (int64_t)(c0 - ob0) * wb.ldw; inv_ld = wb.ldw; }
          }
          const int row_end = wide ? ob_end : F.ms;      // wide fronts: only the diagonal block of the outer block
          if (st.kind == FStep::POTRF) {
            pb.potrf.push_back({F.P + c0 + c0 * F.ld, inv, (int32_t)F.ld, nb, F.f + c0, (int32_t)inv_ld});
            sch.flops += (double)nb * nb * nb / 3.0;
          } else if (st.kind == FStep::TRSM) {
            // rows below the diagonal block:  X = X * inv^T   (in place, one tile column)
            pb.add(make_op(F.P + c1 + c0 * F.ld, 1, F.ld, F.P + c1 + c0 * F.ld, 1, F.ld, inv, 1, inv_ld, row_end - c1, nb,
                           nb, 0));
          } else {
            // update the rest of the current outer block with this inner block
            pb.add(make_op(F.P + c1 + c1 * F.ld, 1, F.ld, F.P + c1 + c0 * F.ld, 1, F.ld, F.P + c1 + c0 * F.ld, 1, F.ld,
                           row_end - c1, ob_end - c1, nb, GF_LOWER | GF_ACCUM | GF_NEG));
          }
        } else if (st.kind == FStep::WINV1 || st.kind == FStep::WINV2) {
          // recursive doubling: inv([A 0; C B]) = [A^-1 0; -B^-1 (C A^-1)  B^-1], pairs of blocks of size m
          const OuterBlock wb = outer_block(h, F, st.a);
          const int m = st.b, o0 = wb.o0;
          double* T = h->wscratch.get() + h->wscratch_off[F.s];
          int pair = 0;
          for (int lo = 0; lo + m < wb.nbo; lo += 2 * m, pair++) {
            const int m2 = std::min(m, wb.nbo - lo - m);
            double* Tp = T + (int64_t)pair * m * m;
            double* Ainv = wb.winv + lo + (int64_t)lo * wb.ldw;
            double* Binv = wb.winv + (lo + m) + (int64_t)(lo + m) * wb.ldw;
            double* X21 = wb.winv + (lo + m) + (int64_t)lo * wb.ldw;
            if (st.kind == FStep::WINV1)       // T = C A^-1
              pb.add(make_op(Tp, 1, m2, F.P + (o0 + lo + m) + (int64_t)(o0 + lo) * F.ld, 1, F.ld, Ainv, wb.ldw, 1, m2, m,
                             m, 0));
            else                               // X21 = -B^-1 T
              pb.add(make_op(X21, 1, wb.ldw, Binv, 1, wb.ldw, Tp, m2, 1, m2, m, m2, GF_NEG));
          }
        } else if (st.kind == FStep::CPANEL) {
          // rows below the outer block: L21[:, j-th 128 columns] = A21[:, 0:K) W[j-th rows, 0:K)'  (W lower triangular)
          const OuterBlock wb = outer_block(h, F, st.a);
          const int o0 = wb.o0, o1 = o0 + wb.nbo, j0 = 128 * st.b, nj = std::min(128, wb.nbo - j0);
          const int K = std::min(wb.nbo, j0 + 128);
          pb.add(make_op(F.P + o1 + (int64_t)(o0 + j0) * F.ld, 1, F.ld, F.P + o1 + (int64_t)o0 * F.ld, 1, F.ld, wb.winv + j0,
                         1, wb.ldw, F.ms - o1, nj, K, GF_BIGTILE));
        } else if (st.kind == FStep::OUTER) {
          // outer block finished: update all remaining panel columns, K = block width.
          // Look-ahead: the columns of the NEXT outer block are updated on the main stream (they gate the next
          // panel factorization); the columns beyond it go to the bulk stream and overlap with that panel
          // factorization, whose diagonal-block steps leave almost every SM idle.
          const int ob0 = st.a * NBO, c1 = std::min(F.ns, ob0 + NBO);
          outer_done = true;
          const int nx = std::min(F.ns, c1 + NBO);
          const bool split = (F.ns - nx) >= NBO;
          const int ncols = split ? nx - c1 : F.ns - c1;
          // Of the next block's columns only the square diagonal part gates the chain (the 64-column steps of the
          // next outer block); the rows below it are needed when that block's triangular panel multiply starts, so
          // they go to the bulk stream with their own event.
          const int below = F.ms - c1 - ncols;
          pb.add(make_op(F.P + c1 + c1 * F.ld, 1, F.ld, F.P + c1 + ob0 * F.ld, 1, F.ld, F.P + c1 + ob0 * F.ld, 1, F.ld,
                         ncols, ncols, c1 - ob0, GF_LOWER | GF_ACCUM | GF_NEG));
          if (below > 0)
            la.below.add(make_op(F.P + (c1 + ncols) + c1 * F.ld, 1, F.ld, F.P + (c1 + ncols) + ob0 * F.ld, 1, F.ld,
                                 F.P + c1 + ob0 * F.ld, 1, F.ld, below, ncols, c1 - ob0, GF_ACCUM | GF_NEG));
          if (split)
            la.bulk.add(make_op(F.P + nx + nx * F.ld, 1, F.ld, F.P + nx + ob0 * F.ld, 1, F.ld, F.P + nx + ob0 * F.ld, 1, F.ld,
                                F.ms - nx, F.ns - nx, c1 - ob0, GF_LOWER | GF_ACCUM | GF_NEG));
        } else {                      // SCHUR: panel done, U = -L21 L21'
          double* U = h->arena[d & 1].get() + h->uptr[F.s];
          pb.add(make_op(U, 1, F.rs, F.P + F.ns, 1, F.ld, F.P + F.ns, 1, F.ld, F.rs, F.rs, F.ns, GF_LOWER | GF_NEG));
        }
      }
      // a trailing update writes entries the previous bulk updates may still be writing; the triangular panel
      // multiply (and the Schur complement) read rows the bulk stream updated
      la.flush_phase(sch, outer_done, needs_below);
    }
    la.end_level(sch);
    add_pull_items(sch, S, h->uptr, d, 1, Launch::PULL_MAT, 8, 0, 512);
    add_pull_items(sch, S, h->uptr, d, 1, Launch::PULL_MAT_BIG, 4, 512);
  }
  // ---- batched triangular inversion of the NBO-wide diagonal blocks of the NARROW fronts (64 < ns <= NBO; all
  //      supernodes at once, off every front's critical path; wide fronts built theirs above).  W = I, then forward
  //      substitution by NBI blocks:  W[t,:] = inv_t W[t,:];  W[t+1:,:] -= L[t+1:,t] W[t,:].  The multi-RHS solves
  //      then need 2 GEMMs per NBO columns instead of per 64.
  if (!h->wblocks.empty()) {
    sch.add(Launch::INIT_W, 0, (int32_t)h->wblocks.size(), (int32_t)h->wblocks.size(), 0.0, 0);
    for (int t = 0; t < NBO / NBI; t++) {
      for (int half = 0; half < 2; half++) {
        for (int s2 = 0; s2 < S.nsuper; s2++) {
          const Front F = front(h, s2);
          if (F.ns <= NBI || F.ns > NBO) continue;
          for (int ob = 0; ob < num_outer(F.ns); ob++) {
            const OuterBlock b = outer_block(h, F, ob);
            if (b.nbo <= NBI || t * NBI >= b.nbo) continue;
            const int r0 = t * NBI, nbt = std::min(NBI, b.nbo - r0), ncols = std::min(b.nbo, r0 + NBI);
            double* inv64 = h->inv.get() + h->invptr[s2] + (int64_t)((b.o0 + r0) / NBI) * NBI * NBI;
            if (half == 0) {
              pb.add(make_op(b.winv + r0, 1, b.ldw, inv64, 1, NBI, b.winv + r0, b.ldw, 1, nbt, ncols, nbt, 0));
            } else if (r0 + nbt < b.nbo) {
              pb.add(make_op(b.winv + r0 + nbt, 1, b.ldw, F.P + (b.o0 + r0 + nbt) + (int64_t)(b.o0 + r0) * F.ld, 1, F.ld,
                             b.winv + r0, b.ldw, 1, b.nbo - r0 - nbt, ncols, nbt, GF_ACCUM | GF_NEG));
            }
          }
        }
        pb.flush(sch);
      }
    }
  }
  sch.upload();
}

static SolvePlan* get_plan(slmm_chol* h, int nrhs) {
  // Plans (X / X2 / contribution arenas / split-K workspace / launch graphs) are keyed by the RHS width AND by the
  // stream section they serve: a solve inside an auxiliary section runs beside the one on stream 0, so the two must
  // never share buffers even when their widths coincide (c+1 == local probe width).
  const int key = nrhs * 2 + (h->cur != nullptr ? 1 : 0);
  auto it = h->plans.find(key);
  if (it != h->plans.end()) return it->second.get();
  // keep a few widths resident (probe block, deterministic RHS, compute_hess stages)
  if (h->plans.size() >= 6) {
    CUDA_OK(cudaDeviceSynchronize());
    h->plans.clear();
  }
  const Symbolic& S = h->S;
  std::unique_ptr<SolvePlan> pl(new SolvePlan());
  pl->nrhs = nrhs;
  const int n = S.n;
  pl->X = dev_alloc<double>((size_t)n * nrhs);
  pl->X2 = dev_alloc<double>((size_t)n * nrhs);
  std::vector<int64_t> vptr(S.nsuper, 0);
  int64_t asz[2] = {0, 0};
  for (int d = 0; d < S.nlevels; d++) {
    int64_t off = 0;
    for (int q = S.level_ptr[d]; q < S.level_ptr[d + 1]; q++) {
      const int s = S.level_sn[q];
      vptr[s] = off;
      off += (int64_t)(S.sn_nrow[s] - (S.sn_first[s + 1] - S.sn_first[s])) * nrhs;
    }
    asz[d & 1] = std::max(asz[d & 1], off);
  }
  pl->arena[0] = dev_alloc<double>(asz[0]);
  pl->arena[1] = dev_alloc<double>(asz[1]);
  pl->d_vptr = dev_upload(vptr.data(), vptr.size());
  pl->bytes = ((size_t)2 * n * nrhs + asz[0] + asz[1]) * 8;
  const int64_t R = nrhs;
  LookAhead la;
  PhaseBuilder& pb = la.chain;
  // bulk-stream ops run beside the chain's: their split-K partials get a workspace of their own.  The bulk updates of
  // consecutive diagonal blocks are serialised (same rows), and the late ones have far fewer tiles than SMs: without
  // split-K each still costs one full-K tile latency (170 us at the 250K config whatever its size)
  la.bulk.ws_id = 1;
  // narrow blocks, up to 32 columns (the local probe block at 4 GPUs): HBM-streaming kernels instead of DMMA tiles
  // (skinny_ops.cuh).  Measured at the 250K config, solve / L*Z in ms, tiles -> streaming: 32 columns 7.7 -> 6.3 /
  // 3.6 -> 2.2; 64 columns 8.2 -> 9.6 / 3.9 -> 3.7 (16 DMMA per streamed fragment: the tensor pipe, not HBM, bounds
  // the stream there).
  if (nrhs <= 32) pb.skinny_mt = nrhs <= 1 ? 1 : nrhs <= 2 ? 2 : nrhs <= 4 ? 4 : nrhs <= 8 ? 8 : nrhs <= 16 ? 16 : 32;
  const bool lookahead = nrhs >= 64;     // narrow solves are launch-latency chains: nothing to overlap with
  // ---------------- forward:  L y = b  (levels deepest first).  X holds b and the running updates, the solved
  //                  blocks y land in X2 (out of place: Y = Winv * X per NBO-wide diagonal block).
  for (int d = S.nlevels - 1; d >= 0; d--) {
    add_pull_items(pl->fwd, S, vptr, d, 0, Launch::PULL_VEC, 4);
    const int max_nob = max_outer(S, d);
    for (int ph = 0; ph < 2 * max_nob + 1; ph++) {
      bool updated = false;
      for (int q = S.level_ptr[d]; q < S.level_ptr[d + 1]; q++) {
        const Front F = front(h, S.level_sn[q]);
        const int nob = num_outer(F.ns);
        double* Xs = pl->X.get() + (int64_t)F.f * R;
        double* Ys = pl->X2.get() + (int64_t)F.f * R;
        if (ph == 2 * nob) {                       // contribution block  u = -L21 y   (rs x nrhs)
          if (F.rs > 0)
            pb.add(make_op(pl->arena[d & 1].get() + vptr[F.s], 1, R, Ys, 1, R, F.P + F.ns, 1, F.ld, nrhs, F.rs, F.ns,
                           GF_NEG));
          continue;
        }
        if (ph > 2 * nob) continue;
        const OuterBlock b = outer_block(h, F, ph / 2);
        const int o1 = b.o0 + b.nbo;
        if (ph % 2 == 0) {                         // y_b = Winv * x_b      (transposed view: Y^T = X^T Winv^T)
          pb.add(make_op(Ys + (int64_t)b.o0 * R, 1, R, Xs + (int64_t)b.o0 * R, 1, R, b.winv, 1, b.ldw, nrhs, b.nbo,
                         b.nbo, 0));
        } else if (o1 < F.ns) {                    // x[o1:ns] -= L[o1:ns, o0:o1] y_b
          // Look-ahead (wide fronts, many RHS): only the rows of the next diagonal block gate the chain; the rows
          // beyond go to the bulk stream and overlap with the next diagonal steps (a few tiles each).
          updated = true;
          const int nx = std::min(F.ns, o1 + NBO);
          const bool split = lookahead && (F.ns - nx) >= NBO;
          pb.add(make_op(Xs + (int64_t)o1 * R, 1, R, Ys + (int64_t)b.o0 * R, 1, R, F.P + o1 + (int64_t)b.o0 * F.ld, 1,
                         F.ld, nrhs, (split ? nx : F.ns) - o1, b.nbo, GF_ACCUM | GF_NEG));
          if (split)
            la.bulk.add(make_op(Xs + (int64_t)nx * R, 1, R, Ys + (int64_t)b.o0 * R, 1, R, F.P + nx + (int64_t)b.o0 * F.ld,
                                1, F.ld, nrhs, F.ns - nx, b.nbo, GF_ACCUM | GF_NEG));
        }
      }
      la.flush_phase(pl->fwd, updated);
    }
    la.end_level(pl->fwd);
    add_pull_items(pl->fwd, S, vptr, d, 1, Launch::PULL_VEC, 4);
  }
  // ---------------- backward:  L' x = y  (roots first).  X2 holds y and the running updates, the solved blocks x
  //                  land in X; ancestors' final rows are read from X through the row lists.
  for (int d = 0; d < S.nlevels; d++) {
    const int max_nob = max_outer(S, d);
    for (int ph = 0; ph < 2 * max_nob + 1; ph++) {
      bool updated = false;
      for (int q = S.level_ptr[d]; q < S.level_ptr[d + 1]; q++) {
        const Front F = front(h, S.level_sn[q]);
        const int nob = num_outer(F.ns);
        double* Xs = pl->X.get() + (int64_t)F.f * R;
        double* Ys = pl->X2.get() + (int64_t)F.f * R;
        if (ph == 0) {                             // y_top -= L21' x[rows below]   (gathered rows of X)
          if (F.rs > 0)
            pb.add(make_op(Ys, 1, R, pl->X.get(), 1, R, F.P + F.ns, F.ld, 1, nrhs, F.ns, F.rs, GF_ACCUM | GF_NEG,
                           h->d_rows.get() + S.sn_rowptr[F.s] + F.ns));
          continue;
        }
        const int step = ph - 1, r = step / 2;     // outer blocks in reverse order
        if (r >= nob) continue;
        const OuterBlock b = outer_block(h, F, nob - 1 - r);
        if (step % 2 == 0) {                       // x_b = Winv' * y_b
          pb.add(make_op(Xs + (int64_t)b.o0 * R, 1, R, Ys + (int64_t)b.o0 * R, 1, R, b.winv, b.ldw, 1, nrhs, b.nbo,
                         b.nbo, 0));
        } else if (b.o0 > 0) {                     // y[0:o0] -= L[o0:o1, 0:o0]' x_b
          updated = true;
          const int p0 = b.o0 - NBO;               // the block solved next is [p0, o0)
          const bool split = lookahead && p0 >= NBO;
          const int lo = split ? p0 : 0;
          pb.add(make_op(Ys + (int64_t)lo * R, 1, R, Xs + (int64_t)b.o0 * R, 1, R, F.P + b.o0 + (int64_t)lo * F.ld, F.ld,
                         1, nrhs, b.o0 - lo, b.nbo, GF_ACCUM | GF_NEG));
          if (split)
            la.bulk.add(make_op(Ys, 1, R, Xs + (int64_t)b.o0 * R, 1, R, F.P + b.o0, F.ld, 1, nrhs, p0, b.nbo,
                                GF_ACCUM | GF_NEG));
        }
      }
      la.flush_phase(pl->bwd, updated);
    }
    la.end_level(pl->bwd);
  }
  // ---------------- L * Z  (same dataflow as the forward sweep, products instead of solves)
  for (int d = S.nlevels - 1; d >= 0; d--) {
    for (int q = S.level_ptr[d]; q < S.level_ptr[d + 1]; q++) {
      const Front F = front(h, S.level_sn[q]);
      // out_top = L11 z_top (upper part of the diagonal block is stored as zeros)
      pb.add(make_op(pl->X2.get() + (int64_t)F.f * R, 1, R, pl->X.get() + (int64_t)F.f * R, 1, R, F.P, 1, F.ld, nrhs, F.ns,
                     F.ns, GF_TRIL_B));
      if (F.rs > 0)
        pb.add(make_op(pl->arena[d & 1].get() + vptr[F.s], 1, R, pl->X.get() + (int64_t)F.f * R, 1, R, F.P + F.ns, 1, F.ld,
                       nrhs, F.rs, F.ns, 0));
    }
    pb.flush(pl->lmul);
    add_pull_items(pl->lmul, S, vptr, d, 2, Launch::PULL_VEC, 4);
  }
  pl->fwd.upload();
  pl->bwd.upload();
  pl->lmul.upload();
  pl->bytes += pl->fwd.device_bytes() + pl->bwd.device_bytes() + pl->lmul.device_bytes();
  SolvePlan* raw = pl.get();
  h->plans[key] = std::move(pl);
  return raw;
}

}  // namespace slmm

template <typename T>
static void copy_out(T* dst, const std::vector<T>& v) { if (dst && !v.empty()) memcpy(dst, v.data(), v.size() * sizeof(T)); }

// =========================================================================================================
extern "C" {

const char* slmm_last_error(void) { return slmm::last_error().c_str(); }
int slmm_version(void) { return 100; }
int slmm_device_count(int* out) {
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess) { c = 0; cudaGetLastError(); }
  *out = c;
  return SLMM_OK;
}

int slmm_chol_analyze(int32_t n, const int32_t* indptr, const int32_t* indices, int32_t ordering,
                      const int32_t* user_perm, slmm_chol_t** out) {
  SLMM_TRY
  if (n <= 0 || !indptr || !indices || !out) throw std::invalid_argument("slmm_chol_analyze: bad arguments");
  std::unique_ptr<slmm_chol> h(new slmm_chol());
  SymbolicOptions opt;
  opt.ordering = ordering;
  analyze(n, indptr, indices, user_perm, opt, h->S);
  const Symbolic& S = h->S;
  init_kernel_attributes();
  // update-matrix and inverse-slot offsets
  h->uptr.assign(S.nsuper, 0);
  h->invptr.assign(S.nsuper + 1, 0);
  for (int d = 0; d < S.nlevels; d++) {
    int64_t off = 0;
    for (int q = S.level_ptr[d]; q < S.level_ptr[d + 1]; q++) {
      const int s = S.level_sn[q];
      const int64_t rs = S.sn_nrow[s] - (S.sn_first[s + 1] - S.sn_first[s]);
      h->uptr[s] = off;
      off += rs * rs;
    }
    h->arena_size[d & 1] = std::max(h->arena_size[d & 1], off);
  }
  h->exported_nnz = 0;
  h->wptr.assign(S.nsuper + 1, 0);
  h->wscratch_off.assign(S.nsuper, 0);
  int64_t wscratch_total = 0;
  for (int s = 0; s < S.nsuper; s++) {
    const int64_t ns = S.sn_first[s + 1] - S.sn_first[s], ms = S.sn_nrow[s];
    h->invptr[s + 1] = h->invptr[s] + ((ns + NBI - 1) / NBI) * NBI * NBI;
    h->exported_nnz += ns * ms - ns * (ns - 1) / 2;
    int64_t w = 0;
    for (int ob = 0; ob < num_outer((int)ns); ob++) {
      const int nbo = (int)std::min<int64_t>(ns, (int64_t)(ob + 1) * NBO) - ob * NBO;
      if (nbo > NBI) {
        if (ns <= NBO) h->wblocks.push_back({h->wptr[s] + w, nbo, 0});   // wide fronts build W during the factorization
        w += ((int64_t)nbo * nbo + 1) & ~(int64_t)1;      // every slot starts on a 16-byte boundary (TMA operands)
      }
    }
    h->wptr[s + 1] = h->wptr[s] + w;
    h->wscratch_off[s] = wscratch_total;
    if (ns > NBO) wscratch_total += (int64_t)(NBO / 2) * (NBO / 2);       // C A^-1 products of one doubling level
  }
  h->d_sn_first = dev_upload(S.sn_first.data(), S.sn_first.size());
  h->d_sn_nrow = dev_upload(S.sn_nrow.data(), S.sn_nrow.size());
  h->d_rows = dev_upload(S.rows.data(), S.rows.size());
  h->d_rel = dev_upload(S.rel.data(), S.rel.size());
  h->d_child_ptr = dev_upload(S.child_ptr.data(), S.child_ptr.size());
  h->d_child_idx = dev_upload(S.child_idx.data(), S.child_idx.size());
  h->d_col2sn = dev_upload(S.col2sn.data(), S.col2sn.size());
  h->d_perm = dev_upload(S.perm.data(), S.perm.size());
  h->d_iperm = dev_upload(S.iperm.data(), S.iperm.size());
  h->d_sn_rowptr = dev_upload(S.sn_rowptr.data(), S.sn_rowptr.size());
  h->d_sn_lptr = dev_upload(S.sn_lptr.data(), S.sn_lptr.size());
  h->d_sn_uptr = dev_upload(h->uptr.data(), h->uptr.size());
  h->Lx = dev_alloc<double>(S.lsize);
  h->inv = dev_alloc<double>(h->invptr[S.nsuper]);
  h->W = dev_alloc<double>(h->wptr[S.nsuper]);
  CUDA_OK(cudaMemset(h->W.get(), 0, std::max<int64_t>(1, h->wptr[S.nsuper]) * sizeof(double)));   // upper blocks of wide fronts' W stay zero
  h->wscratch = dev_alloc<double>(wscratch_total);
  h->d_wblocks = dev_upload(h->wblocks.data(), h->wblocks.size());
  h->arena[0] = dev_alloc<double>(h->arena_size[0]);
  h->arena[1] = dev_alloc<double>(h->arena_size[1]);
  h->d_info = dev_alloc<int>(1);
  h->d_partial = dev_alloc<double>(1024);
  {
    int least = 0, greatest = 0;
    CUDA_OK(cudaDeviceGetStreamPriorityRange(&least, &greatest));
    auto make_stream = [](int priority) {
      cudaStream_t s = nullptr;
      CUDA_OK(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, priority));
      return Stream(s);
    };
    h->s_main = make_stream(greatest);
    h->s_bulk = make_stream(least);
    h->s_aux = make_stream(least);
    h->ev_aux = make_event(cudaEventDisableTiming);
    h->ev_fork = make_event(cudaEventDisableTiming);
    h->ev_join = make_event(cudaEventDisableTiming);
    h->tl_fork = make_event(cudaEventDefault);
    h->tl_join = make_event(cudaEventDefault);
  }
  CUDA_OK(cudaMemset(h->Lx.get(), 0, S.lsize * sizeof(double)));
  build_factor_schedule(h.get());
  h->bytes = (S.lsize + h->invptr[S.nsuper] + h->wptr[S.nsuper] + h->arena_size[0] + h->arena_size[1]) * 8 +
             (S.rows.size() * 2 + S.sn_first.size() * 8) * 4 + h->fact.device_bytes();
  CUDA_OK(cudaDeviceSynchronize());
  *out = h.release();
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_destroy(slmm_chol_t* h) {
  delete h;
  return SLMM_OK;
}

int slmm_chol_stats(const slmm_chol_t* h, int64_t* i, double* d) {
  SLMM_TRY
  if (!h) throw std::invalid_argument("null handle");
  const Symbolic& S = h->S;
  if (i) {
    i[0] = S.n; i[1] = S.nsuper; i[2] = S.nlevels; i[3] = S.nnzL; i[4] = S.lsize; i[5] = h->exported_nnz;
    i[6] = S.max_front_rows; i[7] = S.max_super_cols; i[8] = S.ncomponents;
    i[9] = (int64_t)h->fact.launches.size();
    size_t b = h->bytes;
    for (auto& kv : h->plans) b += kv.second->bytes;
    for (auto& m : h->maps) b += m.nnz * 8;
    i[10] = (int64_t)b;
  }
  if (d) { d[0] = S.flops; d[1] = S.t_order; d[2] = S.t_symbolic; d[3] = h->fact.flops; }
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_perm(const slmm_chol_t* h, int32_t* perm) {
  SLMM_TRY
  if (!h || !perm) throw std::invalid_argument("null argument");
  memcpy(perm, h->S.perm.data(), sizeof(int32_t) * h->S.n);
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_device_perm(const slmm_chol_t* h, const int32_t** d_perm, const int32_t** d_iperm) {
  if (!h || !d_perm || !d_iperm) return SLMM_ERR_INVALID;
  *d_perm = h->d_perm.get();
  *d_iperm = h->d_iperm.get();
  return SLMM_OK;
}

int slmm_chol_register_pattern_tri(slmm_chol_t* h, const int32_t* indptr, const int32_t* indices, int32_t tri,
                                   int32_t* map_id) {
  SLMM_TRY
  if (!h || !indptr || !indices || !map_id) throw std::invalid_argument("null argument");
  const int64_t nnz = indptr[h->S.n];
  std::vector<int64_t> tgt(nnz);
  entry_map(h->S, indptr, indices, tgt.data(), tri);
  EntryMap m;
  m.nnz = nnz;
  m.d_map = dev_upload(tgt.data(), tgt.size());
  CUDA_OK(cudaDeviceSynchronize());
  h->maps.push_back(std::move(m));
  *map_id = (int32_t)h->maps.size() - 1;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_register_pattern(slmm_chol_t* h, const int32_t* indptr, const int32_t* indices, int32_t* map_id) {
  return slmm_chol_register_pattern_tri(h, indptr, indices, 0, map_id);
}

int slmm_chol_register_pattern_device(slmm_chol_t* h, const int32_t* d_indptr, const int32_t* d_indices, int64_t nnz,
                                      int32_t tri, int32_t* map_id) {
  SLMM_TRY
  if (!h || !d_indptr || !d_indices || !map_id || nnz < 0) throw std::invalid_argument("bad arguments");
  EntryMap m;
  m.nnz = nnz;
  m.d_map = dev_alloc<int64_t>((size_t)nnz);
  DevPtr<int> d_bad = dev_alloc<int>(1);
  CUDA_OK(cudaMemsetAsync(d_bad.get(), 0, sizeof(int), 0));
  const int n = h->S.n;
  entry_map_kernel<<<std::max(1, std::min(148 * 8, (n + 7) / 8)), 256>>>(d_indptr, d_indices, n, h->d_iperm.get(), h->d_col2sn.get(),
                                                                       h->devsym(), tri, m.d_map.get(), d_bad.get());
  g_launch_count++;
  int bad = 0;
  CUDA_OK(cudaMemcpy(&bad, d_bad.get(), sizeof(int), cudaMemcpyDeviceToHost));
  if (bad) throw std::invalid_argument("matrix entry outside the analysed pattern");
  h->maps.push_back(std::move(m));
  *map_id = (int32_t)h->maps.size() - 1;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_add_values(slmm_chol_t* h, int32_t map_id, const double* d_values, double sigma, int32_t first) {
  SLMM_TRY
  if (!h || map_id < 0 || map_id >= (int)h->maps.size()) throw std::invalid_argument("bad map id");
  if (first) CUDA_OK(cudaMemsetAsync(h->Lx.get(), 0, h->S.lsize * sizeof(double), 0));
  const EntryMap& m = h->maps[map_id];
  if (m.nnz > 0) {
    const int grid = (int)std::min<int64_t>((m.nnz + 255) / 256, 148 * 16);
    scatter_axpy_kernel<<<grid, 256>>>(m.d_map.get(), d_values, sigma, h->Lx.get(), m.nnz);
    g_launch_count++;
  }
  CUDA_OK(cudaGetLastError());
  h->factored = false;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_add_values2(slmm_chol_t* h, int32_t map_id, const double* d_values0, double sigma0,
                          const double* d_values1, double sigma1, int32_t first) {
  SLMM_TRY
  if (!h || map_id < 0 || map_id >= (int)h->maps.size() || !d_values0 || !d_values1) throw std::invalid_argument("bad arguments");
  if (first) CUDA_OK(cudaMemsetAsync(h->Lx.get(), 0, h->S.lsize * sizeof(double), 0));
  const EntryMap& m = h->maps[map_id];
  if (m.nnz > 0) {
    const int grid = (int)std::min<int64_t>((m.nnz + 255) / 256, 148 * 16);
    scatter_axpy2_kernel<<<grid, 256>>>(m.d_map.get(), d_values0, sigma0, d_values1, sigma1, h->Lx.get(), m.nnz);
    g_launch_count++;
  }
  CUDA_OK(cudaGetLastError());
  h->factored = false;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_factorize(slmm_chol_t* h, int32_t* fail_col) {
  SLMM_TRY
  if (!h) throw std::invalid_argument("null handle");
  const int big = 0x7fffffff;
  CUDA_OK(cudaMemcpyAsync(h->d_info.get(), &big, sizeof(int), cudaMemcpyHostToDevice, 0));
  run_schedule(h, h->fact, nullptr, nullptr, nullptr, 0);
  int info = 0;
  CUDA_OK(cudaMemcpy(&info, h->d_info.get(), sizeof(int), cudaMemcpyDeviceToHost));
  if (info != big) {
    if (fail_col) *fail_col = info - 1;
    set_last_error("matrix is not positive definite (non-positive pivot at permuted column " + std::to_string(info - 1) + ")");
    return SLMM_ERR_NOT_POSDEF;
  }
  if (fail_col) *fail_col = -1;
  h->factored = true;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_logdet(slmm_chol_t* h, double* out) {
  SLMM_TRY
  if (!h || !out) throw std::invalid_argument("null argument");
  if (!h->factored) throw std::invalid_argument("factorize first");
  const int grid = std::min(1024, (h->S.n + 255) / 256);
  logdet_kernel<<<grid, 256>>>(h->Lx.get(), h->d_col2sn.get(), h->d_sn_first.get(), h->d_sn_nrow.get(), h->d_sn_lptr.get(), h->S.n, h->d_partial.get());
  g_launch_count++;
  std::vector<double> part(grid);
  CUDA_OK(cudaMemcpy(part.data(), h->d_partial.get(), grid * sizeof(double), cudaMemcpyDeviceToHost));
  double s = 0;
  for (double v : part) s += v;
  *out = 2.0 * s;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_solve(slmm_chol_t* h, double* d_B, int32_t nrhs, int32_t mode) {
  SLMM_TRY
  if (!h || !d_B || nrhs <= 0) throw std::invalid_argument("bad arguments");
  if (mode < 0 || mode > 3) throw std::invalid_argument("slmm_chol_solve: mode must be 0, 1, 2 or 3");
  if (!h->factored) throw std::invalid_argument("factorize first");
  SolvePlan* pl = get_plan(h, nrhs);
  const int n = h->S.n;
  const int64_t total = (int64_t)n * nrhs;
  const int grid = (int)std::min<int64_t>((total + 255) / 256, 148 * 32);
  // forward consumes X and leaves y in X2; backward consumes X2 and leaves x in X.  Mode 3 takes B in the factor's
  // row order, so it goes into X2 as it is.
  if (mode == 3) {
    CUDA_OK(cudaMemcpyAsync(pl->X2.get(), d_B, total * sizeof(double), cudaMemcpyDeviceToDevice, h->cur));
  } else {
    gather_rows_kernel<<<grid, 256, 0, h->cur>>>(d_B, mode == 2 ? pl->X2.get() : pl->X.get(), h->d_perm.get(), n, nrhs, 0);
    g_launch_count++;
  }
  if (mode == 0 || mode == 1) run_schedule(h, pl->fwd, pl->X.get(), pl->arena, pl->d_vptr.get(), nrhs);
  if (mode != 1) run_schedule(h, pl->bwd, pl->X.get(), pl->arena, pl->d_vptr.get(), nrhs);
  gather_rows_kernel<<<grid, 256, 0, h->cur>>>(mode == 1 ? pl->X2.get() : pl->X.get(), d_B, h->d_perm.get(), n, nrhs, 1);
  g_launch_count++;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_lmul(slmm_chol_t* h, const double* d_Z, double* d_out, int32_t nrhs) {
  SLMM_TRY
  if (!h || !d_Z || !d_out || nrhs <= 0) throw std::invalid_argument("bad arguments");
  if (!h->factored) throw std::invalid_argument("factorize first");
  SolvePlan* pl = get_plan(h, nrhs);
  const int n = h->S.n;
  const int64_t total = (int64_t)n * nrhs;
  CUDA_OK(cudaMemcpyAsync(pl->X.get(), d_Z, total * sizeof(double), cudaMemcpyDeviceToDevice, h->cur));
  run_schedule(h, pl->lmul, pl->X2.get(), pl->arena, pl->d_vptr.get(), nrhs);
  const int grid = (int)std::min<int64_t>((total + 255) / 256, 148 * 32);
  gather_rows_kernel<<<grid, 256, 0, h->cur>>>(pl->X2.get(), d_out, h->d_perm.get(), n, nrhs, 1);
  g_launch_count++;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_probe_normals(double* d_out, int64_t n, int32_t ncols, int32_t col_begin, uint64_t seed, uint64_t stream) {
  SLMM_TRY
  if (!d_out || n <= 0 || ncols <= 0 || col_begin < 0) throw std::invalid_argument("bad arguments");
  const int64_t total = n * ncols;
  const int grid = (int)std::min<int64_t>((total + 255) / 256, 148 * 16);
  probe_normals_kernel<<<grid, 256>>>(d_out, n, ncols, col_begin, seed, stream);
  g_launch_count++;
  CUDA_OK(cudaGetLastError());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_export_L(slmm_chol_t* h, int64_t* colptr, int32_t* rowidx, double* values) {
  SLMM_TRY
  if (!h || !colptr || !rowidx || !values) throw std::invalid_argument("null argument");
  if (!h->factored) throw std::invalid_argument("factorize first");
  const Symbolic& S = h->S;
  std::vector<double> Lh(S.lsize);
  CUDA_OK(cudaMemcpy(Lh.data(), h->Lx.get(), S.lsize * sizeof(double), cudaMemcpyDeviceToHost));
  int64_t q = 0;
  for (int s = 0; s < S.nsuper; s++) {
    const Front F = front(h, s);
    const int32_t* rows = S.rows.data() + S.sn_rowptr[s];
    const double* P = Lh.data() + S.sn_lptr[s];
    for (int c = 0; c < F.ns; c++) {
      colptr[F.f + c] = q;
      for (int r = c; r < F.ms; r++) { rowidx[q] = rows[r]; values[q] = P[r + (int64_t)c * F.ld]; q++; }
    }
  }
  colptr[S.n] = q;
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_aux_begin(slmm_chol_t* h) {
  SLMM_TRY
  if (!h || !h->s_aux) throw std::invalid_argument("null handle");
  if (h->cur != nullptr) throw std::invalid_argument("auxiliary section already open");
  CUDA_OK(cudaEventRecord(h->ev_aux.get(), 0));         // everything issued so far (the factorization) comes first
  CUDA_OK(cudaStreamWaitEvent(h->s_aux.get(), h->ev_aux.get(), 0));
  h->cur = h->s_aux.get();
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_aux_end(slmm_chol_t* h) {
  if (!h) return SLMM_ERR_INVALID;
  h->cur = nullptr;
  return SLMM_OK;
}

int slmm_chol_aux_join(slmm_chol_t* h) {
  SLMM_TRY
  if (!h || !h->s_aux) throw std::invalid_argument("null handle");
  CUDA_OK(cudaEventRecord(h->ev_aux.get(), h->s_aux.get()));
  CUDA_OK(cudaStreamWaitEvent(0, h->ev_aux.get(), 0));
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_copy_panels(slmm_chol_t* h, double* host_out) {
  SLMM_TRY
  if (!h || !host_out) throw std::invalid_argument("null argument");
  CUDA_OK(cudaMemcpy(host_out, h->Lx.get(), h->S.lsize * sizeof(double), cudaMemcpyDeviceToHost));
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_launch_count(int64_t* out, int32_t reset) {
  if (out) *out = g_launch_count;
  if (reset) g_launch_count = 0;
  return SLMM_OK;
}

int slmm_chol_set_profiling(slmm_chol_t* h, int32_t on) {
  if (!h) return SLMM_ERR_INVALID;
  h->profiling = on != 0;
  for (int k = 0; k < 16; k++) { h->prof_ms[k] = 0; h->prof_flops[k] = 0; h->prof_n[k] = 0; }
  h->prof_launch_ms.clear(); h->prof_launch_flops.clear(); h->prof_launch_kind.clear(); h->prof_launch_grid.clear();
  return SLMM_OK;
}

int slmm_chol_set_timeline(slmm_chol_t* h, int32_t on) {
  if (!h) return SLMM_ERR_INVALID;
  h->timeline = on != 0;
  return SLMM_OK;
}

int slmm_chol_get_timeline(slmm_chol_t* h, int32_t max_n, int32_t* n_out, float* ms, int32_t* stream) {
  SLMM_TRY
  if (!h || !n_out) throw std::invalid_argument("null argument");
  // entry q >= 2: event q-2 of the last two-stream schedule run in timeline mode (ms since the fork; stream that
  // recorded it); entry 1: the join
  const int n = h->tl_count;
  *n_out = n;
  if (ms) {
    std::vector<int> rec_stream(std::max(0, n - 2), 0);
    for (const Launch& L : h->fact.launches)
      if (L.kind == Launch::EV_RECORD && L.event() + 2 < n) rec_stream[L.event()] = L.stream;
    for (int q = 0; q < n && q < max_n; q++) {
      float v = 0.f;
      if (q > 0) CUDA_OK(cudaEventElapsedTime(&v, h->tl_fork.get(), (q == 1 ? h->tl_join : h->tl_events[q - 2]).get()));
      ms[q] = v;
      if (stream) stream[q] = q >= 2 ? rec_stream[q - 2] : 0;
    }
  }
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_get_launch_timeline(slmm_chol_t* h, int32_t max_n, int32_t* n_out, float* end_ms, int32_t* stream,
                                  int32_t* kind, int32_t* grid, double* flops) {
  SLMM_TRY
  if (!h || !n_out) throw std::invalid_argument("null argument");
  std::vector<const Launch*> ks;
  for (const Launch& L : h->fact.launches) if (is_kernel(L)) ks.push_back(&L);
  const int n = (int)std::min(ks.size(), h->tl_launch.size());
  *n_out = n;
  for (int q = 0; q < n && q < max_n; q++) {
    if (end_ms) { float v = 0.f; CUDA_OK(cudaEventElapsedTime(&v, h->tl_fork.get(), h->tl_launch[q].get())); end_ms[q] = v; }
    if (stream) stream[q] = ks[q]->stream;
    if (kind) kind[q] = (int)ks[q]->kind;
    if (grid) grid[q] = work_size(*ks[q]);
    if (flops) flops[q] = ks[q]->flops;
  }
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_chol_get_profile(const slmm_chol_t* h, double* ms6, double* flops6, int64_t* n6) {
  if (!h || !ms6 || !flops6 || !n6) return SLMM_ERR_INVALID;
  for (int k = 0; k < 6; k++) { ms6[k] = h->prof_ms[k]; flops6[k] = h->prof_flops[k]; n6[k] = h->prof_n[k]; }
  return SLMM_OK;
}

int slmm_chol_get_profile_ex(const slmm_chol_t* h, int32_t nkinds, double* ms, double* flops, int64_t* n) {
  if (!h || !ms || !flops || !n || nkinds < 0 || nkinds > 16) return SLMM_ERR_INVALID;
  for (int k = 0; k < nkinds; k++) { ms[k] = h->prof_ms[k]; flops[k] = h->prof_flops[k]; n[k] = h->prof_n[k]; }
  return SLMM_OK;
}

int slmm_chol_get_launch_profile(const slmm_chol_t* h, int64_t max_n, int64_t* n_out, float* ms, double* flops,
                                 int32_t* kind, int32_t* grid) {
  if (!h || !n_out) return SLMM_ERR_INVALID;
  const int64_t n = (int64_t)h->prof_launch_ms.size();
  *n_out = n;
  for (int64_t i = 0; i < n && i < max_n; i++) {
    if (ms) ms[i] = h->prof_launch_ms[i];
    if (flops) flops[i] = h->prof_launch_flops[i];
    if (kind) kind[i] = h->prof_launch_kind[i];
    if (grid) grid[i] = h->prof_launch_grid[i];
  }
  return SLMM_OK;
}

struct slmm_symbolic { Symbolic S; };

int slmm_symbolic_create(int32_t n, const int32_t* indptr, const int32_t* indices, int32_t ordering,
                         const int32_t* user_perm, slmm_symbolic_t** out) {
  SLMM_TRY
  if (n <= 0 || !indptr || !indices || !out) throw std::invalid_argument("slmm_symbolic_create: bad arguments");
  std::unique_ptr<slmm_symbolic> h(new slmm_symbolic());
  SymbolicOptions opt;
  opt.ordering = ordering;
  analyze(n, indptr, indices, user_perm, opt, h->S);
  *out = h.release();
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_symbolic_destroy(slmm_symbolic_t* s) { delete s; return SLMM_OK; }

int slmm_symbolic_stats(const slmm_symbolic_t* h, int64_t* i, double* d) {
  SLMM_TRY
  if (!h) throw std::invalid_argument("null handle");
  const Symbolic& S = h->S;
  if (i) {
    int64_t exported = 0;
    for (int s = 0; s < S.nsuper; s++) {
      const int64_t ns = S.sn_first[s + 1] - S.sn_first[s], ms = S.sn_nrow[s];
      exported += ns * ms - ns * (ns - 1) / 2;
    }
    i[0] = S.n; i[1] = S.nsuper; i[2] = S.nlevels; i[3] = S.nnzL; i[4] = S.lsize; i[5] = exported;
    i[6] = S.max_front_rows; i[7] = S.max_super_cols; i[8] = S.ncomponents; i[9] = (int64_t)S.rows.size();
  }
  if (d) { d[0] = S.flops; d[1] = S.t_order; d[2] = S.t_symbolic; d[3] = 0; }
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_symbolic_arrays(const slmm_symbolic_t* h, int32_t* perm, int32_t* parent, int32_t* colcount,
                         int32_t* sn_first, int32_t* sn_nrow, int32_t* sn_parent, int64_t* sn_rowptr,
                         int64_t* sn_lptr, int32_t* rows, int32_t* rel, int32_t* level_ptr, int32_t* level_sn) {
  SLMM_TRY
  if (!h) throw std::invalid_argument("null handle");
  const Symbolic& S = h->S;
  copy_out(perm, S.perm); copy_out(parent, S.parent); copy_out(colcount, S.colcount);
  copy_out(sn_first, S.sn_first); copy_out(sn_nrow, S.sn_nrow); copy_out(sn_parent, S.sn_parent);
  copy_out(sn_rowptr, S.sn_rowptr); copy_out(sn_lptr, S.sn_lptr); copy_out(rows, S.rows); copy_out(rel, S.rel);
  copy_out(level_ptr, S.level_ptr); copy_out(level_sn, S.level_sn);
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_symbolic_entry_map_tri(const slmm_symbolic_t* h, const int32_t* indptr, const int32_t* indices, int32_t tri,
                                int64_t* target) {
  SLMM_TRY
  if (!h || !indptr || !indices || !target) throw std::invalid_argument("null argument");
  entry_map(h->S, indptr, indices, target, tri);
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_symbolic_entry_map(const slmm_symbolic_t* h, const int32_t* indptr, const int32_t* indices, int64_t* target) {
  SLMM_TRY
  if (!h || !indptr || !indices || !target) throw std::invalid_argument("null argument");
  entry_map(h->S, indptr, indices, target);
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_gemm_selftest_ex(int32_t M, int32_t N, int32_t K, const double* d_A, int64_t lda, const double* d_B, int64_t ldb,
                          double* d_C, int64_t ldc, int32_t flags, int32_t copies) {
  SLMM_TRY
  // `copies` identical ops C (+/-)= A B' in ONE launch (several ops per launch, as in the factorization); column-major
  // operands with explicit leading dimensions, so that panel-like strides and odd base offsets can be exercised
  init_kernel_attributes();
  Schedule sch;
  PhaseBuilder pb;
  pb.allow_split = false;
  for (int c = 0; c < copies; c++)
    pb.add(make_op(d_C + (int64_t)c * ldc * N, 1, ldc, d_A, 1, lda, d_B, 1, ldb, M, N, K, flags & (GF_LOWER | GF_ACCUM | GF_NEG)));
  pb.flush(sch);
  sch.upload();
  slmm_chol dummy;
  run_schedule(&dummy, sch, nullptr, nullptr, nullptr, 0);
  CUDA_OK(cudaDeviceSynchronize());
  return SLMM_OK;
  SLMM_CATCH
}

int slmm_gemm_selftest(int32_t M, int32_t N, int32_t K, const double* d_A, const double* d_B, double* d_C,
                       int32_t lower, int32_t reps, float* ms_out) {
  SLMM_TRY
  init_kernel_attributes();
  Schedule sch;
  PhaseBuilder pb;
  pb.add(make_op(d_C, 1, M, d_A, 1, M, d_B, 1, N, M, N, K, lower ? GF_LOWER : 0));
  pb.flush(sch);
  sch.upload();
  const Event e0 = make_event(cudaEventDefault), e1 = make_event(cudaEventDefault);
  slmm_chol dummy;
  run_schedule(&dummy, sch, nullptr, nullptr, nullptr, 0);
  CUDA_OK(cudaEventRecord(e0.get(), 0));
  for (int r = 0; r < reps; r++) run_schedule(&dummy, sch, nullptr, nullptr, nullptr, 0);
  CUDA_OK(cudaEventRecord(e1.get(), 0));
  CUDA_OK(cudaEventSynchronize(e1.get()));
  float ms = 0;
  CUDA_OK(cudaEventElapsedTime(&ms, e0.get(), e1.get()));
  if (ms_out) *ms_out = reps > 0 ? ms / reps : 0.f;
  return SLMM_OK;
  SLMM_CATCH
}

}  // extern "C"
