/*
 * scilmm_b200 — C-ABI of the B200-native estimation engine behind SciLMM's SparseCholesky path.
 *
 * The reference is pure Python (scilmm/SparseCholesky.py); its "FFI" for this path is the set of calls it
 * makes into sksparse.cholmod / scipy.sparse.  Each entry point below names the reference call site(s) it
 * replaces.  All pointers are plain host or device pointers (no torch / numpy types); `d_` = device memory
 * on the current CUDA device, `h_` = host memory.  All matrices are FP64 with int32 indices (the reference
 * hard-codes use_long=False, SparseCholesky.py:17).  Dense multi-column blocks are C-ordered n x k
 * (the layout numpy hands the reference), i.e. the k values of one individual are contiguous.
 *
 * Every function returns SLMM_OK (0) or an error code; slmm_last_error() gives the message.
 * Handles are not thread-safe; all work is issued on the legacy default stream (ordered with torch's
 * default stream).  There is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef SCILMM_B200_H
#define SCILMM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLMM_OK 0
#define SLMM_ERR_INVALID 1
#define SLMM_ERR_CUDA 2
#define SLMM_ERR_NOT_POSDEF 3   /* CholmodNotPositiveDefiniteError analogue */
#define SLMM_ERR_INTERNAL 4

#define SLMM_ORDER_NATURAL 0
#define SLMM_ORDER_GIVEN 1
#define SLMM_ORDER_METIS 2      /* nested dissection, the reference default ordering_method='nesdis' (:17) */
#define SLMM_ORDER_MINDEG 3
#define SLMM_ORDER_METIS_FAST 4 /* nested dissection, one separator per bisection: shorter analysis, ~2 % more flops */

typedef struct slmm_chol slmm_chol_t;       /* symbolic analysis + numeric supernodal factor */
typedef struct slmm_matset slmm_matset_t;   /* K device-resident CSR relationship matrices */

const char* slmm_last_error(void);
int slmm_version(void);
int slmm_device_count(int* out);

/* ------------------------------------------------------------------ sparse relationship matrices ------ */
/* K CSR matrices (n x n, sorted indices, both triangles), the `mats` / `mat_list` arguments of
 * HE / REML / compute_gradients (SparseCholesky.py:62,177,192). */
int slmm_matset_create(int32_t n, int32_t K, slmm_matset_t** out);
int slmm_matset_destroy(slmm_matset_t* ms);
/* copy matrix k from host CSR arrays; identical patterns are detected and shared on the device */
int slmm_matset_upload(slmm_matset_t* ms, int32_t k, const int32_t* h_indptr, const int32_t* h_indices,
                       const double* h_data);
/* borrow device-resident CSR arrays for matrix k (same_as >= 0: pattern identical to matrix same_as) */
int slmm_matset_bind_device(slmm_matset_t* ms, int32_t k, const int32_t* d_indptr, const int32_t* d_indices,
                            const double* d_data, int64_t nnz, int32_t same_as);
/* Row-block shard of the HE path (SparseCholesky.py:215-232 moments, SURVEY 8e): the set holds only rows
 * [row_begin, row_end) of every matrix.  Call before binding; the arrays then bound are the rows' slices (indptr of
 * row_end - row_begin + 1 entries starting at 0, indices / data of the block, columns global).  Such a set serves
 * slmm_he_moments only. */
int slmm_matset_set_row_range(slmm_matset_t* ms, int32_t row_begin, int32_t row_end);
/* Symmetry of a sharded matrix: h_out2[0] / h_out2[1] = order-independent 64-bit hash sums of the stored entries
 * above / below the diagonal under the key (min, max, value bits).  Sum both over all shards (wrapping add): the
 * matrix equals its transpose iff the two totals agree; then tell every shard with slmm_matset_set_symmetric. */
int slmm_matset_symmetry_hash(slmm_matset_t* ms, int32_t k, uint64_t* h_out2);
int slmm_matset_set_symmetric(slmm_matset_t* ms, int32_t k, int32_t flag);
/* Pageable host array -> device through a ring of persistent pinned buffers filled by `threads` worker threads
 * (0 = default 4); ordered with the default stream on both sides.  The e2e upload of the scipy CSR arrays. */
int slmm_upload_h2d(void* d_dst, const void* h_src, int64_t nbytes, int32_t threads);
/* Pitched host block -> pitched device block (`rows` pieces of `width_bytes`): the local probe columns of a host
 * n x s block Z (the reference's np.random.randn(n, sim_num), SparseCholesky.py:98) go up without packing the slice
 * on the host.  Pinned or pageable source; returns when the copy is done. */
int slmm_upload_h2d_2d(void* d_dst, int64_t dst_pitch, const void* h_src, int64_t src_pitch, int64_t width_bytes,
                       int64_t rows);
/* The same two uploads issued on `stream` (a cudaStream_t; NULL = the legacy default stream) instead of the default
 * stream: the genotype blocks of the association scan go up on a copy stream while the previous block is swept. */
int slmm_upload_h2d_on(void* d_dst, const void* h_src, int64_t nbytes, int32_t threads, void* stream);
int slmm_upload_h2d_2d_on(void* d_dst, int64_t dst_pitch, const void* h_src, int64_t src_pitch, int64_t width_bytes,
                          int64_t rows, void* stream);
int slmm_matset_nnz(const slmm_matset_t* ms, int32_t k, int64_t* out);
int slmm_matset_values(const slmm_matset_t* ms, int32_t k, const double** d_data_out);

/* Haseman-Elston moments over rows [row_begin,row_end) (row-block shard), replaces the scipy calls
 *   y.dot(A_i.dot(y)) - A_i.diagonal().dot(y**2)                       SparseCholesky.py:223
 *   (A_i.multiply(A_j)).sum() - A_i.diagonal().dot(A_j.diagonal())     SparseCholesky.py:229 (and :237,:241)
 * d_out (device, 2K + 2K*K doubles): [q_off(K) | q_diag(K) | S_off(K*K) | S_diag(K*K)], where *_off sums
 * entries with row != col and *_diag the diagonal ones.  Partial sums of different shards simply add. */
int slmm_he_moments(slmm_matset_t* ms, const double* d_y, int32_t row_begin, int32_t row_end, double* d_out);
/* whole fit from host buffers (H2D of y, kernels, D2H of the moments): the e2e path */
int slmm_he_moments_host(slmm_matset_t* ms, const double* h_y, double* h_out);

/* out = A_k X for a C-ordered n x ncols block (mats[i].dot(X), SparseCholesky.py:65,66,70,157,161) */
int slmm_spmm(slmm_matset_t* ms, int32_t k, const double* d_X, int32_t ncols, double* d_out);
/* d_out[c] = sum_i X[i,c] (A_k X)[i,c] over rows [row_begin,row_end) without materialising A_k X:
 * np.sum(mats[i].dot(sim_vec) * sim_vec, axis=0) and invV_y.dot(mats[i].dot(invV_y)) (SparseCholesky.py:65-66) */
int slmm_spmm_coldot(slmm_matset_t* ms, int32_t k, const double* d_X, int32_t ncols, int32_t row_begin,
                     int32_t row_end, double* d_out);

/* Fused variant for nk (1 or 2) matrices sharing one sparsity pattern (pattern ids from
 * slmm_matset_pattern_id): one pass reads the indices and the gathered X rows once for all of them.
 * d_dots[g*ncols + c] = sum_i X[i,c] (A_ks[g] X)[i,c];  columns c >= store_from of A_ks[g] X are also written to
 * d_store[g][n][ncols - store_from] (C-ordered), which is what the REML trace correction needs
 * (invV_C.T.dot(mats[i].dot(invV_C)), SparseCholesky.py:70).  ncols <= 160. */
int slmm_spmm_coldot_multi(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* d_X, int32_t ncols,
                           int32_t store_from, double* d_store, int32_t row_begin, int32_t row_end, double* d_dots);
/* Quadratic forms only (no stored product): d_dots[g*ncols + c] = x_c' A_ks[g] x_c over rows [row_begin,row_end).
 * Symmetric matrices (checked once per matrix on the device, pattern and values) are traversed on and below the
 * diagonal only, which halves the gathered-row traffic; others take the general pass.  Replaces
 * np.sum(mats[i].dot(sim_vec) * sim_vec, axis=0) / invV_y.dot(mats[i].dot(invV_y)) (SparseCholesky.py:65-66). */
int slmm_quadform_multi(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* d_X, int32_t ncols,
                        int32_t row_begin, int32_t row_end, double* d_dots);
/* Same pass with a narrow block riding along: XB is n x nb (nb <= 16), C-ordered, typically [V^-1 C | V^-1 y].
 * d_gram_half[g][nb][nb] receives Mh with XB' A_ks[g] XB = Mh + Mh' - every c x c quantity of the REML gradient
 * (invV_C.T.dot(mats[i].dot(invV_C)), SparseCholesky.py:70, and by linearity invV_y.dot(mats[i].dot(invV_y)), :66)
 * without a second pass over the matrix.  Symmetric matrices only. */
int slmm_quadform_gram_multi(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* d_X, int32_t ncols,
                             const double* d_XB, int32_t nb, int32_t row_begin, int32_t row_end, double* d_dots,
                             double* d_gram_half);
/* CSR sanity check on the device: *flags_out = 0 when every row is strictly increasing and in range
 * (bit 1: unsorted or duplicate column, bit 2: index / pointer out of range).  scipy hands the reference canonical
 * CSR (Numerator.py:38 .tocsr()); the engine verifies instead of trusting, without a host scan. */
int slmm_matset_validate(slmm_matset_t* ms, int32_t k, int32_t* flags_out);
/* *out = 1 when two device int32 arrays are equal (used to share one pattern between matrices). */
int slmm_device_arrays_equal_i32(const int32_t* d_a, const int32_t* d_b, int64_t count, int32_t* out);
/* *out = 1 when A_k equals its transpose bit for bit (device check, cached). */
int slmm_matset_is_symmetric(slmm_matset_t* ms, int32_t k, int32_t* out);
int slmm_matset_pattern_id(const slmm_matset_t* ms, int32_t k, int32_t* out);

/* Tiled variant of the quadratic-form / Gram pass for SYMMETRIC matrices (the production path of
 * compute_gradients, SparseCholesky.py:62-74).  slmm_matset_build_tiles cuts the lower triangle of matrix k, in the
 * fill-reducing order of a factor (d_perm[new] = old, d_iperm[old] = new: slmm_chol_device_perm), into tiles of 64
 * permuted rows x 64 distinct columns - once per session, on the device; matrices sharing a pattern share the tiling.
 * slmm_quadform_tiled then takes X = [XB | W] (C-ordered n x ncols, ncols <= 160; the first nb <= 16 columns are
 * the narrow block [V^-1 C | V^-1 r]) in the ORIGINAL row order and returns
 *   d_dots[g*ncols + c]  = x_c' A_ks[g] x_c            (np.sum(mats[i].dot(sim_vec) * sim_vec, axis=0), :65)
 *   d_gram_half[g][nb][nb] with XB' A XB = half + half'   (:66 and :70)
 * reading every gathered row of X once per tile from shared memory instead of once per entry through L2. */
int slmm_matset_build_tiles(slmm_matset_t* ms, int32_t k, const int32_t* d_perm, const int32_t* d_iperm);
/* out4: tiles, entries on/below the diagonal, distinct (row block, column) pairs, CTAs of the pass */
int slmm_matset_tile_stats(const slmm_matset_t* ms, int32_t k, int64_t* out4);
/* Developer profile of the last tiled pass: out[c*4 + 0..3] = tiles, non-empty rows, entries of CTA c's tile range and
 * the clock64 span the CTA took (what the partition's cost model is fitted to). */
int slmm_matset_tile_cta_profile(const slmm_matset_t* ms, int32_t k, int64_t* out, int32_t ncta);
int slmm_quadform_tiled(slmm_matset_t* ms, int32_t nk, const int32_t* ks, const double* d_X, int32_t ncols, int32_t nb,
                        double* d_dots, double* d_gram_half);
/* *out = 1 when the n x n CSR matrix in device memory equals its transpose bit for bit (pattern and values).
 * Guards the factor input: the engine keeps one triangle after the fill-reducing permutation, which is only
 * CHOLMOD's answer (it reads the lower triangle, SparseCholesky.py:23-26) when both triangles agree. */
int slmm_device_csr_is_symmetric(const int32_t* d_indptr, const int32_t* d_indices, const double* d_data, int32_t n,
                                 int32_t* out);
/* *out = 1 when every entry of pattern A is present in pattern B (sorted rows, device arrays): lets the host pick
 * the union pattern of V = sum_k sigma_k A_k (matrices_weighted_sum, SparseCholesky.py:55-59) without sparse adds. */
int slmm_device_pattern_subset(const int32_t* d_indptr_a, const int32_t* d_indices_a, const int32_t* d_indptr_b,
                               const int32_t* d_indices_b, int32_t n, int32_t* out);

/* ------------------------------------------------------------------ sparse Cholesky ------------------- */
/* Symbolic analysis of a symmetric pattern given as CSR/CSC with both triangles (host arrays).  Replaces the
 * analyze half of sksparse.cholmod.cholesky (SparseCholesky.py:22-26); done once per pattern.
 * h_user_perm (perm[new] = old) is read when ordering == SLMM_ORDER_GIVEN. */
int slmm_chol_analyze(int32_t n, const int32_t* h_indptr, const int32_t* h_indices, int32_t ordering,
                      const int32_t* h_user_perm, slmm_chol_t** out);
int slmm_chol_destroy(slmm_chol_t* h);
/* i[0]=n i[1]=nsuper i[2]=nlevels i[3]=nnz(L) (sum of column counts) i[4]=stored panel doubles
 * i[5]=exported nnz of L() i[6]=max front rows i[7]=max supernode cols i[8]=components
 * i[9]=kernel launches per factorization i[10]=device bytes held
 * d[0]=flops (sum colcount^2) d[1]=ordering seconds d[2]=symbolic seconds d[3]=dense flops actually issued */
int slmm_chol_stats(const slmm_chol_t* h, int64_t* i_out, double* d_out);
/* factor.P() (SparseCholesky.py:93): A[P][:,P] = L L' */
int slmm_chol_perm(const slmm_chol_t* h, int32_t* h_perm);
/* the same permutation and its inverse in device memory (owned by the handle) */
int slmm_chol_device_perm(const slmm_chol_t* h, const int32_t** d_perm, const int32_t** d_iperm);

/* Register the pattern of one input matrix (any CSR/CSC subset of the analysed pattern, host arrays) and get a
 * scatter map id; values with that pattern can then be streamed into the factor storage. */
int slmm_chol_register_pattern(slmm_chol_t* h, const int32_t* h_indptr, const int32_t* h_indices, int32_t* map_id);
/* Same with an explicit triangle rule.  tri == 0: both triangles are stored with identical values (the caller has
 * verified it, e.g. slmm_device_csr_is_symmetric).  tri != 0: CHOLMOD's rule - sksparse.cholmod.cholesky reads only
 * the lower triangle of the CSC matrix it is given (SparseCholesky.py:23-26): tri > 0 keeps the entries with
 * index >= row of the given arrays (lower triangle of CSC arrays), tri < 0 those with index <= row (lower triangle
 * of CSR arrays); the other triangle is ignored. */
int slmm_chol_register_pattern_tri(slmm_chol_t* h, const int32_t* h_indptr, const int32_t* h_indices, int32_t tri,
                                   int32_t* map_id);
/* Same from device-resident CSR arrays (e.g. those of a slmm_matset_t): the scatter map is built by a kernel, no
 * host pass over the entries and no 8-byte-per-entry upload. */
int slmm_chol_register_pattern_device(slmm_chol_t* h, const int32_t* d_indptr, const int32_t* d_indices, int64_t nnz,
                                      int32_t tri, int32_t* map_id);
/* V assembly (matrices_weighted_sum, SparseCholesky.py:55-59), fused with the scatter into the permuted
 * supernodal panels:  panels = 0 ; panels += sigma * values  for each call, in call order (rounded multiply then
 * rounded add, the order scipy uses).  first != 0 clears the panels before adding. */
int slmm_chol_add_values(slmm_chol_t* h, int32_t map_id, const double* d_values, double sigma, int32_t first);
/* Same for two matrices sharing one registered pattern (A and A o A): V += sigma0*A0 + sigma1*A1 in one pass over
 * the scatter map, rounded exactly like two consecutive slmm_chol_add_values calls. */
int slmm_chol_add_values2(slmm_chol_t* h, int32_t map_id, const double* d_values0, double sigma0,
                          const double* d_values1, double sigma1, int32_t first);
/* numeric supernodal LL' (the factorize half of sksparse.cholmod.cholesky).  On a non-positive pivot returns
 * SLMM_ERR_NOT_POSDEF and *fail_col = failing column in permuted order. */
int slmm_chol_factorize(slmm_chol_t* h, int32_t* fail_col);
/* factor.logdet() (SparseCholesky.py:40) */
int slmm_chol_logdet(slmm_chol_t* h, double* h_out);
/* factor(b) = solve_A (SparseCholesky.py:30,32,52,100,149,153): in-place on a C-ordered n x nrhs device block,
 * original ordering.  mode 0: V^-1 b;  1: forward half only (L^-1 P b, permuted order);  2: backward half only;
 * 3: backward half from the factor's row order (P' L^-T b: b is taken in permuted order, the result comes back in
 * original order).  With Z in permuted order, mode 3 on Z gives V^-1 (slmm_chol_lmul of Z), the probe block of
 * simulate_vector, without forming L Z.  Any other mode is SLMM_ERR_INVALID. */
int slmm_chol_solve(slmm_chol_t* h, double* d_B, int32_t nrhs, int32_t mode);
/* (factor.L().dot(Z))[argsort(P)]  (SparseCholesky.py:50-51): d_out in original ordering, C-ordered n x nrhs */
int slmm_chol_lmul(slmm_chol_t* h, const double* d_Z, double* d_out, int32_t nrhs);
/* Z = np.random.randn(n, sim_num) of simulate_vector (SparseCholesky.py:50) drawn on the device: columns
 * [col_begin, col_begin + ncols) of the n x sim_num block of evaluation `stream`, written C-ordered n x ncols.
 * Counter-based (Philox4x32-10, Box-Muller): the value of (row, global column) depends only on (seed, stream), never
 * on how the columns are split over GPUs.  Distribution-equivalent to, not stream-identical with, numpy's MT19937. */
int slmm_probe_normals(double* d_out, int64_t n, int32_t ncols, int32_t col_begin, uint64_t seed, uint64_t stream);
/* factor.L() as host CSC (colptr int64[n+1], rowidx int32[nnz], values double[nnz]; nnz = stats i[5]) */
int slmm_chol_export_L(slmm_chol_t* h, int64_t* h_colptr, int32_t* h_rowidx, double* h_values);

/* Instrumentation.  slmm_launch_count: kernels launched by this library since the last reset.
 * Profiling mode brackets every launch of the factor / solve schedules with CUDA events on the launching stream and
 * sums the time per kernel kind: 0 potrf+inverse, 1 DMMA GEMM 128x128 tiles, 2 DMMA GEMM 64x64 tiles,
 * 3 extend-add (warp per item), 4 RHS pull, 5 extend-add (CTA per item, large parents).  flops6 = dense flops issued per kind. */
/* Two solves side by side.  Between slmm_chol_aux_begin and slmm_chol_aux_end, slmm_chol_solve / slmm_chol_lmul
 * are issued on an auxiliary stream (ordered after everything already queued on stream 0, e.g. the
 * factorization) instead of stream 0, so that a narrow solve (the c+1 fixed-effect columns, SparseCholesky.py:30,32)
 * - a launch-latency-bound chain that leaves the SMs idle - overlaps the probe pipeline (:50-52) the caller issues
 * on stream 0 next.  slmm_chol_aux_join makes stream 0 wait for the auxiliary work; the solved block must not be
 * read (or freed) before it.  Solve plans (work buffers, launch graphs) are kept per (RHS width, section), so the
 * two solves may have the same width. */
int slmm_chol_aux_begin(slmm_chol_t* h);
int slmm_chol_aux_end(slmm_chol_t* h);
int slmm_chol_aux_join(slmm_chol_t* h);
/* raw supernodal panels (lsize doubles, layout of slmm_symbolic_arrays' sn_lptr / sn_nrow): parity tests compare
 * them supernode by supernode with the CPU oracle */
int slmm_chol_copy_panels(slmm_chol_t* h, double* host_out);
int slmm_launch_count(int64_t* out, int32_t reset);
int slmm_chol_set_profiling(slmm_chol_t* h, int32_t on);
int slmm_chol_get_profile(const slmm_chol_t* h, double* ms6, double* flops6, int64_t* n6);
/* same for the first nkinds <= 16 kinds: ... 6 identity init, 7 split-K reduce, 10 / 11 narrow-RHS streaming kernels
 * (flavour 1 / 2), 12 DMMA GEMM 128x128 tiles with TMA-staged operands */
int slmm_chol_get_profile_ex(const slmm_chol_t* h, int32_t nkinds, double* ms, double* flops, int64_t* n);
/* Timeline mode: the factorization's two-stream schedule is issued with TIMED events; after a factorization
 * slmm_chol_get_timeline returns, per event of the schedule, the ms since the fork and the stream that recorded it
 * (0 chain / 1 bulk; entry 0 = fork, entry 1 = join).  Shows whether the panel chain or the bulk updates are the
 * critical path of each outer block. */
int slmm_chol_set_timeline(slmm_chol_t* h, int32_t on);
int slmm_chol_get_timeline(slmm_chol_t* h, int32_t max_n, int32_t* n_out, float* ms, int32_t* stream);
/* ... and per kernel launch of that run: completion time (ms since the fork), stream, kind (as in the profile),
 * CTAs / items, dense flops */
int slmm_chol_get_launch_timeline(slmm_chol_t* h, int32_t max_n, int32_t* n_out, float* end_ms, int32_t* stream,
                                  int32_t* kind, int32_t* grid, double* flops);
/* per-launch records of the profiled runs (time, issued flops, kind, CTAs or work items); *n_out = available */
int slmm_chol_get_launch_profile(const slmm_chol_t* h, int64_t max_n, int64_t* n_out, float* ms, double* flops,
                                 int32_t* kind, int32_t* grid);

/* Host-only view of the symbolic analysis (no CUDA device needed): used by the host-logic tests and to size a
 * problem before touching the GPU.  i_out as slmm_chol_stats i[0..8] plus i[9]=total rows entries; the array
 * getters may be NULL. */
typedef struct slmm_symbolic slmm_symbolic_t;
int slmm_symbolic_create(int32_t n, const int32_t* h_indptr, const int32_t* h_indices, int32_t ordering,
                         const int32_t* h_user_perm, slmm_symbolic_t** out);
int slmm_symbolic_destroy(slmm_symbolic_t* s);
int slmm_symbolic_stats(const slmm_symbolic_t* s, int64_t* i_out, double* d_out);
int slmm_symbolic_arrays(const slmm_symbolic_t* s, int32_t* perm, int32_t* parent, int32_t* colcount,
                         int32_t* sn_first, int32_t* sn_nrow, int32_t* sn_parent, int64_t* sn_rowptr,
                         int64_t* sn_lptr, int32_t* rows, int32_t* rel, int32_t* level_ptr, int32_t* level_sn);
/* scatter map of a registered pattern into the panel storage (what slmm_chol_register_pattern uploads) */
int slmm_symbolic_entry_map(const slmm_symbolic_t* s, const int32_t* h_indptr, const int32_t* h_indices,
                            int64_t* h_target);
int slmm_symbolic_entry_map_tri(const slmm_symbolic_t* s, const int32_t* h_indptr, const int32_t* h_indices,
                                int32_t tri, int64_t* h_target);

/* ------------------------------------------------------------------ association scan ------------------ */
/* Mixed-model association test of genotyped variants at fixed variance components (GCTA --mlma, EMMAX).  The
 * reference has no counterpart: its users loop over variants with one sparse solve each.  Per block of b variants:
 *   slmm_assoc_genotypes: int8 allele counts d_G (0, 1, 2; negative = missing) of n individuals x b variants, element
 *     (i, j) at d_G[i*row_stride + j*col_stride] (one stride 1: C- or Fortran-ordered host blocks).  Writes the
 *     per-variant non-missing count d_nobs[b] and allele sum d_sum[b], x~ = x - mean (0 where missing) as the
 *     C-ordered n x b block d_X (original row order, ready for slmm_chol_solve mode 1), and d_proj[k*b + j] =
 *     P[:,k]' x~_j for the C-ordered n x np block P = [V^-1 C | V^-1 r] (np <= 32).  Any other entry value returns
 *     SLMM_ERR_INVALID (checked on the device; nothing faults).
 *   slmm_assoc_colsumsq: d_out[j] = sum_i F[i,j]^2 of a C-ordered n x b block (after the forward half-sweep, F = L^-1
 *     P x~, so d_out[j] = x~_j' V^-1 x~_j; any row order).
 * Reductions run over fixed row chunks: a variant's results do not depend on b or on the memory order. */
int slmm_assoc_genotypes(const int8_t* d_G, int64_t n, int32_t b, int64_t row_stride, int64_t col_stride,
                         const double* d_P, int32_t np, double* d_X, double* d_proj, int64_t* d_nobs, int64_t* d_sum);
int slmm_assoc_colsumsq(const double* d_F, int64_t n, int32_t b, double* d_out);

/* ------------------------------------------------------------------ IBD matrix construction ----------- */
/* The step before the path (SURVEY 8f-1): numerator relationship matrix from a child -> parents matrix, replacing
 * Matrices/Numerator.py LD() :5-34 (per-individual Python loop) and create_numerator() :37-38 (L D L').  h_rel_*:
 * host CSR of the boolean relationship matrix (row = child, columns = its <= 2 parents, parents precede children -
 * the output of Relationship.topo_sort).  Bit-identical to the reference (same operation order, no FMA). */
typedef struct slmm_ibd slmm_ibd_t;
int slmm_ibd_build(int32_t n, const int32_t* h_rel_indptr, const int32_t* h_rel_indices, slmm_ibd_t** out);
int slmm_ibd_sizes(const slmm_ibd_t* h, int64_t* nnz_L, int64_t* nnz_A, int32_t* nlevels);
/* L of LD() (row i: 1 on the diagonal, path weights to its ancestors), sorted CSR */
int slmm_ibd_copy_L(const slmm_ibd_t* h, int32_t* h_indptr, int32_t* h_indices, double* h_data);
/* diagonal of D and the inbreeding coefficients F (either may be NULL) */
int slmm_ibd_copy_DF(const slmm_ibd_t* h, double* h_D, double* h_F);
/* A = L D L' (create_numerator), sorted CSR, both triangles */
int slmm_ibd_copy_A(const slmm_ibd_t* h, int32_t* h_indptr, int32_t* h_indices, double* h_data);
int slmm_ibd_destroy(slmm_ibd_t* h);

/* FP64 DMMA self-test / microbenchmark of the tile GEMM (C = A B^T, column-major); returns elapsed ms */
int slmm_gemm_selftest(int32_t M, int32_t N, int32_t K, const double* d_A, const double* d_B, double* d_C,
                       int32_t lower, int32_t reps, float* ms_out);

/* `copies` identical operations C_c (+/-)= A B^T in one launch, column-major operands with explicit leading
 * dimensions (C_c = d_C + c*ldc*N); flags: 1 lower-masked, 2 accumulate, 4 negate.  Test hook for the tile kernels
 * (several ops per launch, panel-like strides, operands that start on an odd element). */
int slmm_gemm_selftest_ex(int32_t M, int32_t N, int32_t K, const double* d_A, int64_t lda, const double* d_B, int64_t ldb,
                          double* d_C, int64_t ldc, int32_t flags, int32_t copies);

#ifdef __cplusplus
}
#endif
#endif
