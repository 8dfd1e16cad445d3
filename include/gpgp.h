/*
 * gpgp.h -- C ABI of libgpgp.so: the B200 (sm_100a) implementation of the Gaussian-process log-likelihood hot
 * path of ameli/gaussian-process-param-estimation (reference package `gaussian_proc`).
 *
 * The reference has no C ABI of its own (SURVEY.md section 8b): its only native surface are the Cython `cdef`
 * functions of gaussian_proc/generate_correlation/_kernels.pxd:5-13 and the six duck-typed MixedCorrelation
 * methods. Every entry point below therefore cites the reference function whose arithmetic it replaces.
 *
 * Conventions
 *  - all matrix / vector pointers are DEVICE pointers owned by the caller (e.g. torch CUDA tensors) unless the
 *    parameter name ends in `_host`; sizes are int64_t; matrices are row-major; `stream` is a cudaStream_t
 *    passed as void* (NULL = legacy default stream).
 *  - dense square matrices live in a PADDED buffer: npad = gp_padded_size(n) (next multiple of 128), leading
 *    dimension npad, with the padding block equal to the identity (zero off-diagonal). Cholesky, inverse and
 *    log-determinant of the padded matrix restrict exactly to those of the n x n matrix.
 *  - return value: 0 ok; > 0 LAPACK-style info (1-based index of the first non-positive pivot, or the Lanczos /
 *    CG breakdown step); < 0 bad argument (-1..-99) or CUDA error (-1000 - cudaError).
 *  - every entry point that takes a correlation scale (scale_host, d entries) and nu checks them before anything is
 *    enqueued: -3 when a scale entry is not > 0 (NaN included); -4 when a d/d(rho) is requested, which needs an isotropic
 *    scale, and the entries differ; -5 when nu takes the general (Bessel) branch and is not > 0.
 *  - nothing here allocates persistent device memory; the caller passes workspaces sized by the matching
 *    *_workspace_bytes query. Calls are stream-ordered and re-entrant per (device, stream).
 */
#ifndef GPGP_H
#define GPGP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* library / build identification: returns 100 (the sm_100a build) */
int gp_abi_version(void);
/* npad for a matrix of size n */
int64_t gp_padded_size(int64_t n);
/* number of CUDA kernels this library has launched in this process (bench.py reports the delta as gpu_launches) */
unsigned long long gp_launch_count(void);
/* Measurement hooks for bench.py's roofline leg: while enabled, every DMMA GEMM launch is bracketed by CUDA events on
 * its own stream; gp_gemm_profile_read synchronises the device and returns the summed kernel milliseconds, the length
 * of the union of the launch intervals (launches on the helper streams overlap), the tile flops those launches
 * executed and their count (host pointers). */
int gp_gemm_profile_enable(int on);
int gp_gemm_profile_read(double* ms_sum_host, double* ms_union_host, double* flops_host, long long* launches_host);

/* ---------------------------------------------------------------------------------------------------------
 * Correlation generation  (reference: generate_correlation/_kernels.pyx:17-136,
 *                          _generate_dense_correlation.pyx:23-162, _generate_sparse_correlation.pyx:35-594)
 * nu selects the Matern branch exactly as _kernels.pyx:73-93: 0.5, 1.5, 2.5 closed forms, nu >= 100 Gaussian;
 * other nu (Bessel K_nu branch, _kernels.pyx:83-88) is evaluated with a device K_nu (Temme series / Steed CF2).
 * ------------------------------------------------------------------------------------------------------- */

/* K[i][j] = matern(||(p_i - p_j) / scale||, nu) into a padded buffer (ldk = npad; padding = identity).
 * dK (optional, may be NULL) receives dK/d(rho) for an isotropic scale rho = scale_host[0]; its padding is zero.
 * points: (n, d) row-major. */
int gp_matern_dense(const double* points, int64_t n, int64_t d, const double* scale_host, double nu,
                    double* K, int64_t ldk, double* dK, void* stream);

/* Rectangular block out[r][c] = matern(||(prow_r - pcol_c) / scale||, nu) of a larger (block-cyclic distributed) padded
 * matrix: row_gidx / col_gidx (device int32) carry the GLOBAL indices, n the unpadded global size; entries with a global
 * index >= n form the identity padding, the global diagonal is exactly 1 + eta. nr % 64 == 0, nc % 128 == 0. */
int gp_matern_cross(const double* prow, const double* pcol, const int* row_gidx, const int* col_gidx, int64_t nr,
                    int64_t nc, int64_t n, int64_t d, const double* scale_host, double nu, double eta, double* out,
                    int64_t ld, void* stream);
/* the same block of dK/d rho (isotropic correlation scale; zero on the global diagonal and in the padding) */
int gp_matern_cross_dk(const double* prow, const double* pcol, const int* row_gidx, const int* col_gidx, int64_t nr,
                       int64_t nc, int64_t n, int64_t d, const double* scale_host, double nu, double* out, int64_t ld,
                       void* stream);
/* Cross-correlation between two point sets (prediction at new points): P[i][j] = matern(||(p_i - q_j) / scale||, nu) for the
 * n points p (n, d) and the m points q (m, d), row-major npad x mpad (npad = gp_padded_size(n), mpad = gp_padded_size(m)),
 * ldp >= mpad and even, P 16-byte aligned. Entries with i >= n or j >= m are exactly 0 (no identity padding); a zero
 * distance gives exactly 1. The distance is evaluated like gp_matern_dense's, so P(points, points) equals its K bit for bit.
 * scale_host: d entries (anisotropic allowed), d <= 8. */
int gp_matern_cross_points(const double* p, int64_t n, const double* q, int64_t m, int64_t d, const double* scale_host,
                           double nu, double* P, int64_t ldp, void* stream);

/* ---- helpers of the distributed dense path (gaussian_proc/_blockcyclic.py; replaces what a ScaLAPACK-style build of the
 * reference's dposv / inverse would provide; the reference itself is single-node, _linear_solver.py:71) ---------------- */
/* Y (M x p) = alpha X (M x N, ldx) R (N x p) + beta Y: skinny product with a rectangular slab, p <= 16 */
int gp_rect_apply(const double* X, int64_t M, int64_t N, int64_t ldx, const double* R, int64_t p, int64_t ldr, double* Y,
                  int64_t ldy, double alpha, double beta, void* stream);
/* S (N x p) = alpha X^T Y + beta S; ws: gp_rect_workspace_bytes(M, N, p) bytes; fixed-order two-stage reduction */
int64_t gp_rect_workspace_bytes(int64_t M, int64_t N, int64_t p);
int gp_rect_apply_t(const double* X, int64_t M, int64_t N, int64_t ldx, const double* Y, int64_t p, int64_t ldy, double* S,
                    int64_t lds, double alpha, double beta, void* ws, void* stream);
/* accum_dev[0] += sum_{r < rows_w1} <A_r, B_r> + w_rest * sum_{r >= rows_w1} <A_r, B_r> over `cols` columns
 * (ws: gp_rect_workspace_bytes(1, 1, 1) bytes suffice) */
int gp_pair_dot(const double* A, int64_t lda, const double* B, int64_t ldb, int64_t rows, int64_t cols, int64_t rows_w1,
                double w_rest, double* accum_dev, void* ws, void* stream);
/* V (n x p, lds) = dK/drho S with dK/drho regenerated from the points (isotropic scale), rows >= n of V zero up to the
 * padded size */
int gp_dk_apply(const double* points, int64_t n, int64_t d, const double* scale_host, double nu, const double* S, int64_t p,
                int64_t lds, double* V, void* stream);

/* tau = matern(kernel_radius(density), nu): host-only, bit-follows _estimate_kernel_threshold
 * (_generate_sparse_correlation.pyx:294-413, with the missing `dimension` argument of :390 supplied).
 * Returns -10 when density * n < 1 (the reference raises ValueError, :378-383). */
int gp_kernel_threshold(int64_t n, int64_t d, double density, const double* scale_host, double nu, double* tau_host);

/* Sparse generator, two calls around the caller's allocation of indices/data (the reference guesses max_nnz and
 * retries with doubled buffers, :548-577): count -> indptr (device int32, n + 1) and nnz (host); fill -> indices
 * (int32, sorted within each row), data and optionally ddata = d/d(rho) values on the same pattern.
 * points: device (n, d); points_host: the same array on the host (bounding box + host re-decision of the pairs with
 * |K - tau| <= 8 ulp, which makes the pattern bit-exact). ws: gp_sparse_workspace_bytes(n, d), shared by both calls.
 * row_pos_dev: NULL for every row. Otherwise (device int32, n) only the rows i with row_first <= row_pos_dev[i] < row_last
 * are generated - one slab of the spatially ordered operator on the row-slab engine, with row_pos = the position of a row
 * in that order - and the other rows stay empty; indptr keeps n + 1 entries and the column ids stay global. Work, memory
 * and time are then those of the slab. Both calls must get the same rows. */
int64_t gp_sparse_workspace_bytes(int64_t n, int64_t d);
int gp_matern_sparse_count(const double* points, const double* points_host, int64_t n, int64_t d,
                           const double* scale_host, double nu, double tau, void* ws, int* indptr_dev,
                           int64_t* nnz_host, const int* row_pos_dev, int64_t row_first, int64_t row_last, void* stream);
/* Space-filling-curve keys of the points over the bounding box [lo_host, hi_host] (d = 2: Hilbert index; otherwise
 * Z-order over the first min(d,3) coordinates): a stable sort by key is the deterministic, spatially local row order the
 * row-blocked sparse operator (gp_bcsr_*) uses. */
int gp_spatial_keys(const double* points, int64_t n, int64_t d, const double* lo_host, const double* hi_host,
                    int64_t* keys_dev, void* stream);
/* sort_rows = 1: canonical CSR (rows sorted by column). sort_rows = 0: rows are left in generation order - enough for
 * the device operators (gp_csr_spmm, the hash path of gp_bcsr_*); gp_csr_sort_rows canonicalises later, on demand. */
int gp_matern_sparse_fill(const double* points, const double* points_host, int64_t n, int64_t d,
                          const double* scale_host, double nu, double tau, void* ws, const int* indptr_dev,
                          int* indices_dev, double* data_dev, double* ddata_dev, int sort_rows, const int* row_pos_dev,
                          int64_t row_first, int64_t row_last, void* stream);
/* Sorts every row of a CSR matrix by column (data / ddata follow); flags_dev: 2 device ints of scratch. */
int gp_csr_sort_rows(int64_t n, const int* indptr_dev, int* indices_dev, double* data_dev, double* ddata_dev,
                     int* flags_dev, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Dense FP64 linear algebra on K + eta*I  (reference: _mixed_correlation/mixed_correlation.py:155-335 and
 * _linear_solver.py:71 scipy.linalg.solve(assume_a='pos'), i.e. LAPACK dposv; imate 'cholesky' logdet/traceinv)
 * ------------------------------------------------------------------------------------------------------- */

/* General DMMA GEMM used by everything below; exported for tests and the roofline microbenchmark.
 * C[MxN] = beta*C + alpha*op(A)*op(B); at/bt: 0 -> operand stored [mn][k], 1 -> stored [k][mn].
 * krange / tmask: see gp_internal.h (0 / 0 = plain GEMM). M,N multiples of 128, K multiple of 32; K == 0 gives
 * C = beta*C on the tiles tmask covers (beta == 0: C is not read).
 * C may alias an operand in one form only, the in-place C = beta*C + alpha*C*op(B) with C == A, ldc == lda,
 * at == bt == 0 and N == 128 (a 128-wide block column, e.g. a Cholesky panel times an inverted diagonal block). Any
 * other C == A or C == B returns -6 before anything is launched, since tiles would read what other tiles write.
 * Returns -7 when the driver's tensor-map encoder (cuTensorMapEncodeTiled) is unavailable. */
int gp_dgemm_f64(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda, const double* B,
                 int64_t ldb, int64_t M, int64_t N, int64_t K, double alpha, double beta, int krange, int tmask,
                 void* stream);
/* The same product with per-row-tile k ranges: output rows [128 t, 128 t + 128) use k in [kbeg_tab[t], kend_tab[t])
 * (DEVICE int arrays of M / 128 entries, either may be NULL): the staircase operands of the distributed inverse
 * (gaussian_proc/_blockcyclic.py). Table entries must be multiples of 16 (the kernel's k-slab; a kbeg is rounded down
 * to one and a partial slab before kend is dropped); a kbeg beyond K or a kend beyond K is clamped to K, and an empty
 * range (kend <= kbeg), like K == 0, gives C = beta*C for that row tile. C must not alias an operand (-6). */
int gp_dgemm_ktab_f64(int at, int bt, double* C, int64_t ldc, const double* A, int64_t lda, const double* B,
                      int64_t ldb, int64_t M, int64_t N, int64_t K, double alpha, double beta, const int* kbeg_tab,
                      const int* kend_tab, void* stream);

/* A (npad x npad, lower triangle referenced) := K + eta*I on the first n diagonal entries (padding diagonal
 * stays exactly 1); replaces `Kn = K + eta*I` of mixed_correlation.py:184,251,296. */
int gp_shift_copy(const double* K, int64_t n, int64_t npad, double eta, double* A, void* stream);

/* bytes of workspace for gp_potrf_f64 (holds the inverted 128x128 diagonal blocks of L) */
int64_t gp_potrf_workspace_bytes(int64_t npad);
/* In-place lower Cholesky A = L L^T (right-looking, blocked; trailing update on the FP64 tensor pipe).
 * info_dev: device int, 0 or 1-based index of the first non-positive pivot. ws keeps inv(L_jj) blocks that
 * gp_potrs_f64 / gp_trtri_f64 reuse. */
int gp_potrf_f64(double* A, int64_t n, int64_t npad, int* info_dev, void* ws, void* stream);

/* logdet(A) = 2 * sum_i log L_ii over the first n rows; out_dev: device double */
int gp_logdet_from_chol(const double* L, int64_t n, int64_t npad, double* out_dev, void* stream);

/* Solve (L L^T) X = B in place. B is (npad x nrhs) row-major with ldb >= nrhs, rows >= n zero. nrhs <= 16. */
int gp_potrs_f64(const double* L, int64_t npad, const void* potrf_ws, double* B, int64_t nrhs, int64_t ldb,
                 void* stream);

/* workspace for gp_potri_f64 */
int64_t gp_potri_workspace_bytes(int64_t npad);
/* W := inv(L) (lower, npad x npad, separate buffer) and Ainv_lower := W^T W written over the lower triangle of
 * `A` (which held L). */
int gp_potri_f64(double* A, double* W, int64_t npad, const void* potrf_ws, void* ws, void* stream);
/* the two halves of gp_potri_f64: W := inv(L) (recursive triangular products); Ainv_lower := W^T W */
int gp_trtri_f64(const double* L, double* W, int64_t npad, const void* potrf_ws, void* ws, void* stream);
int gp_lauum_f64(const double* W, double* Ainv, int64_t npad, void* stream);

/* Traces of the inverse from the triangular / symmetric inverse (imate 'cholesky' traceinv restated,
 * mixed_correlation.py:183-191). kind 0: M = inv(L) -> out[1] = ||M||_F^2 = tr Kn^-1.
 * kind 1: M = Kn^-1 (lower triangle stored) -> out[1] = tr Kn^-1, out[2] = ||Kn^-1||_F^2 = tr Kn^-2.
 * out_dev: device, >= 5 doubles (same layout as gp_loglik_dense's out[0..4]). */
int64_t gp_traces_workspace_bytes(int64_t npad);
int gp_inverse_traces(const double* M, int64_t n, int64_t npad, int kind, double* out_dev, void* ws, void* stream);

/* Y (npad x p) = K * X for a skinny X (npad x p, p <= 16, rows >= n ignored): K_mixed.dot(0, x) of
 * mixed_correlation.py:305-335 (the eta*x term is added by the caller). */
int gp_symm_skinny(const double* K, int64_t n, int64_t npad, const double* X, int64_t p, double* Y, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Sparse (CSR, int32 indices) operator K + eta*I on n x B row-major column blocks, B in {1,2,4,8,16,32}
 * (reference: mixed_correlation.py:193-209,263-268 imate 'hutchinson' / 'slq'; _linear_solver.py:49-68 CG, tol 1e-6)
 * ------------------------------------------------------------------------------------------------------- */
/* Y = (K + eta I) X */
int gp_csr_spmm(const int* indptr, const int* indices, const double* data, int64_t n, double eta, const double* X,
                int64_t B, double* Y, void* stream);
/* V[i][c] = +-1 from a counter-based hash of (seed, probe_offset + c, row): identical for any batching / rank count.
 * row = row_map[i] when row_map (device int32, n) is given (internally permuted operators), else i. */
int gp_rademacher(double* V, int64_t n, int64_t B, uint64_t seed, int64_t probe_offset, const int* row_map,
                  void* stream);
/* Row-blocked form of a (symmetrically permuted) CSR matrix: 16 consecutive rows share one list of block-columns
 * (16 x 1 blocks, zero filled; the list is padded with zero blocks to a multiple of 4 = one DMMA.8x8x4 k-step). New row r =
 * old row order[r], new column = inv_order[old column] (both NULL: no permutation); the source rows must be sorted. With a
 * spatially local order
 * (gp_spatial_keys) neighbouring rows have nearly the same pattern: one gathered row of X then serves 16 rows of K and the
 * index is amortised. n rows are built; order may point into a longer order (one slab: order + first row).
 *   gp_bcsr_count: nblk[rb] = number of block-columns of row block rb (ceil(n/16) entries); the caller's exclusive
 *                  prefix sum gives bptr (int64, ceil(n/16)+1). needs_sorted_dev (device int, may be NULL) is set to 1
 *                  when some row block exceeded the shared-memory hash table and used the binary-search path, which
 *                  requires SORTED source rows (the hash path does not).
 *   gp_bcsr_fill : nblocks = bptr[last]; bidx (int32, nblocks), bvals / bdvals (f64, 16 * nblocks): every group of four
 *                  block-columns is stored in DMMA A-fragment order (one 8-row fragment after the other), value
 *                  (slot s, row k) at 64 (s/4) + 32 (k/8) + 4 (k%8) + s%4. */
int gp_bcsr_count(int64_t n, const int* order, const int* inv_order, const int* indptr, const int* indices, int* nblk,
                  int* needs_sorted_dev, void* stream);
int gp_bcsr_fill(int64_t n, const int* order, const int* inv_order, const int* indptr, const int* indices, const double* data,
                 const double* ddata, const int64_t* bptr, int64_t nblocks, int* bidx, double* bvals, double* bdvals,
                 void* stream);
/* The row-blocked drivers (gp_bcsr_spmm, gp_col_dot, gp_bcsr_lanczos, gp_bcsr_cg_solve) take `peer`: NULL on one GPU.
 * Otherwise it is this rank's arena (gp_peer_create) of the row-slab operator: the row blocks are this rank's rows with
 * encoded columns (gp_slab_encode_columns), n is the number of those rows, vectors are the rank's rows (n x B), and alpha,
 * beta and dot products are summed over the ranks - identical on every rank.
 * Y = (K + eta I) X on the row-blocked operator (FP64 tensor-core MMAs: 4 block-columns x 8 rows x 8 columns; two MMAs
 * share each gathered fragment of X). Tuned for B <= 16. With a peer, X is copied into exchange vector 2 between two
 * cross-GPU barriers. */
int gp_bcsr_spmm(void* peer, const int64_t* bptr, const int* bidx, const double* bvals, int64_t n, double eta,
                 const double* X, int64_t B, double* Y, void* stream);
/* workspace for gp_col_dot / gp_lanczos / gp_cg_solve */
int64_t gp_krylov_workspace_bytes(int64_t n, int64_t B);
/* out_dev[c] = sum_i X[i][c] Y[i][c] (deterministic two-stage reduction) */
int gp_col_dot(void* peer, const double* X, const double* Y, int64_t n, int64_t B, double* out_dev, void* ws, void* stream);
/* m Lanczos steps per column started from V (normalised internally); alpha_dev, beta_dev: (m x B) device arrays of
 * the tridiagonal coefficients (beta[j] couples steps j and j+1). The quadrature itself is host-side.
 * basis_dev: NULL, or m x n x B doubles that receive the unnormalised Lanczos vectors u_j = beta_{j-1} q_j. */
int gp_lanczos(const int* indptr, const int* indices, const double* data, int64_t n, double eta, const double* V,
               int64_t B, int64_t m, double* alpha_dev, double* beta_dev, double* basis_dev, void* ws, void* stream);
/* Batched CG from a zero start: X = (K + eta I)^-1 R0 column by column, stop at ||r|| <= tol ||b||. R0 is
 * overwritten. Returns 0; 1 when maxiter was reached first; 2 when p^T A p <= 0 was met (K + eta I not positive
 * definite: the hard-thresholded Matern matrix is indefinite, _generate_sparse_correlation.pyx:516-523). */
int gp_cg_solve(const int* indptr, const int* indices, const double* data, int64_t n, double eta, double* R0, double* X,
                int64_t B, double tol, int64_t maxiter, int64_t* iters_host, void* ws, void* stream);
/* Skinny Gram matrix out_dev[a*B + b] = sum_i X[i][a] Y[i][b] of two n x B row-major blocks (B <= 16); fixed summation
 * order. Used for G = R^T S, H = S^T S, Q = S^T dK S of the sparse likelihood evaluation (_direct_likelihood.py:113-150). */
int64_t gp_gram_workspace_bytes(int64_t B);
int gp_gram_skinny(const double* X, const double* Y, int64_t n, int64_t B, double* out_dev, void* ws, void* stream);
/* the same two Krylov drivers on the row-blocked operator */
int gp_bcsr_lanczos(void* peer, const int64_t* bptr, const int* bidx, const double* bvals, int64_t n, double eta,
                    const double* V, int64_t B, int64_t m, double* alpha_dev, double* beta_dev, double* basis_dev, void* ws,
                    void* stream);
/* X[i][c] = sum_j coef_dev[j][c] basis[j][i][c] (coef: m x B). With coef[j][c] = ||v_c|| y_jc / beta_{j-1,c} and
 * y = T^-1 e_1 this is the Lanczos solution of (K + eta I) x = v from the vectors kept by gp_*_lanczos: the Hutchinson
 * tr(Kn^-1 dK) estimator reuses the SLQ run instead of a second Krylov solve. B in {1,2,4,8,16,32} and any degree
 * m >= 1 (the sum runs over j = 0 .. m - 1 in order); -1 otherwise. */
int gp_block_combine(const double* basis, int64_t n, int64_t B, int64_t m, const double* coef_dev, double* X, void* stream);
int gp_bcsr_cg_solve(void* peer, const int64_t* bptr, const int* bidx, const double* bvals, int64_t n, double eta,
                     double* R0, double* X, int64_t B, double tol, int64_t maxiter, int64_t* iters_host, void* ws,
                     void* stream);

/* ---- direct generation of the row-blocked operator (csrc/gp_sparse.cu, sparse_blocks_kernel) -------------------------------
 * The consumer of a sparse K in the likelihood is the operator, not the CSR (the reference hands scipy's CSR to imate / cg,
 * _generate_sparse_correlation.pyx:472-594 -> mixed_correlation.py:193-209): these two passes emit the 16-row blocks of the
 * spatially ordered matrix straight from the cell lists - same kernel arithmetic and pattern rule (K > tau) as
 * gp_matern_sparse_count / fill, no CSR, no hash build. Rows [row_first, row_last) of the ordered operator (row_first a
 * multiple of 16; one slab per GPU, or 0 .. n). ws: gp_sparse_workspace_bytes(n, d).
 * count: nblk_dev[rb] = block-columns of row block rb (padded to a multiple of 4); stats_host[0] = entries in the pattern
 * (nnz of these rows), stats_host[1] = pairs inside the 8-ulp borderline band. Returns 3 when the direct path does not
 * apply (borderline pairs, or a threshold without finite support): use the CSR path + gp_bcsr_count / fill for this matrix.
 * fill: after gp_scan_counts(nblk) -> bptr and allocation of bidx (total), bvals [, bdvals] (16 * total doubles). */
int gp_matern_blocks_count(const double* points, int64_t n, int64_t d, const double* scale_host, double nu, double tau, void* ws,
                           const int* order_dev, const int* inv_order_dev, int64_t row_first, int64_t row_last, int* nblk_dev,
                           int64_t* stats_host, void* stream);
int gp_matern_blocks_fill(const double* points, int64_t n, int64_t d, const double* scale_host, double nu, double tau, void* ws,
                          const int* order_dev, const int* inv_order_dev, int64_t row_first, int64_t row_last,
                          const int64_t* bptr_dev, int* bidx_dev, double* bvals_dev, double* bdvals_dev, void* stream);
/* Per-dimension derivative streams of a built row-blocked operator (either build path): for the operator rows
 * [row_first, row_first + rows) (row_first a multiple of 16) with blocks bptr / bidx (operator positions, not slab-encoded) /
 * bvals of nblocks block-columns, writes d streams of 16 * nblocks doubles, stream k at dvals_dev + 16 * nblocks * k:
 * dK/d scale[k] in the fragment order of bvals, zero wherever bvals is zero. Operator row r is point order_dev[r]; points is
 * the device (n x d) array. dK/d scale[k] = g(x) u_k^2 / (x^2 scale[k]) with u_k = Delta_k / scale[k], x = ||u||,
 * g(x) = -x K'(x); 0 at x = 0 (as gp_loglik_dense_dscale). The scale may be anisotropic (never -4); -1 for a null pointer,
 * d outside [1, 8] or a row_first that is not a multiple of 16. */
int gp_bcsr_dscale_fill(const int64_t* bptr_dev, const int* bidx_dev, const double* bvals_dev, int64_t nblocks, int64_t row_first,
                        int64_t rows, const int* order_dev, const double* points, int64_t n, int64_t d, const double* scale_host,
                        double nu, double* dvals_dev, void* stream);

/* ---- row-slab sparse operator on several GPUs (csrc/gp_peer.cu, gp_sparse_la.cu) ------------------------------------------
 * One process per GPU. The reference evaluates one sparse likelihood on one host (imate SLQ + scipy CG over the whole matrix,
 * gaussian_proc/_mixed_correlation/mixed_correlation.py:193-209, 263-299); here the rows of the (spatially ordered) operator
 * are cut into contiguous slabs, one per GPU. Each rank allocates an ARENA (mailboxes + 3 exchange vectors), exports it as a
 * CUDA IPC handle (gp_peer_handle), receives the handles of its peers through the caller's process group and maps them
 * (gp_peer_connect). Kernels then gather halo rows of the Krylov vectors straight from the owner's arena over NVLink and sum
 * the Lanczos / CG reductions by pushing partial sums into every rank's mailbox - no library collective on the path. */
int64_t gp_peer_handle_bytes(void);
void* gp_peer_create(int64_t rank, int64_t world, int64_t nloc_max);      /* world <= 8; NULL on failure */
int gp_peer_handle(void* peer, unsigned char* handle_out);
int gp_peer_connect(void* peer, const unsigned char* handles);            /* world x gp_peer_handle_bytes(), rank-major */
int gp_peer_destroy(void* peer);
double* gp_peer_vec(void* peer, int64_t k);                               /* this rank's exchange vector k (0..2) */
int gp_peer_barrier(void* peer, void* stream);                            /* cross-GPU barrier in stream order */
int gp_peer_allreduce(void* peer, double* values_dev, int64_t count, void* stream);   /* count <= 256, in place, rank order */
int gp_peer_error(void* peer, void* stream);                              /* 1: a wait timed out (ranks diverged) */
/* bidx: global operator-space column (< n) -> (owner << 28 | row within the owner's slab) for uniform slabs of `slab` rows.
 * halo_host (optional, 2 entries, needs ws >= 16 + 4 * ceil(n / 32) bytes): [0] block-columns owned by another rank (rows
 * gathered over NVLink per SpMM), [1] distinct remote rows among them (what a bulk halo exchange would move) */
int gp_slab_encode_columns(int* bidx, int64_t total, int64_t slab, int64_t rank, int64_t n, int64_t* halo_host, void* ws,
                           void* stream);
/* The row-blocked drivers take this rank's arena as `peer` (gp_bcsr_spmm, gp_col_dot, gp_bcsr_lanczos, gp_bcsr_cg_solve). */

/* ---- index plumbing of the sparse operator build (csrc/gp_index.cu): own kernels instead of library sort / scan ------ */
/* out_host[0..d) = column minima, out_host[d..2d) = column maxima of the device points; ws >= (148 * d * 2 + 2 * d) doubles;
 * synchronises the stream */
int gp_points_bbox(const double* points, int64_t n, int64_t d, double* out_host, void* ws, void* stream);
/* stable LSD radix sort: order_out[i] = index of the i-th smallest key; keys_dev (low key_bits bits significant) is used as
 * scratch. ws: gp_sort_workspace_bytes(n). Replaces the stable sort of the spatial keys (a CSR from the reference's generator,
 * _generate_sparse_correlation.pyx:472-594, has no spatial order; this is the operator-internal permutation). */
int64_t gp_sort_workspace_bytes(int64_t n);
int gp_sort_keys_u64(unsigned long long* keys_dev, int64_t n, int key_bits, int* order_out, void* ws, void* stream);
int gp_inverse_permutation(const int* order, int64_t n, int* inv, void* stream);
/* offsets[0] = 0, offsets[i + 1] = counts[0] + ... + counts[i] */
int gp_scan_counts(const int* counts, int64_t n, int64_t* offsets, void* stream);
int gp_scan_counts_i32(const int* counts, int64_t n, int* offsets, void* stream);     /* 32-bit offsets (CSR row pointers) */
/* out[i][:] = in[map[i]][:] for rows of B doubles (in != out) */
int gp_gather_rows(const double* in, const int* map, int64_t n, int64_t B, double* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Symmetric eigenvalue path (imate_method = 'eigenvalue', the reference's default: _likelihood/likelihood.py:41,
 * _mixed_correlation/mixed_correlation.py:76-79 -> scipy.linalg.eigh(K, eigvals_only=True); :127-136,172-181,239-248 reduce
 * over lam + eta). csrc/gp_eig.cu.
 * ------------------------------------------------------------------------------------------------------- */
/* K = Q T Q^T. A (n x n, lda even, BOTH triangles valid) is overwritten: row k right of the diagonal keeps Householder
 * vector k (v[k+1] = 1). d (n), e (n; n-1 used), tau (n) on the device. ws: gp_sytrd_workspace_bytes(n). */
int64_t gp_sytrd_workspace_bytes(int64_t n);
int gp_sytrd_f64(double* A, int64_t n, int64_t lda, double* d, double* e, double* tau, void* ws, void* stream);
/* all eigenvalues (ascending) of the tridiagonal (d, e) by bisection; ws: (n + 8) doubles; synchronises the stream once */
int gp_stebz_f64(const double* d, const double* e, int64_t n, double* lam, void* ws, void* stream);
/* R (n x p, p <= 16) <- Q^T R (trans != 0) or Q R (trans == 0), Q from gp_sytrd_f64 */
int gp_ormtr_skinny(const double* A, int64_t n, int64_t lda, const double* tau, int trans, double* R, int64_t p, int64_t ldr,
                    void* stream);
/* Y <- (T + eta I)^-1 B (n x p); out (device, 2): log det (T + eta I), number of non-positive pivots; ws: n doubles */
int gp_tridiag_solve(const double* d, const double* e, int64_t n, double eta, const double* B, int64_t p, int64_t ldb, double* Y,
                     int64_t ldy, void* ws, double* out, void* stream);
/* out (device, 4): sum log(lam + eta), sum (lam + eta)^-1, sum (lam + eta)^-2, count of lam + eta <= 0 */
int gp_eig_reduce(const double* lam, int64_t n, double eta, double* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Fused log-likelihood (+ gradient ingredients) evaluation at one (rho, eta)
 * (reference: _likelihood/_direct_likelihood.py:31-157 log_likelihood + log_likelihood_jacobian,
 *  _likelihood/_profile_likelihood.py:38-132 log_likelihood + log_likelihood_der1_eta; the d/drho terms are the
 *  extension named in BASELINE.json's north_star, SURVEY 8a A9/A10).
 *
 * Inputs : K (padded, read-only), R = [X z] (npad x p row-major, rows >= n zero, p = m + 1 <= 16), eta.
 * Work   : A, W (npad x npad scratch each; W may be NULL when flags & 3 == 0), potrf_ws, ws.
 * flags  : bit0 (1) tr Kn^-1 via ||inv(L)||_F^2       (enough for d/d eta)
 *          bit1 (2) full inverse: tr Kn^-1, tr Kn^-2  (needed for d/d rho and the Hessian traces)
 *          bit2 (4) d/d rho reductions, needs bit1 and points/d/scale_host/nu (dK/drho is re-evaluated on the fly; -8
 *                   otherwise); without it points, d, scale_host and nu are not read
 *          bit3 (8) third moments T3 = R^T Kn^-3 R from one more skinny solve batch (Hessian _direct_likelihood.py:163-270,
 *                   second eta-derivative _profile_likelihood.py:138-192); needs bit0 or bit1 (-9 otherwise)
 * Output : out (DEVICE, gp_loglik_out_len(p) doubles):
 *          out[0] logdet(K + eta I)   out[1] tr Kn^-1   out[2] tr Kn^-2   out[3] tr(Kn^-1 dK/drho)
 *          out[4] potrf info (0 = ok) out[5..7] reserved
 *          out[8 ..]            G = R^T Kn^-1 R        (p x p)
 *          out[8 + p^2 ..]      H = R^T Kn^-2 R        (p x p)
 *          out[8 + 2 p^2 ..]    Q = (Kn^-1 R)^T dK/drho (Kn^-1 R)   (p x p; zero unless bit2)
 *          out[8 + 3 p^2 ..]    T3 = R^T Kn^-3 R       (p x p; zero unless bit3)
 * The remaining (m+1)x(m+1) algebra is host-side (gaussian_proc/_likelihood/_fused.py).
 * ------------------------------------------------------------------------------------------------------- */
int64_t gp_loglik_workspace_bytes(int64_t npad);
int64_t gp_loglik_out_len(int64_t p);
int gp_loglik_dense(const double* K, int64_t n, int64_t npad, const double* R, int64_t p, double eta, int flags,
                    const double* points, int64_t d, const double* scale_host, double nu, double* A, double* W,
                    void* potrf_ws, void* ws, double* out, void* stream);
/* Anisotropic gradient (one correlation scale per dimension, generate_correlation/_kernels.pyx:107-136): called after
 * gp_loglik_dense(flags & 2) with the same A (= Kn^-1, lower) and ws. out_dim (DEVICE, 1 + p^2 doubles):
 * out_dim[0] = tr(Kn^-1 dK/d scale[dim]), out_dim[1..] = S^T (dK/d scale[dim]) S. */
int gp_loglik_dense_dscale(const double* Ainv, int64_t n, int64_t npad, int64_t p, const double* points, int64_t d,
                           const double* scale_host, double nu, int64_t dim, void* ws, double* out_dim, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Kriging at new points (gaussian_proc/_predict.py; the reference has no prediction). For mc test points with
 * cross block P = gp_matern_cross_points(training points, test points) and the factor of Kn = K + eta I:
 *   V = W P                      (V: npad x mcpad, ldv; W = inv(L) from gp_trtri_f64, identity padding)
 *   out[j*(p+1) + c] = P[:, j]^T S[:, c]  for c < p,    out[j*(p+1) + p] = ||V[:, j]||^2      (j < mc)
 * S = Kn^-1 [X z] (npad x p, ld = p, rows >= n zero; gp_potrs_f64), p = m + 1 <= 16. mcpad = ceil(mc / 128) * 128; P and V
 * have ld >= mcpad (even) and P's columns mc .. mcpad zero, as gp_matern_cross_points leaves them. A column's results do
 * not depend on mc (fixed-order reduction over 2048-row chunks). ws: gp_predict_workspace_bytes(npad, mc, p) bytes
 * (-1 for invalid sizes). No host synchronisation. The host turns out[] into mean and variance; the covariance is
 * K** - V^T V plus a rank-m term, two more gp_dgemm_f64 calls.
 * ------------------------------------------------------------------------------------------------------- */
int64_t gp_predict_workspace_bytes(int64_t npad, int64_t mc, int64_t p);
int gp_predict_dense(const double* W, int64_t n, int64_t npad, const double* S, int64_t p, const double* P, int64_t mc,
                     int64_t ldp, double* V, int64_t ldv, double* out, void* ws, void* stream);
/* Gradients of the kriging mean and variance with respect to the test-point coordinates. With
 * G_k[i][j] = dP[i][j]/dq_jk = h(x) (p_ik - q_jk) / scale_k^2, x = ||(p_i - q_j) / scale||, h(x) = -matern'(x) / x,
 * regenerated from the n training points (n, d) and the mc test points q (mc, d) and never stored:
 *   out[(j*d + k)*(p+1) + c] = G_k[:, j]^T S[:, c]  for c < p,    out[(j*d + k)*(p+1) + p] = G_k[:, j]^T U[:, j]
 * (0 when U == NULL: mean gradients only). S as for gp_predict_dense (ld = p); U: n x mc (ld ldu >= mc), normally
 * Kn^-1 P = W^T V, one gp_dgemm_ktab_f64(1, 1, ...) with kbeg_tab[t] = 128 t. Rows i >= n of S and U and columns j >= mc of
 * U are never read. A pair at distance exactly 0 contributes exactly 0: the true derivative for nu > 1/2, the symmetric
 * derivative for nu = 1/2, where the correlation has a kink. scale_host, nu and d <= 8 as gp_matern_cross_points,
 * p <= 16. A column's results do not depend on mc (fixed-order reduction over 2048-row chunks).
 * ws: gp_predict_grad_workspace_bytes(n, mc, d, p) bytes (-1 for invalid sizes). No host synchronisation. */
int64_t gp_predict_grad_workspace_bytes(int64_t n, int64_t mc, int64_t d, int64_t p);
int gp_predict_grad_dense(const double* points, int64_t n, const double* q, int64_t mc, int64_t d, const double* scale_host,
                          double nu, const double* S, int64_t p, const double* U, int64_t ldu, double* out, void* ws,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPGP_H */
