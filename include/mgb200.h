/*
 * mgb200.h -- C ABI of libmgb200.so, the B200 (sm_100a) multigrid V-cycle engine.
 *
 * The reference (claudiotomasi/LearnMultigrid) is pure Python; its "FFI" for the hot path is the set of
 * native kernels it reaches through SciPy sparsetools, PyAMG amg_core and SuperLU from
 * learn_multigrid/solvers/Multigrid.py.  Every entry point below names the reference call site it
 * replaces.  Conventions:
 *   - all pointers named d_* are DEVICE pointers (fp64 values, int32 column indices, int64 slice offsets);
 *     h_* are HOST pointers; no torch types anywhere;
 *   - every function returns 0 on success, a negative mg_status otherwise, never throws; the text of the
 *     last failure on the calling thread is returned by mg_last_error();
 *   - nothing allocates device memory: outputs and workspaces are passed in (sizes from the *_size calls);
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued, not synchronised, unless stated.
 */
#ifndef MGB200_H
#define MGB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    MG_OK = 0,
    MG_ERR_INVALID = -1,   /* bad argument                                  */
    MG_ERR_CUDA = -2,      /* a CUDA runtime call or launch failed          */
    MG_ERR_UNSUPPORTED = -3,
    MG_ERR_OVERFLOW = -4,  /* an index would not fit the int32 contract     */
    MG_ERR_SINGULAR = -5   /* zero pivot in the coarsest-level inversion    */
} mg_status;

/* ------------------------------------------------------------------------------------------------ */
/* library                                                                                          */
int mg_version(void);
const char *mg_last_error(void);
/* sizeof of the ABI structs as compiled (0 mg_sell, 1 mg_level, 2 mg_cycle_params, 3 mg_bcr, 4 mg_comm, 5 mg_xfer,
 * 6 mg_dist_level, 7 mg_bcr_dist, 8 mg_dist_norm, 9 mg_gmres): lets a binding verify its own layout */
int64_t mg_struct_size(int which);
/* 1 (default): the kernels of the cycle are launched with programmatic stream serialization (each kernel waits for
 * its predecessor with griddepcontrol.wait and lets its successor be scheduled early); 0: plain stream order.
 * Affects launches (and graph captures) made afterwards; returns the previous setting.  Results are identical. */
int mg_set_pdl(int enabled);
/* fills sm_count / total global memory (bytes) / compute capability (e.g. 100) of the current device */
int mg_device_info(int *sm_count, int64_t *global_mem, int *cc);

/* ------------------------------------------------------------------------------------------------ */
/* CSR kernels (natural ordering).  CSR = (d_indptr[n+1], d_indices[nnz], d_values[nnz]).           */

/* y = A x.   Replaces SciPy csr_matvec / csc_matvec:  Multigrid.py:62,90 (A.dot), :93 (i.T @ res, pass the
 * CSR of Q^T), :115 (i @ u_coarse).  Row sums are accumulated in storage order with separate multiply and
 * add (no FMA) so results are bit-identical to SciPy's. */
int mg_spmv_csr(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                const double *d_x, double *d_y, void *stream);
/* r = b - A x.   Multigrid.py:62 and :90 (rhs - A.dot(u)). */
int mg_residual_csr(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                    const double *d_x, const double *d_b, double *d_r, void *stream);
/* x_out = x + omega * (dinv * (b - A x)), out of place.  omega = 1 is Jacobi.py:35
 * (self.solution += inv_d * self.residual_vector); the damped form is the smoother the commented dispatch at
 * Multigrid.py:85-86,119-120 would call. */
int mg_jacobi_sweep_csr(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                        const double *d_dinv, const double *d_x, const double *d_b, double *d_x_out,
                        double omega, void *stream);
/* One multicolour Gauss-Seidel sweep, in place: for c in 0..ncolors-1, for every row i in
 * d_color_rows[h_color_ptr[c] .. h_color_ptr[c+1]):  x_i = (b_i - sum_{j != i} A_ij x_j) / A_ii  (rows with a
 * zero diagonal are skipped).  Per-row arithmetic is PyAMG amg_core::gauss_seidel's (call sites
 * Multigrid.py:88,121); the row ORDER is the colour order instead of the index order. */
int mg_gs_multicolor_sweep_csr(int64_t n, const int32_t *d_indptr, const int32_t *d_indices,
                               const double *d_values, double *d_x, const double *d_b,
                               const int64_t *h_color_ptr, const int32_t *d_color_rows, int ncolors,
                               void *stream);
/* Exact lexicographic (index-order) Gauss-Seidel = PyAMG gauss_seidel(A, x, b, iterations, 'forward'),
 * Multigrid.py:88,121, parallelised by dependency levels: rows of d_level_rows[h_level_ptr[l]..h_level_ptr[l+1])
 * only depend on rows of earlier levels.  `iterations` full sweeps.  Bit-identical to the serial kernel. */
int mg_gs_lex_sweep_csr(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                        double *d_x, const double *d_b, const int64_t *d_level_ptr,
                        const int32_t *d_level_rows, int64_t nlevels, int iterations, void *stream);
/* u = u + Q e.   Multigrid.py:115 (u + i @ u_coarse): t = Q e from zero in storage order, then u + t. */
int mg_prolong_correct_csr(int64_t n, const int32_t *d_indptr, const int32_t *d_indices,
                           const double *d_values, const double *d_e, double *d_u, void *stream);

/* ------------------------------------------------------------------------------------------------ */
/* SELL-32 kernels (the hot-path format).  A matrix is stored in slices of 32 consecutive rows; slice s
 * holds len_s = (slice_ptr[s+1]-slice_ptr[s])/32 entries per row, column-major inside the slice:
 * entry k of row r sits at slice_ptr[r/32] + 32*k + r%32.  Entries keep their CSR order; padding entries
 * have value 0.0 and any valid column (the builder repeats the row's last column), so they add an exact
 * zero to every row sum and are ignored by the diagonal detection of the Gauss-Seidel kernel.  The builder pads
 * all slices to the longest one ("uniform") when that costs <= 3 % extra entries (structured grids), or <= 25 % for rows of one or two entries (linear transfer operators).      */
typedef struct {
    int64_t nrows;
    int64_t ncols;
    int64_t nslices;            /* ceil(nrows/32)                                  */
    const int64_t *d_slice_ptr; /* [nslices+1], entry offsets (multiples of 32)    */
    const int32_t *d_cols;
    const double *d_vals;
    int64_t max_slice_len;      /* longest slice (entries per row); 0 = unknown (generic kernel)           */
    int64_t uniform_len;        /* > 0: EVERY slice has exactly this many entries per row (= max_slice_len), so
                                   slice offsets are computed, not loaded; 0 = lengths vary, use d_slice_ptr */
    /* optional implied columns (NULL: none): d_slice_rec[s] = id of the offset record of slice s -- every one of its 32
     * rows has the columns row + d_rec_table[8 * id + j] -- or 0xffff for a slice that is not regular (a boundary node
     * among its rows, the ragged tail: the kernels then read its column indices).  Built from mg_sell_slice_offsets by
     * deduplicating the records (structured levels have a handful; at most 65534).  h_spec_*: optional host-side hints, for launches
     * over the rows [h_spec_row[k], h_spec_row[k+1]) the record most of those slices use is h_spec_rec[9 * k] (its id)
     * with the offsets h_spec_rec[9 * k + 1 .. 9 * k + 8]; the launch passes it by value and the kernel gathers with
     * it BEFORE the slice's id has arrived (n_spec = 0: record 0, the most frequent one, is assumed).
     * nrec < 0: the same fields hold -nrec SLICE PATTERNS instead (transfer operators, whose columns live in another
     * level's numbering; L = uniform_len <= 8): entry j of lane l of a slice s with id r has the column base[s] +
     * d_rec_table[(r * L + j) * 32 + l] and the value d_rec_vals[(r * L + j) * 32 + l]; base[s] = the slice's first
     * stored column (entry 0 of lane 0) = d_rec_table[-nrec * L * 32 + s].  h_spec_rec[9 * k] is the pattern most slices
     * of block k use, h_spec_rec[9 * k + 1] how many of them do in per mille (the other 7 ints unused), h_spec_vals
     * unused. */
    const uint16_t *d_slice_rec;
    const int32_t *d_rec_table;
    int32_t nrec, n_spec;
    const int64_t *h_spec_row;
    const int32_t *h_spec_rec;
    /* optional value dictionary (NULL: none; mg_value_dict_build on d_vals): d_vals[p] == d_val_table[d_val_idx[p]] for
     * every stored entry p, at most 256 table entries.  Kernels on rows of at most 8 entries then stream one byte per
     * entry instead of eight (mg_set_value_dict); the doubles are the same, so are the results. */
    const unsigned char *d_val_idx;
    const double *d_val_table;
    /* optional implied values (NULL: none; needs the two above): the 32 rows of every slice with a record id also hold
     * the same VALUE per entry, d_rec_vals[8 * id + j] -- on a constant-coefficient stencil level the record stands for
     * the whole slice of the matrix, and a slice that is regular in its columns but not in its values carries 0xffff.
     * h_spec_vals[8 * k + j]: the values of the record h_spec_rec[9 * k], passed by value like its offsets. */
    const double *d_rec_vals;
    const double *h_spec_vals;
} mg_sell;

/* Implied columns (default on; results identical): on a uniform matrix with <= 8 entries per row, slices whose
 * 32 rows all have the columns row + off[j] (structured stencil levels: all slices but those holding a boundary node)
 * read 4 bytes of offset per entry index instead of 128 bytes of column indices, and the x gathers of a warp become
 * contiguous 256-byte reads.  mg_sell_slice_offsets fills d_off[nslices * 8] (one 32-byte record per slice, entries
 * beyond uniform_len zero; irregular slices: d_off[s * 8] = INT32_MIN) -- the raw material of mg_sell.d_slice_rec /
 * d_rec_table -- and adds the number of regular slices to *d_nregular (device int64, zeroed by the
 * caller; may be NULL). */
int mg_sell_slice_offsets(const mg_sell *A, int32_t *d_off, int64_t *d_nregular, void *stream);
/* Value dictionary (csrc/valdict.cu): finite-element operators on uniform meshes and interpolation operators hold few
 * DISTINCT values (5-point Laplacian: 4, -1, 1, 0; linear interpolation: 1, 0.5, 0).  mg_value_dict_build looks for at
 * most 256 distinct bit patterns among d_vals[0..n): *h_count = how many (d_table[0..count) and d_index[0..n) are
 * written), or -1 if there are more (nothing is written; found after a few thousand entries).  d_work:
 * mg_value_dict_workspace() bytes.  Synchronises.  mg_set_value_dict(0) makes the kernels ignore dictionaries
 * (default 1); returns the previous setting. */
int64_t mg_value_dict_workspace(void);
int mg_value_dict_build(int64_t n, const double *d_vals, unsigned char *d_index, double *d_table, void *d_work,
                        int *h_count, void *stream);
int mg_set_value_dict(int enabled);
/* Implied values (default 1; results identical): launches over matrices that carry value records (mg_sell.d_rec_vals)
 * read nothing per row of a regular slice but the vectors; 0: they read the dictionary bytes.  Returns the previous
 * setting. */
int mg_set_implied_values(int enabled);
int mg_set_implied_columns(int enabled);
/* Implied transfer columns (default 1; results identical): SpMV (restriction) and prolongation launches over matrices
 * that carry slice patterns (mg_sell.nrec < 0) read a record id and a base column per slice instead of the columns and
 * values of its rows (launches of at least mg_set_implied_min_rows rows).  Returns the previous setting; a negative
 * argument only returns it. */
int mg_set_implied_transfers(int enabled);
/* launches of fewer rows keep loading their columns (one dependent load less on latency-bound launches); returns the
 * previous floor (default 2^19) */
int64_t mg_set_implied_min_rows(int64_t rows);
/* y = A x */
int mg_sell_spmv(const mg_sell *A, const double *d_x, double *d_y, void *stream);
/* r = b - A x; _rows: only the rows [row0,row1) of r are written */
int mg_sell_residual(const mg_sell *A, const double *d_x, const double *d_b, double *d_r, void *stream);
int mg_sell_residual_rows(const mg_sell *A, const double *d_x, const double *d_b, double *d_r, int64_t row0,
                          int64_t row1, void *stream);
/* fused: *d_norm2 = sum_i (b - A x)_i^2 without storing r (outer loop Multigrid.py:62-63); d_partials is a
 * workspace of mg_norm_workspace_size(nrows) = ceil(nrows/32)+66 doubles (the worst case over the kernel variants: one
 * partial per CTA, the warps-per-slice kernel has one CTA per slice, and mg_vcycle_norm writes two runs of partials);
 * deterministic two-stage reduction. */
int mg_sell_residual_norm2(const mg_sell *A, const double *d_x, const double *d_b, double *d_partials,
                           double *d_norm2, void *stream);
int64_t mg_norm_workspace_size(int64_t n);
/* launches that cover at least `rows` rows use the bulk-async (TMA) staged kernel; 0 = never.  Returns the
 * previous threshold (default 0 = off).  Both kernels give bit-identical results. */
int64_t mg_set_tma_min_rows(int64_t rows);
/* matrices whose longest slice has at least `len` entries per row (and at most 64) run the warps-per-slice
 * kernel: loads of a row spread over four or eight warps, products added in storage order (same bits); 0 = never.  Returns
 * the previous threshold (default 9: the 19- and 37-point Galerkin stencils of quasi-L2 transfers). */
int64_t mg_set_wide_min_len(int64_t len);
/* SpMV / prolongation with matrices of at most two entries per row (linear transfer operators): launches of at least
 * mg_set_short_min_rows rows (default 2^18) take r in {1, 2, 4} rows per thread (default 2; 1 = the ordinary kernel), all
 * loads of a stage issued for all of them first.  Same bits.  Both return the previous value. */
int mg_set_short_rows_per_thread(int r);
int64_t mg_set_short_min_rows(int64_t rows);
/* ... and only for launches of at most `rows` rows (default 2^18): larger launches keep enough rows in flight for the
 * thread-per-row kernel, which then streams at the DRAM limit.  Returns the previous value. */
int64_t mg_set_wide_max_rows(int64_t rows);
/* x_out = x + omega*(dinv*(b - A x)) */
int mg_sell_jacobi(const mg_sell *A, const double *d_dinv, const double *d_x, const double *d_b,
                   double *d_x_out, double omega, void *stream);
/* One step of the Chebyshev smoother (all rows): t = dinv*(b - A x) with the residual in storage order,
 * dn = c_r*t (first != 0: step 0, d only written) or dn = (c_d*d) + (c_r*t) (first == 0, c_d != 0), then
 * x_out = x + dn and d = dn (in place); every product and sum rounded on its own.  x_out must not alias x. */
int mg_sell_chebyshev(const mg_sell *A, const double *d_dinv, const double *d_x, const double *d_b, double *d_d,
                      double *d_x_out, double c_d, double c_r, int first, void *stream);
/* Step 0 of the Chebyshev smoother on a zero iterate without the matrix: d = c_r*(dinv*b), x_out = 0 + d over n
 * entries -- the bits of mg_sell_chebyshev(first = 1) with x = 0. */
int mg_chebyshev_zero_first(int64_t n, double c_r, const double *d_dinv, const double *d_b, double *d_d,
                            double *d_x_out, void *stream);
/* Gauss-Seidel update of the rows [row0,row1) in place (one colour of a colour-blocked ordering). */
int mg_sell_gs_rows(const mg_sell *A, double *d_x, const double *d_b, int64_t row0, int64_t row1,
                    void *stream);
/* The same sweep, which also leaves what the NEXT operation of a V-cycle needs from these rows, computed from the
 * registers that still hold each row (no second pass over the matrix): tail = 1: d_r[i] = (b - A x)_i with the new
 * x_i, for i in [row0,row1); tail = 2: per-CTA partial sums of (b - A x)_i^2 over these rows in d_partials,
 * *h_nblocks of them; tail = 0: mg_sell_gs_rows.  Exact (the bits of a residual pass after the sweep) when no row of
 * the range has a non-zero entry in the column of another row of the range -- a proper colouring.  Available for
 * rows of at most 8 entries, or launches the warps-per-slice kernel takes: mg_sell_gs_tail_ok. */
int mg_sell_gs_rows_tail(const mg_sell *A, double *d_x, const double *d_b, int64_t row0, int64_t row1, int tail,
                         double *d_r, double *d_partials, int *h_nblocks, void *stream);
int mg_sell_gs_tail_ok(const mg_sell *A, int64_t row0, int64_t row1);
/* First colour sweep on a zero iterate without the matrix: x[0..n_vec) = 0 except x_i = b_i / d_diag[i] for i in
 * [row0,row1) with d_diag[i] != 0 -- the bits of mg_fill(0) followed by mg_sell_gs_rows(row0,row1). */
int mg_sell_gs_zero_first(int64_t n_vec, int64_t row0, int64_t row1, const double *d_diag, const double *d_b,
                          double *d_x, void *stream);
/* u_out = u + Q e  (u_out may alias u); _rows: only the rows [row0,row1) */
int mg_sell_prolong_correct(const mg_sell *Q, const double *d_e, const double *d_u, double *d_u_out,
                            void *stream);
int mg_sell_prolong_correct_rows(const mg_sell *Q, const double *d_e, const double *d_u, double *d_u_out, int64_t row0,
                                 int64_t row1, void *stream);

/* ------------------------------------------------------------------------------------------------ */
/* vector kernels (Multigrid.py:63 np.linalg.norm; CG.py:30-48 dots and updates)                     */
int mg_dot(int64_t n, const double *d_x, const double *d_y, double *d_partials, double *d_out, void *stream);
int mg_axpby(int64_t n, double a, const double *d_x, double b, const double *d_y, double *d_out, void *stream);
int mg_fill(int64_t n, double value, double *d_x, void *stream);
/* out[i] = in[idx[i]] (permute into a level's ordering) and out[idx[i]] = in[i] (back) */
int mg_gather(int64_t n, const int32_t *d_idx, const double *d_in, double *d_out, void *stream);
int mg_scatter(int64_t n, const int32_t *d_idx, const double *d_in, double *d_out, void *stream);

/* ------------------------------------------------------------------------------------------------ */
/* coarsest level: dense direct solve.  Replaces spsolve(A_coarse, res_coarse) (SuperLU), Multigrid.py:106,
 * which the reference refactorises in every cycle; here the inverse is formed once.                 */
/* in: d_a row-major n x n (destroyed); out: d_ainv row-major n x n.  d_work: mg_dense_inverse_workspace(n)
 * bytes.  Gauss-Jordan with partial pivoting, cooperative multi-CTA.  Synchronises the stream. */
int mg_dense_inverse(int64_t n, double *d_a, double *d_ainv, void *d_work, void *stream);
int64_t mg_dense_inverse_workspace(int64_t n);
/* y = M x for a dense row-major n x m matrix (the coarse solve u = A^-1 r) */
int mg_dense_gemv(int64_t n, int64_t m, const double *d_m, const double *d_x, double *d_y, void *stream);
/* Banded coarsest operators too large for an explicit inverse: block cyclic reduction with dense m x m blocks
 * (m >= half bandwidth).  The host side forms all factors once with the three setup entry points below and
 * fills an mg_bcr; mg_bcr_solve (also reached from mg_vcycle through mg_level.coarse_bcr) then performs
 * x = A^-1 rhs in 2*nlevels+3 launches that stream the factors once.  Level s has na[s] active blocks;
 * block position p of level s is original block p << s; odd positions are eliminated.  The reduction stops when
 * tail_na blocks are left; that small block-tridiagonal system is solved through its dense inverse (one launch
 * instead of a chain of latency-bound ones). */
typedef struct {
    int64_t n, n_pad, m, nb;      /* unknowns, padded unknowns (nb*m), block size, number of blocks          */
    int32_t nlevels, pad_;
    const double *d_GL[32], *d_GU[32];   /* per level: [ceil(na/2)][m][m]  f_p -= GL f_{p-1} + GU f_{p+1}     */
    const double *d_Dinv[32], *d_HL[32], *d_HU[32]; /* per level: [na/2][m][m]  x_p = Dinv f_p - HL x_{p-1} - HU x_{p+1} */
    int64_t na[32];
    const double *d_last_inv;     /* dense inverse of what is left after nlevels reductions: (tail_na*m)^2     */
    double *d_f, *d_x;            /* work vectors, n_pad doubles each                                          */
    int64_t tail_na;              /* blocks left after the reductions (<= 1: a single block)                   */
    double *d_tail;               /* work vector, max(tail_na,1)*m doubles                                     */
    const int32_t *d_perm;        /* optional (NULL: identity): the factors are those of P A P^T, row i of which is row
                                     d_perm[i] of A (a bandwidth-reducing ordering); the solve gathers rhs and
                                     scatters x accordingly                                                    */
} mg_bcr;
int mg_bcr_blocks_from_csr(int64_t n, int64_t n_pad, int64_t m, const int32_t *d_indptr, const int32_t *d_indices,
                           const double *d_values, double *d_D, double *d_L, double *d_U, int32_t *d_bad,
                           void *stream);
/* batch of dense inverses, one CTA per matrix (Gauss-Jordan, partial pivoting); d_work: batch*m*2m doubles */
int mg_dense_inverse_batched(int64_t m, int64_t batch, const double *d_a, int64_t stride_a, double *d_out,
                             int64_t stride_out, double *d_work, int32_t *d_singular, void *stream);
/* C[b] = alpha*A[b]*B[b] + beta*C[b], m x m row-major, strides in elements */
int mg_dense_gemm_batched(int64_t m, int64_t batch, const double *d_a, int64_t stride_a, const double *d_b,
                          int64_t stride_b, double *d_c, int64_t stride_c, double alpha, double beta, void *stream);
int mg_bcr_solve(const mg_bcr *bcr, const double *d_rhs, double *d_x, void *stream);
/* scatter a CSR matrix into a zeroed dense row-major n x n buffer */
int mg_csr_to_dense(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                    double *d_dense, void *stream);

/* ------------------------------------------------------------------------------------------------ */
/* hierarchy setup on the device.  Galerkin coarse operators A_c = Q^T A Q replace `csr_matrix(i.T @ A @ i)`
 * (SciPy csr_matmat_maxnnz + csr_matmat twice + tocsr, Multigrid.py:97-98, repeated by the reference in every
 * cycle).  The two-pass SpGEMM accumulates every output entry in SciPy's order without FMA and drops exact
 * zeros, so values and sparsity patterns are bit-identical to SciPy's:  T = A^T Q,  C = Q^T T,  A_c = C^T. */
int64_t mg_scan_workspace_size(int64_t n);
/* d_out[0] = 0, d_out[i+1] = d_in[0..i] summed (int32 row pointer); *d_total (device int64) = total.
 * Synchronises; MG_ERR_OVERFLOW if the total does not fit int32. */
int mg_exclusive_scan_i32(int64_t n, const int32_t *d_in, int32_t *d_out, int64_t *d_total, void *d_temp,
                          int64_t temp_bytes, void *stream);
/* symbolic pass: d_row_count[i] = distinct columns of row i of A*B; group in {4,8,16,32} lanes per row;
 * per-row hash table of 2^log2_table slots in shared memory; *d_overflow = 1 if a table filled up. */
int mg_spgemm_symbolic(int64_t nrows, const int32_t *d_a_indptr, const int32_t *d_a_indices,
                       const int32_t *d_b_indptr, const int32_t *d_b_indices, int group, int log2_table,
                       int32_t *d_row_count, int32_t *d_overflow, void *stream);
/* numeric pass: sorted columns + values into [d_c_indptr[i], d_c_indptr[i+1]); d_row_nonzeros[i] = entries != 0 */
int mg_spgemm_numeric(int64_t nrows, const int32_t *d_a_indptr, const int32_t *d_a_indices, const double *d_a_values,
                      const int32_t *d_b_indptr, const int32_t *d_b_indices, const double *d_b_values, int group,
                      int log2_table, const int32_t *d_c_indptr, int32_t *d_c_indices, double *d_c_values,
                      int32_t *d_row_nonzeros, int32_t *d_overflow, void *stream);
/* prune exact zeros, keeping entry order (what SciPy's numeric pass does) */
int mg_csr_compact_nonzeros(int64_t nrows, const int32_t *d_in_indptr, const int32_t *d_in_indices,
                            const double *d_in_values, const int32_t *d_out_indptr, int32_t *d_out_indices,
                            double *d_out_values, void *stream);
int64_t mg_sort_workspace_size(int64_t n);
/* stable argsort of int32 keys (LSD radix sort on key_bits bits): d_perm_out[i] = position of the i-th key */
int mg_stable_argsort_i32(int64_t n, const int32_t *d_keys, int32_t *d_keys_sorted, int32_t *d_perm_out,
                          int32_t *d_iota_tmp, int key_bits, void *d_temp, int64_t temp_bytes, void *stream);
int64_t mg_csr_transpose_workspace(int64_t nnz);
/* CSR of A^T with row entries in ascending original-row order (the order SciPy's csc kernels add them in,
 * Multigrid.py:93 `i.T @ res`) */
int mg_csr_transpose(int64_t nrows, int64_t ncols, int64_t nnz, const int32_t *d_indptr, const int32_t *d_indices,
                     const double *d_values, int32_t *d_t_indptr, int32_t *d_t_indices, double *d_t_values,
                     void *d_work, void *stream);
int mg_invert_permutation(int64_t n, const int32_t *d_perm, int32_t *d_iperm, void *stream);
int mg_csr_row_lengths(int64_t n, const int32_t *d_indptr, const int32_t *d_perm, int32_t *d_lens, void *stream);
/* new row i = old row perm[i] (NULL = identity), column j -> col_iperm[j] (NULL = identity), entry order kept */
int mg_csr_permute(int64_t n, const int32_t *d_in_indptr, const int32_t *d_in_indices, const double *d_in_values,
                   const int32_t *d_perm, const int32_t *d_col_iperm, const int32_t *d_out_indptr,
                   int32_t *d_out_indices, double *d_out_values, void *stream);
/* SELL-32 build: layout (slice pointers, padded size returned on the host; synchronises) then fill */
int mg_sell_layout(int64_t n, const int32_t *d_indptr, int32_t *d_slice_len_tmp, int64_t *d_slice_ptr,
                   int64_t *h_total_out, int64_t *h_max_len_out, int64_t *h_uniform_len_out, void *d_temp,
                   int64_t temp_bytes, void *stream);
int mg_sell_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                 const int64_t *d_slice_ptr, int32_t *d_cols, double *d_vals, void *stream);
/* d_dinv[i] = 1 / A[perm[i], perm[i]] (Jacobi.py:22-23 inverts the diagonal) */
int mg_extract_dinv(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                    const int32_t *d_perm, double *d_dinv, void *stream);

/* ------------------------------------------------------------------------------------------------ */
/* multi-GPU: exchanges between the row blocks of a distributed level over peer-mapped memory (NVLink / NVSwitch).
 * No reference counterpart (the reference is single-process); the contract is SURVEY.md 8e.
 *
 * Every rank owns an ARENA (mg_comm_alloc, exported with CUDA IPC and mapped by its peers):
 *     [0]    u64 epoch | u32 error                                                   (header, 4096 bytes)
 *     [4096] u64 flags[world][max_sites]          flags[q][s]: handshake word of rank q for site s (empty messages)
 *     [...]  staging[world][2][region_bytes]      packets from rank q, double-buffered by epoch parity
 * A PROGRAM is the launch sequence between mg_comm_begin and mg_comm_end (e.g. one V-cycle; capturable in a CUDA
 * graph).  Every rank enqueues the same sequence of exchange SITES.  One fused kernel per site: gather the
 * outgoing values and store them straight into each peer's staging area as 16-byte packets (every double split into
 * two 8-byte words, each carrying 4 data bytes and the epoch as a tag), then poll the own staging area until the
 * peers' packets carry this program's tag and unpack them.  An aligned 8-byte store is atomic, so no fence and no
 * separate flag is needed: one NVLink traversal of latency per site.  Pushes never wait, so no ordering of the
 * ranks can deadlock; a wait longer than timeout_s sets the error word instead of hanging.
 * Peer sets must be symmetric at every site (zero-length messages are fine).  Every program contains at least one
 * site at which all pairs of ranks talk (mg_comm_end appends an empty one if none occurred): together with the parity
 * double-buffering this is what makes it safe for a rank to run ahead into the next program.
 * Several ranks inside ONE process (virtual ranks on one device, used by the tests): CUDA loads kernels lazily and a
 * first-time load can wait for the device to drain, which never happens while another rank's exchange kernel spins on
 * a message this thread has yet to launch.  Run every program once with dry_run = 1 (all kernels get loaded, exchanges
 * neither push nor wait, the epoch stands still) before the first real one. */
#define MG_MAX_RANKS 8
typedef struct {
    int32_t rank, world;
    int32_t max_sites, dry_run;        /* dry_run != 0: exchanges are launched as no-ops (kernel warm-up, below)  */
    int64_t region_bytes;              /* staging bytes per (sender, parity)                                     */
    void *d_arena[MG_MAX_RANKS];       /* every rank's arena as mapped into THIS process ([rank] = the own one)  */
    double timeout_s;                  /* <= 0: 10 s                                                             */
    /* running state of the program being enqueued (host side; reset by mg_comm_begin) */
    int32_t site, all_pairs;           /* all_pairs: an all-ranks site occurred (else mg_comm_end adds a fence)  */
    int64_t bump_send[MG_MAX_RANKS], bump_recv[MG_MAX_RANKS];
} mg_comm;
/* one exchange site: for peer k, send src[d_send_idx[k][i]] (NULL: src[send_off[k]+i]), i < send_cnt[k], and
 * receive recv_cnt[k] values into dst[d_recv_idx[k][i]] (NULL: dst[recv_off[k]+i]) */
typedef struct {
    int32_t npeers, pad_;
    int32_t peer[MG_MAX_RANKS];
    const int32_t *d_send_idx[MG_MAX_RANKS];
    int64_t send_off[MG_MAX_RANKS], send_cnt[MG_MAX_RANKS];
    const int32_t *d_recv_idx[MG_MAX_RANKS];
    int64_t recv_off[MG_MAX_RANKS], recv_cnt[MG_MAX_RANKS];
} mg_xfer;
int64_t mg_comm_arena_bytes(int32_t world, int32_t max_sites, int64_t region_bytes);
int mg_comm_alloc(int64_t bytes, void **d_ptr_out);          /* cudaMalloc'ed (IPC needs a whole allocation), zeroed */
int mg_comm_free(void *d_ptr);
int mg_comm_export(void *d_ptr, unsigned char *h_handle64);  /* 64-byte CUDA IPC handle                              */
int mg_comm_import(const unsigned char *h_handle64, void **d_peer_ptr_out);
int mg_comm_unmap(void *d_peer_ptr);
int mg_comm_init(mg_comm *comm, void *stream);               /* epoch = 1, error = 0 in the own arena                */
int mg_comm_begin(mg_comm *comm);
int mg_comm_exchange(mg_comm *comm, const mg_xfer *xfer, const double *d_src, double *d_dst, void *stream);
/* *d_out = sum over ranks of *d_value, added in rank order (identical bits on every rank); d_slots: world doubles */
int mg_comm_allreduce_sum(mg_comm *comm, const double *d_value, double *d_slots, double *d_out, void *stream);
/* d_out[i] = sum over ranks of d_values[i], i < k, added in rank order at ONE exchange site; d_slots: world * k doubles.
 * mg_comm_allreduce_sum is its k = 1 case. */
int mg_comm_allreduce_sum_n(mg_comm *comm, const double *d_values, int32_t k, double *d_slots, double *d_out,
                            void *stream);
int mg_comm_end(mg_comm *comm, void *stream);                /* epoch += 1                                           */
/* synchronises the stream; *h_error = 0, or 1 + the first site whose wait timed out */
int mg_comm_error(mg_comm *comm, int32_t *h_error, void *stream);
/* relabel the columns of a row block: c in [c0,c1) -> d_own_iperm[c-c0] (NULL: c-c0), else n_own + d_slot_of[c] */
int mg_csr_remap_cols(int64_t nnz, const int32_t *d_cols_in, int64_t c0, int64_t c1, const int32_t *d_own_iperm,
                      int64_t n_own, const int32_t *d_slot_of, int32_t *d_cols_out, int32_t *d_missing, void *stream);
/* Coarsest-level BCR solve with its large steps split over the ranks (the level itself is replicated): rank r
 * computes the block rows [j0,j1) of a reduction level / the rows [i0,i1) of the dense tail, then all ranks gather
 * what the others computed (xfer: an all-pairs site with index lists into the padded work vectors).  xfer == NULL:
 * the step runs replicated.  Same per-row arithmetic as the replicated solve, hence the same bits. */
typedef struct {
    int64_t fwd_j0[32], fwd_j1[32];
    const mg_xfer *fwd_xfer[32];
    int64_t bwd_j0[32], bwd_j1[32];
    const mg_xfer *bwd_xfer[32];
    int64_t tail_i0, tail_i1;
    const mg_xfer *tail_xfer;
} mg_bcr_dist;
int mg_bcr_solve_dist(mg_comm *comm, const mg_bcr *bcr, const mg_bcr_dist *dist, const double *d_rhs, double *d_x,
                      void *stream);
/* what a distributed level adds to mg_level (mg_level.dist): level vectors are laid out [owned rows | halo] */
typedef struct {
    int64_t n_halo;
    int32_t ncolors, pad_;
    const mg_xfer *xfer_color;          /* [ncolors] boundary values of one colour (multicolour Gauss-Seidel)       */
    const mg_xfer *xfer_all;            /* all boundary values                                                      */
    /* hand-off to the replicated coarse levels (set on the LAST distributed level only): the restriction writes the
     * owned block of the coarse right-hand side to d_gather_tmp, which is then gathered into every rank's full vector */
    const mg_xfer *xfer_gather;
    double *d_gather_tmp;
    const int32_t *d_gather_self_idx;   /* positions of the own block in the full coarse vector                     */
    int64_t n_gather_own;
    /* per slice of A / Q / Q^T: 1 if the slice reads halo columns (mg_sell_halo_mask).  With these, an exchange is not
     * launched on its own but rides on the next SELL kernel that reads the exchanged vector (mg_set_fused_exchange):
     * extra CTAs in front push / poll / unpack, the compute CTAs of masked slices wait for them, all others overlap
     * the exchange.  NULL: every slice waits. */
    const unsigned char *d_mask_A, *d_mask_Q, *d_mask_QT;
} mg_dist_level;
/* d_mask[s] = 1 if slice s of the SELL matrix holds a column >= first_halo_col */
int mg_sell_halo_mask(const mg_sell *A, int64_t first_halo_col, unsigned char *d_mask, void *stream);
/* 1 (default): in mg_vcycle_dist with multicolour Gauss-Seidel the halo exchanges ride on the following SELL kernel
 * (see mg_dist_level); 0: every exchange is a kernel of its own.  Same results.  Returns the previous setting. */
int mg_set_fused_exchange(int enabled);

/* ------------------------------------------------------------------------------------------------ */
/* P1 assembly on the device (csrc/assembly_kernels.cu).  Replaces the per-element Python loops of
 * MassMatrix.compute_mass_2d (MassMatrix.py:21-35), StiffnessMatrix.compute_stiffness_2d (StiffnessMatrix.py:21-36),
 * LoadVector.compute_rhs_2d (LoadVector.py:20-51) and the Dirichlet row replacement thesis_structured_2d.py:407-414. */
/* nine (row, col, value) contributions per element, element-major.  kind 0 mass: h_const = c[3][3]; kind 1 stiffness:
 * h_const = g[3][2], w[3], number of quadrature points (10 doubles); d_coef optional per-element coefficient */
int mg_assemble_p1_2d(int64_t ne, const double *d_points, const int32_t *d_conn, int kind, const double *h_const,
                      const double *d_coef, int32_t *d_rows, int32_t *d_cols, double *d_vals, void *stream);
int mg_assemble_load_p1_2d(int64_t ne, const double *d_points, const int32_t *d_conn, const double *h_c3,
                           int32_t *d_nodes, double *d_vals, void *stream);
/* sum the runs of equal (row, col) of contributions sorted stably by (row, col), in order (= element order, the order
 * of the reference's `+=`); runs whose sum is exactly 0 are dropped (d_head = 0).  mg_nn_emit writes the triplets. */
int mg_coo_fold_sum(int64_t m, const int32_t *d_rows, const int32_t *d_cols, const double *d_vals,
                    const int32_t *d_order, int32_t *d_head, double *d_folded, void *stream);
int mg_vector_from_runs(int64_t m, const int32_t *d_rows, const int32_t *d_order, const int32_t *d_head,
                        const double *d_folded, double *d_out, void *stream);
/* Semi-geometric coupling operator B[f,c] = int phi_f phi_c between two P1 triangle meshes, integrated on the
 * triangle-triangle intersections (finishes the reference's 2D stub L2Projection.py:17-24 along the 1D recipe
 * CouplingOperator.py:31-69): nine contributions per candidate pair of elements (+ the overlap area, optional).
 * Fold with mg_coo_fold_sum.  (mg_host_coupling_pairs_p1_2d, testing library only: the same per-pair code run serially on
 * host arrays, for the CPU tests.) */
/* Candidate (fine, coarse) element pairs = overlapping bounding boxes, found on the device by binning both meshes on one
 * G x G grid (lower corner h_lo, cell (p - lo) * h_inv_size): mg_tri_boxes_2d writes the boxes (and how many cells each
 * covers), mg_tri_incidence_2d the (cell, triangle) incidences of the coarse mesh at d_ptr[t] (sort them stably by cell
 * to get the per-cell lists), mg_tri_pairs_2d counts (d_pair_c NULL) and then writes the pairs of every fine triangle,
 * coarse ids ascending; a pair is reported in the one cell that holds the lower-left corner of the boxes' intersection. */
int mg_tri_boxes_2d(int64_t ne, const double *d_points, const int32_t *d_conn, const double *h_lo, const double *h_inv_size,
                    int32_t G, double *d_box, int32_t *d_ncells, void *stream);
int mg_tri_incidence_2d(int64_t ne, const double *d_box, const double *h_lo, const double *h_inv_size, int32_t G,
                        const int32_t *d_ptr, int32_t *d_inc_cell, int32_t *d_inc_tri, void *stream);
int mg_tri_pairs_2d(int64_t nf, const double *d_box_f, const double *d_box_c, const double *h_lo, const double *h_inv_size,
                    int32_t G, const int32_t *d_cell_ptr, const int32_t *d_cell_tri, int32_t *d_count,
                    const int32_t *d_ptr, int32_t *d_pair_f, int32_t *d_pair_c, void *stream);
int mg_coupling_pairs_p1_2d(int64_t npairs, const int32_t *d_pair_f, const int32_t *d_pair_c, const double *d_pf,
                            const int32_t *d_tf, const double *d_pc, const int32_t *d_tc, int32_t *d_rows,
                            int32_t *d_cols, double *d_vals, double *d_area, void *stream);
#ifdef MGB_TESTING      /* libmgb200_testing.so only: not exported by the product library */
int mg_host_coupling_pairs_p1_2d(int64_t npairs, const int32_t *h_pair_f, const int32_t *h_pair_c, const double *h_pf,
                                 const int32_t *h_tf, const double *h_pc, const int32_t *h_tc, int32_t *h_rows,
                                 int32_t *h_cols, double *h_vals, double *h_area);
#endif
/* A[nodes,:] = I[nodes,:] for the rows flagged in d_flag: count pass, scan, fill pass */
int mg_csr_dirichlet_count(int64_t n, const int32_t *d_indptr, const int32_t *d_flag, int32_t *d_count, void *stream);
int mg_csr_dirichlet_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                          const int32_t *d_flag, const int32_t *d_out_indptr, int32_t *d_out_indices,
                          double *d_out_values, void *stream);

/* ------------------------------------------------------------------------------------------------ */
/* NN-predicted transfer operators in 2D: the device form of NeuralMG_2D.define_hierarchy and its helpers
 * (learn_multigrid/solvers/Multigrid.py:401-765; csrc/nn_kernels.cu).  CSR inputs with sorted columns, int32 ids.
 * Supported regime: at most 6 positive off-diagonal entries per row (MG_ERR_UNSUPPORTED otherwise, no fallback). */
/* coarsening (:401-426): lexicographically first maximal independent set; input = CSR of M^T; d_state: 1 coarse /
 * 2 fine; d_work: n+1 int32; synchronises; returns the number of rounds or a negative status */
int mg_nn_coarsen(int64_t n, const int32_t *d_t_indptr, const int32_t *d_t_indices, const double *d_t_values,
                  int32_t *d_state, int32_t *d_work, void *stream);
/* map_coarse (:679-684): with d_scan = exclusive scan of (state == 1): cmap[i] = coarse id or -1, clist[k] = node */
int mg_nn_compact(int64_t n, const int32_t *d_state, const int32_t *d_scan, int32_t *d_cmap, int32_t *d_clist,
                  void *stream);
/* extract_patches (:591-677): [nc][43] features and [nc][31] fill indices (-1 padded); synchronises.  For a coarse node
 * with more than 6 neighbours this is patch variant 0 (the 6 largest mass entries kept) */
int mg_nn_extract_patches(int64_t nc, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                          const int32_t *d_cmap, const int32_t *d_clist, double *d_patches, int32_t *d_fill,
                          int32_t *d_err, void *stream);
/* extra patch variants of coarse nodes with 6 + a neighbours (:631-663): d_extra[k] = a; with d_extra_ptr = exclusive
 * scan of d_extra (nc + 1 entries, total T) variants 1..a of every such node go to rows nc .. nc+T-1 of d_patches /
 * d_fill (node order), and d_not_last ([nc + T], zeroed by the caller) is set for every patch of such a node but its
 * last variant, whose d_neighs row is the one fill_B keeps.  a <= 6.  mg_nn_extract_variants synchronises. */
int mg_nn_count_variants(int64_t nc, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                         const int32_t *d_clist, int32_t *d_extra, void *stream);
int mg_nn_extract_variants(int64_t nc, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                           const int32_t *d_cmap, const int32_t *d_clist, const int32_t *d_extra_ptr,
                           double *d_patches, int32_t *d_fill, int32_t *d_not_last, int32_t *d_err, void *stream);
/* fill_B (:687-732) in three steps: contributions [np][31] in application order (unused: row = unused_row >= rows)
 * + d_neighs table [ncoarse][6]; fold of the runs of equal (row, col) given the stable (row, col) sort order with the
 * reference's running mean (d_head marks run heads with a non-zero result); emission of the COO triplets of B */
int mg_nn_contributions(int64_t np_, const int32_t *d_fill, const double *d_pred, const int32_t *d_cmap,
                        const int32_t *d_not_last /* nullable */, int32_t unused_row, int32_t *d_rows, int32_t *d_cols,
                        double *d_vals, int32_t *d_dneigh, void *stream);
int mg_nn_fold(int64_t m, int32_t unused_row, const int32_t *d_rows, const int32_t *d_cols, const double *d_vals,
               const int32_t *d_order, int32_t *d_head, double *d_folded, void *stream);
int mg_nn_emit(int64_t m, const int32_t *d_rows, const int32_t *d_cols, const int32_t *d_order, const int32_t *d_head,
               const int32_t *d_slot, const double *d_folded, int32_t *d_out_rows, int32_t *d_out_cols,
               double *d_out_vals, void *stream);
/* Q = B / rowsum(B) in place (:758-759) */
int mg_nn_row_normalise(int64_t n, const int32_t *d_indptr, double *d_values, void *stream);
/* pre_process (:735-739): keep of row i the diagonal and the columns d_dneigh[i][0..5]; count pass, scan, fill pass */
int mg_nn_cut_count(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                    const int32_t *d_dneigh, int32_t *d_keep, int32_t *d_count, void *stream);
int mg_nn_cut_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                   const int32_t *d_keep, const int32_t *d_out_indptr, int32_t *d_out_indices, double *d_out_values,
                   void *stream);
#ifdef MGB_TESTING      /* libmgb200_testing.so only: not exported by the product library */
/* the same per-node code run serially on HOST arrays: lets the CPU test-suite check the extraction and contribution
 * logic against the reference's golden vectors without a GPU; not called by the product */
int mg_host_nn_coarsen(int64_t n, const int32_t *h_t_indptr, const int32_t *h_t_indices, const double *h_t_values,
                       int32_t *h_cmap, int32_t *h_clist);
/* returns the number of patch rows = nc + extra variants (outputs may be null to only count), or a negative status */
int mg_host_nn_extract_patches(int64_t nc, const int32_t *h_indptr, const int32_t *h_indices, const double *h_values,
                               const int32_t *h_cmap, const int32_t *h_clist, double *h_patches, int32_t *h_fill);
int mg_host_nn_contributions(int64_t np_, const int32_t *h_fill, const double *h_pred, const int32_t *h_cmap,
                             int32_t unused_row, int32_t *h_rows, int32_t *h_cols, double *h_vals, int32_t *h_dneigh);
#endif

/* ------------------------------------------------------------------------------------------------ */
/* Classical AMG setup (csrc/amg_kernels.cu, driven by learnmultigrid_b200/amg.py): strength of connection on negative
 * couplings, PMIS C/F splitting, direct interpolation.  CSR inputs with sorted columns, int32 ids, one thread per row;
 * the definitions are in DESIGN.md §4.10 and tests/amg_oracle.py restates them.  States: 0 undecided, 1 C, 2 F. */
/* strength S: j != i with -a_ij > 0 and -a_ij >= theta * max_{k!=i}(-a_ik), theta in [0, 1).  Count pass (d_count[n]),
 * exclusive scan by the caller, fill pass (pattern + the values a_ij, columns ascending) */
int mg_amg_strength_count(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                          double theta, int32_t *d_count, void *stream);
int mg_amg_strength_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                         double theta, const int32_t *d_s_indptr, int32_t *d_s_indices, double *d_s_values,
                         void *stream);
/* PMIS rounds on S and S^T (d_t_*: its transpose) with weights d_weights: points with an empty S^T row start F; per
 * round `select` (an undecided point whose (w, i) beats every undecided point of its S and S^T rows turns C) and
 * `mark` (an undecided point with a C point in its S row turns F), until nothing is undecided.  d_work: n + 1 int32.
 * One host read-back per round (synchronises); returns the number of rounds (>= 0) or a negative status. */
int mg_amg_pmis(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_t_indptr,
                const int32_t *d_t_indices, const double *d_weights, int32_t *d_state, int32_t *d_work, void *stream);
/* promotion pass on the final states: an F point with a non-empty S row and no C point in it turns C.  d_state_out
 * must not alias d_state; d_work: 1 int32.  Synchronises; returns the number of promoted points or a negative status. */
int mg_amg_promote(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_state,
                   int32_t *d_state_out, int32_t *d_work, void *stream);
/* direct interpolation Q (n x n_c): count pass (1 per C row, |S_i n C| per F row), exclusive scan by the caller, fill
 * pass with d_cmap from mg_nn_compact.  The fill synchronises; if a_ii + (sum of the positive off-diagonal entries) is 0
 * in an F row that interpolates, *h_bad_row receives the smallest such row and MG_ERR_SINGULAR is returned (else -1).
 * d_work: 1 int32. */
int mg_amg_interp_count(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_state,
                        int32_t *d_count, void *stream);
int mg_amg_interp_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                       const int32_t *d_s_indptr, const int32_t *d_s_indices, const double *d_s_values,
                       const int32_t *d_state, const int32_t *d_cmap, const int32_t *d_q_indptr,
                       int32_t *d_q_indices, double *d_q_values, int32_t *d_work, int64_t *h_bad_row, void *stream);

/* ------------------------------------------------------------------------------------------------ */
/* Smoothed aggregation setup (csrc/sa_kernels.cu, driven by learnmultigrid_b200/sa.py): symmetric strength of
 * connection, MIS(2) roots, aggregation, tentative prolongator, Jacobi-smoothing scale.  CSR inputs with sorted
 * columns, int32 ids, one thread per row (or aggregate); the definitions are in DESIGN.md §4.11 and tests/sa_oracle.py
 * restates them.  MIS(2) states: 0 OUT, 1 undecided, 2 IN (root). */
/* d_diag[i] = the stored a_ii (0 where none is stored) */
int mg_sa_diagonal(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                   double *d_diag, void *stream);
/* strength S: j != i with a_ij != 0 and a_ij * a_ij >= theta^2 * (|a_ii| * |a_jj|), theta in [0, 1) (theta^2 formed
 * once on the host), d_diag from mg_sa_diagonal.  Count pass (d_count[n]), exclusive scan by the caller, fill pass
 * (pattern + the values a_ij, columns ascending) */
int mg_sa_strength_count(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                         const double *d_diag, double theta, int32_t *d_count, void *stream);
int mg_sa_strength_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                        const double *d_diag, double theta, const int32_t *d_s_indptr, int32_t *d_s_indices,
                        double *d_s_values, void *stream);
/* MIS(2) on the graph S u S^T (d_t_*: the transpose of S): isolated points start OUT, the others undecided; per round
 * two passes propagate the maximum key (state, hash(i)) over {i} u S_i u S^T_i, and an undecided point turns IN if the
 * maximum is its own key, OUT if the maximum's state is IN.  d_work: n + 1 int32, d_keys: 2n uint64.  One host read-back
 * per round (synchronises); returns the number of rounds (>= 0) or a negative status. */
int mg_sa_mis2(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_t_indptr,
               const int32_t *d_t_indices, int32_t *d_state, int32_t *d_work, uint64_t *d_keys, void *stream);
/* aggregates d_agg[n] (-1: isolated) from the final MIS(2) states and d_cmap (mg_nn_compact over the roots): pass 1
 * joins a point to the root among its neighbours, pass 2 an unassigned one to its pass-1 neighbour of largest
 * (hash(j), j).  d_work: n + 2 int32.  Synchronises; a point with two distinct roots among its neighbours, or a
 * non-isolated point left unassigned, is MG_ERR_INVALID with the smallest such point in *h_bad_row (else -1). */
int mg_sa_aggregate(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_t_indptr,
                    const int32_t *d_t_indices, const int32_t *d_state, const int32_t *d_cmap, int32_t *d_agg,
                    int32_t *d_work, int64_t *h_bad_row, void *stream);
/* nu_a = sqrt(sum of the squares of row a of T^T, in storage order); one thread per aggregate */
int mg_sa_aggregate_norm(int64_t nc, const int32_t *d_tt_indptr, const double *d_tt_values, double *d_nu,
                         void *stream);
/* tentative prolongator T (n x n_c, one entry per aggregated row): column d_agg[i], value d_b[i] / d_nu[d_agg[i]], or
 * d_b[i] where d_nu is NULL (the pattern pass whose transpose gives nu); d_t_indptr: exclusive scan of d_agg >= 0 */
int mg_sa_tentative_fill(int64_t n, const int32_t *d_agg, const int32_t *d_t_indptr, const double *d_b,
                         const double *d_nu, int32_t *d_t_indices, double *d_t_values, void *stream);
/* the values of I - omega_hat D^-1 A on A's pattern (d_out_values[nnz]): -(s_i * a_ij) off the diagonal,
 * 1 - s_i * a_ii on it, s_i = omega_hat / a_ii */
int mg_sa_smooth_scale(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                       const double *d_diag, double omega_hat, double *d_out_values, void *stream);

/* ------------------------------------------------------------------------------------------------ */
/* host-side (serial, HOST pointers) setup helpers                                                    */
/* First-fit greedy colouring in index order on the symmetrised pattern of A; returns ncolors (>0) or <0.
 * The colour order defines the multicolour Gauss-Seidel that replaces PyAMG's index-order sweep
 * (Multigrid.py:88,121); the same colours are handed to the CPU oracle. */
int mg_host_greedy_color(int64_t n, const int32_t *h_indptr, const int32_t *h_indices, int32_t *h_colors);
/* The same colouring on a ROW BLOCK, one phase per call, for a setup in which no process holds the global pattern
 * (learnmultigrid_b200/partition_setup.py drives the blocks in rank order and gets the colours of the call above).
 * Columns are block-local: own rows 0..n_own-1, external node k at n_own + k with colour h_ext_color[k] (-1 = not
 * coloured yet).  h_forbidden_lo / _hi: n_own + n_ext words each, bit c = colour c (lo) / 64 + c (hi) is taken by a
 * coloured row that reaches the node through its own row only; in for the own rows, out for the external nodes.
 * phase 0: rows with off-diagonal entries (h_colors is reset to -1 first); phase 1: the remaining rows.
 * Returns the largest colour used in the block + 1 (0 if none) or a negative status. */
int mg_host_greedy_color_block(int64_t n_own, int64_t n_ext, const int32_t *h_indptr, const int32_t *h_indices,
                               const int32_t *h_ext_color, uint64_t *h_forbidden_lo, uint64_t *h_forbidden_hi,
                               int32_t *h_colors, int phase);
/* The colouring of mg_host_greedy_color computed on the device (csrc/color_kernels.cu): rounds of a Jones-Plassmann
 * sweep whose priority is the row's place in the first-fit order, on the patterns of A and A^T (device CSR index arrays).
 * Identical colours, entry for entry.  d_work: mg_color_workspace_size(n) bytes.  A round is one launch (a group of 8
 * lanes per row, programmatic dependent launches); a setup-time call: it synchronises the stream every 128 rounds.
 * MG_ERR_UNSUPPORTED if more than max_rounds rounds (long dependency chains, e.g. a 1D mesh numbered end to end: use
 * the host helper) or more than 128 colours would be needed. */
int64_t mg_color_workspace_size(int64_t n);
/* Is a colouring proper for the operator, and has every row a diagonal (mg_level.flags)?  Rows [0,nrows) of a CSR block
 * whose row i is global row row0 + i; d_color is indexed by GLOBAL row / column id.  *d_flags (device int32, zeroed by
 * the caller) |= 1 if a row has a non-zero entry in the column of another row of its own colour, |= 2 if a row has no
 * non-zero diagonal entry. */
int mg_csr_coloring_flags(int64_t nrows, int64_t row0, const int32_t *d_indptr, const int32_t *d_indices,
                          const double *d_values, const int32_t *d_color, int32_t *d_flags, void *stream);
int mg_color_first_fit(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const int32_t *d_t_indptr,
                       const int32_t *d_t_indices, int32_t *d_colors, void *d_work, int64_t work_bytes,
                       int64_t max_rounds, int64_t *h_rounds, void *stream);
#ifdef MGB_TESTING      /* libmgb200_testing.so only: not exported by the product library */
/* the same rounds run serially on HOST arrays with the same per-row code (CPU test-suite; not called by the product) */
int mg_host_color_rounds(int64_t n, const int32_t *h_indptr, const int32_t *h_indices, const int32_t *h_t_indptr,
                         const int32_t *h_t_indices, int32_t *h_colors, void *h_work, int64_t *h_rounds);
#endif
/* dependency level of every row for an exact index-order sweep (see mg_gs_lex_sweep_csr); returns nlevels */
int64_t mg_host_lex_levels(int64_t n, const int32_t *h_indptr, const int32_t *h_indices, int32_t *h_level);

/* ------------------------------------------------------------------------------------------------ */
/* The V-cycle (Multigrid.v_cycle, Multigrid.py:77-124) over a prebuilt hierarchy.                   */
enum { MG_SMOOTH_JACOBI = 0, MG_SMOOTH_MCGS = 1, MG_SMOOTH_LEXGS = 2, MG_SMOOTH_CHEBY = 3 };
enum { MG_COARSE_DENSE = 0, MG_COARSE_BCR = 1 };

typedef struct {
    int64_t n;                 /* rows on this level                                                     */
    mg_sell A;                 /* operator in this level's ordering                                      */
    const double *d_dinv;      /* 1/diag(A) (Jacobi)                                                     */
    int32_t ncolors;           /* multicolour GS: colour c owns rows [h_color_ptr[c], h_color_ptr[c+1])  */
    const int64_t *h_color_ptr;
    /* exact lexicographic GS (parity mode): CSR + dependency levels, both in this level's ordering      */
    const int32_t *d_csr_indptr, *d_csr_indices;
    const double *d_csr_values;
    const int64_t *d_lex_level_ptr;
    const int32_t *d_lex_level_rows;
    int64_t lex_nlevels;
    mg_sell Q;                 /* n x n_coarse, prolongation  (absent on the coarsest level)             */
    mg_sell QT;                /* n_coarse x n, restriction = explicit transpose                         */
    double *d_x, *d_b, *d_r, *d_tmp;  /* level vectors; on level 0 d_x/d_b are the caller's                */
    /* coarsest level only */
    int32_t coarse_kind;
    const double *d_coarse_inv;       /* MG_COARSE_DENSE: row-major n x n inverse                         */
    const void *coarse_bcr;           /* MG_COARSE_BCR: handle from mg_bcr_create                         */
    /* row-partitioned level (multi-GPU): n = OWNED rows, vectors hold n + dist->n_halo entries; NULL otherwise */
    const mg_dist_level *dist;
    const mg_bcr_dist *coarse_bcr_dist;   /* optional: split the BCR solve over the ranks (mg_vcycle_dist only)      */
    /* what mg_level_inspect established about A and the colouring (0 = nothing: the cycle then does no work-saving
     * fusion on this level); on partitioned levels the facts must hold for the GLOBAL operator                      */
    uint32_t flags;                       /* MG_LEVEL_*                                                              */
    uint32_t pad_;
    const double *d_diag;                 /* the diagonal as the Gauss-Seidel kernel finds it (0: none); optional    */
    /* Chebyshev smoother (MG_SMOOTH_CHEBY): the polynomial's degree and a HOST table of cheb_degree pairs
     * (c_d, c_r), step k at [2k, 2k+1] (c_d of step 0 unused); the step's d lives in d_r                           */
    int32_t cheb_degree;
    int32_t pad2_;
    const double *h_cheb_coef;
    /* singular operator with a declared null vector (coarsest level solved by block cyclic reduction only; NULL
     * otherwise): the cycle runs mg_project_out(n, d_null, null_inv_nn, null_pin, d_b) before the solve and
     * mg_project_out(n, d_null, null_inv_nn, -1, d_x) after it, with d_tmp as the partials workspace */
    const double *d_null;
    double null_inv_nn;                   /* 1 / (nu^T nu)                                                           */
    int64_t null_pin;                     /* the pinned row of the factor, in this level's ordering                  */
} mg_level;
/* multicolour Gauss-Seidel only.  PROPER_COLORING: no row has a non-zero entry in the column of ANOTHER row of its own
 * colour.  NONZERO_DIAG: every row has a non-zero diagonal entry (so a colour sweep overwrites every row it visits). */
enum { MG_LEVEL_PROPER_COLORING = 1, MG_LEVEL_NONZERO_DIAG = 2 };
/* d_diag[i] (optional) = last non-zero stored entry of row i on the diagonal (0 if none) -- what mg_sell_gs_rows divides
 * by; *d_flags (device int32, zeroed by the caller) |= 1 if the colouring given by d_color_ptr[ncolors+1] (device) is
 * NOT proper, |= 2 if some row has no non-zero diagonal.  ncolors = 0: only the diagonal is examined. */
int mg_level_inspect(const mg_sell *A, int ncolors, const int64_t *d_color_ptr, double *d_diag, int32_t *d_flags,
                     void *stream);

typedef struct {
    int32_t smoother;          /* MG_SMOOTH_*                                                            */
    int32_t nu_pre, nu_post;   /* smooth_steps (the reference uses the same number before and after)     */
    double omega;              /* Jacobi damping                                                         */
    int32_t zero_guess_skip;   /* 1: skip A*0 work on coarse levels (results identical)                  */
    int32_t reverse_post;      /* 1: multicolour post-smoothing visits the colours in reverse order, which makes
                                  the V-cycle a symmetric operator (preconditioner for CG); 0: reference order  */
    int32_t x0_zero;           /* 1: the iterate on levels[0] is to be taken as zero (d_x need not be initialised):
                                  z = M^-1 r of a preconditioner application without a memset and the A*0 work    */
    int32_t pad_;
} mg_cycle_params;

/* One V-cycle starting on levels[0]: pre-smooth, residual, restrict, recurse / coarsest solve,
 * prolong + correct, post-smooth.  Launches only; capturable in a CUDA graph. */
int mg_vcycle(const mg_level *levels, int nlevels, const mg_cycle_params *params, void *stream);
/* The same cycle, then *d_norm2 = ||b - A x||_2^2 of the NEW iterate on levels[0] -- what the next outer iteration of
 * Multigrid.solve evaluates first (Multigrid.py:62-63).  With multicolour Gauss-Seidel on a properly coloured level
 * the last colour sweep sums the squared residuals of its own rows from registers, and only the other colours' rows
 * are passed over again.  d_partials: mg_norm_workspace_size(n) doubles. */
int mg_vcycle_norm(const mg_level *levels, int nlevels, const mg_cycle_params *params, double *d_partials,
                   double *d_norm2, void *stream);
/* 1 (default): the multicolour cycle skips work whose result is never read or is already in registers (residual of the
 * last pre-smoothing colour from its sweep, no prolongation onto the colour the post-smoothing overwrites first, first
 * sweep on a zero iterate without the matrix); needs mg_level.flags.  0: every operation is a pass of its own.  The
 * results are bit-identical.  Returns the previous setting. */
int mg_set_cycle_fusion(int enabled);
/* The same cycle over a hierarchy whose first levels are row-partitioned across the ranks of `comm` (levels with
 * mg_level.dist set) and whose remaining levels are replicated.  Enqueues ONE program (mg_comm_begin .. mg_comm_end):
 * if `norm` is given, first the fused residual + squared 2-norm of level 0 summed over all ranks into *d_norm2 (the
 * outer loop of Multigrid.solve, Multigrid.py:62-63); then, if `params` is given, the V-cycle. */
typedef struct {
    double *d_partials;        /* mg_norm_workspace_size(owned rows) doubles                                */
    double *d_local;           /* 1 double: this rank's sum of squares                                      */
    double *d_slots;           /* MG_MAX_RANKS doubles: the other ranks' sums land here                     */
    double *d_norm2;           /* 1 double: the global sum, identical bits on every rank                    */
    int32_t after;             /* 0: the norm of the iterate the program STARTS from; 1: of the iterate the cycle
                                  leaves (fused into the last sweep as in mg_vcycle_norm; needs params)          */
    int32_t pad_;
} mg_dist_norm;
int mg_vcycle_dist(mg_comm *comm, const mg_level *levels, int nlevels, const mg_cycle_params *params,
                   const mg_dist_norm *norm, void *stream);
/* Conjugate gradients preconditioned by one V-cycle per iteration, statement order of learn_multigrid/solvers/CG.py:12-50
 * (x0 = 0) with z = M^-1 r inserted (BASELINE.json configs[4]).  The residual r lives in levels[0].d_b (the caller puts
 * the right-hand side there), z in levels[0].d_x.  All scalars stay on the device:
 *     d_scalars[8]: [0] r.z  [1] p.Ap  [2] alpha  [3] beta  [4] r.r  [5..7] scratch
 * mg_pcg_start: x = 0, [4] = r.r.  mg_pcg_iterate (first != 0 on the first call): z = M^-1 r (params == NULL: z = r),
 * beta, p = z + beta p, Ap = A p together with p.Ap, alpha, x += alpha p and r -= alpha Ap together with r.r.  Launches
 * only (one CUDA graph per value of `first`); the host reads [4] afterwards to test convergence.  comm != NULL: levels[0]
 * is row-partitioned (d_p then holds n + n_halo entries), every call is one program and the dot products are summed over
 * the ranks in rank order. */
typedef struct {
    double *d_x;          /* n: the solution being built, level-0 ordering                   */
    double *d_p;          /* n (+ halo): search direction                                    */
    double *d_Ap;         /* n                                                               */
    double *d_scalars;    /* 8 doubles                                                       */
    double *d_partials;   /* mg_norm_workspace_size(n) doubles                               */
    double *d_slots;      /* MG_MAX_RANKS doubles (partitioned runs; NULL otherwise)         */
} mg_pcg;
int mg_pcg_start(mg_comm *comm, const mg_level *levels, const mg_pcg *pcg, void *stream);
int mg_pcg_iterate(mg_comm *comm, const mg_level *levels, int nlevels, const mg_cycle_params *params, const mg_pcg *pcg,
                   int first, void *stream);
/* Restarted GMRES, right-preconditioned by one V-cycle per step (z_j = M^-1 v_j, w = A z_j; params == NULL: z_j = v_j),
 * everything in the level-0 ordering and on the device; the right-hand side is in levels[0].d_b.  Column-major buffers:
 * basis vector k of V (Z) starts at d_V + k * ld (d_Z + k * ld); the Hessenberg matrix d_H is (restart+1) x restart
 * with leading dimension restart + 1.  Arnoldi uses classical Gram-Schmidt in one pass, the least-squares problem is
 * kept triangular by Givens rotations.  Scalars:
 *     d_scalars[8]: [0] the squared residual the host reads  [1] divisor of the next basis vector  [2..7] scratch
 * mg_gmres_start: v_0 = r / beta with r = b - A x, beta = ||r|| (x's halo exchanged first when partitioned), g = beta e_1,
 *     [0] = beta^2; beta == 0 divides nothing.
 * mg_gmres_iterate(j): z_j = M^-1 v_j (one V-cycle from zero on the level-0 struct with d_b = v_j, d_x = z_j: nothing
 *     is copied), w = A z_j into slot j+1 of V, h = V^T w (multi-dot), w -= sum h_k v_k together with ||w||^2
 *     (multi-axpy), the Givens step (h_{j+1,j} = ||w||, rotations, g), v_{j+1} = w / h_{j+1,j} unless that is 0;
 *     [0] = |g_{j+1}|^2.  Launches only: one call can be captured in a CUDA graph.
 * mg_gmres_finish(k): R y = g over the first k columns, x += sum_{c<k} y_c z_c (params == NULL: v_c).
 * comm != NULL: levels[0] is row-partitioned (d_x, d_V and d_Z vectors hold n + n_halo entries, ld >= that); start and
 * iterate are one program each and the dot products are summed over the ranks in rank order. */
typedef struct {
    double *d_x;          /* ld: the solution, level-0 ordering                                          */
    double *d_V, *d_Z;    /* (restart + 1) * ld each                                                     */
    int64_t ld;           /* >= n (+ halo), a multiple of 32                                             */
    int32_t restart, pad_;
    double *d_H;          /* (restart + 1) * restart                                                     */
    double *d_g, *d_cs, *d_sn;  /* restart + 1 each                                                      */
    double *d_y;          /* restart + 1: y; during an iteration the rank's own dot products             */
    double *d_scalars;    /* 8 doubles                                                                   */
    double *d_partials;   /* max(mg_norm_workspace_size(n), mg_krylov_partials(n, restart + 1)) doubles  */
    double *d_slots;      /* MG_MAX_RANKS * (restart + 1) doubles (partitioned runs; NULL otherwise)     */
} mg_gmres;
int mg_gmres_start(mg_comm *comm, const mg_level *levels, const mg_gmres *gmres, void *stream);
int mg_gmres_iterate(mg_comm *comm, const mg_level *levels, int nlevels, const mg_cycle_params *params,
                     const mg_gmres *gmres, int j, void *stream);
int mg_gmres_finish(const mg_level *levels, const mg_cycle_params *params, const mg_gmres *gmres, int k, void *stream);
/* The building blocks (csrc/krylov_kernels.cu) on their own; V holds m vectors of n entries at a stride ld.
 * mg_krylov_partials: doubles of d_partials the two below need for n rows and m vectors. */
int64_t mg_krylov_partials(int64_t n, int32_t m);
/* d_out[k] = v_k . w, k < m, in a fixed order */
int mg_multi_dot(int64_t n, const double *d_V, int64_t ld, int32_t m, const double *d_w, double *d_partials,
                 double *d_out, void *stream);
/* w -= h_k v_k for k = 0, 1, ..., m-1 (each product and difference rounded), then *d_norm2 = ||w||^2 */
int mg_multi_axpy_norm(int64_t n, const double *d_V, int64_t ld, int32_t m, const double *d_h, double *d_w,
                       double *d_partials, double *d_norm2, void *stream);
/* v /= *d_h, nothing when *d_h == 0 */
int mg_scale_inv(int64_t n, const double *d_h, double *d_v, void *stream);
/* y = R^-1 g (R: upper triangle of the first k columns of d_H, leading dimension ldh), then x += y_c z_c, c = 0..k-1 */
int mg_gmres_solve_update(int64_t n, const double *d_H, int32_t ldh, const double *d_g, int32_t k, double *d_y,
                          const double *d_Z, int64_t ld, double *d_x, void *stream);
/* v <- v - (nu^T v * inv_nn) nu, then v[pin] = 0 if pin >= 0 (removes the null vector nu of a singular symmetric
 * operator; inv_nn = 1 / nu^T nu).  The dot is accumulated in double-double and rounded once, so it does not depend on
 * how the rows are split; d_dot (optional) receives it.  d_partials: mg_project_workspace_size(n) doubles.  Two
 * launches, capturable.  mg_project_out_dist: the same on this rank's row block of a row-partitioned vector, the dot
 * summed over the ranks of comm in rank order (one program; d_slots: 2 * world doubles); every rank gets the same bits. */
int64_t mg_project_workspace_size(int64_t n);
int mg_project_out(int64_t n, const double *d_nu, double inv_nn, int64_t pin, double *d_v, double *d_partials,
                   double *d_dot, void *stream);
int mg_project_out_dist(mg_comm *comm, int64_t n, const double *d_nu, double inv_nn, int64_t pin, double *d_v,
                        double *d_partials, double *d_slots, double *d_dot, void *stream);
/* number of kernels the last mg_vcycle call on this thread launched (bench.py's gpu_launches) */
int64_t mg_last_launch_count(void);
/* CUDA-graph helpers: capture whatever is enqueued on `stream` between begin and end. */
int mg_graph_begin(void *stream);
int mg_graph_end(void *stream, void **graph_exec_out);
int mg_graph_launch(void *graph_exec, void *stream);
int mg_graph_destroy(void *graph_exec);

#ifdef __cplusplus
}
#endif
#endif /* MGB200_H */
