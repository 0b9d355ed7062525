// sell_kernels.cu -- SELL-32 hot path: tunables, the small helper kernels, the SpMV / residual / norm launches and the
// C ABI of the whole family.  The streaming kernels themselves are templates in sell_core.cuh; the Gauss-Seidel modes
// are instantiated in sell_modes_gs.cu, Jacobi and prolongation in sell_modes_vec.cu.
#include "sell_core.cuh"

namespace mgb {

int64_t g_wide_min_len = 9;          // slices at least this long use sell_wide_kernel (0 = never)
// ... for launches of at most this many rows; larger launches have enough rows in flight for the thread-per-row kernel,
// which then streams at the DRAM limit (measured: profiles/r01_launches_c3_quasi_*.txt)
int64_t g_wide_max_rows = 1 << 18;
int64_t g_tma_min_rows = 0;          // off by default: the register-staged kernel is as fast (see sell_tma.cu)
// implied columns: on (matrices that carry an offset table, launches of at least g_implied_min_rows rows).  Measured on
// B200 (profiles/r02_bench_implied_columns_8193sq_first.json): fine-level colour sweep 0.429 -> 0.358 ms, SpMV on 1 M
// rows 11.8 -> 9.9 us, but 263 k rows 3.5 -> 4.8 us (one more dependent load in a latency-bound launch): hence the floor.
int g_implied_columns = 1;
int64_t g_implied_min_rows = 1 << 19;
int g_value_dict = 1;                // value dictionaries (valdict.cu) are used where a matrix carries one
int g_implied_values = 1;            // value records (sell_core.cuh, IMPV) are used where a matrix carries them
int g_implied_transfers = 1;         // slice patterns (sell_core.cuh, sell_pattern_kernel) where a matrix carries them
// rows of one or two entries (linear transfers): R rows per thread on large launches (sell_short_kernel)
int g_short_rows_per_thread = 2;
int64_t g_short_min_rows = 1 << 18;

__global__ void __launch_bounds__(kBlock)
sell_slice_offsets_kernel(int64_t nslices, int64_t nrows, int len, const int32_t *__restrict__ cols,
                          int32_t *__restrict__ off, unsigned long long *__restrict__ nregular) {
    const int64_t w = ((int64_t)blockIdx.x * kBlock + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= nslices) return;
    const int64_t row = w * kSlice + lane;
    bool regular = (w + 1) * kSlice <= nrows;
    for (int j = 0; j < kOffStride; ++j) {
        int64_t rel0 = 0;
        if (j < len) {
            const int64_t rel = (int64_t)cols[(w * len + j) * kSlice + lane] - row;
            rel0 = __shfl_sync(0xffffffffu, rel, 0);
            regular = __all_sync(0xffffffffu, rel == rel0) && regular;
        }
        if (lane == 0) off[w * kOffStride + j] = (int32_t)rel0;
    }
    if (lane == 0) {
        if (!regular) off[w * kOffStride] = kSliceIrregular;
        else if (nregular) atomicAdd(nregular, 1ull);
    }
}

// mask[s] = 1 if slice s holds a column >= first_halo_col (one warp per slice)
__global__ void __launch_bounds__(kBlock)
sell_halo_mask_kernel(int64_t nslices, const int64_t *__restrict__ slice_ptr, int64_t uniform_len,
                      const int32_t *__restrict__ cols, int64_t first_halo_col, unsigned char *__restrict__ mask) {
    const int64_t s = ((int64_t)blockIdx.x * kBlock + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (s >= nslices) return;
    const int64_t base = uniform_len > 0 ? s * kSlice * uniform_len : slice_ptr[s];
    const int64_t end = uniform_len > 0 ? base + kSlice * uniform_len : slice_ptr[s + 1];
    int hit = 0;
    for (int64_t p = base + lane; p < end; p += 32) hit |= cols[p] >= first_halo_col;
    hit = __any_sync(0xffffffffu, hit);
    if (lane == 0) mask[s] = hit ? 1 : 0;
}

// second stage of the deterministic norm / dot: one CTA sums the per-block partials in a fixed order
__global__ void __launch_bounds__(1024) reduce_partials_kernel(const double *__restrict__ partials, int64_t n,
                                                               double *__restrict__ out) {
    pdl_prologue();
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) s += partials[i];
    s = block_sum<1024>(s);
    if (threadIdx.x == 0) *out = s;
}

// What the cycle may assume about a level (mg_level_inspect): diag[i] = the value the Gauss-Seidel kernel divides row i
// by (the last non-zero stored entry on the diagonal, 0 if there is none); flags[0] |= 1 if some row couples, through a
// non-zero entry, to ANOTHER row of its own colour block (the colouring is not proper: a colour sweep is then not
// independent of the order inside the colour); flags[0] |= 2 if some row has no non-zero diagonal.
__global__ void __launch_bounds__(kBlock)
sell_inspect_kernel(int64_t nrows, const int64_t *__restrict__ slice_ptr, int64_t uniform_len,
                    const int32_t *__restrict__ cols, const double *__restrict__ vals, int ncolors,
                    const int64_t *__restrict__ color_ptr, double *__restrict__ diag_out, int32_t *__restrict__ flags) {
    const int64_t row = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (row >= nrows) return;
    const int64_t slice = row >> 5;
    const int lane = (int)(row & 31);
    const int64_t base = uniform_len > 0 ? slice * kSlice * uniform_len : slice_ptr[slice];
    const int len = uniform_len > 0 ? (int)uniform_len : (int)((slice_ptr[slice + 1] - base) >> 5);
    int64_t c0 = 0, c1 = -1;                       // colour block of this row
    for (int c = 0; c < ncolors; ++c)
        if (row >= color_ptr[c] && row < color_ptr[c + 1]) { c0 = color_ptr[c]; c1 = color_ptr[c + 1]; }
    double diag = 0.0;
    int bad = 0;
    for (int k = 0; k < len; ++k) {
        const int64_t col = cols[base + (int64_t)k * kSlice + lane];
        const double v = vals[base + (int64_t)k * kSlice + lane];
        if (v == 0.0) continue;
        if (col == row) diag = v;
        else if (col >= c0 && col < c1) bad |= 1;
    }
    if (diag == 0.0) bad |= 2;
    if (diag_out) diag_out[row] = diag;
    if (bad) atomicOr(flags, bad);
}

// see sell_gs_zero_first: two entries per thread, 128-bit accesses where both lie inside the colour
__global__ void __launch_bounds__(kBlock)
gs_zero_first_kernel(int64_t n_vec, int64_t row0, int64_t row1, const double *__restrict__ diag,
                     const double *__restrict__ b, double *__restrict__ x) {
    pdl_prologue();
    const int64_t i = 2 * ((int64_t)blockIdx.x * kBlock + threadIdx.x);
    if (i >= n_vec) return;
    double v0 = 0.0, v1 = 0.0;
    if (i >= row0 && i + 1 < row1) {
        const double2 d = *reinterpret_cast<const double2 *>(diag + i);
        const double2 r = *reinterpret_cast<const double2 *>(b + i);
        if (d.x != 0.0) v0 = __ddiv_rn(__dsub_rn(r.x, 0.0), d.x);
        if (d.y != 0.0) v1 = __ddiv_rn(__dsub_rn(r.y, 0.0), d.y);
    } else {
        if (i >= row0 && i < row1) { const double d = diag[i]; if (d != 0.0) v0 = __ddiv_rn(__dsub_rn(b[i], 0.0), d); }
        if (i + 1 >= row0 && i + 1 < row1) { const double d = diag[i + 1]; if (d != 0.0) v1 = __ddiv_rn(__dsub_rn(b[i + 1], 0.0), d); }
    }
    if (i + 1 < n_vec) *reinterpret_cast<double2 *>(x + i) = make_double2(v0, v1);
    else x[i] = v0;
}

bool sell_fusable(const mg_sell *A, int64_t row0, int64_t row1) {
    if (row1 <= row0 || g_tma_min_rows > 0) return false;
    return !sell_uses_wide(A, row0, row1);
}
bool sell_gs_tail_ok(const mg_sell *A, int64_t row0, int64_t row1) {
    if (row1 <= row0) return false;
    const int64_t ml = A->max_slice_len;
    return (ml >= 1 && ml <= 8) || sell_uses_wide(A, row0, row1);
}

int sell_spmv(const mg_sell *A, const double *x, double *y, int64_t row0, int64_t row1, const SellFuse *fuse, cudaStream_t st) {
    return launch_sell<SPMV>(A, x, nullptr, nullptr, y, 0.0, nullptr, row0, row1, st, "sell_spmv", nullptr, fuse);
}
// first stage of a long reduction: CTA g sums the contiguous chunk [g * chunk, (g+1) * chunk) in a fixed order
__global__ void __launch_bounds__(1024) reduce_chunks_kernel(const double *__restrict__ partials, int64_t n, int64_t chunk,
                                                             double *__restrict__ out) {
    pdl_prologue();
    const int64_t lo = (int64_t)blockIdx.x * chunk, hi = lo + chunk < n ? lo + chunk : n;
    double s = 0.0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += 1024) s += partials[i];
    s = block_sum_last<1024>(s);
    if (threadIdx.x == 0) out[blockIdx.x] = s;
}

constexpr int kReduceChunks = 64;       // CTAs of the first stage (the workspace holds that many doubles behind the partials)

int sell_reduce_partials(const double *partials, int64_t n, double *out, cudaStream_t st) {
    if (n > 32768) {                    // one CTA would take tens of microseconds (262 k partials: 28 us)
        double *tmp = const_cast<double *>(partials) + n;
        const int64_t chunk = (n + kReduceChunks - 1) / kReduceChunks;
        launch_k(reduce_chunks_kernel, (unsigned)kReduceChunks, 1024u, st, partials, n, chunk, tmp);
        MG_CHECK_LAUNCH("reduce_chunks");
        launch_k(reduce_partials_kernel, 1u, 1024u, st, (const double *)tmp, (int64_t)kReduceChunks, out);
        MG_CHECK_LAUNCH("reduce_partials");
        return MG_OK;
    }
    launch_k(reduce_partials_kernel, 1u, 1024u, st, partials, n, out);
    MG_CHECK_LAUNCH("reduce_partials");
    return MG_OK;
}
int sell_residual_norm2(const mg_sell *A, const double *x, const double *b, double *partials, double *out,
                        cudaStream_t st) {
    int nblocks = 0;
    if (int rc = sell_residual_partials(A, x, b, partials, 0, A->nrows, &nblocks, nullptr, st)) return rc;
    return sell_reduce_partials(partials, nblocks, out, st);
}
int sell_gs_zero_first(int64_t n_vec, int64_t row0, int64_t row1, const double *diag, const double *b, double *x,
                       cudaStream_t st) {
    if (n_vec <= 0) return MG_OK;
    if ((((uintptr_t)diag | (uintptr_t)b | (uintptr_t)x) & 15) != 0) return set_error(MG_ERR_INVALID, "gs_zero_first", "vectors must be 16-byte aligned");
    launch_k(gs_zero_first_kernel, (unsigned)(((n_vec + 1) / 2 + kBlock - 1) / kBlock), kBlock, st, n_vec, row0, row1, diag, b, x);
    MG_CHECK_LAUNCH("gs_zero_first");
    return MG_OK;
}

}  // namespace mgb

using namespace mgb;

extern "C" {

static int check_sell(const mg_sell *A) {
    if (!A || A->nrows < 0 || (A->nrows > 0 && (!A->d_slice_ptr || !A->d_cols || !A->d_vals)))
        return set_error(MG_ERR_INVALID, "mg_sell", "null or negative-sized SELL matrix");
    if (A->nslices != (A->nrows + kSlice - 1) / kSlice)
        return set_error(MG_ERR_INVALID, "mg_sell", "nslices != ceil(nrows/32)");
    return MG_OK;
}
static int check_rows(const mg_sell *A, int64_t row0, int64_t row1) {
    if (int rc = check_sell(A)) return rc;
    if (!(row0 >= 0 && row1 <= A->nrows && row0 <= row1)) return set_error(MG_ERR_INVALID, "mg_sell", "row range outside the matrix");
    return MG_OK;
}

int mg_sell_spmv(const mg_sell *A, const double *d_x, double *d_y, void *stream) {
    if (int rc = check_sell(A)) return rc;
    return sell_spmv(A, d_x, d_y, 0, A->nrows, nullptr, (cudaStream_t)stream);
}
int mg_sell_residual(const mg_sell *A, const double *d_x, const double *d_b, double *d_r, void *stream) {
    if (int rc = check_sell(A)) return rc;
    return sell_residual(A, d_x, d_b, d_r, 0, A->nrows, nullptr, (cudaStream_t)stream);
}
int mg_sell_residual_rows(const mg_sell *A, const double *d_x, const double *d_b, double *d_r, int64_t row0,
                          int64_t row1, void *stream) {
    if (int rc = check_rows(A, row0, row1)) return rc;
    return sell_residual(A, d_x, d_b, d_r, row0, row1, nullptr, (cudaStream_t)stream);
}
/* worst case over the kernels that write partials: the warps-per-slice kernel with eight warps per slice has one CTA
 * (one partial) per 32 rows; a sweep with a fused norm followed by the norm of the remaining rows writes two runs;
 * the first stage of a long second-stage reduction parks its 64 sums behind the partials */
int64_t mg_norm_workspace_size(int64_t n) { return (n + kSlice - 1) / kSlice + 2 + kReduceChunks; }
int mg_sell_halo_mask(const mg_sell *A, int64_t first_halo_col, unsigned char *d_mask, void *stream) {
    MG_REQUIRE(A && d_mask && A->nrows > 0, "null argument");
    const int64_t ns = A->nslices;
    sell_halo_mask_kernel<<<(unsigned)((ns * 32 + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(
        ns, A->d_slice_ptr, A->uniform_len, A->d_cols, first_halo_col, d_mask);
    MG_CHECK_LAUNCH("sell_halo_mask");
    return MG_OK;
}
/* per-slice column offsets of a UNIFORM matrix (uniform_len <= 8 entries per row): one record of 8 ints per slice,
 * d_off[s * 8 + j] (32-byte aligned: cudaMalloc'ed); slices that are not regular get d_off[s * 8] = INT32_MIN (see
 * sell_core.cuh); *d_nregular (device, zeroed by the caller, may be NULL) counts the regular slices */
int mg_sell_slice_offsets(const mg_sell *A, int32_t *d_off, int64_t *d_nregular, void *stream) {
    if (int rc = check_sell(A)) return rc;
    MG_REQUIRE(d_off && A->uniform_len > 0 && A->uniform_len == A->max_slice_len && A->uniform_len <= kOffStride,
               "uniform SELL matrix with at most 8 entries per row expected");
    MG_REQUIRE(((uintptr_t)d_off & 31) == 0, "offset table must be 32-byte aligned");
    if (A->nslices == 0) return MG_OK;
    sell_slice_offsets_kernel<<<(unsigned)((A->nslices * 32 + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(
        A->nslices, A->nrows, (int)A->uniform_len, A->d_cols, d_off, (unsigned long long *)d_nregular);
    MG_CHECK_LAUNCH("sell_slice_offsets");
    return MG_OK;
}
int mg_level_inspect(const mg_sell *A, int ncolors, const int64_t *d_color_ptr, double *d_diag, int32_t *d_flags,
                     void *stream) {
    if (int rc = check_sell(A)) return rc;
    MG_REQUIRE(d_flags && ncolors >= 0 && (ncolors == 0 || d_color_ptr), "null argument");
    if (A->nrows == 0) return MG_OK;
    sell_inspect_kernel<<<(unsigned)((A->nrows + kBlock - 1) / kBlock), kBlock, 0, (cudaStream_t)stream>>>(
        A->nrows, A->d_slice_ptr, A->uniform_len > 0 && A->uniform_len == A->max_slice_len ? A->uniform_len : 0, A->d_cols,
        A->d_vals, ncolors, d_color_ptr, d_diag, d_flags);
    MG_CHECK_LAUNCH("sell_inspect");
    return MG_OK;
}
int mg_set_implied_columns(int enabled) {
    const int prev = g_implied_columns;
    g_implied_columns = enabled ? 1 : 0;
    return prev;
}
int mg_set_implied_transfers(int enabled) {
    const int prev = g_implied_transfers;
    if (enabled >= 0) g_implied_transfers = enabled ? 1 : 0;
    return prev;
}
int64_t mg_set_implied_min_rows(int64_t rows) {
    const int64_t prev = g_implied_min_rows;
    g_implied_min_rows = rows < 0 ? 0 : rows;
    return prev;
}
int mg_set_value_dict(int enabled) {
    const int prev = g_value_dict;
    g_value_dict = enabled ? 1 : 0;
    return prev;
}
int mg_set_implied_values(int enabled) {
    const int prev = g_implied_values;
    g_implied_values = enabled ? 1 : 0;
    return prev;
}
int mg_set_short_rows_per_thread(int r) {
    const int prev = g_short_rows_per_thread;
    g_short_rows_per_thread = r >= 4 ? 4 : r >= 2 ? 2 : 1;
    return prev;
}
int64_t mg_set_short_min_rows(int64_t rows) {
    const int64_t prev = g_short_min_rows;
    g_short_min_rows = rows < 0 ? 0 : rows;
    return prev;
}
int64_t mg_set_wide_min_len(int64_t len) {
    const int64_t prev = g_wide_min_len;
    g_wide_min_len = len < 0 ? 0 : len;
    return prev;
}
int64_t mg_set_wide_max_rows(int64_t rows) {
    const int64_t prev = g_wide_max_rows;
    g_wide_max_rows = rows < 0 ? 0 : rows;
    return prev;
}
int64_t mg_set_tma_min_rows(int64_t rows) {
    const int64_t old = g_tma_min_rows;
    g_tma_min_rows = rows;
    return old;
}
int mg_sell_residual_norm2(const mg_sell *A, const double *d_x, const double *d_b, double *d_partials,
                           double *d_norm2, void *stream) {
    if (int rc = check_sell(A)) return rc;
    if (A->nrows == 0) return mg_fill(1, 0.0, d_norm2, stream);
    return sell_residual_norm2(A, d_x, d_b, d_partials, d_norm2, (cudaStream_t)stream);
}
int mg_sell_jacobi(const mg_sell *A, const double *d_dinv, const double *d_x, const double *d_b,
                   double *d_x_out, double omega, void *stream) {
    if (int rc = check_sell(A)) return rc;
    MG_REQUIRE(d_x != d_x_out, "Jacobi is out of place: x_out must not alias x");
    return sell_jacobi(A, d_dinv, d_x, d_b, d_x_out, omega, (cudaStream_t)stream);
}
int mg_sell_gs_rows(const mg_sell *A, double *d_x, const double *d_b, int64_t row0, int64_t row1,
                    void *stream) {
    if (int rc = check_rows(A, row0, row1)) return rc;
    return sell_gs_rows(A, d_x, d_b, row0, row1, nullptr, TAIL_NONE, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}
int mg_sell_gs_rows_tail(const mg_sell *A, double *d_x, const double *d_b, int64_t row0, int64_t row1, int tail,
                         double *d_r, double *d_partials, int *h_nblocks, void *stream) {
    if (int rc = check_rows(A, row0, row1)) return rc;
    MG_REQUIRE(tail == TAIL_NONE || (tail == TAIL_RESIDUAL && d_r) || (tail == TAIL_NORM && d_partials && h_nblocks),
               "tail output missing");
    if (h_nblocks) *h_nblocks = 0;
    if (tail != TAIL_NONE && row1 > row0 && !sell_gs_tail_ok(A, row0, row1))
        return set_error(MG_ERR_UNSUPPORTED, "mg_sell_gs_rows_tail", "rows too long for a sweep with a fused residual (mg_sell_gs_tail_ok)");
    return sell_gs_rows(A, d_x, d_b, row0, row1, nullptr, tail, d_r, d_partials, h_nblocks, (cudaStream_t)stream);
}
int mg_sell_gs_tail_ok(const mg_sell *A, int64_t row0, int64_t row1) {
    if (check_rows(A, row0, row1)) return 0;
    return sell_gs_tail_ok(A, row0, row1) ? 1 : 0;
}
int mg_sell_gs_zero_first(int64_t n_vec, int64_t row0, int64_t row1, const double *d_diag, const double *d_b,
                          double *d_x, void *stream) {
    MG_REQUIRE(n_vec >= 0 && row0 >= 0 && row0 <= row1 && row1 <= n_vec && d_diag && d_b && d_x, "bad argument");
    return sell_gs_zero_first(n_vec, row0, row1, d_diag, d_b, d_x, (cudaStream_t)stream);
}
int mg_sell_prolong_correct(const mg_sell *Q, const double *d_e, const double *d_u, double *d_u_out,
                            void *stream) {
    if (int rc = check_sell(Q)) return rc;
    return sell_prolong(Q, d_e, d_u, d_u_out, 0, Q->nrows, nullptr, (cudaStream_t)stream);
}
int mg_sell_prolong_correct_rows(const mg_sell *Q, const double *d_e, const double *d_u, double *d_u_out, int64_t row0,
                                 int64_t row1, void *stream) {
    if (int rc = check_rows(Q, row0, row1)) return rc;
    return sell_prolong(Q, d_e, d_u, d_u_out, row0, row1, nullptr, (cudaStream_t)stream);
}

}  // extern "C"
