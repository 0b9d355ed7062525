// amg_kernels.cu -- classical algebraic multigrid setup on the device: strength of connection, PMIS C/F splitting and
// direct interpolation (learnmultigrid_b200/amg.py drives them level by level; DESIGN.md §4.10).
//
// Every step is one thread per row over CSR with sorted columns; the per-row logic is written once as a __device__
// function that reads like the definition in DESIGN.md, so that tests/amg_oracle.py (NumPy, written from the same
// definition) and the device agree bit for bit:
//   strength     j != i is strong for i iff -a_ij > 0 and -a_ij >= theta * max_{k != i}(-a_ik);
//   PMIS         rounds of select (an undecided i becomes C iff its (w_i, i) beats every undecided j in S_i and S^T_i)
//                and mark (an undecided i with a C point in S_i becomes F), then one promotion pass (an F point with a
//                non-empty S_i and no C point in it becomes C);
//   interpolate  C row: 1 at cmap[i]; F row: coef * a_ij for j in S_i n C with coef = -(sn_all / sn_str) / (a_ii + sp_all).
// Products, sums and quotients are rounded one at a time (__dmul_rn / __dadd_rn / __ddiv_rn: no FMA contraction).
#include "common.cuh"

namespace mgb {

enum AmgState : int32_t { AMG_UNDECIDED = 0, AMG_C = 1, AMG_F = 2 };   // AMG_C = 1: mg_nn_compact's coarse flag

// theta * max_{k != i}(-a_ik) of row i; rows whose off-diagonal entries are all >= 0 give 0 (and have no strong entry,
// since a strong entry needs -a_ij > 0)
__device__ inline double amg_strength_threshold(const int32_t *indptr, const int32_t *indices, const double *values,
                                                int64_t i, double theta) {
    double m = 0.0;
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p) {
        const double na = -values[p];
        if (indices[p] != i && na > m) m = na;
    }
    return __dmul_rn(theta, m);
}

__device__ inline bool amg_is_strong(int64_t i, int32_t j, double a_ij, double threshold) {
    return j != i && -a_ij > 0.0 && -a_ij >= threshold;
}

// (w_i, i) > (w_j, j) lexicographically
__device__ inline bool amg_beats(const double *w, int64_t i, int32_t j) {
    return w[i] > w[j] || (w[i] == w[j] && i > j);
}

// select: an undecided i becomes C iff no undecided j in S_i or S^T_i has a larger (w_j, j)
__device__ inline bool amg_select_row(const int32_t *s_ptr, const int32_t *s_idx, const int32_t *t_ptr,
                                      const int32_t *t_idx, const double *w, const int32_t *state, int64_t i) {
    for (int32_t p = s_ptr[i]; p < s_ptr[i + 1]; ++p) {
        const int32_t j = s_idx[p];
        if (state[j] == AMG_UNDECIDED && !amg_beats(w, i, j)) return false;
    }
    for (int32_t p = t_ptr[i]; p < t_ptr[i + 1]; ++p) {
        const int32_t j = t_idx[p];
        if (state[j] == AMG_UNDECIDED && !amg_beats(w, i, j)) return false;
    }
    return true;
}

__device__ inline bool amg_has_strong_c(const int32_t *s_ptr, const int32_t *s_idx, const int32_t *state, int64_t i) {
    for (int32_t p = s_ptr[i]; p < s_ptr[i + 1]; ++p)
        if (state[s_idx[p]] == AMG_C) return true;
    return false;
}

// direct interpolation weight of F row i: coef such that Q[i, cmap[j]] = coef * a_ij for j in S_i n C.  Sums in storage
// order.  Returns false if d = a_ii + sp_all is zero.
__device__ inline bool amg_direct_coef(const int32_t *indptr, const int32_t *indices, const double *values,
                                       const int32_t *s_ptr, const int32_t *s_idx, const double *s_val,
                                       const int32_t *state, int64_t i, double &coef) {
    double sn_all = 0.0, sp_all = 0.0, a_ii = 0.0;
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p) {
        const double a = values[p];
        if (indices[p] == i) a_ii = a;
        else if (a < 0.0) sn_all = __dadd_rn(sn_all, a);
        else if (a > 0.0) sp_all = __dadd_rn(sp_all, a);
    }
    double sn_str = 0.0;
    for (int32_t p = s_ptr[i]; p < s_ptr[i + 1]; ++p)
        if (state[s_idx[p]] == AMG_C) sn_str = __dadd_rn(sn_str, s_val[p]);
    const double alpha = __ddiv_rn(sn_all, sn_str);
    const double d = __dadd_rn(a_ii, sp_all);
    if (d == 0.0) return false;
    coef = __ddiv_rn(-alpha, d);
    return true;
}

// ---- kernels ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
amg_strength_count_kernel(int64_t n, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                          const double *__restrict__ values, double theta, int32_t *__restrict__ count) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const double thr = amg_strength_threshold(indptr, indices, values, i, theta);
    int32_t c = 0;
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p)
        if (amg_is_strong(i, indices[p], values[p], thr)) ++c;
    count[i] = c;
}

__global__ void __launch_bounds__(kBlock)
amg_strength_fill_kernel(int64_t n, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                         const double *__restrict__ values, double theta, const int32_t *__restrict__ s_ptr,
                         int32_t *__restrict__ s_idx, double *__restrict__ s_val) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const double thr = amg_strength_threshold(indptr, indices, values, i, theta);
    int32_t q = s_ptr[i];
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p) {
        const int32_t j = indices[p];
        const double a = values[p];
        if (amg_is_strong(i, j, a, thr)) {
            s_idx[q] = j;
            s_val[q] = a;
            ++q;
        }
    }
}

// points that influence nobody (empty S^T_i) start as F, the others undecided.  *any_undecided: set to 1 if a point
// is left undecided (every writer stores the same value, so a plain store is enough)
__global__ void __launch_bounds__(kBlock)
amg_pmis_init_kernel(int64_t n, const int32_t *__restrict__ t_ptr, int32_t *__restrict__ state,
                     int32_t *__restrict__ any_undecided) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const bool u = t_ptr[i + 1] > t_ptr[i];
    state[i] = u ? AMG_UNDECIDED : AMG_F;
    if (u) *any_undecided = 1;
}

// reads the states of the round's start, writes the new C points to another buffer (a point that turns C in this
// round must still count as undecided for its neighbours' comparisons)
__global__ void __launch_bounds__(kBlock)
amg_pmis_select_kernel(int64_t n, const int32_t *__restrict__ s_ptr, const int32_t *__restrict__ s_idx,
                       const int32_t *__restrict__ t_ptr, const int32_t *__restrict__ t_idx,
                       const double *__restrict__ w, const int32_t *__restrict__ state_in,
                       int32_t *__restrict__ state_out) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    int32_t s = state_in[i];
    if (s == AMG_UNDECIDED && amg_select_row(s_ptr, s_idx, t_ptr, t_idx, w, state_in, i)) s = AMG_C;
    state_out[i] = s;
}

// in place: only undecided -> F is written, only C is read, so the order of the threads does not matter
__global__ void __launch_bounds__(kBlock)
amg_pmis_mark_kernel(int64_t n, const int32_t *__restrict__ s_ptr, const int32_t *__restrict__ s_idx,
                     int32_t *__restrict__ state, int32_t *__restrict__ any_undecided) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    if (state[i] != AMG_UNDECIDED) return;
    if (amg_has_strong_c(s_ptr, s_idx, state, i)) state[i] = AMG_F;
    else *any_undecided = 1;
}

__global__ void __launch_bounds__(kBlock)
amg_promote_kernel(int64_t n, const int32_t *__restrict__ s_ptr, const int32_t *__restrict__ s_idx,
                   const int32_t *__restrict__ state_in, int32_t *__restrict__ state_out,
                   int32_t *__restrict__ promoted) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    int32_t s = state_in[i];
    if (s == AMG_F && s_ptr[i + 1] > s_ptr[i] && !amg_has_strong_c(s_ptr, s_idx, state_in, i)) {
        s = AMG_C;
        atomicAdd(promoted, 1);
    }
    state_out[i] = s;
}

__global__ void __launch_bounds__(kBlock)
amg_interp_count_kernel(int64_t n, const int32_t *__restrict__ s_ptr, const int32_t *__restrict__ s_idx,
                        const int32_t *__restrict__ state, int32_t *__restrict__ count) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    int32_t c = 0;
    if (state[i] == AMG_C) {
        c = 1;
    } else {
        for (int32_t p = s_ptr[i]; p < s_ptr[i + 1]; ++p)
            if (state[s_idx[p]] == AMG_C) ++c;
    }
    count[i] = c;
}

__global__ void __launch_bounds__(kBlock)
amg_interp_fill_kernel(int64_t n, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                       const double *__restrict__ values, const int32_t *__restrict__ s_ptr,
                       const int32_t *__restrict__ s_idx, const double *__restrict__ s_val,
                       const int32_t *__restrict__ state, const int32_t *__restrict__ cmap,
                       const int32_t *__restrict__ q_ptr, int32_t *__restrict__ q_idx, double *__restrict__ q_val,
                       int32_t *__restrict__ bad_row) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    int32_t q = q_ptr[i];
    if (state[i] == AMG_C) {
        q_idx[q] = cmap[i];
        q_val[q] = 1.0;
        return;
    }
    if (q_ptr[i + 1] == q) return;                 // empty S_i: no interpolation entries
    double coef;
    if (!amg_direct_coef(indptr, indices, values, s_ptr, s_idx, s_val, state, i, coef)) {
        atomicMin(bad_row, (int32_t)i);
        return;
    }
    for (int32_t p = s_ptr[i]; p < s_ptr[i + 1]; ++p) {
        const int32_t j = s_idx[p];
        if (state[j] != AMG_C) continue;
        q_idx[q] = cmap[j];
        q_val[q] = __dmul_rn(coef, s_val[p]);
        ++q;
    }
}

constexpr int32_t kAmgNoRow = 0x7f7f7f7f;     // "no failing row": every byte 0x7f, so one memset sets it

inline unsigned amg_grid(int64_t n) { return (unsigned)((n + kBlock - 1) / kBlock); }

}  // namespace mgb

using namespace mgb;

extern "C" {

int mg_amg_strength_count(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                          double theta, int32_t *d_count, void *stream) {
    MG_REQUIRE(n > 0 && d_indptr && d_indices && d_values && d_count, "null argument");
    MG_REQUIRE(theta >= 0.0 && theta < 1.0, "theta must be in [0, 1)");
    amg_strength_count_kernel<<<amg_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, d_indptr, d_indices, d_values,
                                                                                  theta, d_count);
    MG_CHECK_LAUNCH("amg_strength_count");
    return MG_OK;
}

int mg_amg_strength_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                         double theta, const int32_t *d_s_indptr, int32_t *d_s_indices, double *d_s_values,
                         void *stream) {
    MG_REQUIRE(n > 0 && d_indptr && d_indices && d_values && d_s_indptr, "null argument");
    MG_REQUIRE(theta >= 0.0 && theta < 1.0, "theta must be in [0, 1)");
    amg_strength_fill_kernel<<<amg_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, d_indptr, d_indices, d_values,
                                                                                 theta, d_s_indptr, d_s_indices,
                                                                                 d_s_values);
    MG_CHECK_LAUNCH("amg_strength_fill");
    return MG_OK;
}

int mg_amg_pmis(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_t_indptr,
                const int32_t *d_t_indices, const double *d_weights, int32_t *d_state, int32_t *d_work,
                void *stream) {
    MG_REQUIRE(n > 0 && d_s_indptr && d_t_indptr && d_weights && d_state && d_work, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    int32_t *sel = d_work, *flag = d_work + n;
    const unsigned grid = amg_grid(n);
    MG_CHECK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), st));
    amg_pmis_init_kernel<<<grid, kBlock, 0, st>>>(n, d_t_indptr, d_state, flag);
    MG_CHECK_LAUNCH("amg_pmis_init");
    int32_t undecided = 0;                         // 0 or 1: is any point undecided?
    MG_CHECK_CUDA(cudaMemcpyAsync(&undecided, flag, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MG_CHECK_CUDA(cudaStreamSynchronize(st));
    int rounds = 0;
    while (undecided > 0) {
        // the global maximum of (w, i) over the undecided points always turns C, so every round decides a point
        if (rounds > n) return set_error(MG_ERR_INVALID, "mg_amg_pmis", "no progress");
        amg_pmis_select_kernel<<<grid, kBlock, 0, st>>>(n, d_s_indptr, d_s_indices, d_t_indptr, d_t_indices,
                                                         d_weights, d_state, sel);
        MG_CHECK_LAUNCH("amg_pmis_select");
        MG_CHECK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), st));
        amg_pmis_mark_kernel<<<grid, kBlock, 0, st>>>(n, d_s_indptr, d_s_indices, sel, flag);
        MG_CHECK_LAUNCH("amg_pmis_mark");
        MG_CHECK_CUDA(cudaMemcpyAsync(d_state, sel, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        MG_CHECK_CUDA(cudaMemcpyAsync(&undecided, flag, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MG_CHECK_CUDA(cudaStreamSynchronize(st));
        ++rounds;
    }
    return rounds;
}

int mg_amg_promote(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_state,
                   int32_t *d_state_out, int32_t *d_work, void *stream) {
    MG_REQUIRE(n > 0 && d_s_indptr && d_state && d_state_out && d_work && d_state != d_state_out, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    MG_CHECK_CUDA(cudaMemsetAsync(d_work, 0, sizeof(int32_t), st));
    amg_promote_kernel<<<amg_grid(n), kBlock, 0, st>>>(n, d_s_indptr, d_s_indices, d_state, d_state_out, d_work);
    MG_CHECK_LAUNCH("amg_promote");
    int32_t promoted = 0;
    MG_CHECK_CUDA(cudaMemcpyAsync(&promoted, d_work, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MG_CHECK_CUDA(cudaStreamSynchronize(st));
    return promoted;
}

int mg_amg_interp_count(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_state,
                        int32_t *d_count, void *stream) {
    MG_REQUIRE(n > 0 && d_s_indptr && d_state && d_count, "null argument");
    amg_interp_count_kernel<<<amg_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, d_s_indptr, d_s_indices, d_state,
                                                                                d_count);
    MG_CHECK_LAUNCH("amg_interp_count");
    return MG_OK;
}

int mg_amg_interp_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                       const int32_t *d_s_indptr, const int32_t *d_s_indices, const double *d_s_values,
                       const int32_t *d_state, const int32_t *d_cmap, const int32_t *d_q_indptr,
                       int32_t *d_q_indices, double *d_q_values, int32_t *d_work, int64_t *h_bad_row, void *stream) {
    MG_REQUIRE(n > 0 && n < kAmgNoRow && d_indptr && d_indices && d_values && d_s_indptr && d_state && d_cmap &&
               d_q_indptr && d_work && h_bad_row, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    MG_CHECK_CUDA(cudaMemsetAsync(d_work, 0x7f, sizeof(int32_t), st));      // kAmgNoRow
    amg_interp_fill_kernel<<<amg_grid(n), kBlock, 0, st>>>(n, d_indptr, d_indices, d_values, d_s_indptr, d_s_indices,
                                                            d_s_values, d_state, d_cmap, d_q_indptr, d_q_indices,
                                                            d_q_values, d_work);
    MG_CHECK_LAUNCH("amg_interp_fill");
    int32_t bad = kAmgNoRow;
    MG_CHECK_CUDA(cudaMemcpyAsync(&bad, d_work, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MG_CHECK_CUDA(cudaStreamSynchronize(st));
    *h_bad_row = bad == kAmgNoRow ? -1 : (int64_t)bad;
    if (bad != kAmgNoRow) {
        char msg[96];
        snprintf(msg, sizeof(msg), "a_ii + sum of positive off-diagonal entries is 0 in row %d", (int)bad);
        return set_error(MG_ERR_SINGULAR, "mg_amg_interp_fill", msg);
    }
    return MG_OK;
}

}  // extern "C"
