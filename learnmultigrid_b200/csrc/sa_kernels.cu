// sa_kernels.cu -- smoothed aggregation setup on the device: symmetric strength of connection, MIS(2) by the tuple
// algorithm of Bell, Dalton and Olson (2012), aggregation around the MIS(2) roots, the tentative prolongator and the
// Jacobi smoothing of its operator (learnmultigrid_b200/sa.py drives them level by level; DESIGN.md §4.11).
//
// One thread per row (or per aggregate) over CSR with sorted columns, in the style of amg_kernels.cu, so that
// tests/sa_oracle.py (NumPy, written from the definition in DESIGN.md) and the device agree bit for bit:
//   strength   j != i is strong for i iff a_ij != 0 and a_ij * a_ij >= theta^2 * (|a_ii| * |a_jj|);
//   MIS(2)     keys (state, r_i, i), OUT = 0 < UNDECIDED = 1 < IN = 2; per round two max-propagation passes over
//              {i} u S_i u S^T_i and one update (an undecided i turns IN if the propagated maximum is its own key, OUT
//              if the maximum's state is IN);
//   aggregate  pass 1: a point with a root among its neighbours joins it; pass 2: a point still unassigned joins the
//              aggregate of its pass-1 neighbour with the largest (r_j, j);
//   tentative  nu_a = sqrt(sum_{i in a} B_i * B_i) in ascending i, T[i, agg(i)] = B_i / nu_agg(i);
//   smoothing  s_i = omega_hat / a_ii, At_ij = -(s_i * a_ij) (j != i), At_ii = 1 - s_i * a_ii.
// Products, sums, quotients and square roots are rounded one at a time (no FMA contraction).
//
// r_i = formats.chebyshev_start_vector(i) + 0.5 is h(i) / 2^32 for a 32-bit integer hash h.  Every step of h (a product
// with an odd constant mod 2^32, a xor-shift) is a bijection of the 32-bit integers, so h never ties for indices below
// 2^31: the key (state, r_i, i) is ordered exactly as the 64-bit integer (state << 32) | h(i), which is what the passes
// propagate.
#include "common.cuh"

namespace mgb {

enum SaState : int32_t { SA_OUT = 0, SA_UNDECIDED = 1, SA_IN = 2 };

// formats.chebyshev_start_vector's hash (mod 2^32 arithmetic)
__device__ inline uint32_t sa_hash(int64_t i) {
    uint32_t h = (uint32_t)i * 2654435761u;
    h ^= h >> 16;
    h *= 0x45d9f3bu;
    h ^= h >> 16;
    h *= 0x45d9f3bu;
    h ^= h >> 16;
    return h;
}

__device__ inline uint64_t sa_key(int32_t state, int64_t i) {
    return ((uint64_t)(uint32_t)state << 32) | (uint64_t)sa_hash(i);
}

__device__ inline bool sa_is_strong(int64_t i, int32_t j, double a_ij, double a_ii, double a_jj, double theta2) {
    return j != i && a_ij != 0.0 && __dmul_rn(a_ij, a_ij) >= __dmul_rn(theta2, __dmul_rn(fabs(a_ii), fabs(a_jj)));
}

__device__ inline bool sa_isolated(const int32_t *s_ptr, const int32_t *t_ptr, int64_t i) {
    return s_ptr[i + 1] == s_ptr[i] && t_ptr[i + 1] == t_ptr[i];
}

// ---- kernels ---------------------------------------------------------------------------------------------------------
// the stored diagonal entry of every row (0 where none is stored)
__global__ void __launch_bounds__(kBlock)
sa_diagonal_kernel(int64_t n, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                   const double *__restrict__ values, double *__restrict__ diag) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    double d = 0.0;
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p)
        if (indices[p] == i) d = values[p];
    diag[i] = d;
}

__global__ void __launch_bounds__(kBlock)
sa_strength_count_kernel(int64_t n, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                         const double *__restrict__ values, const double *__restrict__ diag, double theta2,
                         int32_t *__restrict__ count) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const double a_ii = diag[i];
    int32_t c = 0;
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p) {
        const int32_t j = indices[p];
        if (sa_is_strong(i, j, values[p], a_ii, diag[j], theta2)) ++c;
    }
    count[i] = c;
}

__global__ void __launch_bounds__(kBlock)
sa_strength_fill_kernel(int64_t n, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                        const double *__restrict__ values, const double *__restrict__ diag, double theta2,
                        const int32_t *__restrict__ s_ptr, int32_t *__restrict__ s_idx, double *__restrict__ s_val) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const double a_ii = diag[i];
    int32_t q = s_ptr[i];
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p) {
        const int32_t j = indices[p];
        const double a = values[p];
        if (sa_is_strong(i, j, a, a_ii, diag[j], theta2)) {
            s_idx[q] = j;
            s_val[q] = a;
            ++q;
        }
    }
}

// isolated points (empty S_i and S^T_i) start OUT, the others undecided; *any_undecided = 1 if a point is undecided
__global__ void __launch_bounds__(kBlock)
sa_mis2_init_kernel(int64_t n, const int32_t *__restrict__ s_ptr, const int32_t *__restrict__ t_ptr,
                    int32_t *__restrict__ state, int32_t *__restrict__ any_undecided) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const bool u = !sa_isolated(s_ptr, t_ptr, i);
    state[i] = u ? SA_UNDECIDED : SA_OUT;
    if (u) *any_undecided = 1;
}

// k_out[i] = max over {i} u S_i u S^T_i of the keys: those of the round's states (kFirst) or k_in
template <bool kFirst>
__global__ void __launch_bounds__(kBlock)
sa_mis2_propagate_kernel(int64_t n, const int32_t *__restrict__ s_ptr, const int32_t *__restrict__ s_idx,
                         const int32_t *__restrict__ t_ptr, const int32_t *__restrict__ t_idx,
                         const int32_t *__restrict__ state, const uint64_t *__restrict__ k_in,
                         uint64_t *__restrict__ k_out) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    uint64_t m = kFirst ? sa_key(state[i], i) : k_in[i];
    for (int32_t p = s_ptr[i]; p < s_ptr[i + 1]; ++p) {
        const int32_t j = s_idx[p];
        const uint64_t k = kFirst ? sa_key(state[j], j) : k_in[j];
        m = k > m ? k : m;
    }
    for (int32_t p = t_ptr[i]; p < t_ptr[i + 1]; ++p) {
        const int32_t j = t_idx[p];
        const uint64_t k = kFirst ? sa_key(state[j], j) : k_in[j];
        m = k > m ? k : m;
    }
    k_out[i] = m;
}

// reads the round's states, writes another buffer
__global__ void __launch_bounds__(kBlock)
sa_mis2_update_kernel(int64_t n, const int32_t *__restrict__ state_in, const uint64_t *__restrict__ k2,
                      int32_t *__restrict__ state_out, int32_t *__restrict__ any_undecided) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    int32_t s = state_in[i];
    if (s == SA_UNDECIDED) {
        const uint64_t m = k2[i];
        if (m == sa_key(SA_UNDECIDED, i)) s = SA_IN;
        else if ((int32_t)(m >> 32) == SA_IN) s = SA_OUT;
        else *any_undecided = 1;
    }
    state_out[i] = s;
}

// pass 1: a root keeps its own aggregate; a non-root with a root in S_i u S^T_i joins that root's (the root must be
// unique: two distinct roots flag the row in bad[0]); every other point is left unassigned (-1)
__global__ void __launch_bounds__(kBlock)
sa_aggregate_pass1_kernel(int64_t n, const int32_t *__restrict__ s_ptr, const int32_t *__restrict__ s_idx,
                          const int32_t *__restrict__ t_ptr, const int32_t *__restrict__ t_idx,
                          const int32_t *__restrict__ state, const int32_t *__restrict__ cmap,
                          int32_t *__restrict__ agg, int32_t *__restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    if (state[i] == SA_IN) {
        agg[i] = cmap[i];
        return;
    }
    int32_t root = -1;
    bool twice = false;
    for (int32_t p = s_ptr[i]; p < s_ptr[i + 1]; ++p) {
        const int32_t j = s_idx[p];
        if (state[j] == SA_IN) {
            twice |= root >= 0 && root != j;
            root = j;
        }
    }
    for (int32_t p = t_ptr[i]; p < t_ptr[i + 1]; ++p) {
        const int32_t j = t_idx[p];
        if (state[j] == SA_IN) {
            twice |= root >= 0 && root != j;
            root = j;
        }
    }
    if (twice) atomicMin(bad, (int32_t)i);
    agg[i] = root >= 0 ? cmap[root] : -1;
}

// pass 2, from the pass-1 results only: an unassigned non-isolated point joins the aggregate of its assigned neighbour
// with the largest (r_j, j); one that has none flags its row in bad[1]
__global__ void __launch_bounds__(kBlock)
sa_aggregate_pass2_kernel(int64_t n, const int32_t *__restrict__ s_ptr, const int32_t *__restrict__ s_idx,
                          const int32_t *__restrict__ t_ptr, const int32_t *__restrict__ t_idx,
                          const int32_t *__restrict__ agg1, int32_t *__restrict__ agg, int32_t *__restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    int32_t a = agg1[i];
    if (a < 0 && !sa_isolated(s_ptr, t_ptr, i)) {
        uint64_t best = 0;                          // keys of assigned points are h(j) + 1 >= 1
        for (int32_t p = s_ptr[i]; p < s_ptr[i + 1]; ++p) {
            const int32_t j = s_idx[p], aj = agg1[j];
            const uint64_t k = (uint64_t)sa_hash(j) + 1;
            if (aj >= 0 && k > best) { best = k; a = aj; }
        }
        for (int32_t p = t_ptr[i]; p < t_ptr[i + 1]; ++p) {
            const int32_t j = t_idx[p], aj = agg1[j];
            const uint64_t k = (uint64_t)sa_hash(j) + 1;
            if (aj >= 0 && k > best) { best = k; a = aj; }
        }
        if (a < 0) atomicMin(bad + 1, (int32_t)i);
    }
    agg[i] = a;
}

// one thread per aggregate over the rows of T^T (members ascending, values B_i): nu_a = sqrt(sum B_i * B_i)
__global__ void __launch_bounds__(kBlock)
sa_aggregate_norm_kernel(int64_t nc, const int32_t *__restrict__ tt_ptr, const double *__restrict__ tt_val,
                         double *__restrict__ nu) {
    const int64_t a = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (a >= nc) return;
    double s = 0.0;
    for (int32_t p = tt_ptr[a]; p < tt_ptr[a + 1]; ++p) s = __dadd_rn(s, __dmul_rn(tt_val[p], tt_val[p]));
    nu[a] = __dsqrt_rn(s);
}

// T's row i: column agg[i], value B_i / nu[agg[i]] (B_i itself where nu is null); rows with agg[i] < 0 are empty
__global__ void __launch_bounds__(kBlock)
sa_tentative_fill_kernel(int64_t n, const int32_t *__restrict__ agg, const int32_t *__restrict__ t_ptr,
                         const double *__restrict__ b, const double *__restrict__ nu, int32_t *__restrict__ t_idx,
                         double *__restrict__ t_val) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const int32_t a = agg[i];
    if (a < 0) return;
    const int32_t q = t_ptr[i];
    t_idx[q] = a;
    t_val[q] = nu ? __ddiv_rn(b[i], nu[a]) : b[i];
}

// the values of I - omega_hat D^-1 A on A's pattern
__global__ void __launch_bounds__(kBlock)
sa_smooth_scale_kernel(int64_t n, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                       const double *__restrict__ values, const double *__restrict__ diag, double omega_hat,
                       double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= n) return;
    const double s = __ddiv_rn(omega_hat, diag[i]);
    for (int32_t p = indptr[i]; p < indptr[i + 1]; ++p) {
        const double sa = __dmul_rn(s, values[p]);
        out[p] = indices[p] == i ? __dadd_rn(1.0, -sa) : -sa;
    }
}

constexpr int32_t kSaNoRow = 0x7f7f7f7f;     // "no flagged row": every byte 0x7f, so one memset sets it

inline unsigned sa_grid(int64_t n) { return (unsigned)((n + kBlock - 1) / kBlock); }

}  // namespace mgb

using namespace mgb;

extern "C" {

int mg_sa_diagonal(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                   double *d_diag, void *stream) {
    MG_REQUIRE(n > 0 && d_indptr && d_indices && d_values && d_diag, "null argument");
    sa_diagonal_kernel<<<sa_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, d_indptr, d_indices, d_values, d_diag);
    MG_CHECK_LAUNCH("sa_diagonal");
    return MG_OK;
}

int mg_sa_strength_count(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                         const double *d_diag, double theta, int32_t *d_count, void *stream) {
    MG_REQUIRE(n > 0 && d_indptr && d_indices && d_values && d_diag && d_count, "null argument");
    MG_REQUIRE(theta >= 0.0 && theta < 1.0, "theta must be in [0, 1)");
    sa_strength_count_kernel<<<sa_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, d_indptr, d_indices, d_values,
                                                                                d_diag, theta * theta, d_count);
    MG_CHECK_LAUNCH("sa_strength_count");
    return MG_OK;
}

int mg_sa_strength_fill(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                        const double *d_diag, double theta, const int32_t *d_s_indptr, int32_t *d_s_indices,
                        double *d_s_values, void *stream) {
    MG_REQUIRE(n > 0 && d_indptr && d_indices && d_values && d_diag && d_s_indptr, "null argument");
    MG_REQUIRE(theta >= 0.0 && theta < 1.0, "theta must be in [0, 1)");
    sa_strength_fill_kernel<<<sa_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, d_indptr, d_indices, d_values, d_diag,
                                                                               theta * theta, d_s_indptr, d_s_indices,
                                                                               d_s_values);
    MG_CHECK_LAUNCH("sa_strength_fill");
    return MG_OK;
}

int mg_sa_mis2(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_t_indptr,
               const int32_t *d_t_indices, int32_t *d_state, int32_t *d_work, uint64_t *d_keys, void *stream) {
    MG_REQUIRE(n > 0 && n < (int64_t)1 << 31 && d_s_indptr && d_t_indptr && d_state && d_work && d_keys,
               "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    int32_t *next = d_work, *flag = d_work + n;
    uint64_t *k1 = d_keys, *k2 = d_keys + n;
    const unsigned grid = sa_grid(n);
    MG_CHECK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), st));
    sa_mis2_init_kernel<<<grid, kBlock, 0, st>>>(n, d_s_indptr, d_t_indptr, d_state, flag);
    MG_CHECK_LAUNCH("sa_mis2_init");
    int32_t undecided = 0;                         // 0 or 1: is any point undecided?
    MG_CHECK_CUDA(cudaMemcpyAsync(&undecided, flag, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MG_CHECK_CUDA(cudaStreamSynchronize(st));
    int rounds = 0;
    while (undecided > 0) {
        // the undecided point with the largest key turns IN or has an IN point within distance 2: every round decides
        if (rounds > n) return set_error(MG_ERR_INVALID, "mg_sa_mis2", "no progress");
        sa_mis2_propagate_kernel<true><<<grid, kBlock, 0, st>>>(n, d_s_indptr, d_s_indices, d_t_indptr, d_t_indices,
                                                                d_state, nullptr, k1);
        MG_CHECK_LAUNCH("sa_mis2_propagate");
        sa_mis2_propagate_kernel<false><<<grid, kBlock, 0, st>>>(n, d_s_indptr, d_s_indices, d_t_indptr,
                                                                 d_t_indices, nullptr, k1, k2);
        MG_CHECK_LAUNCH("sa_mis2_propagate");
        MG_CHECK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), st));
        sa_mis2_update_kernel<<<grid, kBlock, 0, st>>>(n, d_state, k2, next, flag);
        MG_CHECK_LAUNCH("sa_mis2_update");
        MG_CHECK_CUDA(cudaMemcpyAsync(d_state, next, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        MG_CHECK_CUDA(cudaMemcpyAsync(&undecided, flag, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MG_CHECK_CUDA(cudaStreamSynchronize(st));
        ++rounds;
    }
    return rounds;
}

int mg_sa_aggregate(int64_t n, const int32_t *d_s_indptr, const int32_t *d_s_indices, const int32_t *d_t_indptr,
                    const int32_t *d_t_indices, const int32_t *d_state, const int32_t *d_cmap, int32_t *d_agg,
                    int32_t *d_work, int64_t *h_bad_row, void *stream) {
    MG_REQUIRE(n > 0 && n < kSaNoRow && d_s_indptr && d_t_indptr && d_state && d_cmap && d_agg && d_work &&
               h_bad_row, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    int32_t *agg1 = d_work, *bad = d_work + n;
    MG_CHECK_CUDA(cudaMemsetAsync(bad, 0x7f, 2 * sizeof(int32_t), st));      // kSaNoRow, twice
    sa_aggregate_pass1_kernel<<<sa_grid(n), kBlock, 0, st>>>(n, d_s_indptr, d_s_indices, d_t_indptr, d_t_indices,
                                                             d_state, d_cmap, agg1, bad);
    MG_CHECK_LAUNCH("sa_aggregate_pass1");
    sa_aggregate_pass2_kernel<<<sa_grid(n), kBlock, 0, st>>>(n, d_s_indptr, d_s_indices, d_t_indptr, d_t_indices,
                                                             agg1, d_agg, bad);
    MG_CHECK_LAUNCH("sa_aggregate_pass2");
    int32_t hb[2] = {kSaNoRow, kSaNoRow};
    MG_CHECK_CUDA(cudaMemcpyAsync(hb, bad, sizeof(hb), cudaMemcpyDeviceToHost, st));
    MG_CHECK_CUDA(cudaStreamSynchronize(st));
    *h_bad_row = -1;
    char msg[96];
    if (hb[0] != kSaNoRow) {
        *h_bad_row = hb[0];
        snprintf(msg, sizeof(msg), "point %d has two roots among its neighbours", (int)hb[0]);
        return set_error(MG_ERR_INVALID, "mg_sa_aggregate", msg);
    }
    if (hb[1] != kSaNoRow) {
        *h_bad_row = hb[1];
        snprintf(msg, sizeof(msg), "point %d is left unassigned", (int)hb[1]);
        return set_error(MG_ERR_INVALID, "mg_sa_aggregate", msg);
    }
    return MG_OK;
}

int mg_sa_aggregate_norm(int64_t nc, const int32_t *d_tt_indptr, const double *d_tt_values, double *d_nu,
                         void *stream) {
    MG_REQUIRE(nc > 0 && d_tt_indptr && d_tt_values && d_nu, "null argument");
    sa_aggregate_norm_kernel<<<sa_grid(nc), kBlock, 0, (cudaStream_t)stream>>>(nc, d_tt_indptr, d_tt_values, d_nu);
    MG_CHECK_LAUNCH("sa_aggregate_norm");
    return MG_OK;
}

int mg_sa_tentative_fill(int64_t n, const int32_t *d_agg, const int32_t *d_t_indptr, const double *d_b,
                         const double *d_nu, int32_t *d_t_indices, double *d_t_values, void *stream) {
    MG_REQUIRE(n > 0 && d_agg && d_t_indptr && d_b && d_t_indices && d_t_values, "null argument");
    sa_tentative_fill_kernel<<<sa_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, d_agg, d_t_indptr, d_b, d_nu,
                                                                                d_t_indices, d_t_values);
    MG_CHECK_LAUNCH("sa_tentative_fill");
    return MG_OK;
}

int mg_sa_smooth_scale(int64_t n, const int32_t *d_indptr, const int32_t *d_indices, const double *d_values,
                       const double *d_diag, double omega_hat, double *d_out_values, void *stream) {
    MG_REQUIRE(n > 0 && d_indptr && d_indices && d_values && d_diag && d_out_values, "null argument");
    sa_smooth_scale_kernel<<<sa_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, d_indptr, d_indices, d_values, d_diag,
                                                                              omega_hat, d_out_values);
    MG_CHECK_LAUNCH("sa_smooth_scale");
    return MG_OK;
}

}  // extern "C"
