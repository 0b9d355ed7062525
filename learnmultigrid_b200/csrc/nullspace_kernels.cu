// nullspace_kernels.cu -- removal of a declared null vector from a level vector (singular symmetric operators).
//   v <- v - (nu^T v / nu^T nu) nu, then v[pin] = 0 when pin >= 0
// The dot is accumulated in double-double (error-free products and sums, ~106 bits): per CTA a (hi, lo) pair, then
// one pass in which every CTA sums the same pairs in the same order -- so all CTAs hold the same bits -- and updates its
// rows.  Rounded to a double, the dot then does not depend on how the rows were split into CTAs or over ranks (unless
// the exact value lies within ~1e-30 relative of a rounding boundary): a row-partitioned level 0 removes exactly what
// one GPU removes, and partitioned iterates stay bit-identical to one GPU's.  One GPU: two launches; row-partitioned
// (mg_project_out_dist): the pairs of the ranks are exchanged through the all-reduce site and summed in rank order.
#include "sell_api.cuh"

namespace mgb {

__device__ __forceinline__ void dd_add(double &hi, double &lo, double bh, double bl) {
    const double s = hi + bh;                      // two-sum of the high parts
    const double bb = s - hi;
    const double e = (hi - (s - bb)) + (bh - bb);
    const double t = e + lo + bl;
    hi = s + t;                                    // renormalise
    lo = t - (hi - s);
}

// (hi, lo) summed over the CTA (fixed tree); valid in thread 0
template <int BLOCK>
__device__ __forceinline__ void dd_block_sum(double &hi, double &lo) {
    __shared__ double sh[2][BLOCK];
    sh[0][threadIdx.x] = hi;
    sh[1][threadIdx.x] = lo;
    __syncthreads();
#pragma unroll
    for (int s = BLOCK / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            double h = sh[0][threadIdx.x], l = sh[1][threadIdx.x];
            dd_add(h, l, sh[0][threadIdx.x + s], sh[1][threadIdx.x + s]);
            sh[0][threadIdx.x] = h;
            sh[1][threadIdx.x] = l;
        }
        __syncthreads();
    }
    hi = sh[0][0];
    lo = sh[1][0];
    __syncthreads();
}

// pairs[2 * blockIdx.x .. +1] = the CTA's share of nu^T v in double-double
__global__ void __launch_bounds__(kBlock)
dd_dot_partials_kernel(int64_t n, const double *__restrict__ nu, const double *__restrict__ v, double *__restrict__ pairs) {
    pdl_prologue();
    double hi = 0.0, lo = 0.0;
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
        const double p = nu[i] * v[i];
        const double pe = fma(nu[i], v[i], -p);    // error-free product
        dd_add(hi, lo, p, pe);
    }
    dd_block_sum<kBlock>(hi, lo);
    if (threadIdx.x == 0) {
        pairs[2 * blockIdx.x] = hi;
        pairs[2 * blockIdx.x + 1] = lo;
    }
}

// the sum of npairs (hi, lo) pairs in a fixed order, by every thread of the CTA (same bits in every CTA)
__device__ __forceinline__ double dd_sum_pairs(const double *__restrict__ pairs, int npairs) {
    double hi = 0.0, lo = 0.0;
    for (int i = threadIdx.x; i < npairs; i += kBlock) dd_add(hi, lo, pairs[2 * i], pairs[2 * i + 1]);
    dd_block_sum<kBlock>(hi, lo);
    return hi + lo;
}

// one CTA: out[0..1] = the sum of the pairs as a pair; copy[0..1] too (a rank's own slot of the all-reduce)
__global__ void __launch_bounds__(kBlock) dd_reduce_pairs_kernel(const double *__restrict__ pairs, int npairs,
                                                                 double *__restrict__ out, double *__restrict__ copy) {
    pdl_prologue();
    double hi = 0.0, lo = 0.0;
    for (int i = threadIdx.x; i < npairs; i += kBlock) dd_add(hi, lo, pairs[2 * i], pairs[2 * i + 1]);
    dd_block_sum<kBlock>(hi, lo);
    if (threadIdx.x == 0) {
        out[0] = hi;
        out[1] = lo;
        copy[0] = hi;
        copy[1] = lo;
    }
}

__global__ void __launch_bounds__(kBlock)
project_out_kernel(int64_t n, const double *__restrict__ nu, double inv_nn, int64_t pin, double *__restrict__ v,
                   const double *__restrict__ pairs, int npairs, double *__restrict__ dot_out) {
    pdl_prologue();
    const double s = dd_sum_pairs(pairs, npairs);
    if (dot_out && blockIdx.x == 0 && threadIdx.x == 0) *dot_out = s;
    const double c = __dmul_rn(s, inv_nn);
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride)
        v[i] = (i == pin) ? 0.0 : __dadd_rn(v[i], -__dmul_rn(c, nu[i]));
}

static inline unsigned project_grid(int64_t n) {
    int64_t g = (n + kBlock - 1) / kBlock;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

int null_project(int64_t n, const double *nu, double inv_nn, int64_t pin, double *v, double *partials, cudaStream_t st,
                 double *dot_out) {
    if (n <= 0) return MG_OK;
    const unsigned g = project_grid(n);
    launch_k(dd_dot_partials_kernel, g, (unsigned)kBlock, st, n, nu, (const double *)v, partials);
    MG_CHECK_LAUNCH("dd_dot_partials");
    launch_k(project_out_kernel, g, (unsigned)kBlock, st, n, nu, inv_nn, pin, v, (const double *)partials, (int)g,
             dot_out);
    MG_CHECK_LAUNCH("project_out");
    return MG_OK;
}

}  // namespace mgb

using namespace mgb;

extern "C" {

int64_t mg_project_workspace_size(int64_t n) { return 2 * (int64_t)project_grid(n < 1 ? 1 : n) + 4; }

int mg_project_out(int64_t n, const double *d_nu, double inv_nn, int64_t pin, double *d_v, double *d_partials,
                   double *d_dot, void *stream) {
    MG_REQUIRE(n >= 0 && pin < n, "bad size or pin");
    MG_REQUIRE(n == 0 || (d_nu && d_v && d_partials), "null pointer");
    return null_project(n, d_nu, inv_nn, pin, d_v, d_partials, (cudaStream_t)stream, d_dot);
}

int mg_project_out_dist(mg_comm *comm, int64_t n, const double *d_nu, double inv_nn, int64_t pin, double *d_v,
                        double *d_partials, double *d_slots, double *d_dot, void *stream) {
    MG_REQUIRE(comm && d_nu && d_v && d_partials && d_slots, "null pointer");
    MG_REQUIRE(n > 0 && pin < n, "bad size or pin");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned g = project_grid(n);
    int rc = mg_comm_begin(comm);
    if (rc) return rc;
    launch_k(dd_dot_partials_kernel, g, (unsigned)kBlock, st, n, d_nu, (const double *)d_v, d_partials);
    MG_CHECK_LAUNCH("dd_dot_partials");
    // this rank's pair goes to d_partials[2g..2g+1] (sent) and to its own slot of d_slots (the others' land there)
    double *local = d_partials + 2 * (int64_t)g;
    launch_k(dd_reduce_pairs_kernel, 1u, (unsigned)kBlock, st, (const double *)d_partials, (int)g, local,
             d_slots + 2 * comm->rank);
    MG_CHECK_LAUNCH("dd_reduce_pairs");
    if (comm->world > 1) {
        rc = mg_comm_allreduce_sum_n(comm, local, 2, d_slots, local + 2, stream);   // the others' pairs -> d_slots
        if (rc) return rc;
    }
    launch_k(project_out_kernel, g, (unsigned)kBlock, st, n, d_nu, inv_nn, pin, d_v, (const double *)d_slots,
             (int)comm->world, d_dot);
    MG_CHECK_LAUNCH("project_out");
    return mg_comm_end(comm, stream);
}

}  // extern "C"
