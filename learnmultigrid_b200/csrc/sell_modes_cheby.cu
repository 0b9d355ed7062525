// sell_modes_cheby.cu -- the Chebyshev smoother step of the SELL-32 streaming kernels (sell_core.cuh, mode CHEBY) and
// its first step on a zero iterate, which needs no pass over the matrix.
//
// One step k of the degree-m polynomial in D^-1 A over [lo, hi] (coefficients: formats.chebyshev_coefficients):
//   t  = dinv_i (b_i - sum_j a_ij x_j)      (the residual in the residual kernel's storage order)
//   dn = c_r t                 (k = 0)
//   dn = (c_d d_i) + (c_r t)   (k >= 1)
//   x_out_i = x_i + dn,  d_i = dn
// every product and sum rounded on its own.  The step is out of place in x (other rows read x_j) and in place in d
// (row i alone reads and writes d_i).
#include <string.h>
#include "sell_core.cuh"

namespace mgb {

int sell_chebyshev(const mg_sell *A, const double *dinv, const double *x, const double *b, double *d, double *xo,
                   double c_d, double c_r, bool first, cudaStream_t st) {
    // c_d travels as the bit pattern of the `partials` slot; zero bits mark step 0 (d not read)
    uintptr_t bits = 0;
    if (!first) {
        static_assert(sizeof(uintptr_t) == sizeof(double), "64-bit pointers");
        memcpy(&bits, &c_d, sizeof(bits));
        if (bits == 0) return set_error(MG_ERR_INVALID, "sell_chebyshev", "c_d = +0 after step 0");
    }
    return launch_sell<CHEBY>(A, x, b, dinv, xo, c_r, reinterpret_cast<double *>(bits), 0, A->nrows, st,
                              "sell_chebyshev", nullptr, nullptr, d);
}

// step 0 on a zero iterate: the matrix step with x = 0 has s = +0, r = b - 0 = b, so dn = c_r (dinv b) and
// x_out = 0 + dn -- the same bits without reading the matrix
__global__ void __launch_bounds__(kBlock)
cheby_zero_first_kernel(int64_t n, double c_r, const double *__restrict__ dinv, const double *__restrict__ b,
                        double *__restrict__ d, double *__restrict__ xo) {
    pdl_prologue();
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
        const double dn = __dmul_rn(c_r, __dmul_rn(dinv[i], __dsub_rn(b[i], 0.0)));
        d[i] = dn;
        xo[i] = __dadd_rn(0.0, dn);
    }
}

int sell_chebyshev_zero_first(int64_t n, double c_r, const double *dinv, const double *b, double *d, double *xo,
                              cudaStream_t st) {
    if (n <= 0) return MG_OK;
    int64_t grid = (n + kBlock - 1) / kBlock;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (grid > cap) grid = cap;
    launch_k(cheby_zero_first_kernel, (unsigned)grid, (unsigned)kBlock, st, n, c_r, dinv, b, d, xo);
    MG_CHECK_LAUNCH("cheby_zero_first");
    return MG_OK;
}

}  // namespace mgb

using namespace mgb;

extern "C" {

int mg_sell_chebyshev(const mg_sell *A, const double *d_dinv, const double *d_x, const double *d_b, double *d_d,
                      double *d_x_out, double c_d, double c_r, int first, void *stream) {
    MG_REQUIRE(A && A->nrows >= 0 && (A->nrows == 0 || (A->d_slice_ptr && A->d_cols && A->d_vals)), "null or negative-sized SELL matrix");
    MG_REQUIRE(A->nslices == (A->nrows + kSlice - 1) / kSlice, "nslices != ceil(nrows/32)");
    MG_REQUIRE(d_dinv && d_x && d_b && d_d && d_x_out, "null vector");
    MG_REQUIRE(d_x != d_x_out, "the Chebyshev step is out of place: x_out must not alias x");
    MG_REQUIRE(first || c_d != 0.0, "c_d must be non-zero after step 0");
    return sell_chebyshev(A, d_dinv, d_x, d_b, d_d, d_x_out, c_d, c_r, first != 0, (cudaStream_t)stream);
}

int mg_chebyshev_zero_first(int64_t n, double c_r, const double *d_dinv, const double *d_b, double *d_d,
                            double *d_x_out, void *stream) {
    MG_REQUIRE(n >= 0 && d_dinv && d_b && d_d && d_x_out, "bad argument");
    return sell_chebyshev_zero_first(n, c_r, d_dinv, d_b, d_d, d_x_out, (cudaStream_t)stream);
}

}  // extern "C"
