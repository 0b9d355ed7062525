// sell_api.cuh -- what the SELL translation units (sell_kernels.cu, sell_modes_gs.cu, sell_modes_vec.cu) offer to the
// cycle (cycle.cu) and to each other.  Row ranges [row0,row1) are in the matrix' own (colour-blocked) ordering; `fuse`
// is an exchange site riding on the launch (multi-GPU) or NULL.
#pragma once
#include "exchange.cuh"

namespace mgb {

enum SweepTail { TAIL_NONE = 0, TAIL_RESIDUAL = 1, TAIL_NORM = 2 };

// y = A x
int sell_spmv(const mg_sell *A, const double *x, double *y, int64_t row0, int64_t row1, const SellFuse *fuse, cudaStream_t st);
// y = A x and per-CTA partial sums of w . y over the rows (*nblocks of them): the p . A p of conjugate gradients
int sell_spmv_dot(const mg_sell *A, const double *x, const double *w, double *y, double *partials, int *nblocks,
                  const SellFuse *fuse, cudaStream_t st);
// r = b - A x
int sell_residual(const mg_sell *A, const double *x, const double *b, double *r, int64_t row0, int64_t row1,
                  const SellFuse *fuse, cudaStream_t st);
// per-CTA partial sums of (b - A x)_i^2 over the rows; *nblocks = how many were written
int sell_residual_partials(const mg_sell *A, const double *x, const double *b, double *partials, int64_t row0,
                           int64_t row1, int *nblocks, const SellFuse *fuse, cudaStream_t st);
// *out = sum of n partials, fixed order (one CTA)
int sell_reduce_partials(const double *partials, int64_t n, double *out, cudaStream_t st);
int sell_residual_norm2(const mg_sell *A, const double *x, const double *b, double *partials, double *out, cudaStream_t st);
int sell_jacobi(const mg_sell *A, const double *dinv, const double *x, const double *b, double *xo, double omega,
                cudaStream_t st);
// one Chebyshev step (sell_modes_cheby.cu): x_out = x + dn, d = dn; `first` = step 0 (c_d unused, d only written)
int sell_chebyshev(const mg_sell *A, const double *dinv, const double *x, const double *b, double *d, double *xo,
                   double c_d, double c_r, bool first, cudaStream_t st);
// step 0 on a zero iterate without the matrix: d = c_r (dinv b), x_out = 0 + d over n entries
int sell_chebyshev_zero_first(int64_t n, double c_r, const double *dinv, const double *b, double *d, double *xo,
                              cudaStream_t st);
// Gauss-Seidel on the rows of one colour, in place.  tail: also write the residual of these rows (with their new
// values) to r_out, or their squared residuals as per-CTA partial sums (*nblocks of them) -- see sell_gs_tail_ok.
int sell_gs_rows(const mg_sell *A, double *x, const double *b, int64_t row0, int64_t row1, const SellFuse *fuse,
                 int tail, double *r_out, double *partials, int *nblocks, cudaStream_t st);
// uo = u + Q e on the rows
int sell_prolong(const mg_sell *Q, const double *e, const double *u, double *uo, int64_t row0, int64_t row1,
                 const SellFuse *fuse, cudaStream_t st);
// first colour sweep on a zero iterate without the matrix: x = 0 everywhere (n_vec entries) except rows [row0,row1),
// which get b/diag (rows with a zero diagonal stay 0) -- the bits of fill + sweep
int sell_gs_zero_first(int64_t n_vec, int64_t row0, int64_t row1, const double *diag, const double *b, double *x,
                       cudaStream_t st);
bool sell_fusable(const mg_sell *A, int64_t row0, int64_t row1);
bool sell_gs_tail_ok(const mg_sell *A, int64_t row0, int64_t row1);

}  // namespace mgb
