// krylov_kernels.cu -- the vector work of restarted GMRES (cycle.cu mg_gmres_*): Gram-Schmidt against many basis
// vectors per pass, the Givens step, the scaling of the new basis vector and the final update of x.
// The basis is one column-major buffer: vector k starts at V + k * ld.  Every sum runs in a fixed order (each CTA owns
// fixed row chunks, the per-CTA partials are added in index order), so a run repeats its bits; every product, sum,
// quotient and square root is rounded on its own, as in tests/gmres_oracle.py.
#include "common.cuh"

namespace mgb {

// Basis vectors one thread accumulates in registers per pass over w (8 doubles = 16 registers; ptxas -v: no spills).
constexpr int kDotTile = 8;

static inline unsigned krylov_grid(int64_t n) {
    int64_t g = (n + kBlock - 1) / kBlock;
    const int64_t cap = (int64_t)sm_count() * 8;   // 8 resident CTAs of 256 threads per SM
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

// partials[k * nb + c] = sum over the rows of CTA c of V[k][i] * w[i], k < m.  CTA blockIdx.x = tile * nb + c handles
// the vectors [tile * kDotTile, ...) and reads w once for all of them.
__global__ void __launch_bounds__(kBlock)
multi_dot_kernel(int64_t n, const double *__restrict__ V, int64_t ld, int m, int nb, const double *__restrict__ w,
                 double *__restrict__ partials) {
    pdl_prologue();
    const int tile = blockIdx.x / nb, c = blockIdx.x - tile * nb;
    const int k0 = tile * kDotTile;
    const int mt = m - k0 < kDotTile ? m - k0 : kDotTile;
    double acc[kDotTile];
#pragma unroll
    for (int t = 0; t < kDotTile; ++t) acc[t] = 0.0;
    const double *Vt = V + (int64_t)k0 * ld;
    const int64_t stride = (int64_t)nb * kBlock;
    for (int64_t i = (int64_t)c * kBlock + threadIdx.x; i < n; i += stride) {
        const double wi = w[i];
#pragma unroll
        for (int t = 0; t < kDotTile; ++t)
            if (t < mt) acc[t] = mul_add_unfused(acc[t], Vt[(int64_t)t * ld + i], wi);
    }
    __shared__ double sh[kDotTile][kBlock / 32];
    const int wp = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll
    for (int t = 0; t < kDotTile; ++t) {
        double v = acc[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (l == 0) sh[t][wp] = v;
    }
    __syncthreads();
    if (threadIdx.x < mt) {
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < kBlock / 32; ++q) s += sh[threadIdx.x][q];
        partials[(int64_t)(k0 + threadIdx.x) * nb + c] = s;
    }
}

// out[k] = sum of partials[k * nb .. (k+1) * nb) in a fixed order, one CTA per column (nb <= 8 * SMs: one stage)
__global__ void __launch_bounds__(1024)
reduce_columns_kernel(const double *__restrict__ partials, int nb, double *__restrict__ out) {
    pdl_prologue();
    const double *p = partials + (int64_t)blockIdx.x * nb;
    double s = 0.0;
    for (int i = threadIdx.x; i < nb; i += 1024) s += p[i];
    s = block_sum<1024>(s);
    if (threadIdx.x == 0) out[blockIdx.x] = s;
}

// w -= h_0 v_0, w -= h_1 v_1, ... (classical Gram-Schmidt, one pass) and the per-CTA partials of ||w||^2 of the result
__global__ void __launch_bounds__(kBlock)
multi_axpy_norm_kernel(int64_t n, const double *__restrict__ V, int64_t ld, int m, const double *__restrict__ h,
                       double *__restrict__ w, double *__restrict__ partials) {
    pdl_prologue();
    double acc = 0.0;
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
        double wi = w[i];
        int k = 0;
        for (; k + kDotTile <= m; k += kDotTile) {
            double v[kDotTile];
#pragma unroll
            for (int t = 0; t < kDotTile; ++t) v[t] = V[(int64_t)(k + t) * ld + i];     // all loads in flight first
#pragma unroll
            for (int t = 0; t < kDotTile; ++t) wi = __dsub_rn(wi, __dmul_rn(h[k + t], v[t]));
        }
        for (; k < m; ++k) wi = __dsub_rn(wi, __dmul_rn(h[k], V[(int64_t)k * ld + i]));
        w[i] = wi;
        acc += wi * wi;
    }
    acc = block_sum_last<kBlock>(acc);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}

// v /= *h, skipped when *h == 0 (lucky breakdown: the new vector is zero and is never used)
__global__ void __launch_bounds__(kBlock) scale_inv_kernel(int64_t n, const double *__restrict__ h, double *__restrict__ v) {
    pdl_prologue();
    const double d = *h;
    if (d == 0.0) return;
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) v[i] = __ddiv_rn(v[i], d);
}

// Scalars s[]: [0] the squared residual the host reads (beta^2 after a start, |g_{j+1}|^2 after step j)  [1] the
// divisor of the next basis vector (beta, or h_{j+1,j})  [2] this rank's sum of squares  [3] the sum over the ranks.
// Start of a cycle: g = beta e_1 with beta = sqrt(*nrm2).
__global__ void gmres_start_kernel(const double *nrm2, double *g, int restart, double *s) {
    pdl_prologue();
    if (blockIdx.x != 0) return;
    const double r2 = *nrm2, beta = __dsqrt_rn(r2);
    for (int i = threadIdx.x; i <= restart; i += blockDim.x) g[i] = i == 0 ? beta : 0.0;
    if (threadIdx.x == 0) {
        s[0] = r2;
        s[1] = beta;
    }
}

// Step j of the Hessenberg QR: h_{j+1,j} = sqrt(*nrm2), the j earlier rotations applied to column j, the new rotation
// (t = sqrt(a a + b b), c = a / t, s = b / t) and g updated.  H is column-major with leading dimension ldh.
__global__ void gmres_givens_kernel(double *H, int ldh, int j, double *cs, double *sn, double *g, const double *nrm2,
                                    double *s) {
    pdl_prologue();
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double *h = H + (int64_t)j * ldh;
    const double hn = __dsqrt_rn(*nrm2);
    for (int i = 0; i < j; ++i) {
        const double a = h[i], b = h[i + 1], c = cs[i], sg = sn[i];
        h[i] = __dadd_rn(__dmul_rn(c, a), __dmul_rn(sg, b));
        h[i + 1] = __dadd_rn(__dmul_rn(-sg, a), __dmul_rn(c, b));
    }
    const double a = h[j], b = hn;
    const double t = __dsqrt_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)));
    const double c = t == 0.0 ? 1.0 : __ddiv_rn(a, t), sg = t == 0.0 ? 0.0 : __ddiv_rn(b, t);
    cs[j] = c;
    sn[j] = sg;
    h[j] = t;
    h[j + 1] = 0.0;
    const double gj = g[j], gn = __dmul_rn(-sg, gj);
    g[j] = __dmul_rn(c, gj);
    g[j + 1] = gn;
    s[0] = __dmul_rn(gn, gn);
    s[1] = hn;
}

// R y = g by back substitution over the k x k upper triangle of H: y_i = (g_i - sum_{c>i} R_ic y_c) / R_ii, the sum
// taken for c = i+1, i+2, ... (one thread: k is the restart length)
__global__ void gmres_backsub_kernel(const double *H, int ldh, const double *g, int k, double *y) {
    pdl_prologue();
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    for (int i = k - 1; i >= 0; --i) {
        double r = g[i];
        for (int c = i + 1; c < k; ++c) r = __dsub_rn(r, __dmul_rn(H[(int64_t)c * ldh + i], y[c]));
        y[i] = __ddiv_rn(r, H[(int64_t)i * ldh + i]);
    }
}

// x += y_0 z_0, x += y_1 z_1, ... in one pass over the basis
__global__ void __launch_bounds__(kBlock)
multi_axpy_update_kernel(int64_t n, const double *__restrict__ Z, int64_t ld, int k, const double *__restrict__ y,
                         double *__restrict__ x) {
    pdl_prologue();
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
        double xi = x[i];
        int c = 0;
        for (; c + kDotTile <= k; c += kDotTile) {
            double v[kDotTile];
#pragma unroll
            for (int t = 0; t < kDotTile; ++t) v[t] = Z[(int64_t)(c + t) * ld + i];
#pragma unroll
            for (int t = 0; t < kDotTile; ++t) xi = __dadd_rn(xi, __dmul_rn(y[c + t], v[t]));
        }
        for (; c < k; ++c) xi = __dadd_rn(xi, __dmul_rn(y[c], Z[(int64_t)c * ld + i]));
        x[i] = xi;
    }
}

int64_t krylov_partials(int64_t n, int m) { return (int64_t)krylov_grid(n) * (m > 1 ? m : 1); }

int krylov_multi_dot(int64_t n, const double *V, int64_t ld, int m, const double *w, double *partials, double *out,
                     cudaStream_t st) {
    if (m <= 0) return MG_OK;
    const unsigned nb = krylov_grid(n), tiles = (unsigned)((m + kDotTile - 1) / kDotTile);
    launch_k(multi_dot_kernel, nb * tiles, (unsigned)kBlock, st, n, V, ld, m, (int)nb, w, partials);
    MG_CHECK_LAUNCH("multi_dot");
    launch_k(reduce_columns_kernel, (unsigned)m, 1024u, st, (const double *)partials, (int)nb, out);
    MG_CHECK_LAUNCH("reduce_columns");
    return MG_OK;
}
int krylov_multi_axpy_norm(int64_t n, const double *V, int64_t ld, int m, const double *h, double *w, double *partials,
                           double *norm2, cudaStream_t st) {
    const unsigned nb = krylov_grid(n);
    launch_k(multi_axpy_norm_kernel, nb, (unsigned)kBlock, st, n, V, ld, m, h, w, partials);
    MG_CHECK_LAUNCH("multi_axpy_norm");
    launch_k(reduce_columns_kernel, 1u, 1024u, st, (const double *)partials, (int)nb, norm2);
    MG_CHECK_LAUNCH("reduce_columns");
    return MG_OK;
}
int krylov_scale_inv(int64_t n, const double *h, double *v, cudaStream_t st) {
    launch_k(scale_inv_kernel, krylov_grid(n), (unsigned)kBlock, st, n, h, v);
    MG_CHECK_LAUNCH("scale_inv");
    return MG_OK;
}
int krylov_gmres_start(const double *nrm2, double *g, int restart, double *s, cudaStream_t st) {
    launch_k(gmres_start_kernel, 1u, 128u, st, nrm2, g, restart, s);
    MG_CHECK_LAUNCH("gmres_start");
    return MG_OK;
}
int krylov_givens(double *H, int ldh, int j, double *cs, double *sn, double *g, const double *nrm2, double *s,
                  cudaStream_t st) {
    launch_k(gmres_givens_kernel, 1u, 32u, st, H, ldh, j, cs, sn, g, nrm2, s);
    MG_CHECK_LAUNCH("gmres_givens");
    return MG_OK;
}
int krylov_solve_update(int64_t n, const double *H, int ldh, const double *g, int k, double *y, const double *Z,
                        int64_t ld, double *x, cudaStream_t st) {
    if (k <= 0) return MG_OK;
    launch_k(gmres_backsub_kernel, 1u, 32u, st, H, ldh, g, k, y);
    MG_CHECK_LAUNCH("gmres_backsub");
    launch_k(multi_axpy_update_kernel, krylov_grid(n), (unsigned)kBlock, st, n, Z, ld, k, (const double *)y, x);
    MG_CHECK_LAUNCH("multi_axpy_update");
    return MG_OK;
}

}  // namespace mgb

using namespace mgb;

extern "C" {

int64_t mg_krylov_partials(int64_t n, int32_t m) { return n < 0 || m < 0 ? -1 : krylov_partials(n, m); }

int mg_multi_dot(int64_t n, const double *d_V, int64_t ld, int32_t m, const double *d_w, double *d_partials,
                 double *d_out, void *stream) {
    MG_REQUIRE(n >= 1 && m >= 0 && ld >= n, "bad sizes");
    MG_REQUIRE(d_V && d_w && d_partials && d_out, "null argument");
    return krylov_multi_dot(n, d_V, ld, m, d_w, d_partials, d_out, (cudaStream_t)stream);
}
int mg_multi_axpy_norm(int64_t n, const double *d_V, int64_t ld, int32_t m, const double *d_h, double *d_w,
                       double *d_partials, double *d_norm2, void *stream) {
    MG_REQUIRE(n >= 1 && m >= 0 && ld >= n, "bad sizes");
    MG_REQUIRE(d_V && d_h && d_w && d_partials && d_norm2, "null argument");
    return krylov_multi_axpy_norm(n, d_V, ld, m, d_h, d_w, d_partials, d_norm2, (cudaStream_t)stream);
}
int mg_scale_inv(int64_t n, const double *d_h, double *d_v, void *stream) {
    MG_REQUIRE(n >= 1 && d_h && d_v, "bad argument");
    return krylov_scale_inv(n, d_h, d_v, (cudaStream_t)stream);
}
int mg_gmres_solve_update(int64_t n, const double *d_H, int32_t ldh, const double *d_g, int32_t k, double *d_y,
                          const double *d_Z, int64_t ld, double *d_x, void *stream) {
    MG_REQUIRE(n >= 1 && k >= 0 && ldh >= k && ld >= n, "bad sizes");
    MG_REQUIRE(d_H && d_g && d_y && d_Z && d_x, "null argument");
    return krylov_solve_update(n, d_H, ldh, d_g, k, d_y, d_Z, ld, d_x, (cudaStream_t)stream);
}

}  // extern "C"
