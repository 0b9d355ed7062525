// cycle.cu -- V-cycle orchestration over a prebuilt device hierarchy, CUDA-graph helpers, library globals.
// Statement order follows Multigrid.v_cycle (learn_multigrid/solvers/Multigrid.py:77-124):
//   pre-smooth (:88) -> residual (:90) -> restrict (:93) -> recurse (:102-104) or coarsest solve (:106)
//   -> prolong + correct (:115) -> post-smooth (:121).
// The Galerkin product (:97-98) and the coarse factorisation (:106), which the reference repeats in every
// cycle, are hoisted to setup; the arithmetic of a cycle is unchanged.
#include "sell_api.cuh"

#include <vector>

namespace mgb {

int comm_prepare(mg_comm *, const mg_xfer *, const double *, double *, ExArgs *, int *);
int g_fused_exchange = 1;
// Work the multicolour cycle does not have to do (mg_set_cycle_fusion; results are the same bits either way):
//  * the last colour sweep of the pre-smoothing also writes the residual of its own rows, so the residual pass only
//    covers the other colours; likewise the last sweep of the post-smoothing on level 0 yields its rows' share of
//    ||b - A x||^2 when the caller wants the norm of the new iterate (mg_vcycle_norm);
//  * the prolongation skips the rows of the colour the post-smoothing sweeps first: a Gauss-Seidel update does not read
//    the row's own old value, so whatever the correction added there is overwritten unread;
//  * the first colour sweep on a zero iterate is x = b / diag without a pass over the matrix.
// The first two need a proper colouring (no non-zero coupling inside a colour), the second also a non-zero diagonal in
// every row: mg_level.flags, established by mg_level_inspect on the operator as stored.
int g_cycle_fusion = 1;

thread_local char g_last_error[512] = "";
thread_local int64_t g_launch_count = 0;
thread_local int64_t g_last_cycle_launches = 0;
int g_pdl = 1;

int vec_axpby(int64_t, double, const double *, double, const double *, double *, cudaStream_t);
int vec_fill(int64_t, double, double *, cudaStream_t);
int vec_diag_scale(int64_t, double, const double *, const double *, double *, cudaStream_t);
int dense_gemv(int64_t, int64_t, const double *, const double *, double *, cudaStream_t);
int csr_gs_lex(const int32_t *, const int32_t *, const double *, double *, const double *, const int64_t *,
               const int32_t *, int64_t, int64_t, int, cudaStream_t);
int bcr_solve(const void *handle, const mg_bcr_dist *dist, mg_comm *comm, const double *rhs, double *x, cudaStream_t st);
int vec_scatter(int64_t, const int32_t *, const double *, double *, cudaStream_t);
int vec_dot_partials(int64_t, const double *, const double *, double *, int *, cudaStream_t);
int vec_pcg_direction(int64_t, const double *, double *, const double *, int, cudaStream_t);
int vec_pcg_update(int64_t, const double *, const double *, double *, double *, const double *, double *, int *, cudaStream_t);
int vec_pcg_scalar(int, int, double *, const double *, cudaStream_t);
int comm_exchange(mg_comm *, const mg_xfer *, const double *, double *, cudaStream_t);
int krylov_multi_dot(int64_t, const double *, int64_t, int, const double *, double *, double *, cudaStream_t);
int krylov_multi_axpy_norm(int64_t, const double *, int64_t, int, const double *, double *, double *, double *, cudaStream_t);
int krylov_scale_inv(int64_t, const double *, double *, cudaStream_t);
int krylov_gmres_start(const double *, double *, int, double *, cudaStream_t);
int krylov_givens(double *, int, int, double *, double *, double *, const double *, double *, cudaStream_t);
int krylov_solve_update(int64_t, const double *, int, const double *, int, double *, const double *, int64_t, double *,
                        cudaStream_t);

#define MG_TRY(expr)            \
    do {                        \
        int _rc = (expr);       \
        if (_rc) return _rc;    \
    } while (0)

// Deferred exchange: with multicolour Gauss-Seidel an exchange of a level vector is not launched when it is issued
// but handed to the next SELL kernel that gathers from that vector, which carries it as extra CTAs (sell_kernel_fused).
// Anything else that needs the halo first calls flush_pending().
struct Pending {
    const mg_xfer *x = nullptr;
    double *vec = nullptr;
};
static thread_local Pending g_pend;

static int flush_pending(mg_comm *comm, cudaStream_t st) {
    if (!g_pend.x) return MG_OK;
    const mg_xfer *x = g_pend.x;
    double *v = g_pend.vec;
    g_pend.x = nullptr;
    return comm_exchange(comm, x, v, v, st);
}
// issue an exchange of vector v: deferred if allowed, immediate otherwise
static int issue_exchange(mg_comm *comm, const mg_xfer *x, double *v, bool may_defer, cudaStream_t st) {
    MG_TRY(flush_pending(comm, st));
    if (!may_defer || !g_fused_exchange) return comm_exchange(comm, x, v, v, st);
    g_pend.x = x;
    g_pend.vec = v;
    return MG_OK;
}
// before a SELL launch that gathers from `xop` over rows [row0,row1) of M: take the pending exchange along if it is on
// that vector and the launch can carry it; otherwise flush it.  *use tells whether `f` was filled.
static int take_pending(mg_comm *comm, const double *xop, const mg_sell *M, int64_t row0, int64_t row1,
                        const unsigned char *mask, SellFuse *f, bool *use, cudaStream_t st) {
    *use = false;
    if (!g_pend.x) return MG_OK;
    if (g_pend.vec != xop || !sell_fusable(M, row0, row1)) return flush_pending(comm, st);
    const mg_xfer *x = g_pend.x;
    double *v = g_pend.vec;
    g_pend.x = nullptr;
    int grid = 0;
    MG_TRY(comm_prepare(comm, x, v, v, &f->ex, &grid));
    if (grid == 0) return MG_OK;
    f->nex = grid;
    f->mask = mask;
    *use = true;
    return MG_OK;
}

// Row-partitioned levels (mg_level.dist != NULL, SURVEY 8e): L.n counts the OWNED rows, the level vectors carry
// dist->n_halo more entries behind them, and every kernel that changes a vector other ranks read is followed by an
// exchange of the boundary values.  Invariant: the halo of the iterate is current on entry to and on return from
// vcycle_rec, and after every smoothing step.
static inline int64_t vec_len(const mg_level &L) { return L.n + (L.dist ? L.dist->n_halo : 0); }
static inline int halo_all(mg_comm *comm, const mg_level &L, double *v, cudaStream_t st) {
    if (!L.dist) return MG_OK;
    return comm_exchange(comm, L.dist->xfer_all, v, v, st);
}

// What the LAST colour sweep of a smoothing call should produce besides the new values of its rows (multicolour
// Gauss-Seidel on a properly coloured level, see g_cycle_fusion): their residual, or their share of the squared
// residual norm.  On return `done` tells whether it did; the rows [rest0, rest1) are then what a stand-alone pass
// still has to cover.
struct Tail {
    int kind = TAIL_NONE;
    double *r_out = nullptr;
    double *partials = nullptr;
    bool done = false;
    int64_t rest0 = 0, rest1 = 0;
    int nblocks = 0;
};

static inline bool level_proper(const mg_level &L) { return g_cycle_fusion && (L.flags & MG_LEVEL_PROPER_COLORING); }

// `steps` smoothing sweeps on level L.  cur points at the buffer holding the iterate and is updated
// (Jacobi and Chebyshev ping-pong between d_x and d_tmp).  zero_guess: the iterate is known to be exactly zero and the
// buffer has NOT been initialised.
static int smooth(mg_comm *comm, const mg_level &L, const mg_cycle_params &P, int steps, double **cur, double **alt,
                  bool zero_guess, bool reverse, cudaStream_t st, Tail *tail = nullptr) {
    if (steps <= 0) {
        if (zero_guess) MG_TRY(vec_fill(vec_len(L), 0.0, *cur, st));
        return MG_OK;
    }
    if (P.smoother == MG_SMOOTH_JACOBI) {
        int s = 0;
        if (zero_guess) {
            if (P.zero_guess_skip) {
                // x1 = 0 + omega*(dinv*(b - A*0)) = omega*(dinv*b): same bits as a sweep on zeros, no matrix pass
                MG_TRY(vec_diag_scale(L.n, P.omega, L.d_dinv, L.d_b, *alt, st));
                MG_TRY(halo_all(comm, L, *alt, st));
                double *t = *cur; *cur = *alt; *alt = t;
                s = 1;
            } else {
                MG_TRY(vec_fill(vec_len(L), 0.0, *cur, st));
            }
        }
        for (; s < steps; ++s) {
            MG_TRY(sell_jacobi(&L.A, L.d_dinv, *cur, L.d_b, *alt, P.omega, st));
            MG_TRY(halo_all(comm, L, *alt, st));
            double *t = *cur; *cur = *alt; *alt = t;
        }
        return MG_OK;
    }
    if (P.smoother == MG_SMOOTH_CHEBY) {
        // `steps` applications of the degree-m polynomial, each restarting at step 0; d lives in d_r, which is free
        // during the pre-smoothing (the residual is formed after it) and the post-smoothing (the restriction has read it)
        const int deg = L.cheb_degree;
        if (deg < 1 || !L.h_cheb_coef) return set_error(MG_ERR_INVALID, "mg_vcycle", "level has no Chebyshev coefficients");
        for (int s = 0; s < steps; ++s)
            for (int k = 0; k < deg; ++k) {
                const double c_d = L.h_cheb_coef[2 * k], c_r = L.h_cheb_coef[2 * k + 1];
                if (s == 0 && k == 0 && zero_guess) {
                    if (P.zero_guess_skip) {
                        // x = 0 + c_r (dinv b): the bits of the step on zeros, no matrix pass
                        MG_TRY(sell_chebyshev_zero_first(L.n, c_r, L.d_dinv, L.d_b, L.d_r, *alt, st));
                        MG_TRY(halo_all(comm, L, *alt, st));
                        double *t = *cur; *cur = *alt; *alt = t;
                        continue;
                    }
                    MG_TRY(vec_fill(vec_len(L), 0.0, *cur, st));
                }
                MG_TRY(sell_chebyshev(&L.A, L.d_dinv, *cur, L.d_b, L.d_r, *alt, c_d, c_r, k == 0, st));
                MG_TRY(halo_all(comm, L, *alt, st));
                double *t = *cur; *cur = *alt; *alt = t;
            }
        return MG_OK;
    }
    if (P.smoother == MG_SMOOTH_MCGS) {
        if (L.ncolors <= 0 || !L.h_color_ptr) return set_error(MG_ERR_INVALID, "mg_vcycle", "level has no colouring");
        if (L.dist && L.dist->ncolors != L.ncolors) return set_error(MG_ERR_INVALID, "mg_vcycle", "halo plan and colouring disagree");
        for (int s = 0; s < steps; ++s)
            for (int cc = 0; cc < L.ncolors; ++cc) {
                const int c = reverse ? L.ncolors - 1 - cc : cc;
                const int64_t r0 = L.h_color_ptr[c], r1 = L.h_color_ptr[c + 1];
                const bool first = s == 0 && cc == 0, last = s == steps - 1 && cc == L.ncolors - 1;
                int tk = TAIL_NONE;
                if (last && tail && tail->kind != TAIL_NONE && level_proper(L) && sell_gs_tail_ok(&L.A, r0, r1)) tk = tail->kind;
                if (first && zero_guess) {
                    if (g_cycle_fusion && P.zero_guess_skip && L.d_diag && tk == TAIL_NONE && r1 > r0) {
                        // every entry the first colour reads is zero: x = b / diag for its rows, zeros elsewhere, in
                        // one pass over the vector and none over the matrix (the bits of fill + sweep)
                        MG_TRY(sell_gs_zero_first(vec_len(L), r0, r1, L.d_diag, L.d_b, *cur, st));
                        if (L.dist) MG_TRY(issue_exchange(comm, L.dist->xfer_color + c, *cur, true, st));
                        continue;
                    }
                    MG_TRY(vec_fill(vec_len(L), 0.0, *cur, st));
                }
                double *r_out = tk == TAIL_RESIDUAL ? tail->r_out : nullptr;
                double *partials = tk == TAIL_NORM ? tail->partials : nullptr;
                int nb = 0;
                if (L.dist) {
                    SellFuse f;
                    bool use;
                    MG_TRY(take_pending(comm, *cur, &L.A, r0, r1, L.dist->d_mask_A, &f, &use, st));
                    MG_TRY(sell_gs_rows(&L.A, *cur, L.d_b, r0, r1, use ? &f : nullptr, tk, r_out, partials, &nb, st));
                    MG_TRY(issue_exchange(comm, L.dist->xfer_color + c, *cur, true, st));
                } else {
                    MG_TRY(sell_gs_rows(&L.A, *cur, L.d_b, r0, r1, nullptr, tk, r_out, partials, &nb, st));
                }
                if (tk != TAIL_NONE) {
                    tail->done = true;
                    tail->nblocks = nb;
                    // the swept colour is the first or the last block, what is left is one range
                    tail->rest0 = c == 0 ? r1 : 0;
                    tail->rest1 = c == 0 ? L.n : r0;
                    if (c != 0 && c != L.ncolors - 1) return set_error(MG_ERR_INVALID, "mg_vcycle", "internal: tail colour in the middle");
                }
            }
        return MG_OK;
    }
    if (zero_guess) MG_TRY(vec_fill(vec_len(L), 0.0, *cur, st));
    if (P.smoother == MG_SMOOTH_LEXGS) {
        if (L.dist) return set_error(MG_ERR_UNSUPPORTED, "mg_vcycle", "index-order Gauss-Seidel is serial across row blocks; not available on partitioned levels");
        if (!L.d_csr_indptr || !L.d_lex_level_ptr) return set_error(MG_ERR_INVALID, "mg_vcycle", "level has no lexicographic schedule");
        return csr_gs_lex(L.d_csr_indptr, L.d_csr_indices, L.d_csr_values, *cur, L.d_b, L.d_lex_level_ptr,
                          L.d_lex_level_rows, L.lex_nlevels, L.n, steps, st);
    }
    return set_error(MG_ERR_INVALID, "mg_vcycle", "unknown smoother");
}

// the squared residual norm of the iterate the cycle leaves on level 0, as per-CTA partial sums (mg_vcycle_norm)
struct NormOut {
    double *partials;
    int nblocks;
};

static int vcycle_rec(mg_comm *comm, const mg_level *levels, int nlevels, int l, const mg_cycle_params &P,
                      cudaStream_t st, NormOut *norm = nullptr) {
    const mg_level &L = levels[l];
    if (l == nlevels - 1) {   // coarsest: direct solve (Multigrid.py:106)
        if (L.coarse_kind == MG_COARSE_DENSE) {
            if (!L.d_coarse_inv) return set_error(MG_ERR_INVALID, "mg_vcycle", "coarsest level has no inverse");
            return dense_gemv(L.n, L.n, L.d_coarse_inv, L.d_b, L.d_x, st);
        }
        if (L.coarse_kind == MG_COARSE_BCR) return bcr_solve(L.coarse_bcr, L.coarse_bcr_dist, comm, L.d_b, L.d_x, st);
        return set_error(MG_ERR_INVALID, "mg_vcycle", "unknown coarse solver kind");
    }
    const mg_level &C = levels[l + 1];
    const bool jac = P.smoother == MG_SMOOTH_JACOBI;
    const bool cheb = P.smoother == MG_SMOOTH_CHEBY;
    const bool mcgs = P.smoother == MG_SMOOTH_MCGS;
    const bool zero_guess = l > 0 || P.x0_zero != 0;
    double *cur = L.d_x, *alt = L.d_tmp;
    bool prolong_flip = false;
    if (jac || cheb) {
        // Jacobi flips buffers once per sweep, Chebyshev once per step (degree steps per sweep).  The result must end
        // in d_x: on coarse levels choose the start buffer (the zero guess is virtual), on level 0 let the
        // prolongation write out of place.
        const int flips = (cheb ? L.cheb_degree : 1) * (P.nu_pre + P.nu_post);
        if (flips & 1) {
            if (zero_guess) { cur = L.d_tmp; alt = L.d_x; }
            else prolong_flip = true;
        }
    }
    if (!L.dist) MG_TRY(flush_pending(comm, st));                    // replicated level: nothing may be in flight
    const bool defer = mcgs;                                         // exchanges ride on the next SELL kernel
    SellFuse f;
    bool use = false;
    // ---- pre-smoothing; its last colour sweep also writes the residual of its rows
    Tail pre;
    if (mcgs && P.nu_pre > 0) {
        pre.kind = TAIL_RESIDUAL;
        pre.r_out = L.d_r;
    }
    MG_TRY(smooth(comm, L, P, P.nu_pre, &cur, &alt, zero_guess, false, st, &pre));
    int64_t q0 = 0, q1 = L.A.nrows;                                  // rows whose residual is still to be formed
    if (pre.done) { q0 = pre.rest0; q1 = pre.rest1; }
    if (L.dist) {
        const mg_dist_level &D = *L.dist;
        MG_TRY(take_pending(comm, cur, &L.A, q0, q1, D.d_mask_A, &f, &use, st));
        MG_TRY(sell_residual(&L.A, cur, L.d_b, L.d_r, q0, q1, use ? &f : nullptr, st));      // res = rhs - A u
        MG_TRY(issue_exchange(comm, D.xfer_all, L.d_r, defer, st));                  // the restriction reads halo rows
        // last partitioned level: restrict into the owned block of the coarse rhs, then gather it into every
        // rank's full vector (the coarse levels below are replicated)
        double *rc = D.xfer_gather ? D.d_gather_tmp : C.d_b;
        MG_TRY(take_pending(comm, L.d_r, &L.QT, 0, L.QT.nrows, D.d_mask_QT, &f, &use, st));
        MG_TRY(sell_spmv(&L.QT, L.d_r, rc, 0, L.QT.nrows, use ? &f : nullptr, st));  // res_coarse = Q^T res (owned rows)
        if (D.xfer_gather) {
            MG_TRY(vec_scatter(D.n_gather_own, D.d_gather_self_idx, D.d_gather_tmp, C.d_b, st));
            MG_TRY(comm_exchange(comm, D.xfer_gather, D.d_gather_tmp, C.d_b, st));
        }
    } else {
        MG_TRY(sell_residual(&L.A, cur, L.d_b, L.d_r, q0, q1, nullptr, st));         // res = rhs - A u
        MG_TRY(sell_spmv(&L.QT, L.d_r, C.d_b, 0, L.QT.nrows, nullptr, st));          // res_coarse = Q^T res
    }
    mg_cycle_params Pc = P;
    Pc.x0_zero = 0;                                                  // below level 0 the guess is zero anyway
    MG_TRY(vcycle_rec(comm, levels, nlevels, l + 1, Pc, st));        // u_coarse
    double *out = prolong_flip ? alt : cur;                          // u = u + Q u_coarse (out of place when flipping)
    // The colour the post-smoothing sweeps first is overwritten without being read: its rows need no correction.
    int64_t p0 = 0, p1 = L.Q.nrows;
    if (mcgs && P.nu_post > 0 && level_proper(L) && (L.flags & MG_LEVEL_NONZERO_DIAG) && L.ncolors > 0 && L.h_color_ptr) {
        if (P.reverse_post) p1 = L.h_color_ptr[L.ncolors - 1];
        else p0 = L.h_color_ptr[1];
    }
    if (L.dist) {
        // a partitioned coarse level leaves the exchange of its last sweep pending on C.d_x
        MG_TRY(take_pending(comm, C.d_x, &L.Q, p0, p1, L.dist->d_mask_Q, &f, &use, st));
        MG_TRY(sell_prolong(&L.Q, C.d_x, cur, out, p0, p1, use ? &f : nullptr, st));
    } else {
        MG_TRY(sell_prolong(&L.Q, C.d_x, cur, out, p0, p1, nullptr, st));
    }
    if (prolong_flip) { double *t = cur; cur = alt; alt = t; }
    // every boundary value changed.  Deferred, this exchange rides on the first post-smoothing sweep, which rewrites
    // its own colour while the values are being sent: harmless, a colour never reads itself and is sent again right
    // after its sweep.
    if (L.dist) MG_TRY(issue_exchange(comm, L.dist->xfer_all, cur, defer, st));
    // ---- post-smoothing; on level 0 its last colour sweep can yield its rows' share of the new residual norm
    Tail post;
    if (norm && mcgs && P.nu_post > 0) {
        post.kind = TAIL_NORM;
        post.partials = norm->partials;
    }
    MG_TRY(smooth(comm, L, P, P.nu_post, &cur, &alt, false, P.reverse_post != 0, st, &post));
    if (cur != L.d_x) MG_TRY(vec_axpby(vec_len(L), 1.0, cur, 0.0, nullptr, L.d_x, st));   // safety net; not reached
    if (norm) {
        int64_t n0 = 0, n1 = L.A.nrows;
        int nb = 0, nb2 = 0;
        if (post.done) { n0 = post.rest0; n1 = post.rest1; nb = post.nblocks; }
        use = false;
        if (L.dist) MG_TRY(take_pending(comm, L.d_x, &L.A, n0, n1, L.dist->d_mask_A, &f, &use, st));
        MG_TRY(sell_residual_partials(&L.A, L.d_x, L.d_b, norm->partials + nb, n0, n1, &nb2, use ? &f : nullptr, st));
        norm->nblocks = nb + nb2;
    }
    return MG_OK;
}

static int check_levels(const mg_level *levels, int nlevels, const mg_cycle_params *params, bool dist_ok) {
    MG_REQUIRE(levels && params && nlevels >= 2, "need at least two levels (Multigrid.py:78,102: levels=1 is not handled by the reference either)");
    MG_REQUIRE(params->nu_pre >= 0 && params->nu_post >= 0, "negative smoothing steps");
    for (int l = 0; l < nlevels; ++l) {
        MG_REQUIRE(levels[l].n > 0 && levels[l].d_x && levels[l].d_b, "level vectors missing");
        MG_REQUIRE(dist_ok || !levels[l].dist, "partitioned level passed to mg_vcycle; use mg_vcycle_dist");
        if (l + 1 < nlevels) {
            const mg_level &L = levels[l], &C = levels[l + 1];
            MG_REQUIRE(L.d_r && L.d_tmp, "level work vectors missing");
            MG_REQUIRE(!(C.dist && !L.dist), "a partitioned level below a replicated one");
            const int64_t lenL = L.n + (L.dist ? L.dist->n_halo : 0), lenC = C.n + (C.dist ? C.dist->n_halo : 0);
            if (L.dist && !C.dist) {
                MG_REQUIRE(L.dist->xfer_gather && L.dist->d_gather_tmp && L.dist->d_gather_self_idx &&
                               L.QT.nrows == L.dist->n_gather_own, "last partitioned level has no coarse hand-off");
            } else {
                MG_REQUIRE(L.QT.nrows == C.n, "inconsistent level shapes");
            }
            MG_REQUIRE(L.A.nrows == L.n && L.A.ncols == lenL && L.Q.nrows == L.n && L.Q.ncols == lenC && L.QT.ncols == lenL,
                       "inconsistent level shapes");
        }
    }
    return MG_OK;
}

}  // namespace mgb

using namespace mgb;

extern "C" {

int mg_version(void) { return 200; }
int mg_set_fused_exchange(int enabled) {
    const int prev = g_fused_exchange;
    g_fused_exchange = enabled ? 1 : 0;
    return prev;
}
int mg_set_cycle_fusion(int enabled) {
    const int prev = g_cycle_fusion;
    g_cycle_fusion = enabled ? 1 : 0;
    return prev;
}
int mg_set_pdl(int enabled) {
    const int prev = g_pdl;
    g_pdl = enabled ? 1 : 0;
    return prev;
}
int64_t mg_struct_size(int which) {
    switch (which) {
        case 0: return sizeof(mg_sell);
        case 1: return sizeof(mg_level);
        case 2: return sizeof(mg_cycle_params);
        case 3: return sizeof(mg_bcr);
        case 4: return sizeof(mg_comm);
        case 5: return sizeof(mg_xfer);
        case 6: return sizeof(mg_dist_level);
        case 7: return sizeof(mg_bcr_dist);
        case 8: return sizeof(mg_dist_norm);
        case 9: return sizeof(mg_gmres);
        default: return -1;
    }
}
const char *mg_last_error(void) { return g_last_error; }

int mg_device_info(int *sm, int64_t *mem, int *cc) {
    int dev = 0;
    MG_CHECK_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    MG_CHECK_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm) *sm = p.multiProcessorCount;
    if (mem) *mem = (int64_t)p.totalGlobalMem;
    if (cc) *cc = p.major * 10 + p.minor;
    return MG_OK;
}

int mg_vcycle(const mg_level *levels, int nlevels, const mg_cycle_params *params, void *stream) {
    MG_TRY(check_levels(levels, nlevels, params, false));
    const int64_t before = g_launch_count;
    int rc = vcycle_rec(nullptr, levels, nlevels, 0, *params, (cudaStream_t)stream);
    g_last_cycle_launches = g_launch_count - before;
    return rc;
}

int mg_vcycle_norm(const mg_level *levels, int nlevels, const mg_cycle_params *params, double *d_partials,
                   double *d_norm2, void *stream) {
    MG_TRY(check_levels(levels, nlevels, params, false));
    MG_REQUIRE(d_partials && d_norm2, "norm workspace missing");
    const int64_t before = g_launch_count;
    NormOut no{d_partials, 0};
    int rc = vcycle_rec(nullptr, levels, nlevels, 0, *params, (cudaStream_t)stream, &no);
    if (!rc) rc = sell_reduce_partials(d_partials, no.nblocks, d_norm2, (cudaStream_t)stream);
    g_last_cycle_launches = g_launch_count - before;
    return rc;
}

int mg_vcycle_dist(mg_comm *comm, const mg_level *levels, int nlevels, const mg_cycle_params *params,
                   const mg_dist_norm *norm, void *stream) {
    MG_REQUIRE(comm, "null communicator");
    MG_REQUIRE(params || norm, "nothing to do");
    if (params) MG_TRY(check_levels(levels, nlevels, params, true));
    else MG_REQUIRE(levels && nlevels >= 1, "no level");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t before = g_launch_count;
    MG_TRY(mg_comm_begin(comm));
    g_pend.x = nullptr;
    int rc = MG_OK;
    if (norm) MG_REQUIRE(norm->d_partials && norm->d_local && norm->d_slots && norm->d_norm2, "norm workspace missing");
    const bool after = norm && norm->after && params;
    // second stage of a norm whose per-CTA partials are in norm->d_partials, and its all-reduce
    auto finish_norm = [&](int nblocks) -> int {
        int r = sell_reduce_partials(norm->d_partials, nblocks, norm->d_local, st);
        if (!r) r = mg_comm_allreduce_sum(comm, norm->d_local, norm->d_slots, norm->d_norm2, stream);
        return r;
    };
    if (norm && !after) {   // outer loop of Multigrid.solve (:62-63): ||b - A x||^2 over all row blocks
        int nblocks = 0;
        rc = sell_residual_partials(&levels[0].A, levels[0].d_x, levels[0].d_b, norm->d_partials, 0, levels[0].A.nrows,
                                    &nblocks, nullptr, st);
        if (!rc) rc = finish_norm(nblocks);
    }
    NormOut no{norm ? norm->d_partials : nullptr, 0};
    if (!rc && params) rc = vcycle_rec(comm, levels, nlevels, 0, *params, st, after ? &no : nullptr);
    if (!rc && after) {     // the norm of the NEW iterate, its last colour's share already summed by the last sweep
        rc = flush_pending(comm, st);
        if (!rc) rc = finish_norm(no.nblocks);
    }
    if (!rc) rc = flush_pending(comm, st);      // the halo of the iterate is current when the program ends
    g_pend.x = nullptr;
    if (!rc) rc = mg_comm_end(comm, stream);
    g_last_cycle_launches = g_launch_count - before;
    return rc;
}

int64_t mg_last_launch_count(void) { return g_last_cycle_launches; }

/* ---- conjugate gradients preconditioned by one V-cycle per iteration (CG.py:12-50 + BASELINE configs[4]) -------------
 * Everything stays on the device: the scalars live in pcg->d_scalars, every dot product is the by-product of the
 * kernel that produces its operand where there is one (p.Ap from the SpMV, r.r from the update of x and r), and an
 * iteration is one launch sequence (capturable in one CUDA graph) after which the host reads 8 bytes to test
 * convergence.  comm != NULL: levels[0] is row-partitioned, the sequence is one program of the communicator and the
 * dot products are summed over the ranks in rank order. */
static int pcg_reduce(mg_comm *comm, const mg_pcg *S, int nblocks, int op, int first, cudaStream_t st) {
    double *local = S->d_scalars + 6;
    MG_TRY(sell_reduce_partials(S->d_partials, nblocks, local, st));
    const double *in = local;
    if (comm && comm->world > 1) {
        MG_REQUIRE(S->d_slots, "mg_pcg.d_slots missing");
        MG_TRY(flush_pending(comm, st));
        MG_TRY(mg_comm_allreduce_sum(comm, local, S->d_slots, S->d_scalars + 7, st));
        in = S->d_scalars + 7;
    }
    return vec_pcg_scalar(op, first, S->d_scalars, in, st);
}
static int check_pcg(const mg_level *levels, const mg_pcg *S) {
    MG_REQUIRE(levels && S && S->d_x && S->d_p && S->d_Ap && S->d_scalars && S->d_partials, "mg_pcg: null member");
    MG_REQUIRE(levels[0].n > 0 && levels[0].d_x && levels[0].d_b, "level vectors missing");
    return MG_OK;
}
int mg_pcg_start(mg_comm *comm, const mg_level *levels, const mg_pcg *pcg, void *stream) {
    MG_TRY(check_pcg(levels, pcg));
    cudaStream_t st = (cudaStream_t)stream;
    const mg_level &L = levels[0];
    if (comm) {
        MG_TRY(mg_comm_begin(comm));
        g_pend.x = nullptr;
        }
    MG_TRY(vec_fill(L.n, 0.0, pcg->d_x, st));
    int nb = 0;
    MG_TRY(vec_dot_partials(L.n, L.d_b, L.d_b, pcg->d_partials, &nb, st));
    MG_TRY(pcg_reduce(comm, pcg, nb, 0, 0, st));
    if (comm) MG_TRY(mg_comm_end(comm, stream));
    return MG_OK;
}
int mg_pcg_iterate(mg_comm *comm, const mg_level *levels, int nlevels, const mg_cycle_params *params, const mg_pcg *pcg,
                   int first, void *stream) {
    MG_TRY(check_pcg(levels, pcg));
    if (params) MG_TRY(check_levels(levels, nlevels, params, comm != nullptr));
    cudaStream_t st = (cudaStream_t)stream;
    const mg_level &L = levels[0];
    MG_REQUIRE(!L.dist || comm, "partitioned level without a communicator");
    const int64_t before = g_launch_count;
    if (comm) {
        MG_TRY(mg_comm_begin(comm));
        g_pend.x = nullptr;
        }
    double *r = L.d_b;
    const double *z = r;
    if (params) {                               // z = M^-1 r: one V-cycle on (x, b) = (0, r), z lands in d_x
        mg_cycle_params P = *params;
        P.x0_zero = 1;
        MG_TRY(vcycle_rec(comm, levels, nlevels, 0, P, st));
        MG_TRY(flush_pending(comm, st));
        z = L.d_x;
    }
    int nb = 0;
    MG_TRY(vec_dot_partials(L.n, r, z, pcg->d_partials, &nb, st));
    MG_TRY(pcg_reduce(comm, pcg, nb, 1, first, st));                          // beta = r.z / (r.z)_old
    MG_TRY(vec_pcg_direction(L.n, z, pcg->d_p, pcg->d_scalars, first, st));    // p = z + beta p
    SellFuse f;
    bool use = false;
    if (L.dist) {
        MG_TRY(issue_exchange(comm, L.dist->xfer_all, pcg->d_p, true, st));    // the SpMV reads halo entries of p
        MG_TRY(take_pending(comm, pcg->d_p, &L.A, 0, L.A.nrows, L.dist->d_mask_A, &f, &use, st));
    }
    MG_TRY(sell_spmv_dot(&L.A, pcg->d_p, pcg->d_p, pcg->d_Ap, pcg->d_partials, &nb, use ? &f : nullptr, st));
    MG_TRY(pcg_reduce(comm, pcg, nb, 2, 0, st));                              // alpha = r.z / p.Ap
    MG_TRY(vec_pcg_update(L.n, pcg->d_p, pcg->d_Ap, pcg->d_x, r, pcg->d_scalars, pcg->d_partials, &nb, st));
    MG_TRY(pcg_reduce(comm, pcg, nb, 0, 0, st));                              // r.r of the new residual
    if (comm) {
        MG_TRY(flush_pending(comm, st));
        g_pend.x = nullptr;
            MG_TRY(mg_comm_end(comm, stream));
    }
    g_last_cycle_launches = g_launch_count - before;
    return MG_OK;
}

/* ---- restarted GMRES, right-preconditioned by one V-cycle per Arnoldi step (include/mgb200.h, mg_gmres) ---------------
 * Launch sequences only, the scalars on the device; after each call the host reads d_scalars[0] (8 bytes). */
static int check_gmres(const mg_level *levels, const mg_gmres *G) {
    MG_REQUIRE(levels && G && G->d_x && G->d_V && G->d_Z && G->d_H && G->d_g && G->d_cs && G->d_sn && G->d_y &&
                   G->d_scalars && G->d_partials, "mg_gmres: null member");
    MG_REQUIRE(G->restart >= 1, "mg_gmres: restart must be >= 1");
    const mg_level &L = levels[0];
    MG_REQUIRE(L.n > 0 && L.d_b, "level vectors missing");
    MG_REQUIRE(G->ld >= vec_len(L) && G->ld % 32 == 0, "mg_gmres: ld must cover the level vector and be a multiple of 32");
    return MG_OK;
}
// local sums -> the sums over all ranks (in place when there is one rank)
static int gmres_allreduce(mg_comm *comm, const mg_gmres *G, double *local, int k, double *out, cudaStream_t st) {
    MG_REQUIRE(G->d_slots, "mg_gmres.d_slots missing");
    MG_TRY(flush_pending(comm, st));
    return mg_comm_allreduce_sum_n(comm, local, k, G->d_slots, out, st);
}
int mg_gmres_start(mg_comm *comm, const mg_level *levels, const mg_gmres *gmres, void *stream) {
    MG_TRY(check_gmres(levels, gmres));
    cudaStream_t st = (cudaStream_t)stream;
    const mg_level &L = levels[0];
    MG_REQUIRE(!L.dist || comm, "partitioned level without a communicator");
    const bool multi = comm && comm->world > 1;
    if (comm) {
        MG_TRY(mg_comm_begin(comm));
        g_pend.x = nullptr;
    }
    double *r = gmres->d_V, *sc = gmres->d_scalars;
    SellFuse f;
    bool use = false;
    if (L.dist) {
        MG_TRY(issue_exchange(comm, L.dist->xfer_all, gmres->d_x, true, st));       // the residual reads halo entries of x
        MG_TRY(take_pending(comm, gmres->d_x, &L.A, 0, L.A.nrows, L.dist->d_mask_A, &f, &use, st));
    }
    MG_TRY(sell_residual(&L.A, gmres->d_x, L.d_b, r, 0, L.A.nrows, use ? &f : nullptr, st));     // r = b - A x
    MG_TRY(flush_pending(comm, st));
    int nb = 0;
    MG_TRY(vec_dot_partials(L.n, r, r, gmres->d_partials, &nb, st));
    MG_TRY(sell_reduce_partials(gmres->d_partials, nb, sc + 2, st));
    if (multi) MG_TRY(gmres_allreduce(comm, gmres, sc + 2, 1, sc + 3, st));
    MG_TRY(krylov_gmres_start(multi ? sc + 3 : sc + 2, gmres->d_g, gmres->restart, sc, st));   // g = beta e_1
    MG_TRY(krylov_scale_inv(L.n, sc + 1, r, st));                                              // v_0 = r / beta
    if (comm) {
        MG_TRY(flush_pending(comm, st));
        g_pend.x = nullptr;
        MG_TRY(mg_comm_end(comm, stream));
    }
    return MG_OK;
}
int mg_gmres_iterate(mg_comm *comm, const mg_level *levels, int nlevels, const mg_cycle_params *params,
                     const mg_gmres *gmres, int j, void *stream) {
    MG_TRY(check_gmres(levels, gmres));
    MG_REQUIRE(j >= 0 && j < gmres->restart, "mg_gmres_iterate: step outside the cycle");
    if (params) MG_TRY(check_levels(levels, nlevels, params, comm != nullptr));
    cudaStream_t st = (cudaStream_t)stream;
    const mg_level &L = levels[0];
    MG_REQUIRE(!L.dist || comm, "partitioned level without a communicator");
    const bool multi = comm && comm->world > 1;
    const int64_t before = g_launch_count;
    if (comm) {
        MG_TRY(mg_comm_begin(comm));
        g_pend.x = nullptr;
    }
    const int64_t ld = gmres->ld;
    double *vj = gmres->d_V + (int64_t)j * ld, *w = vj + ld, *sc = gmres->d_scalars;
    double *z = vj;
    if (params) {
        // z_j = M^-1 v_j: the cycle runs on a copy of the level structs whose level 0 reads v_j and writes z_j, so
        // neither vector is copied.  Every smoother leaves its result in d_x (vcycle_rec picks the start buffer).
        std::vector<mg_level> lv(levels, levels + nlevels);
        z = gmres->d_Z + (int64_t)j * ld;
        lv[0].d_b = vj;
        lv[0].d_x = z;
        mg_cycle_params P = *params;
        P.x0_zero = 1;
        MG_TRY(vcycle_rec(comm, lv.data(), nlevels, 0, P, st));
    } else if (L.dist) {
        MG_TRY(issue_exchange(comm, L.dist->xfer_all, vj, true, st));             // the SpMV reads halo entries of v_j
    }
    SellFuse f;
    bool use = false;
    if (L.dist) MG_TRY(take_pending(comm, z, &L.A, 0, L.A.nrows, L.dist->d_mask_A, &f, &use, st));
    MG_TRY(sell_spmv(&L.A, z, w, 0, L.A.nrows, use ? &f : nullptr, st));           // w = A z_j in slot j+1
    MG_TRY(flush_pending(comm, st));
    const int m = j + 1, ldh = gmres->restart + 1;
    double *hcol = gmres->d_H + (int64_t)j * ldh;
    MG_TRY(krylov_multi_dot(L.n, gmres->d_V, ld, m, w, gmres->d_partials, multi ? gmres->d_y : hcol, st));
    if (multi) MG_TRY(gmres_allreduce(comm, gmres, gmres->d_y, m, hcol, st));
    MG_TRY(krylov_multi_axpy_norm(L.n, gmres->d_V, ld, m, hcol, w, gmres->d_partials, sc + 2, st));
    if (multi) MG_TRY(gmres_allreduce(comm, gmres, sc + 2, 1, sc + 3, st));
    MG_TRY(krylov_givens(gmres->d_H, ldh, j, gmres->d_cs, gmres->d_sn, gmres->d_g, multi ? sc + 3 : sc + 2, sc, st));
    MG_TRY(krylov_scale_inv(L.n, sc + 1, w, st));                                  // v_{j+1} = w / h_{j+1,j}
    if (comm) {
        MG_TRY(flush_pending(comm, st));
        g_pend.x = nullptr;
        MG_TRY(mg_comm_end(comm, stream));
    }
    g_last_cycle_launches = g_launch_count - before;
    return MG_OK;
}
int mg_gmres_finish(const mg_level *levels, const mg_cycle_params *params, const mg_gmres *gmres, int k, void *stream) {
    MG_TRY(check_gmres(levels, gmres));
    MG_REQUIRE(k >= 0 && k <= gmres->restart, "mg_gmres_finish: more steps than the cycle holds");
    return krylov_solve_update(levels[0].n, gmres->d_H, gmres->restart + 1, gmres->d_g, k, gmres->d_y,
                               params ? gmres->d_Z : gmres->d_V, gmres->ld, gmres->d_x, (cudaStream_t)stream);
}

int mg_graph_begin(void *stream) {
    MG_CHECK_CUDA(cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeThreadLocal));
    return MG_OK;
}
int mg_graph_end(void *stream, void **graph_exec_out) {
    MG_REQUIRE(graph_exec_out, "null output");
    cudaGraph_t graph = nullptr;
    MG_CHECK_CUDA(cudaStreamEndCapture((cudaStream_t)stream, &graph));
    cudaGraphExec_t exec = nullptr;
    cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) return set_error(MG_ERR_CUDA, "cudaGraphInstantiate", cudaGetErrorString(e));
    *graph_exec_out = (void *)exec;
    return MG_OK;
}
int mg_graph_launch(void *graph_exec, void *stream) {
    MG_REQUIRE(graph_exec, "null graph");
    MG_CHECK_CUDA(cudaGraphLaunch((cudaGraphExec_t)graph_exec, (cudaStream_t)stream));
    return MG_OK;
}
int mg_graph_destroy(void *graph_exec) {
    if (graph_exec) MG_CHECK_CUDA(cudaGraphExecDestroy((cudaGraphExec_t)graph_exec));
    return MG_OK;
}

}  // extern "C"
