// sell_core.cuh -- the streaming hot-path kernels on the SELL-32 format (see include/mgb200.h) and their launcher.
//
// One thread per row, one warp per slice.  Entry k of the 32 rows of a slice is contiguous
// (256 B of values + 128 B of columns per warp request), so the matrix streams fully coalesced; the x
// gathers go through L1/L2, which hold the few grid lines a structured stencil touches.
// Every kernel is HBM-bound: algorithmic bytes per row = 12*nnz_row + 4 (CSR yardstick of SURVEY 8d) plus
// the vector traffic listed at each launcher.
//
// The templates are instantiated per group of modes in sell_kernels.cu / sell_modes_gs.cu / sell_modes_vec.cu (three
// translation units so that the ~500 specialisations compile in parallel).
#pragma once
#include <type_traits>
#include "exchange.cuh"
#include "sell_api.cuh"

namespace mgb {

struct SellArgs {
    const int64_t *__restrict__ slice_ptr;
    const int32_t *__restrict__ cols;
    const double *__restrict__ vals;
    const unsigned short *__restrict__ slice_rec;  // implied columns (IMPL kernels): record id per slice, see below
    const int32_t *__restrict__ rec_table;         // ... [nrec][8] column offsets relative to the row
    int32_t spec_id;                               // the record this launch expects (most of its slices use it)
    int32_t spec_off[8];                           // ... and its offsets, by value
    int32_t spec_lo, spec_hi;                      // rows in [lo, hi] keep every row + spec_off[j] inside the vector
    const double *__restrict__ rec_vals;           // implied values (IMPV kernels): [nrec][8] values of a record's entries
    double spec_val[8];                            // ... those of the expected record, by value
    double spec_diag;                              // ... its diagonal entry (the entries with offset 0, bits OR-ed)
    uint32_t spec_dmask;                           // ... and which entries those are (bit j: offset 0, value != 0)
    const unsigned char *__restrict__ vidx;  // value dictionary (VAL8 kernels): one byte per entry, laid out like vals
    const double *__restrict__ vtab;         // ... indexing this table of at most 256 doubles
    int64_t row_begin;   // first row this launch touches
    int64_t row_end;     // one past the last row
    int64_t first_row;   // row of thread 0 of block 0 (row_begin rounded down to a slice)
    int64_t nrows;       // rows of the matrix (rows of the last slice beyond it hold no data)
    double *r_out;       // GS_RES: where the residual of the swept rows goes
};

__host__ __device__ constexpr bool mode_is_gs(int m) { return m == GS || m == GS_RES || m == GS_NORM; }
__host__ __device__ constexpr bool mode_has_partials(int m) { return m == RESNORM || m == GS_NORM || m == SPMV_DOT; }
__host__ __device__ constexpr bool mode_is_tail(int m) { return m == GS_RES || m == GS_NORM; }
// modes whose epilogue reads the row's own old iterate and 1/diag (aux): damped Jacobi, Chebyshev
__host__ __device__ constexpr bool mode_is_jacobi_like(int m) { return m == JACOBI || m == CHEBY; }

// CHEBY: x_out = x + dn, d = dn with dn = c_r (dinv (b - A x)) on step 0 and (c_d d) + (c_r (dinv (b - A x))) after it,
// every product and sum rounded on its own.  The launch carries c_r in `omega`, d in SellArgs::r_out and c_d's bit
// pattern in the `partials` slot (zero bits: step 0, d is written but not read), so that the parameter block of every
// other mode stays as it is.
__device__ __forceinline__ double cheby_dn(double cd, bool has_d, double dv, double cr, double t) {
    const double rt = __dmul_rn(cr, t);
    return has_d ? __dadd_rn(__dmul_rn(cd, dv), rt) : rt;
}
__device__ __forceinline__ double cheby_cd(const double *slot) {
    return __longlong_as_double((long long)(uintptr_t)slot);
}

// ---- implied columns ------------------------------------------------------------------------------------------------
// On a structured stencil level nearly every slice is REGULAR: entry j of every one of its 32 rows has column
// row + off[j] with ONE offset table for the slice (mg_sell_slice_offsets; formats.sell_slice_offsets is the host twin).
// For those slices the IMPL kernels compute the columns instead of streaming them.  A structured level has only a
// handful of DIFFERENT offset tables (one per colour and grid-line parity), so a slice stores two bytes -- the id of its
// record in a small table -- in place of 128*LEN bytes of column indices: 57 instead of 88 bytes per 5-point row, and
// the x gathers of a warp become contiguous 256-byte reads.  The launch carries the record most of its slices use BY
// VALUE: the kernel gathers x with it at once, in the shadow of the load of the slice's id, and only redoes the
// gathers for the few slices that turn out to use another record (or to be irregular: id 0xffff, columns read from
// memory).  Without that, every thread would pay two dependent DRAM round trips (record, then x).  The values, the gathers and the order of the additions are untouched, so the
// results are the same bits; slices that are not regular (a boundary node among the rows, the ragged tail) take the
// ordinary path inside the same kernel.  Uniform matrices with at most 8 entries per row only.
// IMPLIED VALUES (IMPV, on top of implied columns and a value dictionary): on a constant-coefficient stencil level the
// 32 rows of a regular slice also hold the same VALUE per entry, so the record stands for the whole slice of the matrix
// (mg_sell.d_rec_vals): nothing is read per row but the vectors -- 23 instead of 28 bytes per 5-point row -- and the
// values of the expected record are kernel parameters, i.e. operands straight from the constant bank: fifteen
// instructions per row less in kernels that are bound by instruction issue.  Slices of another record take its values
// from the table, irregular ones their dictionary bytes, inside the same kernel; same doubles, same order, same bits.
constexpr int32_t kSliceIrregular = INT32_MIN;
constexpr int kOffStride = 8;      // ints per offset record (rows of at most 8 entries)
constexpr int kRecIrregular = 0xffff; // d_slice_rec value of a slice whose columns are not implied

// What the epilogue of a row needs besides the row sum.
struct SellEp {
    const double *__restrict__ b;
    const double *aux;
    double *y;
    double omega;
    double cd;      // CHEBY: c_d
    bool has_d;     // CHEBY: not step 0 (d is read)
};

// One row of at most LEN entries, everything in registers and in straight-line code: all cols/vals loads are issued
// first, then all x gathers, then the sums in storage order (LEN*12 bytes per thread in flight at ~4 registers per
// entry).  PRED: the slice holds len < LEN entries per row (non-uniform matrices), loads and sums are predicated on
// j < len (warp-uniform).  IMPL: the columns are row + o[j] (regular slice of an implied-columns matrix).
// `halo_wait` (launches carrying an exchange site): this slice reads halo columns, so between the matrix loads (which
// do not depend on the halo and are already in flight) and the x gathers, wait until the launch's exchange CTAs have
// unpacked it.
// Gauss-Seidel modes: the diagonal entry is skipped in the sum and divides it (PyAMG gauss_seidel); GS_RES / GS_NORM
// then form r = b - A x of the row WITH its new value from the registers that still hold the row -- the row's
// residual costs no second pass over the matrix.  That is exact because a properly coloured sweep changes no other
// entry this row reads (cycle.cu only asks for it on such levels), and it adds the products in storage order with the
// diagonal in its place, i.e. it is the residual kernel's arithmetic.
// A Gauss-Seidel row whose new value is stored by the caller (GS_NORM: after the block reduction, so that the
// reduction's barrier does not wait for the store).
struct RowOut {
    double xn;
    bool store;
};

// VAL8: the values come from the matrix' dictionary (valdict.cu): one byte per entry from DRAM, the double from a
// 2 KB table that stays in L1 -- the same doubles, 7 bytes per entry less.
template <int MODE, int LEN, bool PRED, bool IMPL, bool VAL8, bool STAB, bool IMPV = false>
__device__ __forceinline__ void short_row(const SellArgs &A, int64_t ent, int64_t slice, int len, const double *x,
                                          int32_t row, bool active, const SellEp &E, double &contrib,
                                          unsigned char halo_wait, const ExArgs *fx, RowOut &out, double *stab) {
    const int32_t *__restrict__ c = A.cols + ent;
    const double *__restrict__ v = A.vals + ent;
    const unsigned char *__restrict__ vi = A.vidx + ent;
    // STAB: the CTA keeps the value dictionary in shared memory (two instructions per lookup instead of five: the
    // sweeps are bound by instruction issue, ncu: 68-76 % issue-slot utilisation at 4 of 7 TB/s).  Every thread starts
    // the asynchronous copy of one table entry now and waits for it after its own loads have been issued.
    if (STAB) cp_async8(stab + threadIdx.x, A.vtab + threadIdx.x);
    // The row's own vector entries (right-hand side, u of a prolongation, Jacobi's x and 1/diag, the dot product's
    // partner) are asked for HERE, under the matrix loads.  Left to their point of use -- after the gathers have been
    // consumed -- each is a second dependent DRAM round trip per thread (cuobjdump showed the load of b behind the last
    // gather).  A prefetch holds no register (the sweeps sit at the 32-register limit of full occupancy; loading b early
    // spilled it straight back to local memory), the load at the point of use then hits L1.  PROLONG rows are short and
    // have registers to spare: their u is loaded.
    constexpr bool kUsesB = MODE == RESID || MODE == RESNORM || mode_is_jacobi_like(MODE) || mode_is_gs(MODE);
    constexpr bool kUsesAux = mode_is_jacobi_like(MODE) || MODE == SPMV_DOT;
    constexpr bool kEarly = kRowOperands == 3;
    double bv = 0.0, av = 0.0, xr = 0.0, dv = 0.0;
    if (active) {
        if (MODE == PROLONG) av = E.aux[row];
        if (kEarly) {
            if (kUsesB) bv = E.b[row];
            if (kUsesAux) av = E.aux[row];
            if (mode_is_jacobi_like(MODE)) xr = x[row];
            if (MODE == CHEBY && E.has_d) dv = A.r_out[row];
        } else {
            if (kUsesB) prefetch_row_operand(E.b + row);
            if (kUsesAux) prefetch_row_operand(E.aux + row);
            if (mode_is_jacobi_like(MODE)) prefetch_row_operand(x + row);
            if (MODE == CHEBY && E.has_d) prefetch_row_operand(A.r_out + row);
        }
    }
    static_assert(!IMPV || (IMPL && VAL8 && !STAB && !PRED), "implied values ride on implied columns and a dictionary");
    int32_t cc[LEN];
    double vv[LEN], xx[LEN];
    unsigned ii[VAL8 ? LEN : 1];
    if (IMPV) {
        // nothing to load: the values are the launch's record (below) or, for the few other slices, fetched there
    } else if (VAL8) {
#pragma unroll
        for (int j = 0; j < LEN; ++j)
            if (!PRED || j < len) ii[j] = ld_stream_u8(vi + j * kSlice);
#pragma unroll
        for (int j = 0; j < LEN; ++j)
            if (!PRED || j < len) {
                if (!IMPL) cc[j] = ld_stream(c + j * kSlice);
                if (!STAB) vv[j] = __ldg(A.vtab + ii[j]);
            }
    } else {
#pragma unroll
        for (int j = 0; j < LEN; ++j) {
            if (!PRED || j < len) {
                vv[j] = ld_stream(v + j * kSlice);
                if (!IMPL) cc[j] = ld_stream(c + j * kSlice);
            }
        }
    }
    unsigned rec = 0;
    if (IMPL) {
        rec = ld_const_u16(A.slice_rec + slice);   // two bytes, the same for the whole warp; not waited for yet
        // speculative columns: the expected record applied to the row, which is clamped ONCE so that every column stays
        // inside the vector (a slice that really uses the record has all its rows inside [lo, hi]: the clamp is the
        // identity there; any other slice redoes its gathers below)
        const int32_t rs = min(max(row, A.spec_lo), A.spec_hi);
#pragma unroll
        for (int j = 0; j < LEN; ++j) cc[j] = rs + A.spec_off[j];
    }
    if (halo_wait) fused_wait_ready(*fx);
    // A Gauss-Seidel row never uses its own old value (the diagonal entry divides, and a row that is not updated has a
    // zero there): no gather for it -- 8 bytes per row of DRAM reads less (ncu: 65 -> 57 B per 5-point row)
#pragma unroll
    for (int j = 0; j < LEN; ++j)
        if (!PRED || j < len) xx[j] = mode_is_gs(MODE) ? ld_gather_skip(x, cc[j], row) : ld_gather(x, cc[j]);
    if (STAB) {
        // everything this row reads from DRAM is in flight: wait for the table entry, meet the other warps, look the values up
        cp_async_wait_all();
        __syncthreads();
#pragma unroll
        for (int j = 0; j < LEN; ++j)
            if (!PRED || j < len) vv[j] = stab[ii[j]];
    }
    const bool other = IMPL && rec != (unsigned)A.spec_id;
    if (other) {                                   // warp-uniform and rare: this slice uses another record, or none
        if (rec == (unsigned)kRecIrregular) {
#pragma unroll
            for (int j = 0; j < LEN; ++j) cc[j] = ld_stream(c + j * kSlice);
            if (IMPV) {
#pragma unroll
                for (int j = 0; j < LEN; ++j) ii[j] = ld_stream_u8(vi + j * kSlice);
#pragma unroll
                for (int j = 0; j < LEN; ++j) vv[j] = __ldg(A.vtab + ii[j]);
            }
        } else {
            const int32_t *__restrict__ o = A.rec_table + rec * kOffStride;
#pragma unroll
            for (int j = 0; j < LEN; ++j) cc[j] = row + __ldg(o + j);
            if (IMPV) {
                const double *__restrict__ rv = A.rec_vals + rec * kOffStride;
#pragma unroll
                for (int j = 0; j < LEN; ++j) vv[j] = __ldg(rv + j);
            }
        }
#pragma unroll
        for (int j = 0; j < LEN; ++j) xx[j] = (mode_is_gs(MODE) && cc[j] == row) ? 0.0 : x[cc[j]];
    }
    // The rest of the row -- products, sums, epilogue -- as a function of where values, gathered entries and columns
    // come from: the kernels with implied values run it on the launch's value record (kernel parameters: operands
    // straight from the constant bank, no register copies) for the slices that use it and on loaded values for the
    // others; everything else runs it once.
    // `known`: the row belongs to a slice of the launch's record, so which entry is the diagonal and what it holds are
    // launch constants too (spec_diag / spec_dmask) instead of five compares, ten selects and four ORs per row.
    auto finish = [&](auto known, const double (&vv)[LEN], const double (&xx)[LEN], const int32_t (&cc)[LEN]) {
        constexpr bool KD = decltype(known)::value;
        double sum = 0.0;
        // GS_RES keeps the separately rounded products (the slot of the diagonal entry flagged in dmask) instead of the row
        // itself: 2 registers per entry across the division instead of 5.
        // Gauss-Seidel family, branch-free: the diagonal entry was "gathered" as +0.0, so its product is an exact zero, and
        // adding a zero never changes a sum that started at +0.0 (such a sum is never -0.0): the sum has the bits of the
        // oracle's, which skips the entry.  The diagonal VALUE is collected by OR-ing bit patterns: a row has one stored
        // diagonal entry; padding that repeats its column carries +0.0, i.e. no bits (the old test `value != 0`).
        double pp[MODE == GS_RES ? LEN : 1];
        unsigned dmask = KD ? A.spec_dmask : 0u;
        unsigned long long dbits = 0ull;
#pragma unroll
        for (int j = 0; j < LEN; ++j) {
            if (!PRED || j < len) {
                if (mode_is_gs(MODE)) {
                    const bool is_d = cc[j] == row;
                    const double p = __dmul_rn(vv[j], xx[j]);
                    sum = __dadd_rn(sum, p);
                    if (!KD) dbits |= is_d ? (unsigned long long)__double_as_longlong(vv[j]) : 0ull;
                    if (MODE == GS_RES) {
                        pp[j] = p;
                        if (!KD) dmask |= (is_d && vv[j] != 0.0) ? (1u << j) : 0u;
                    }
                } else {
                    sum = mul_add_unfused(sum, vv[j], xx[j]);
                }
            }
        }
        const double diag = KD ? A.spec_diag : __longlong_as_double((long long)dbits);
        if (!active) return;
        if (!kEarly) {
            if (kUsesB) bv = E.b[row];
            if (kUsesAux) av = E.aux[row];
            if (mode_is_jacobi_like(MODE)) xr = x[row];
            if (MODE == CHEBY && E.has_d) dv = A.r_out[row];
        }
        if (MODE == SPMV) {
            E.y[row] = sum;
        } else if (MODE == SPMV_DOT) {
            E.y[row] = sum;
            contrib = av * sum;
        } else if (MODE == RESID) {
            E.y[row] = __dsub_rn(bv, sum);
        } else if (MODE == RESNORM) {
            const double r = __dsub_rn(bv, sum);
            contrib = r * r;
        } else if (MODE == JACOBI) {
            const double r = __dsub_rn(bv, sum);
            E.y[row] = __dadd_rn(xr, __dmul_rn(E.omega, __dmul_rn(av, r)));
        } else if (MODE == CHEBY) {
            const double dn = cheby_dn(E.cd, E.has_d, dv, E.omega, __dmul_rn(av, __dsub_rn(bv, sum)));
            A.r_out[row] = dn;
            E.y[row] = __dadd_rn(xr, dn);
        } else if (MODE == PROLONG) {
            E.y[row] = __dadd_rn(av, sum);   // aux = u (may alias y)
        } else {                             // Gauss-Seidel family
            const bool upd = diag != 0.0;
            double xn = 0.0;
            if (upd) {
                xn = __ddiv_rn(__dsub_rn(bv, sum), diag);
                if (MODE == GS_NORM) {
                    out.xn = xn;
                    out.store = true;
                } else {
                    E.y[row] = xn;
                }
            }
            if (MODE == GS_RES) {
                // residual of the row with its new value: the products in storage order, the diagonal entry times the new
                // iterate in its place (selects, no branches).  A diagonal entry of a row that was not updated is a stored
                // zero: xn is 0 then and the term an exact zero, which changes nothing (a sum that starts at +0 never
                // becomes -0).  These are the bits of the residual pass: the restriction reads them.
                double s2 = 0.0;
                const double dx = __dmul_rn(diag, xn);
#pragma unroll
                for (int j = 0; j < LEN; ++j)
                    if (!PRED || j < len) {
                        const double t = ((dmask >> j) & 1u) ? dx : pp[j];
                        s2 = __dadd_rn(s2, t);
                    }
                A.r_out[row] = __dsub_rn(bv, s2);
            }
            if (MODE == GS_NORM) {
                // The swept row's share of ||b - A x||^2.  Only the NORM is wanted here (a history value compared at
                // 1e-12, summed in an order of its own anyway), so the row's residual is taken as (b - sum) - d x_new in one
                // fused multiply-add instead of re-adding the products in storage order: the row has just been solved, the
                // value is rounding noise of size eps |b| either way, and the kernel stays as light as the plain sweep
                // (ncu: the storage-order version ran at 2.4 TB/s against 3.9 for the sweep).
                const double r = upd ? fma(-diag, xn, __dsub_rn(bv, sum)) : __dsub_rn(bv, sum);
                contrib = r * r;
            }
        }
    };
    if (IMPV && !other) {
        double vs[LEN];
#pragma unroll
        for (int j = 0; j < LEN; ++j) vs[j] = A.spec_val[j];
        finish(std::true_type{}, vs, xx, cc);
    } else {
        finish(std::false_type{}, vv, xx, cc);
    }
}

// CNT consecutive entries of a long row (LEN == 0 kernels): loads first, then gathers, then the sums
template <int MODE, int CNT>
__device__ __forceinline__ void row_chunk(const int32_t *__restrict__ c, const double *__restrict__ v,
                                          const double *x, int64_t row, double &sum, double &diag,
                                          unsigned char halo_wait = 0, const ExArgs *fx = nullptr) {
    int32_t cc[CNT];
    double vv[CNT], xx[CNT];
#pragma unroll
    for (int j = 0; j < CNT; ++j) {
        cc[j] = ld_stream(c + j * kSlice);
        vv[j] = ld_stream(v + j * kSlice);
    }
    if (halo_wait) fused_wait_ready(*fx);
#pragma unroll
    for (int j = 0; j < CNT; ++j) xx[j] = (MODE == GS && cc[j] == row) ? 0.0 : x[cc[j]];
#pragma unroll
    for (int j = 0; j < CNT; ++j) {
        if (MODE == GS) {
            if (cc[j] == row) { if (vv[j] != 0.0) diag = vv[j]; } else sum = mul_add_unfused(sum, vv[j], xx[j]);
        } else {
            sum = mul_add_unfused(sum, vv[j], xx[j]);
        }
    }
}

// LEN   : the matrix' longest slice when it is <= 8 (short_row), 0 for longer rows (chunks of 4 + rolled remainder;
//         not for GS_RES / GS_NORM, which need the whole row in registers).
// UNIFORM: every slice of the matrix has exactly LEN entries, so the slice offset is computed instead of loaded.
// IMPL  : implied columns for the regular slices (UNIFORM matrices only).
// The microbenchmark behind these choices is tools/sellbench.cu (profiles/r01_sellbench.log): occupancy x bytes in
// flight per thread decides; at 32 registers and 60 B per thread the fine-level sweep reaches the DRAM limit
// (6.8 TB/s algorithmic, ~7.1 TB/s of actual traffic), a rolled loop stays at 5.4 TB/s.
template <int MODE, int LEN, bool UNIFORM, bool FUSED, bool IMPL, bool VAL8, bool IMPV = false>
__device__ __forceinline__ void
sell_body(const SellArgs &A, const double *x, const double *__restrict__ b, const double *aux, double *y, double omega,
          double *__restrict__ partials, int64_t bid, const ExArgs *fx, const unsigned char *__restrict__ mask) {
    static_assert(!IMPL || (UNIFORM && LEN > 0), "implied columns need a uniform matrix with short rows");
    static_assert(LEN > 0 || !mode_is_tail(MODE), "fused residual modes need the row in registers");
    static_assert(!VAL8 || LEN > 0, "the value dictionary is for short rows");
    constexpr int BLK = FUSED ? kBlock : kSellBlock;
    // the value dictionary sits in shared memory when every warp of the CTA takes the same path to the barrier that
    // publishes it (uniform matrices) and the CTA has one thread per table entry
    constexpr bool STAB = kSharedDict && VAL8 && UNIFORM && LEN > 0 && BLK == 256 && !IMPV;
    __shared__ double stab[STAB ? 256 : 1];
    // rows are 32-bit here (the launcher refuses matrices of 2^31 rows or more; column indices are int32 anyway): one
    // instruction per address instead of four
    const int32_t raw_row = (int32_t)A.first_row + (int32_t)bid * BLK + (int32_t)threadIdx.x;
    const int32_t row_end = (int32_t)A.row_end;
    const bool active = raw_row >= (int32_t)A.row_begin && raw_row < row_end;
    // a CTA that shares a table meets at a barrier: its threads past the end redo the last row without storing
    const int32_t row = STAB ? min(raw_row, row_end - 1) : raw_row;
    double contrib = 0.0;
    RowOut out{0.0, false};
    if (row < row_end) {   // warp-uniform except in the last slice
        const int64_t slice = row >> 5;
        const int lane = row & 31;
        unsigned char hw = 0;      // fused launch: does this slice read halo columns? (load issued now, used later)
        if (FUSED) hw = mask ? mask[slice] : 1;
        int64_t base;
        int len;
        if (UNIFORM) {
            base = slice * (int64_t)(kSlice * LEN);
            len = LEN;
        } else {
            base = A.slice_ptr[slice];
            len = (int)((A.slice_ptr[slice + 1] - base) >> 5);
        }
        const double *__restrict__ v = A.vals + base + lane;
        const int32_t *__restrict__ c = A.cols + base + lane;
        if (LEN > 0) {
            constexpr int L = LEN > 0 ? LEN : 1;
            const SellEp E{b, aux, y, omega, MODE == CHEBY ? cheby_cd(partials) : 0.0, MODE == CHEBY && partials != nullptr};
            if (IMPL) {
                short_row<MODE, L, false, true, VAL8, STAB, IMPV>(A, base + lane, slice, L, x, row, active, E, contrib, hw, fx, out, stab);
            } else if (UNIFORM || len == L) {
                short_row<MODE, L, false, false, VAL8, STAB>(A, base + lane, slice, L, x, row, active, E, contrib, hw, fx, out, stab);
            } else {
                short_row<MODE, L, true, false, VAL8, false>(A, base + lane, slice, len, x, row, active, E, contrib, hw, fx, out, stab);
            }
        } else {
            double sum = 0.0, diag = 0.0;
            // the row's own vector entries first (see short_row): not one more round trip behind the last chunk
            double bv = 0.0, av = 0.0, xr = 0.0, dv = 0.0;
            if ((MODE == RESID || MODE == RESNORM || mode_is_jacobi_like(MODE) || MODE == GS) && active) bv = b[row];
            if ((MODE == PROLONG || mode_is_jacobi_like(MODE) || MODE == SPMV_DOT) && active) av = aux[row];
            if (mode_is_jacobi_like(MODE) && active) xr = x[row];
            if (MODE == CHEBY && partials != nullptr && active) dv = A.r_out[row];
            int k = 0;
            for (; k + 4 <= len; k += 4) {
                row_chunk<MODE, 4>(c + k * kSlice, v + k * kSlice, x, row, sum, diag, hw, fx);
                hw = 0;
            }
            for (; k < len; ++k) {
                row_chunk<MODE, 1>(c + k * kSlice, v + k * kSlice, x, row, sum, diag, hw, fx);
                hw = 0;
            }
            if (active) {
                if (MODE == SPMV) {
                    y[row] = sum;
                } else if (MODE == SPMV_DOT) {
                    y[row] = sum;
                    contrib = av * sum;
                } else if (MODE == RESID) {
                    y[row] = __dsub_rn(bv, sum);
                } else if (MODE == RESNORM) {
                    const double r = __dsub_rn(bv, sum);
                    contrib = r * r;
                } else if (MODE == JACOBI) {
                    const double r = __dsub_rn(bv, sum);
                    y[row] = __dadd_rn(xr, __dmul_rn(omega, __dmul_rn(av, r)));
                } else if (MODE == CHEBY) {
                    const double dn = cheby_dn(cheby_cd(partials), partials != nullptr, dv, omega,
                                               __dmul_rn(av, __dsub_rn(bv, sum)));
                    A.r_out[row] = dn;
                    y[row] = __dadd_rn(xr, dn);
                } else if (MODE == GS) {
                    if (diag != 0.0) y[row] = __ddiv_rn(__dsub_rn(bv, sum), diag);
                } else if (MODE == PROLONG) {
                    y[row] = __dadd_rn(av, sum);   // aux = u (may alias y)
                }
            }
        }
    }
    if (MODE == GS_NORM && out.store) y[row] = out.xn;
    if (mode_has_partials(MODE)) {
        const double s = block_sum_parked<BLK>(contrib);
        if (threadIdx.x == 0) partials[bid] = s;
    }
}

// resident CTAs per SM the compiler has to leave room for: the sweeps with a fused residual keep the row's products
// alive across the division and take 41-48 registers (5 CTAs) when left alone; capped at 40 (6 CTAs) where ptxas
// manages that without spilling (build/sell_modes_gs.ptxas.log)
__host__ __device__ constexpr int mode_min_ctas(int m, int len, bool uniform, bool impl) {
    if (m == GS_NORM || m == GS_RES) { if (len >= 1 && uniform && len <= 5) return 8; }
    if (mode_is_tail(m)) return (len <= 5 || (uniform && len <= 7)) ? 6 : 1;
    // the plain modes fit 32 registers (full occupancy); the Gauss-Seidel sweep and the implied-column kernels (whose
    // offsets arrive as kernel arguments) do so up to 5 entries per row
    if (len >= 1 && uniform && len <= ((m == GS || impl) ? 5 : 7)) return 8;
    return (impl && len <= 7) ? 6 : 1;
}

template <int MODE, int LEN, bool UNIFORM, bool IMPL, bool VAL8, bool IMPV = false>
__global__ void __launch_bounds__(kSellBlock, mode_min_ctas(MODE, LEN, UNIFORM, IMPL) * (kBlock / kSellBlock))
sell_kernel(SellArgs A, const double *x, const double *__restrict__ b, const double *aux,
            double *y, double omega, double *__restrict__ partials) {
    pdl_prologue();
    sell_body<MODE, LEN, UNIFORM, false, IMPL, VAL8, IMPV>(A, x, b, aux, y, omega, partials, (int64_t)blockIdx.x, nullptr, nullptr);
}

// Very short rows (linear transfer operators: one or two entries): one row per thread keeps only ~30 bytes per thread in
// flight behind a chain of three dependent loads (slice pointer -> column -> vector entry), and the prolongation runs at
// 5.4 instead of 6.8 TB/s (ncu, profiles/r02_ncu_step_sell_kernels.txt).  Here a thread takes R rows, 256 apart, and
// issues every load of a stage for all of them before the first use.  SpMV and prolongation, LEN <= 2, no exchange site.
// UNIFORM: every slice holds exactly LEN entries per row (transfer operators are padded to that when it costs at most a
// quarter more entries, mg_sell_layout), so the slice pointer -- the first of the three round trips -- is computed.
template <int MODE, int LEN, int R, bool VAL8, bool UNIFORM>
__global__ void __launch_bounds__(kBlock, 6)
sell_short_kernel(SellArgs A, const double *x, const double *aux, double *y) {
    static_assert(MODE == SPMV || MODE == PROLONG, "short-row kernel: SpMV and prolongation only");
    pdl_prologue();
    int64_t row[R], base[R];
    int len[R];
    bool act[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        row[r] = A.first_row + ((int64_t)blockIdx.x * R + r) * kBlock + threadIdx.x;
        act[r] = row[r] >= A.row_begin && row[r] < A.row_end;
        base[r] = 0;
        len[r] = 0;
        if (row[r] < A.row_end) {
            const int64_t sl = row[r] >> 5;
            if (UNIFORM) {
                base[r] = sl * (int64_t)(kSlice * LEN) + (row[r] & 31);
                len[r] = LEN;
            } else {
                const int64_t p0 = A.slice_ptr[sl], p1 = A.slice_ptr[sl + 1];
                base[r] = p0 + (row[r] & 31);
                len[r] = (int)((p1 - p0) >> 5);
            }
        }
    }
    int32_t cc[R][LEN];
    double vv[R][LEN], xx[R][LEN], av[R];
    unsigned char ii[R][LEN];
#pragma unroll
    for (int r = 0; r < R; ++r) {
#pragma unroll
        for (int j = 0; j < LEN; ++j)
            if (j < len[r]) {
                cc[r][j] = ld_stream(A.cols + base[r] + j * kSlice);
                if (VAL8) ii[r][j] = ld_stream(A.vidx + base[r] + j * kSlice);
                else vv[r][j] = ld_stream(A.vals + base[r] + j * kSlice);
            }
        av[r] = (MODE == PROLONG && act[r]) ? aux[row[r]] : 0.0;
    }
    if (VAL8) {
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int j = 0; j < LEN; ++j)
                if (j < len[r]) vv[r][j] = __ldg(A.vtab + ii[r][j]);
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < LEN; ++j)
            if (j < len[r]) xx[r][j] = x[cc[r][j]];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < LEN; ++j)
            if (j < len[r]) sum = mul_add_unfused(sum, vv[r][j], xx[r][j]);
        if (act[r]) y[row[r]] = MODE == PROLONG ? __dadd_rn(av[r], sum) : sum;
    }
}

// ---- implied transfer columns: slice patterns ---------------------------------------------------------------------
// A transfer operator's columns live in the other level's colour-blocked numbering, so `col = row + off[j]` (implied
// columns above) never holds.  What does hold, for almost every slice of a structured hierarchy, is that the slice's
// columns are its first stored column (entry 0 of lane 0, the base) plus one of a few LEN x 32 delta patterns, and its
// values one of a few value patterns (linear interpolation: 1, 1/2 and the padding's 0): mg_sell with nrec < 0
// (engine.DeviceSell._attach_patterns, formats.pattern_records).  A slice then reads a two-byte record id and a
// four-byte base, both from dense per-slice arrays that a CTA's warps share in L1, instead of 32*LEN*(4+1) bytes of
// columns and dictionary bytes; the pattern itself comes from L1 (the records of a launch are a few KB).
// SPEC (the restriction: one record covers nearly every slice of a colour block): the launch carries the record most
// slices of each row block use, the thread loads its deltas by lane from L1 at once and issues the x gathers as soon as
// the base arrives, before the slice's own id is known; slices of another record redo their gathers.  Without SPEC (the
// prolongation: its slices split over about four patterns per colour -- grid-line parity x the colour of lane 0 -- so
// three quarters would miss and gather twice) the thread waits for the id and reads that record: base and id (L2 / L1)
// -> deltas (L1) -> x, where the explicit kernel has columns (DRAM) -> x.  Irregular slices (0xffff) read their columns
// and values.  Products are added in storage order from the same doubles: the same bits as sell_kernel and
// sell_short_kernel.  R rows per thread, 256 apart, for the one- and two-entry rows of a prolongation.
constexpr int kPatBlocks = 8;       // row blocks with their own expected record per launch

struct PatArgs {
    const unsigned short *__restrict__ rec;    // [nslices] record id, 0xffff = read the slice's columns and values
    const int32_t *__restrict__ base;          // [nslices] first stored column of the slice
    const int32_t *__restrict__ delta;         // [nrec][LEN][32] column - base
    const double *__restrict__ pvals;          // [nrec][LEN][32] values
    const int32_t *__restrict__ cols;
    const double *__restrict__ vals;
    int32_t spec_row[kPatBlocks];              // block k = rows [spec_row[k], spec_row[k+1]) (unused: INT32_MAX)
    int32_t spec_id[kPatBlocks];               // ... and the record its launch expects (SPEC)
    int32_t row_begin, row_end, first_row;
    uint32_t col_max;                          // ncols - 1: speculative columns are clamped to it
};

template <int MODE, int LEN, int R, bool SPEC>
__global__ void __launch_bounds__(kBlock, LEN >= 8 ? 4 : 5)
sell_pattern_kernel(PatArgs A, const double *x, const double *aux, double *y) {
    static_assert(MODE == SPMV || MODE == PROLONG, "slice patterns: SpMV and prolongation only");
    pdl_prologue();
    const int lane = threadIdx.x & 31;
    int32_t row[R], bs[R], cc[R][LEN];
    unsigned id[R];
    bool in[R];
    double vv[R][LEN], xx[R][LEN], av[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        row[r] = A.first_row + ((int32_t)blockIdx.x * R + r) * kBlock + (int32_t)threadIdx.x;
        in[r] = row[r] < A.row_end;                           // warp-uniform except in the last slice
        bs[r] = in[r] ? __ldg(A.base + (row[r] >> 5)) : 0;
        id[r] = in[r] ? ld_const_u16(A.rec + (row[r] >> 5)) : 0u;
    }
    int spec[R];
    if (SPEC) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            spec[r] = A.spec_id[0];
#pragma unroll
            for (int k = 1; k < kPatBlocks; ++k) spec[r] = row[r] >= A.spec_row[k] ? A.spec_id[k] : spec[r];
#pragma unroll
            for (int j = 0; j < LEN; ++j) cc[r][j] = __ldg(A.delta + (spec[r] * LEN + j) * kSlice + lane);
        }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) av[r] = (MODE == PROLONG && in[r] && row[r] >= A.row_begin) ? aux[row[r]] : 0.0;
    if (SPEC) {
        // speculative gathers: exact for slices of the expected record, clamped into the vector for any other
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (in[r]) {
#pragma unroll
                for (int j = 0; j < LEN; ++j)
                    xx[r][j] = ld_gather(x, (int32_t)min((uint32_t)(bs[r] + cc[r][j]), A.col_max));
            }
    }
    bool redo[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        redo[r] = in[r] && (!SPEC || id[r] != (unsigned)spec[r]);
        if (!in[r]) continue;
        if (SPEC && !redo[r]) {
#pragma unroll
            for (int j = 0; j < LEN; ++j) vv[r][j] = __ldg(A.pvals + (spec[r] * LEN + j) * kSlice + lane);
        } else if (id[r] == (unsigned)kRecIrregular) {        // warp-uniform
            const int64_t ent = (int64_t)(row[r] >> 5) * (kSlice * LEN) + lane;
#pragma unroll
            for (int j = 0; j < LEN; ++j) {
                cc[r][j] = ld_stream(A.cols + ent + j * kSlice);
                vv[r][j] = ld_stream(A.vals + ent + j * kSlice);
            }
        } else {
            const int o = (int)id[r] * LEN * kSlice + lane;
#pragma unroll
            for (int j = 0; j < LEN; ++j) {
                cc[r][j] = bs[r] + __ldg(A.delta + o + j * kSlice);
                vv[r][j] = __ldg(A.pvals + o + j * kSlice);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
        if (redo[r]) {
#pragma unroll
            for (int j = 0; j < LEN; ++j) xx[r][j] = ld_gather(x, cc[r][j]);
        }
#pragma unroll
    for (int r = 0; r < R; ++r) {
        if (!in[r] || row[r] < A.row_begin) continue;
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < LEN; ++j) sum = mul_add_unfused(sum, vv[r][j], xx[r][j]);
        y[row[r]] = MODE == PROLONG ? __dadd_rn(av[r], sum) : sum;
    }
}

// The same kernel carrying an exchange site (multi-GPU, csrc/comm.cu): the first npeers*ctas_per_peer CTAs push the
// boundary values the previous kernel produced, poll for the peers' packets and unpack them into the halo of x; the
// compute CTAs whose slice reads halo columns (mask) wait for that, all others start at once.  The exchange latency
// (NVLink flight + polling) is hidden behind the interior rows, and the site costs no launch of its own.
// (the launches that also carry an exchange site keep 40 registers for the sweeps with a fused residual: ptxas spills at 32)
__host__ __device__ constexpr int fused_min_ctas(int m, int len, bool uniform, bool impl) {
    if (mode_is_tail(m)) return (len <= 5 || (uniform && len <= 7)) ? 6 : 1;
    return mode_min_ctas(m, len, uniform, impl);
}

template <int MODE, int LEN, bool UNIFORM, bool IMPL, bool VAL8, bool IMPV = false>
__global__ void __launch_bounds__(kBlock, fused_min_ctas(MODE, LEN, UNIFORM, IMPL))
sell_kernel_fused(SellArgs A, const double *x, const double *__restrict__ b, const double *aux, double *y, double omega,
                  double *__restrict__ partials, const ExArgs fx, const unsigned char *__restrict__ mask) {
    pdl_prologue();
    const int nex = fx.npeers * fx.ctas_per_peer;
    if ((int)blockIdx.x < nex) {
        fused_exchange_cta(fx, (int)blockIdx.x);
        if (mode_has_partials(MODE)) {}      // exchange CTAs own no partial sum
        return;
    }
    sell_body<MODE, LEN, UNIFORM, true, IMPL, VAL8, IMPV>(A, x, b, aux, y, omega, partials, (int64_t)blockIdx.x - nex, &fx, mask);
}

// ---- long rows: four warps per slice ---------------------------------------------------------------------------------
// With 19- / 37-point Galerkin stencils (quasi-L2 transfers) one thread walking a whole row is a chain of dependent
// (column -> x gather) round trips: ~15 us per launch however small, and half the DRAM rate on large levels.  Here
// the four warps of a slice take every fourth entry each, issue all their loads up front, and park the separately
// rounded products v*x in shared memory; one warp then adds them in STORAGE ORDER, so the row sums keep the oracle's
// bits (the additions are the only order-sensitive part, and they are a few hundred cycles of shared-memory reads).
constexpr int kWideU = 5;          // entries per warp and pass
constexpr int kWideMaxLen = 64;    // products kept in shared memory: 64 entries x 32 rows per slice

// WPS warps share one slice (kBlock/32/WPS slices per CTA); WPS*kWideU entries per pass: 4 warps cover the 19-point
// stencil in one pass, 8 warps the 37-point one.
template <int MODE, int WPS>
__global__ void __launch_bounds__(kBlock)
sell_wide_kernel(SellArgs A, int uniform_len, const double *x, const double *__restrict__ b, const double *aux,
                 double *y, double omega, double *__restrict__ partials) {
    pdl_prologue();
    constexpr int SPC = kBlock / 32 / WPS;
    __shared__ double prod[SPC][kWideMaxLen][kSlice];
    __shared__ unsigned char skip[SPC][kWideMaxLen][kSlice];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sl = warp / WPS, w = warp % WPS;
    const int64_t slice = (A.first_row >> 5) + (int64_t)blockIdx.x * SPC + sl;
    const int64_t row = slice * kSlice + lane;
    int len = 0;
    int64_t base = 0;
    if (slice * kSlice < A.row_end && row < A.nrows) {
        if (uniform_len > 0) {
            base = slice * (int64_t)kSlice * uniform_len;
            len = uniform_len;
        } else {
            base = A.slice_ptr[slice];
            len = (int)((A.slice_ptr[slice + 1] - base) >> 5);
        }
    }
    // the warp that will finish the rows fetches their vector entries now, under the shadow of the matrix loads
    const bool finisher = w == 0 && row >= A.row_begin && row < A.row_end;
    double bv = 0.0, av = 0.0;
    if (finisher) {
        if (MODE != SPMV && MODE != PROLONG && MODE != SPMV_DOT) bv = b[row];
        if (mode_is_jacobi_like(MODE) || MODE == PROLONG || MODE == SPMV_DOT) av = aux[row];
    }
    const double *__restrict__ v = A.vals + base + lane;
    const int32_t *__restrict__ c = A.cols + base + lane;
    for (int k0 = w; k0 < len; k0 += WPS * kWideU) {
        int32_t cc[kWideU];
        double vv[kWideU], xx[kWideU];
#pragma unroll
        for (int j = 0; j < kWideU; ++j) {
            const int k = k0 + j * WPS;
            if (k < len) {
                cc[j] = ld_stream(c + (int64_t)k * kSlice);
                vv[j] = ld_stream(v + (int64_t)k * kSlice);
            }
        }
#pragma unroll
        for (int j = 0; j < kWideU; ++j)
            if (k0 + j * WPS < len) xx[j] = (mode_is_gs(MODE) && cc[j] == row) ? 0.0 : x[cc[j]];
#pragma unroll
        for (int j = 0; j < kWideU; ++j) {
            const int k = k0 + j * WPS;
            if (k < len) {
                const bool is_diag = mode_is_gs(MODE) && cc[j] == row;
                prod[sl][k][lane] = is_diag ? vv[j] : __dmul_rn(vv[j], xx[j]);
                if (mode_is_gs(MODE)) skip[sl][k][lane] = is_diag ? 1 : 0;
            }
        }
    }
    double xr = 0.0, dv = 0.0;
    if (mode_is_jacobi_like(MODE) && finisher) xr = x[row];
    if (MODE == CHEBY && finisher && partials != nullptr) dv = A.r_out[row];
    __syncthreads();
    double contrib = 0.0;
    if (finisher) {
        double sum = 0.0, diag = 0.0;
        for (int k = 0; k < len; ++k) {
            const double p = prod[sl][k][lane];
            if (mode_is_gs(MODE) && skip[sl][k][lane]) { if (p != 0.0) diag = p; }
            else sum = __dadd_rn(sum, p);
        }
        if (MODE == SPMV) {
            y[row] = sum;
        } else if (MODE == SPMV_DOT) {
            y[row] = sum;
            contrib = av * sum;
        } else if (MODE == RESID) {
            y[row] = __dsub_rn(bv, sum);
        } else if (MODE == RESNORM) {
            const double r = __dsub_rn(bv, sum);
            contrib = r * r;
        } else if (MODE == JACOBI) {
            const double r = __dsub_rn(bv, sum);
            y[row] = __dadd_rn(xr, __dmul_rn(omega, __dmul_rn(av, r)));
        } else if (MODE == CHEBY) {
            const double dn = cheby_dn(cheby_cd(partials), partials != nullptr, dv, omega, __dmul_rn(av, __dsub_rn(bv, sum)));
            A.r_out[row] = dn;
            y[row] = __dadd_rn(xr, dn);
        } else if (MODE == PROLONG) {
            y[row] = __dadd_rn(av, sum);
        } else {                       // Gauss-Seidel family, see short_row
            const bool upd = diag != 0.0;
            double xn = 0.0;
            if (upd) {
                xn = __ddiv_rn(__dsub_rn(bv, sum), diag);
                y[row] = xn;
            }
            if (MODE != GS) {
                // the residual of the row with its new value: the parked products in storage order, the diagonal
                // entry (parked as its VALUE) times the new iterate in its place.  A diagonal entry that did not
                // update the row is a stored zero: its product is an exact zero and adding it changes nothing.
                double s2 = 0.0;
                for (int k = 0; k < len; ++k) {
                    const double p = prod[sl][k][lane];
                    s2 = __dadd_rn(s2, skip[sl][k][lane] ? __dmul_rn(p, xn) : p);
                }
                const double r = __dsub_rn(bv, s2);
                if (MODE == GS_RES) A.r_out[row] = r;
                else contrib = r * r;
            }
        }
    }
    if (mode_has_partials(MODE)) {
        const double s = block_sum_last<kBlock>(contrib);
        if (threadIdx.x == 0) partials[blockIdx.x] = s;
    }
}

// ---- launcher ----------------------------------------------------------------------------------------------------------
// tunables (defined in sell_kernels.cu)
extern int64_t g_wide_min_len;      // slices at least this long use sell_wide_kernel (0 = never)
extern int64_t g_wide_max_rows;     // ... for launches of at most this many rows
extern int64_t g_tma_min_rows;      // rows per launch from which the bulk-async staged kernel is used; 0 disables it
extern int g_implied_columns;       // use the offset tables of matrices that carry one
extern int64_t g_implied_min_rows;  // ... for launches of at least this many rows
extern int g_value_dict;            // use the value dictionaries of matrices that carry one
extern int g_implied_values;        // use the value records of matrices that carry them (on top of the two above)
extern int g_short_rows_per_thread; // rows per thread of sell_short_kernel (1 = off, 2 or 4)
extern int64_t g_short_min_rows;    // ... for launches of at least this many rows
extern int g_implied_transfers;     // use the slice patterns of matrices that carry them (sell_pattern_kernel)

inline bool sell_use_patterns(const mg_sell *A, int64_t row0, int64_t row1) {
    const int64_t ml = A->max_slice_len;
    return g_implied_transfers && A->d_slice_rec && A->d_rec_table && A->d_rec_vals && A->nrec < 0 &&
           A->uniform_len == ml && ml >= 1 && ml <= 8 && row1 - row0 >= g_implied_min_rows;
}

template <int MODE>
int launch_sell_pattern(const mg_sell *A, const double *x, const double *aux, double *y, int64_t row0, int64_t row1,
                        cudaStream_t st, const char *name, int *nblocks_out) {
    const int L = (int)A->max_slice_len;
    PatArgs a;
    a.rec = A->d_slice_rec;
    a.delta = A->d_rec_table;
    a.base = A->d_rec_table + (int64_t)(-A->nrec) * L * kSlice;   // the table holds the bases behind the patterns
    a.pvals = A->d_rec_vals;
    a.cols = A->d_cols;
    a.vals = A->d_vals;
    // the expected record of each row block (mg_sell.h_spec_*; without hints record 0, the most frequent one) and how
    // many of the block's slices use it (per mille): the launch speculates when every block it touches is mostly one
    // record
    for (int k = 0; k < kPatBlocks; ++k) {
        a.spec_row[k] = k == 0 ? 0 : INT32_MAX;
        a.spec_id[k] = 0;
    }
    bool spec = false;
    if (A->h_spec_row && A->h_spec_rec && A->n_spec > 0) {
        spec = true;
        for (int k = 0; k < A->n_spec; ++k) {
            if (k < kPatBlocks) {
                a.spec_row[k] = k == 0 ? 0 : (int32_t)A->h_spec_row[k];
                a.spec_id[k] = A->h_spec_rec[9 * k];
            }
            if (A->h_spec_row[k] < row1 && A->h_spec_row[k + 1] > row0 && A->h_spec_rec[9 * k + 1] < 500) spec = false;
        }
    }
    a.row_begin = (int32_t)row0;
    a.row_end = (int32_t)row1;
    a.first_row = (int32_t)(row0 & ~(int64_t)(kSlice - 1));
    a.col_max = (uint32_t)(A->ncols > 0 ? A->ncols - 1 : 0);
    const int R = L <= 2 ? 2 : 1;
    const unsigned grid = (unsigned)(((row1 - a.first_row + kBlock - 1) / kBlock + R - 1) / R);
#define MG_PAT(LL, RR)                                                                                          \
    do {                                                                                                        \
        if (spec) launch_k(sell_pattern_kernel<MODE, LL, RR, true>, grid, kBlock, st, a, x, aux, y);            \
        else launch_k(sell_pattern_kernel<MODE, LL, RR, false>, grid, kBlock, st, a, x, aux, y);                \
    } while (0)
    switch (L) {
        case 1: MG_PAT(1, 2); break;
        case 2: MG_PAT(2, 2); break;
        case 3: MG_PAT(3, 1); break;
        case 4: MG_PAT(4, 1); break;
        case 5: MG_PAT(5, 1); break;
        case 6: MG_PAT(6, 1); break;
        case 7: MG_PAT(7, 1); break;
        default: MG_PAT(8, 1); break;
    }
#undef MG_PAT
    MG_CHECK_LAUNCH(name);
    if (nblocks_out) *nblocks_out = (int)grid;
    return MG_OK;
}

template <int MODE>
int launch_sell_tma(const mg_sell *M, int64_t max_len, const double *x, const double *b, const double *aux, double *y,
                    double omega, double *partials, int64_t row0, int64_t row1, int *grid_out, cudaStream_t st,
                    const char *name);

inline bool sell_uses_wide(const mg_sell *A, int64_t row0, int64_t row1) {
    const int64_t ml = A->max_slice_len;
    return g_wide_min_len > 0 && ml >= g_wide_min_len && ml <= kWideMaxLen && row1 - row0 <= g_wide_max_rows;
}
// which launches can carry an exchange site: the thread-per-row kernel only
bool sell_fusable(const mg_sell *A, int64_t row0, int64_t row1);
// which colour sweeps can also produce the residual / the squared residual norm of their rows (GS_RES / GS_NORM)
bool sell_gs_tail_ok(const mg_sell *A, int64_t row0, int64_t row1);

inline SellArgs sell_args(const mg_sell *A, int64_t row0, int64_t row1, double *r_out) {
    SellArgs a;
    a.slice_ptr = A->d_slice_ptr;
    a.cols = A->d_cols;
    a.vals = A->d_vals;
    a.slice_rec = A->d_slice_rec;
    a.rec_table = A->d_rec_table;
    a.spec_id = 0;
    for (int j = 0; j < 8; ++j) a.spec_off[j] = 0;
    a.spec_lo = 0;
    a.spec_hi = (int32_t)(A->ncols > 0 ? A->ncols - 1 : 0);
    a.vidx = A->d_val_idx;
    a.vtab = A->d_val_table;
    a.rec_vals = A->d_rec_vals;
    for (int j = 0; j < 8; ++j) a.spec_val[j] = 0.0;
    a.spec_diag = 0.0;
    a.spec_dmask = 0;
    a.row_begin = row0;
    a.row_end = row1;
    a.first_row = row0 & ~(int64_t)(kSlice - 1);
    a.nrows = A->nrows;
    a.r_out = r_out;
    return a;
}
inline bool sell_use_dict(const mg_sell *A) {
    const int64_t ml = A->max_slice_len;
    return g_value_dict && A->d_val_idx && A->d_val_table && ml >= 1 && ml <= 8;
}
inline bool sell_use_implied(const mg_sell *A, int64_t row0, int64_t row1) {
    const int64_t ml = A->max_slice_len;
    return g_implied_columns && A->d_slice_rec && A->d_rec_table && A->nrec > 0 && A->uniform_len > 0 &&
           A->uniform_len == ml && ml >= 1 && ml <= 8 && row1 - row0 >= g_implied_min_rows;
}
// the record a launch over [row0,row1) should expect: the hint of the block that holds row0 if the matrix carries
// hints, else record 0 (the most frequent one), whose offsets are then unknown on the host -> no speculation possible,
// the kernel takes the table path for every slice (spec_id = -1)
inline void sell_pick_spec(const mg_sell *A, int64_t row0, SellArgs &a) {
    a.spec_id = -1;
    for (int k = 0; k < A->n_spec && A->h_spec_row && A->h_spec_rec; ++k)
        if (row0 >= A->h_spec_row[k] && row0 < A->h_spec_row[k + 1]) {
            // rows in [lo, hi] keep row + off[j] inside [0, ncols) for every j; the kernel clamps the row to that range
            int64_t omin = 0, omax = 0;
            for (int j = 0; j < 8; ++j) {
                const int64_t o = A->h_spec_rec[9 * k + 1 + j];
                if (o < omin) omin = o;
                if (o > omax) omax = o;
            }
            const int64_t lo = -omin, hi = A->ncols - 1 - omax;
            if (hi < lo) return;                      // a matrix smaller than its stencil: no speculation
            a.spec_id = A->h_spec_rec[9 * k];
            for (int j = 0; j < 8; ++j) a.spec_off[j] = A->h_spec_rec[9 * k + 1 + j];
            a.spec_lo = (int32_t)lo;
            a.spec_hi = (int32_t)hi;
            if (A->h_spec_vals) {
                // the record's diagonal as the kernels find it: the entries in the row's own column, bit patterns OR-ed
                // (a row stores one; padding that repeats the column holds +0.0)
                unsigned long long bits = 0ull;
                for (int j = 0; j < 8; ++j) {
                    const double vj = A->h_spec_vals[8 * k + j];
                    a.spec_val[j] = vj;
                    if (j < A->uniform_len && a.spec_off[j] == 0) {
                        unsigned long long b;
                        memcpy(&b, &vj, sizeof(b));
                        bits |= b;
                        if (vj != 0.0) a.spec_dmask |= 1u << j;
                    }
                }
                memcpy(&a.spec_diag, &bits, sizeof(bits));
            }
            return;
        }
}

template <int MODE>
static int launch_sell(const mg_sell *A, const double *x, const double *b, const double *aux, double *y,
                       double omega, double *partials, int64_t row0, int64_t row1, cudaStream_t st,
                       const char *name, int *nblocks_out = nullptr, const SellFuse *fuse = nullptr,
                       double *r_out = nullptr) {
    if (nblocks_out) *nblocks_out = 0;
    if (fuse && !sell_fusable(A, row0, row1)) return set_error(MG_ERR_INVALID, name, "this launch cannot carry an exchange site");
    if (row1 <= row0) return MG_OK;
    if (A->nrows > 0x7fffffffLL || A->ncols > 0x7fffffffLL) return set_error(MG_ERR_OVERFLOW, name, "2^31 rows or more");
    if (mode_is_tail(MODE) && !sell_gs_tail_ok(A, row0, row1)) return set_error(MG_ERR_INVALID, name, "rows too long for a sweep with a fused residual");
    if constexpr (MODE <= PROLONG) {
        if (g_tma_min_rows > 0 && row1 - row0 >= g_tma_min_rows && A->max_slice_len > 0) {
            int grid = 0;
            const int rc = launch_sell_tma<MODE>(A, A->max_slice_len, x, b, aux, y, omega, partials, row0, row1, &grid, st, name);
            if (rc <= 0) {
                if (nblocks_out) *nblocks_out = grid;
                return rc;
            }
        }
    }
    if constexpr (MODE == SPMV || MODE == PROLONG) {
        if (!fuse && sell_use_patterns(A, row0, row1)) return launch_sell_pattern<MODE>(A, x, aux, y, row0, row1, st, name, nblocks_out);
    }
    SellArgs a = sell_args(A, row0, row1, r_out);
    if (sell_use_implied(A, row0, row1)) sell_pick_spec(A, row0, a);
    const int64_t nthreads = row1 - a.first_row;
    const int64_t ml = A->max_slice_len;
    const bool uni = A->uniform_len > 0 && A->uniform_len == ml;
    if (sell_uses_wide(A, row0, row1)) {
        const int wps = ml <= 4 * kWideU ? 4 : 8;
        const int spc = kBlock / 32 / wps;                            // slices per CTA
        const int64_t nsl = (nthreads + kSlice - 1) / kSlice;
        const int64_t wgrid = (nsl + spc - 1) / spc;
        if (wgrid > 0x7fffffffLL) return set_error(MG_ERR_OVERFLOW, name, "grid too large");
        if (wps == 4)
            launch_k(sell_wide_kernel<MODE, 4>, (unsigned)wgrid, kBlock, st, a, (int)(uni ? ml : 0), x, b, aux, y, omega, partials);
        else
            launch_k(sell_wide_kernel<MODE, 8>, (unsigned)wgrid, kBlock, st, a, (int)(uni ? ml : 0), x, b, aux, y, omega, partials);
        MG_CHECK_LAUNCH(name);
        if (nblocks_out) *nblocks_out = (int)wgrid;
        return MG_OK;
    }
    const int blk = fuse ? kBlock : kSellBlock;     // threads per CTA of the one-row-per-thread kernels
    const int64_t grid = (nthreads + blk - 1) / blk;
    if (grid + (fuse ? fuse->nex : 0) > 0x7fffffffLL) return set_error(MG_ERR_OVERFLOW, name, "grid too large");
    if constexpr (MODE == SPMV || MODE == PROLONG) {
        if (!fuse && ml >= 1 && ml <= 2 && g_short_rows_per_thread > 1 && row1 - row0 >= g_short_min_rows && (uni || A->d_slice_ptr)) {
            const int R = g_short_rows_per_thread >= 4 ? 4 : 2;
            const unsigned sg = (unsigned)(((nthreads + kBlock - 1) / kBlock + R - 1) / R);
            const bool dict = sell_use_dict(A);
#define MG_SHORT(L, RR)                                                                                 \
    do {                                                                                                \
        if (dict && uni) launch_k(sell_short_kernel<MODE, L, RR, true, true>, sg, kBlock, st, a, x, aux, y);    \
        else if (dict) launch_k(sell_short_kernel<MODE, L, RR, true, false>, sg, kBlock, st, a, x, aux, y);    \
        else if (uni) launch_k(sell_short_kernel<MODE, L, RR, false, true>, sg, kBlock, st, a, x, aux, y);     \
        else launch_k(sell_short_kernel<MODE, L, RR, false, false>, sg, kBlock, st, a, x, aux, y);             \
    } while (0)
            if (ml == 1) {
                if (R == 4) MG_SHORT(1, 4);
                else MG_SHORT(1, 2);
            } else {
                if (R == 4) MG_SHORT(2, 4);
                else MG_SHORT(2, 2);
            }
#undef MG_SHORT
            MG_CHECK_LAUNCH(name);
            if (nblocks_out) *nblocks_out = (int)sg;
            return MG_OK;
        }
    }
    const bool impl = sell_use_implied(A, row0, row1);
    const bool dict = sell_use_dict(A);
    // implied values: the launch must carry an expected record (its values travel as kernel parameters)
    const bool impv = impl && dict && g_implied_values && A->d_rec_vals && A->h_spec_vals && a.spec_id >= 0;
#define MG_SELL_LAUNCH(L, U, I, V)                                                                                       \
    do {                                                                                                                 \
        if (fuse) launch_k(sell_kernel_fused<MODE, L, U, I, V>, (unsigned)(grid + fuse->nex), kBlock, st, a, x, b, aux, y, omega, partials, fuse->ex, fuse->mask); \
        else launch_k(sell_kernel<MODE, L, U, I, V>, (unsigned)grid, kSellBlock, st, a, x, b, aux, y, omega, partials);  \
    } while (0)
#define MG_SELL_VARIANT(L, V)                             \
    do {                                                  \
        if (impl) MG_SELL_LAUNCH(L, true, true, V);       \
        else if (uni) MG_SELL_LAUNCH(L, true, false, V);  \
        else MG_SELL_LAUNCH(L, false, false, V);          \
    } while (0)
#define MG_SELL_IMPV(L)                                                                                                  \
    do {                                                                                                                 \
        if (fuse) launch_k(sell_kernel_fused<MODE, L, true, true, true, true>, (unsigned)(grid + fuse->nex), kBlock, st, a, x, b, aux, y, omega, partials, fuse->ex, fuse->mask); \
        else launch_k(sell_kernel<MODE, L, true, true, true, true>, (unsigned)grid, kSellBlock, st, a, x, b, aux, y, omega, partials); \
    } while (0)
#define MG_SELL_CASE(L)                                   \
    case L:                                               \
        if (impv) MG_SELL_IMPV(L);                        \
        else if (dict) MG_SELL_VARIANT(L, true);          \
        else MG_SELL_VARIANT(L, false);                   \
        break
    switch (ml) {
        MG_SELL_CASE(1); MG_SELL_CASE(2); MG_SELL_CASE(3); MG_SELL_CASE(4);
        MG_SELL_CASE(5); MG_SELL_CASE(6); MG_SELL_CASE(7); MG_SELL_CASE(8);
        default:   // long rows, or length unknown (0)
            if constexpr (!mode_is_tail(MODE)) MG_SELL_LAUNCH(0, false, false, false);
            else return set_error(MG_ERR_INVALID, name, "rows too long for a sweep with a fused residual");
    }
#undef MG_SELL_CASE
#undef MG_SELL_IMPV
#undef MG_SELL_VARIANT
#undef MG_SELL_LAUNCH
    MG_CHECK_LAUNCH(name);
    if (nblocks_out) *nblocks_out = (int)grid;
    return MG_OK;
}

}  // namespace mgb
