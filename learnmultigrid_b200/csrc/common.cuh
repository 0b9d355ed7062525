// common.cuh -- shared helpers of libmgb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/mgb200.h"

namespace mgb {

extern thread_local char g_last_error[512];
extern thread_local int64_t g_launch_count;

inline int set_error(int code, const char *what, const char *detail) {
    snprintf(g_last_error, sizeof(g_last_error), "%s: %s", what, detail ? detail : "");
    return code;
}

#define MG_CHECK_CUDA(expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) return mgb::set_error(MG_ERR_CUDA, #expr, cudaGetErrorString(_e)); \
    } while (0)

#define MG_CHECK_LAUNCH(name)                                                                 \
    do {                                                                                      \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess) return mgb::set_error(MG_ERR_CUDA, name, cudaGetErrorString(_e)); \
        ++mgb::g_launch_count;                                                                \
    } while (0)

#define MG_REQUIRE(cond, msg)                                                                 \
    do {                                                                                      \
        if (!(cond)) return mgb::set_error(MG_ERR_INVALID, __func__, msg);                    \
    } while (0)

// GS_RES / GS_NORM: colour sweep that also yields the residual / the squared residual norm of the swept rows
// SPMV_DOT: y = A x and per-CTA partial sums of aux . y (the p . A p of conjugate gradients from the SpMV's registers)
// CHEBY: one step of the Chebyshev smoother (sell_modes_cheby.cu); after PROLONG, so the staged TMA path never sees it
enum SellMode { SPMV = 0, RESID = 1, RESNORM = 2, JACOBI = 3, GS = 4, PROLONG = 5, GS_RES = 6, GS_NORM = 7, SPMV_DOT = 8,
                CHEBY = 9 };

constexpr int kSlice = 32;      // SELL slice height = one warp
constexpr int kBlock = 256;     // threads per CTA of the streaming kernels
#ifndef MGB_SELL_BLOCK
#define MGB_SELL_BLOCK 256
#endif
// threads per CTA of the one-row-per-thread SELL kernels without an exchange site (sell_core.cuh: sell_kernel); the
// occupancy bounds scale with it, so that the SM holds the same 2048 threads in more, smaller CTAs
constexpr int kSellBlock = MGB_SELL_BLOCK;
static_assert(kSellBlock >= 64 && kSellBlock <= kBlock && kBlock % kSellBlock == 0, "MGB_SELL_BLOCK: 64, 128 or 256");

// IEEE multiply / add that the compiler may not contract into an FMA: the CPU oracle (gcc
// -ffp-contract=off, SciPy, PyAMG) rounds the product and the sum separately and we match it bit for bit.
__device__ __forceinline__ double mul_add_unfused(double acc, double a, double b) {
    return __dadd_rn(acc, __dmul_rn(a, b));
}

// streaming (read-once) loads of the matrix arrays: do not pollute L1, which we want for the x gathers
__device__ __forceinline__ double ld_stream(const double *p) { return __ldcs(p); }
__device__ __forceinline__ int32_t ld_stream(const int32_t *p) { return __ldcs(p); }
__device__ __forceinline__ unsigned char ld_stream(const unsigned char *p) { return __ldcs(p); }

// Bring a line towards the SM without holding a register for it (sell_core.cuh: the row's own vector entries).
#ifndef MGB_ROW_OPERANDS
#define MGB_ROW_OPERANDS 1
#endif
// how the one-row-per-thread kernels fetch the row's own vector entries (b, u, 1/diag, x of a Jacobi row):
// 0 = where they are used, 1 = prefetch into L1 under the matrix loads, 2 = prefetch into L2, 3 = load into registers
constexpr int kRowOperands = MGB_ROW_OPERANDS;
__device__ __forceinline__ void prefetch_row_operand(const double *p) {
    if (kRowOperands == 1) asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
    else if (kRowOperands == 2) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// Value dictionaries in shared memory (sell_core.cuh: STAB): two instructions per lookup instead of five, at the price
// of an asynchronous table copy and a CTA barrier in every CTA.  Measured on the 8193^2 cycle: 2.70 ms per step against
// 2.66 ms with the table read through L1 (profiles/r02_variants_*.txt) -- the sweeps are not bound by issue slots
// alone -- so it is off; -DMGB_SHARED_DICT=1 builds it (tools/build_variant.sh).
#ifndef MGB_SHARED_DICT
#define MGB_SHARED_DICT 0
#endif
constexpr bool kSharedDict = MGB_SHARED_DICT != 0;

// dictionary index of one entry: the byte zero-extended into a 32-bit register by the load itself (a C++ unsigned char
// makes the compiler re-mask the index before every table lookup)
// (these loads are volatile asm: the one-row kernels rely on their loads being ISSUED in program order -- all of a row's
// DRAM requests before the first wait, sell_core.cuh -- and ptxas otherwise sinks some of them below that wait)
__device__ __forceinline__ unsigned ld_stream_u8(const unsigned char *p) {
    unsigned v;
    asm volatile("ld.global.cs.u8 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ unsigned ld_const_u16(const unsigned short *p) {
    unsigned v;
    asm volatile("ld.global.nc.u16 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
// x[col], issued here
__device__ __forceinline__ double ld_gather(const double *x, int32_t col) {
    double v;
    asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(x + col));
    return v;
}
// x[col] unless col == skip (a Gauss-Seidel row's own entry): +0.0 then, and no memory access
__device__ __forceinline__ double ld_gather_skip(const double *x, int32_t col, int32_t skip) {
    double v;
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %2, %3;\n\tmov.f64 %0, 0d0000000000000000;\n\t@p ld.global.f64 %0, [%1];\n\t}"
                 : "=d"(v) : "l"(x + col), "r"(col), "r"(skip));
    return v;
}
// asynchronous 8-byte copy global -> shared (no register, no stall at the point of issue)
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- programmatic dependent launch (PDL) --------------------------------------------------------------------------
// The V-cycle is a long chain of short dependent kernels (60-150 per cycle, many of a few microseconds on the coarse
// levels and between exchange sites).  Every kernel of the chain starts with pdl_prologue(): it waits until the
// preceding grid has completed and flushed (griddepcontrol.wait) and then allows the NEXT kernel of the stream to
// be scheduled early (griddepcontrol.launch_dependents), so that its launch latency overlaps this kernel's
// execution; launch_k() marks the launch accordingly.  Since every kernel of the chain waits unconditionally, a grid
// can never complete before all of its predecessors have, which keeps the ordering transitive.  Stream capture turns
// these launches into programmatic graph edges.  mg_set_pdl(0) falls back to plain stream order.
extern int g_pdl;
__device__ __forceinline__ void pdl_prologue() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), unsigned grid, unsigned block, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(block, 1, 1);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);     // errors are picked up by MG_CHECK_LAUNCH
}

inline int sm_count() {
    static int cached = 0;
    if (!cached) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
        if (cached <= 0) cached = 148;
    }
    return cached;
}

// deterministic block reduction (fixed tree), result valid in thread 0
template <int BLOCK>
__device__ __forceinline__ double block_sum(double v) {
    __shared__ double sh[BLOCK / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sh[w] = v;
    __syncthreads();
    if (w == 0) {
        v = (l < BLOCK / 32) ? sh[l] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    }
    __syncthreads();
    return v;
}

// The same sum as the LAST thing a kernel does: only warp 0 waits.  The other warps park their warp sums in shared
// memory, ARRIVE at a named barrier and are done (barrier.cta.arrive / barrier.cta.sync, the producer-consumer pattern of
// the PTX ISA): no warp stalls on the slowest one, which matters when the block holds few warps per SM to hide it
// (ncu on the sweep with a fused norm: 3.3 barrier stalls per issue, 5.5 instead of 6.8 TB/s).  Same tree, same bits.
// Every thread of the block must call it, exactly once, and nothing may follow that needs the other warps.
template <int BLOCK>
__device__ __forceinline__ double block_sum_last(double v) {
    __shared__ double sh[BLOCK / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sh[w] = v;
    if (w != 0) {
        asm volatile("barrier.cta.arrive 1, %0;" ::"n"(BLOCK) : "memory");
        return 0.0;
    }
    asm volatile("barrier.cta.sync 1, %0;" ::"n"(BLOCK) : "memory");
    v = (l < BLOCK / 32) ? sh[l] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// The same job with a quarter of the instructions: every thread parks its value in shared memory (one store), all warps
// but the first arrive and retire, and warp 0 adds the BLOCK values in a fixed order (lane l takes l, l + 32, ..., then
// the warp tree).  The one-row-per-thread kernels are bound by instruction issue (68-76 % of the issue slots at 4 of 7
// TB/s): the five-step shuffle tree in EVERY warp made the sweep with a fused norm a third slower than the plain sweep
// (ncu, level 0 of the 8193^2 step: 284 against 215 us for the same bytes).  -DMGB_PARKED_SUM=0 keeps the tree per warp.
#ifndef MGB_PARKED_SUM
#define MGB_PARKED_SUM 1
#endif
template <int BLOCK>
__device__ __forceinline__ double block_sum_parked(double v) {
    if (!MGB_PARKED_SUM) return block_sum_last<BLOCK>(v);
    __shared__ double sh[BLOCK];
    sh[threadIdx.x] = v;
    if (threadIdx.x >= 32) {
        asm volatile("barrier.cta.arrive 1, %0;" ::"n"(BLOCK) : "memory");
        return 0.0;
    }
    asm volatile("barrier.cta.sync 1, %0;" ::"n"(BLOCK) : "memory");
    double s = sh[threadIdx.x];
#pragma unroll
    for (int k = 1; k < BLOCK / 32; ++k) s = __dadd_rn(s, sh[threadIdx.x + 32 * k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    return s;
}

}  // namespace mgb
