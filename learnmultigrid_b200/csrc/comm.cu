// comm.cu -- exchanges between the row blocks of a distributed level over peer-mapped memory (NVLink/NVSwitch).
//
// There is no reference counterpart (the reference is single-process, SURVEY 2a); the contract is SURVEY 8e.
// Mechanism (arena layout and protocol: include/mgb200.h): every rank owns an arena allocated with cudaMalloc and
// exported with CUDA IPC; peers map it.  One fused kernel per exchange site gathers the boundary values, WRITES them
// straight into each peer's staging area (st.global over NVLink) as self-validating packets tagged with the
// program's epoch, then polls its own staging area until the peers' packets carry the same tag and unpacks them.  It is ordinary stream work, so a whole V-cycle including its exchanges is captured in one CUDA graph; the
// epoch is a device counter the program advances at its end, staging is double-buffered by epoch parity so a rank
// that runs ahead into the next program never overwrites data its peer has not consumed yet.
#include "exchange.cuh"

namespace mgb {

constexpr int64_t kHeaderBytes = 4096;
constexpr int kMaxCtasPerPeer = 16;

__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(kBlock) exchange_kernel(const ExArgs a) {
    pdl_prologue();
    if (a.dry) return;
    exchange_role(a, (int)blockIdx.x);
}

__global__ void comm_init_kernel(unsigned long long *hdr) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        hdr[0] = 1ull;
        ((unsigned int *)hdr)[2] = 0u;
    }
}
__global__ void epoch_advance_kernel(unsigned long long *epoch, unsigned long long delta) {
    pdl_prologue();
    if (threadIdx.x == 0 && blockIdx.x == 0) epoch[0] += delta;
}
// out = sum_q (q == rank ? *value : slots[q]) in rank order
__global__ void sum_slots_kernel(const double *value, const double *slots, int rank, int world, double *out) {
    pdl_prologue();
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.0;
        for (int q = 0; q < world; ++q) s += (q == rank) ? *value : slots[q];
        *out = s;
    }
}
// the same for k values per rank: out[i] = sum_q (q == rank ? value[i] : slots[q * k + i]) in rank order, i < k
__global__ void sum_slots_n_kernel(const double *value, const double *slots, int k, int rank, int world, double *out) {
    pdl_prologue();
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < world; ++q) s += (q == rank) ? value[i] : slots[(int64_t)q * k + i];
        out[i] = s;
    }
}

// column relabelling of a row block: global column -> local [owned (permuted) | halo] index through a lookup table:
// slot_of[c] = halo slot (>= 0) or -1
__global__ void __launch_bounds__(kBlock)
remap_cols_table_kernel(int64_t nnz, const int32_t *__restrict__ cols_in, int64_t c0, int64_t c1,
                        const int32_t *__restrict__ own_iperm, int64_t n_own,
                        const int32_t *__restrict__ slot_of, int32_t *__restrict__ cols_out,
                        int32_t *__restrict__ missing) {
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    for (int64_t p = (int64_t)blockIdx.x * kBlock + threadIdx.x; p < nnz; p += stride) {
        const int64_t c = cols_in[p];
        if (c >= c0 && c < c1) {
            cols_out[p] = own_iperm ? own_iperm[c - c0] : (int32_t)(c - c0);
        } else {
            const int32_t s = slot_of[c];
            if (s < 0) atomicExch(missing, 1);
            cols_out[p] = (int32_t)(n_own + s);
        }
    }
}


static inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }
static inline int64_t flags_offset() { return kHeaderBytes; }
static inline int64_t staging_offset(int world, int max_sites) {
    return align_up(kHeaderBytes + (int64_t)world * max_sites * 8, 4096);
}

// Book the next site of the program for `x` and fill the kernel arguments.  *grid_out = number of exchange CTAs
// (0: nothing to launch, e.g. no peers).  Returns MG_OK or an error.
int comm_prepare(mg_comm *c, const mg_xfer *x, const double *src, double *dst, ExArgs *out, int *grid_out) {
    *grid_out = 0;
    if (!c || !x) return set_error(MG_ERR_INVALID, "mg_comm_exchange", "null argument");
    if (c->site >= c->max_sites) return set_error(MG_ERR_INVALID, "mg_comm_exchange", "program has more exchange sites than the arena has flags");
    const int site = c->site++;
    ExArgs &a = *out;
    memset(&a, 0, sizeof(a));
    char *mine = (char *)c->d_arena[c->rank];
    a.epoch = (const unsigned long long *)mine;
    a.err = (unsigned int *)(mine + 8);
    a.done = (unsigned int *)(mine + 16);
    a.ready = (unsigned long long *)(mine + 24);
    a.timeout_ns = (unsigned long long)((c->timeout_s > 0 ? c->timeout_s : 10.0) * 1e9);
    a.site = (unsigned)site;
    if (c->dry_run) {
        a.dry = 1;
        a.npeers = 1;
        a.ctas_per_peer = 1;
        *grid_out = 1;
        return MG_OK;
    }
    if (x->npeers == 0) return MG_OK;
    if (x->npeers == c->world - 1) c->all_pairs = 1;
    if (x->npeers < 0 || x->npeers > MG_MAX_RANKS) return set_error(MG_ERR_INVALID, "mg_comm_exchange", "bad peer count");
    a.npeers = x->npeers;
    a.src = src;
    a.dst = dst;
    a.parity_stride = c->region_bytes / 16;
    const int64_t stg = staging_offset(c->world, c->max_sites);
    int64_t longest = 1;
    for (int k = 0; k < x->npeers; ++k) {
        const int q = x->peer[k];
        if (q < 0 || q >= c->world || q == c->rank || !c->d_arena[q])
            return set_error(MG_ERR_INVALID, "mg_comm_exchange", "bad peer rank");
        if (x->send_cnt[k] < 0 || x->recv_cnt[k] < 0) return set_error(MG_ERR_INVALID, "mg_comm_exchange", "negative count");
        if ((c->bump_send[q] + x->send_cnt[k]) * 16 > c->region_bytes || (c->bump_recv[q] + x->recv_cnt[k]) * 16 > c->region_bytes)
            return set_error(MG_ERR_INVALID, "mg_comm_exchange", "staging region too small for this program");
        char *theirs = (char *)c->d_arena[q];
        ExPeer &P = a.p[k];
        P.send_idx = x->d_send_idx[k];
        P.send_off = x->send_off[k];
        P.send_cnt = x->send_cnt[k];
        P.peer_stage = (ulonglong2 *)(theirs + stg + (int64_t)c->rank * 2 * c->region_bytes) + c->bump_send[q];
        P.peer_flag = (unsigned long long *)(theirs + flags_offset()) + (int64_t)c->rank * c->max_sites + site;
        P.my_stage = (const ulonglong2 *)(mine + stg + (int64_t)q * 2 * c->region_bytes) + c->bump_recv[q];
        P.my_flag = (const unsigned long long *)(mine + flags_offset()) + (int64_t)q * c->max_sites + site;
        P.recv_idx = x->d_recv_idx[k];
        P.recv_off = x->recv_off[k];
        P.recv_cnt = x->recv_cnt[k];
        c->bump_send[q] += (x->send_cnt[k] + 7) / 8 * 8;          // keep messages 128-byte aligned
        c->bump_recv[q] += (x->recv_cnt[k] + 7) / 8 * 8;
        if (x->send_cnt[k] > longest) longest = x->send_cnt[k];
        if (x->recv_cnt[k] > longest) longest = x->recv_cnt[k];
    }
    int cpp = (int)((longest + 2 * kBlock - 1) / (2 * kBlock));
    if (cpp > kMaxCtasPerPeer) cpp = kMaxCtasPerPeer;
    if (cpp < 1) cpp = 1;
    a.ctas_per_peer = cpp;
    *grid_out = cpp * x->npeers;
    return MG_OK;
}

int comm_exchange(mg_comm *c, const mg_xfer *x, const double *src, double *dst, cudaStream_t st) {
    ExArgs a;
    int grid = 0;
    int rc = comm_prepare(c, x, src, dst, &a, &grid);
    if (rc || grid == 0) return rc;
    launch_k(exchange_kernel, (unsigned)grid, (unsigned)kBlock, st, a);
    MG_CHECK_LAUNCH("exchange");
    return MG_OK;
}

}  // namespace mgb

using namespace mgb;

extern "C" {

int64_t mg_comm_arena_bytes(int32_t world, int32_t max_sites, int64_t region_bytes) {
    if (world < 1 || world > MG_MAX_RANKS || max_sites < 1 || region_bytes < 0 || region_bytes % 128) return -1;
    return staging_offset(world, max_sites) + (int64_t)world * 2 * region_bytes;
}
/* communication arena: cudaMalloc'ed (IPC needs a whole allocation), zero-initialised */
int mg_comm_alloc(int64_t bytes, void **d_ptr_out) {
    MG_REQUIRE(bytes > 0 && d_ptr_out, "bad argument");
    MG_CHECK_CUDA(cudaMalloc(d_ptr_out, (size_t)bytes));
    MG_CHECK_CUDA(cudaMemset(*d_ptr_out, 0, (size_t)bytes));
    MG_CHECK_CUDA(cudaDeviceSynchronize());
    return MG_OK;
}
int mg_comm_free(void *d_ptr) {
    if (d_ptr) MG_CHECK_CUDA(cudaFree(d_ptr));
    return MG_OK;
}
/* 64-byte CUDA IPC handle of an arena (to be sent to the peers) */
int mg_comm_export(void *d_ptr, unsigned char *h_handle64) {
    MG_REQUIRE(d_ptr && h_handle64, "null argument");
    cudaIpcMemHandle_t h;
    MG_CHECK_CUDA(cudaIpcGetMemHandle(&h, d_ptr));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(h_handle64, &h, 64);
    return MG_OK;
}
/* map a peer's arena into this process (enables peer access lazily) */
int mg_comm_import(const unsigned char *h_handle64, void **d_peer_ptr_out) {
    MG_REQUIRE(h_handle64 && d_peer_ptr_out, "null argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, h_handle64, 64);
    MG_CHECK_CUDA(cudaIpcOpenMemHandle(d_peer_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return MG_OK;
}
int mg_comm_unmap(void *d_peer_ptr) {
    if (d_peer_ptr) MG_CHECK_CUDA(cudaIpcCloseMemHandle(d_peer_ptr));
    return MG_OK;
}
int mg_comm_init(mg_comm *comm, void *stream) {
    MG_REQUIRE(comm && comm->world >= 1 && comm->world <= MG_MAX_RANKS && comm->rank >= 0 && comm->rank < comm->world &&
                   comm->d_arena[comm->rank] && comm->max_sites > 0 && comm->region_bytes % 128 == 0, "bad communicator");
    comm_init_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((unsigned long long *)comm->d_arena[comm->rank]);
    MG_CHECK_LAUNCH("comm_init");
    return mg_comm_begin(comm);
}
int mg_comm_begin(mg_comm *comm) {
    MG_REQUIRE(comm, "null communicator");
    comm->site = 0;
    comm->all_pairs = 0;
    for (int q = 0; q < MG_MAX_RANKS; ++q) comm->bump_send[q] = comm->bump_recv[q] = 0;
    return MG_OK;
}
int mg_comm_exchange(mg_comm *comm, const mg_xfer *xfer, const double *d_src, double *d_dst, void *stream) {
    return comm_exchange(comm, xfer, d_src, d_dst, (cudaStream_t)stream);
}
int mg_comm_allreduce_sum_n(mg_comm *comm, const double *d_values, int32_t k, double *d_slots, double *d_out,
                            void *stream) {
    MG_REQUIRE(comm && d_values && d_slots && d_out, "null argument");
    MG_REQUIRE(k >= 1, "need at least one value");
    mg_xfer x;
    memset(&x, 0, sizeof(x));
    for (int q = 0; q < comm->world; ++q) {
        if (q == comm->rank) continue;
        const int p = x.npeers++;
        x.peer[p] = q;
        x.send_cnt[p] = k;
        x.recv_off[p] = (int64_t)q * k;
        x.recv_cnt[p] = k;
    }
    int rc = comm_exchange(comm, &x, d_values, d_slots, (cudaStream_t)stream);
    if (rc) return rc;
    if (k == 1)     // the single-value kernel of the V-cycle norm and of CG
        launch_k(sum_slots_kernel, 1u, 32u, (cudaStream_t)stream, d_values, (const double *)d_slots, comm->rank,
                 comm->world, d_out);
    else
        launch_k(sum_slots_n_kernel, 1u, 32u, (cudaStream_t)stream, d_values, (const double *)d_slots, (int)k,
                 comm->rank, comm->world, d_out);
    MG_CHECK_LAUNCH("sum_slots");
    return MG_OK;
}
int mg_comm_allreduce_sum(mg_comm *comm, const double *d_value, double *d_slots, double *d_out, void *stream) {
    return mg_comm_allreduce_sum_n(comm, d_value, 1, d_slots, d_out, stream);
}
int mg_comm_end(mg_comm *comm, void *stream) {
    MG_REQUIRE(comm && comm->d_arena[comm->rank], "null communicator");
    if (!comm->all_pairs && comm->world > 1) {      // fence: an empty all-pairs site (see mgb200.h)
        mg_xfer x;
        memset(&x, 0, sizeof(x));
        for (int q = 0; q < comm->world; ++q)
            if (q != comm->rank) x.peer[x.npeers++] = q;
        int rc = comm_exchange(comm, &x, nullptr, nullptr, (cudaStream_t)stream);
        if (rc) return rc;
    }
    launch_k(epoch_advance_kernel, (unsigned)(1), (unsigned)32, (cudaStream_t)stream, (unsigned long long *)comm->d_arena[comm->rank],
                                                             comm->dry_run ? 0ull : 1ull);
    MG_CHECK_LAUNCH("epoch_advance");
    return MG_OK;
}
int mg_comm_error(mg_comm *comm, int32_t *h_error, void *stream) {
    MG_REQUIRE(comm && h_error && comm->d_arena[comm->rank], "null argument");
    MG_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    unsigned int e = 0;
    MG_CHECK_CUDA(cudaMemcpy(&e, (char *)comm->d_arena[comm->rank] + 8, 4, cudaMemcpyDeviceToHost));
    *h_error = (int32_t)e;
    return MG_OK;
}
/* relabel the columns of a row block: c in [c0,c1) -> d_own_iperm[c-c0] (NULL: c-c0), otherwise n_own + d_slot_of[c] */
int mg_csr_remap_cols(int64_t nnz, const int32_t *d_cols_in, int64_t c0, int64_t c1, const int32_t *d_own_iperm,
                      int64_t n_own, const int32_t *d_slot_of, int32_t *d_cols_out, int32_t *d_missing, void *stream) {
    MG_REQUIRE(nnz >= 0 && d_slot_of && d_missing, "null argument");
    if (nnz == 0) return MG_OK;
    int64_t g = (nnz + kBlock - 1) / kBlock;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (g > cap) g = cap;
    remap_cols_table_kernel<<<(unsigned)g, kBlock, 0, (cudaStream_t)stream>>>(nnz, d_cols_in, c0, c1, d_own_iperm, n_own,
                                                                             d_slot_of, d_cols_out, d_missing);
    MG_CHECK_LAUNCH("remap_cols");
    return MG_OK;
}

}  // extern "C"
