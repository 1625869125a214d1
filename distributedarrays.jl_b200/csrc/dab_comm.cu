// dab_comm.cu -- the cross-worker combine seam: NCCL over NVLink 5 / NVSwitch + CUDA IPC peer memory.
//
// Replaces Distributed.remotecall_fetch ON THE HOT PATH ONLY (north_star):
//   * asyncmap(procs(d)) do p remotecall_fetch(...) end ; reduce(op, results)   reference src/mapreduce.jl:30-34
//       -> dab_mapreduce_all: chunk kernel, ncclAllGather of the P chunk results, ordered left fold.
//   * mapreducedim_between! pulling the partial slabs of a fibre                  reference src/mapreduce.jl:72-80
//       -> dab_group_start / dab_send / dab_recv / dab_group_end (grouped ncclSend/ncclRecv).
//   * chunk(d, pid) / remotecall_fetch(localpart(d)[idxs...])                    reference src/darray.jl:458,809-815
//       -> dab_ipc_* + dab_copy_box (one-sided peer loads) or dab_send/dab_recv.
// NCCL is resolved with dlopen at first use so that libdab200.so itself loads on a machine without NCCL / a GPU
// (the torch-bundled libnccl.so.2 is reused when the host runtime already loaded it).
#include <dlfcn.h>
#include <nccl.h>

#include "dab_common.cuh"
#include "dab_scalar_ops.cuh"

namespace {

struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    const char* (*GetLastError)(ncclComm_t) = nullptr;
    bool ok = false;
    char why[256] = "";
};

NcclApi& nccl() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api;
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so", nullptr};
    for (int i = 0; names[i] && !api.handle; ++i) api.handle = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
    if (!api.handle) {
        snprintf(api.why, sizeof(api.why), "dlopen(libnccl.so.2) failed: %s", dlerror());
        return api;
    }
#define SYM(field, name)                                                            \
    do {                                                                            \
        *(void**)(&api.field) = dlsym(api.handle, name);                            \
        if (!api.field) {                                                           \
            snprintf(api.why, sizeof(api.why), "libnccl lacks symbol %s", name);    \
            return api;                                                             \
        }                                                                           \
    } while (0)
    SYM(GetUniqueId, "ncclGetUniqueId");
    SYM(CommInitRank, "ncclCommInitRank");
    SYM(CommDestroy, "ncclCommDestroy");
    SYM(AllGather, "ncclAllGather");
    SYM(AllReduce, "ncclAllReduce");
    SYM(Send, "ncclSend");
    SYM(Recv, "ncclRecv");
    SYM(GroupStart, "ncclGroupStart");
    SYM(GroupEnd, "ncclGroupEnd");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    *(void**)(&api.GetLastError) = dlsym(api.handle, "ncclGetLastError");  // optional
    api.ok = true;
    return api;
}

int32_t nccl_fail(dab_ctx* ctx, ncclResult_t r, const char* what) {
    NcclApi& api = nccl();
    const char* last = (api.GetLastError && ctx && ctx->comm) ? api.GetLastError((ncclComm_t)ctx->comm) : "";
    return dab_fail(ctx, DAB_ERR_NCCL, "NCCL error %d (%s) in %s %s", (int)r, api.GetErrorString ? api.GetErrorString(r) : "?", what,
                    last ? last : "");
}

#define DAB_NCCL(ctx, call)                                       \
    do {                                                          \
        ncclResult_t r__ = (call);                                \
        if (r__ != ncclSuccess) return nccl_fail((ctx), r__, #call); \
    } while (0)

#define NEED_NCCL(ctx)                                                           \
    NcclApi& api = nccl();                                                       \
    if (!api.ok) return dab_fail((ctx), DAB_ERR_NCCL, "NCCL unavailable: %s", api.why)

#define NEED_COMM(ctx)                                                                                    \
    NEED_NCCL(ctx);                                                                                       \
    if (!(ctx)->comm) return dab_fail((ctx), DAB_ERR_NCCL, "no communicator: call dab_comm_init_rank first")


// ---- device-side barrier across the ranks (stream-ordered; no host synchronisation, no NCCL launch) ---------------------------------------
// One CTA: thread j stores this rank's arrival number into rank j's counter row (peer store over NVLink, system fence first so that every
// write of the preceding kernels of this stream is visible to a peer that sees the number), then polls its own row until rank j has
// arrived too.  Kernels queued after it on this stream therefore start only when EVERY rank's earlier kernels have completed: the fence
// the reference gets from remotecall_wait / fetch, without leaving the GPU.  A dead peer surfaces after the wall-clock timeout as a status
// word in pinned host memory (checked by dab_sync), not as a hung device.
__global__ void peer_barrier_kernel(void* const* __restrict__ peers, int rank, int nranks, unsigned long long seq, unsigned long long timeout_ns,
                                    volatile unsigned long long* __restrict__ host_status) {
    const int j = threadIdx.x;
    if (j >= nranks) return;
    __threadfence_system();
    volatile unsigned long long* theirs = reinterpret_cast<volatile unsigned long long*>((char*)peers[j] + DAB_MBOX_BARRIER_OFFSET) + rank;
    *theirs = seq;
    volatile unsigned long long* mine = reinterpret_cast<volatile unsigned long long*>((char*)peers[rank] + DAB_MBOX_BARRIER_OFFSET) + j;
    const unsigned long long t0 = dab_globaltimer_ns();
    unsigned int spins = 0;
    while (*mine < seq) {
        if ((++spins & 1023u) == 0 && dab_globaltimer_ns() - t0 > timeout_ns) {
            host_status[0] = 1ull;
            __threadfence_system();
            break;
        }
    }
    __threadfence_system();
}

// y = beta * y (fill 0 when beta == 0, untouched when beta == 1), then y += alpha * stack[j] for j = 0 .. count-1 IN ORDER, each step one
// multiply and one add rounded separately: the rmul!/fill! + add!(localpart(y), R[i,j], alpha) sequence of mul! (reference src/linalg.jl:
// 101-117, 62-76) in ONE launch instead of 1 + 2*count; bit-identical to the separate launches.
template <typename T>
__global__ void __launch_bounds__(256) accumulate_stack_kernel(T* __restrict__ y, size_t n, T beta, int beta_mode, T alpha, int alpha_one,
                                                              const T* __restrict__ stack, size_t stride, int count) {
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
        T v = beta_mode == 0 ? T(0) : (beta_mode == 1 ? y[i] : jl::mul(y[i], beta));
        for (int j = 0; j < count; ++j) {
            const T r = stack[(size_t)j * stride + i];
            v = jl::add(v, alpha_one ? r : jl::mul(alpha, r));
        }
        y[i] = v;
    }
}

}  // namespace

extern "C" {

int32_t dab_comm_unique_id(void* id128) {
    NEED_NCCL(nullptr);
    if (!id128) return dab_fail(nullptr, DAB_ERR_ARG, "null id");
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    DAB_NCCL(nullptr, api.GetUniqueId(&id));
    memcpy(id128, &id, 128);
    return DAB_OK;
}

int32_t dab_comm_init_rank(dab_ctx* ctx, const void* id128, int32_t rank, int32_t nranks) {
    DAB_ENTER(ctx);
    NEED_NCCL(ctx);
    DAB_REQUIRE(ctx, id128 && nranks >= 1 && rank >= 0 && rank < nranks && nranks <= DAB_MAX_RANKS, DAB_ERR_ARG,
                "dab_comm_init_rank: bad rank %d / nranks %d", rank, nranks);
    DAB_REQUIRE(ctx, !ctx->comm, DAB_ERR_ARG, "communicator already initialised");
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclComm_t comm;
    DAB_NCCL(ctx, api.CommInitRank(&comm, nranks, id, rank));
    ctx->comm = (void*)comm;
    ctx->rank = rank;
    ctx->nranks = nranks;
    return DAB_OK;
}

int32_t dab_comm_destroy(dab_ctx* ctx) {
    if (!ctx || !ctx->comm) return DAB_OK;
    NcclApi& api = nccl();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (api.ok) api.CommDestroy((ncclComm_t)ctx->comm);
    ctx->comm = nullptr;
    ctx->rank = 0;
    ctx->nranks = 1;
    return DAB_OK;
}

int32_t dab_allgather(dab_ctx* ctx, const void* send_dev, void* recv_dev, size_t nbytes_per_rank) {
    DAB_ENTER(ctx);
    NEED_COMM(ctx);
    DAB_NCCL(ctx, api.AllGather(send_dev, recv_dev, nbytes_per_rank, ncclInt8, (ncclComm_t)ctx->comm, ctx->stream));
    ctx->launches++;
    return DAB_OK;
}

int32_t dab_allreduce(dab_ctx* ctx, int32_t dtype, int32_t op, const void* send_dev, void* recv_dev, size_t count) {
    DAB_ENTER(ctx);
    NEED_COMM(ctx);
    ncclDataType_t dt;
    switch (dtype) {
        case DAB_F32: dt = ncclFloat32; break;
        case DAB_F64: dt = ncclFloat64; break;
        case DAB_I32: dt = ncclInt32; break;
        case DAB_I64: dt = ncclInt64; break;
        case DAB_U8: dt = ncclUint8; break;
        default: return dab_fail(ctx, DAB_ERR_ARG, "dab_allreduce: bad dtype %d", dtype);
    }
    ncclRedOp_t ro;
    switch (op) {
        case DAB_SUM: ro = ncclSum; break;
        case DAB_PROD: ro = ncclProd; break;
        case DAB_MAX: ro = ncclMax; break;  // NOTE: not NaN-propagating; the DArray path uses allgather + ordered fold
        case DAB_MIN: ro = ncclMin; break;
        default: return dab_fail(ctx, DAB_ERR_ARG, "dab_allreduce: bad op %d", op);
    }
    DAB_NCCL(ctx, api.AllReduce(send_dev, recv_dev, count, dt, ro, (ncclComm_t)ctx->comm, ctx->stream));
    ctx->launches++;
    return DAB_OK;
}

int32_t dab_group_start(dab_ctx* ctx) {
    DAB_ENTER(ctx);
    NEED_COMM(ctx);
    DAB_NCCL(ctx, api.GroupStart());
    return DAB_OK;
}
int32_t dab_group_end(dab_ctx* ctx) {
    DAB_ENTER(ctx);
    NEED_COMM(ctx);
    DAB_NCCL(ctx, api.GroupEnd());
    ctx->launches++;
    return DAB_OK;
}
int32_t dab_send(dab_ctx* ctx, const void* send_dev, size_t nbytes, int32_t peer) {
    DAB_ENTER(ctx);
    NEED_COMM(ctx);
    DAB_NCCL(ctx, api.Send(send_dev, nbytes, ncclInt8, peer, (ncclComm_t)ctx->comm, ctx->stream));
    return DAB_OK;
}
int32_t dab_recv(dab_ctx* ctx, void* recv_dev, size_t nbytes, int32_t peer) {
    DAB_ENTER(ctx);
    NEED_COMM(ctx);
    DAB_NCCL(ctx, api.Recv(recv_dev, nbytes, ncclInt8, peer, (ncclComm_t)ctx->comm, ctx->stream));
    return DAB_OK;
}

}  // extern "C"

namespace {

// The combine of dab_mapreduce_all around one chunk reduce: `launch(slot)` enqueues the kernel that writes this rank's 16-byte result
// slot (dab_reduce, or dab_affine_reduce for the fused broadcast + sum).  rdt: the result dtype.
template <typename Launch>
int32_t mapreduce_all_combine(dab_ctx* ctx, int32_t op, int32_t rdt, size_t n, void* out_host, Launch launch) {
    if ((ctx->mbox_ranks > 1 || !ctx->comm || ctx->nranks == 1) && n > 0) {
        // fused path: ONE kernel = chunk reduce + peer-memory all-gather + ordered fold + scalar into pinned host memory
        ctx->fuse_op = op;
        int32_t st = launch(ctx->result_slot);
        ctx->fuse_op = -1;
        if (st != DAB_OK) return st;
        DAB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const volatile unsigned long long* h = (const volatile unsigned long long*)ctx->host_slot;
        if (h[1] != 0) return dab_fail(ctx, DAB_ERR_NCCL, "fused combine timed out waiting for a peer's chunk result (did every rank call?)");
        unsigned long long bits = h[0];
        memset(out_host, 0, 8);
        memcpy(out_host, &bits, dab_dtype_size(rdt));
        return DAB_OK;
    }
    int32_t st = launch(ctx->result_slot);
    if (st != DAB_OK) return st;
    const int P = ctx->comm ? ctx->nranks : 1;
    const void* src = ctx->result_slot;
    if (P > 1) {
        NEED_COMM(ctx);
        DAB_NCCL(ctx, api.AllGather(ctx->result_slot, ctx->gather_slots, 16, ncclInt8, (ncclComm_t)ctx->comm, ctx->stream));
        ctx->launches++;
        src = ctx->gather_slots;
    }
    DAB_CUDA(ctx, cudaMemcpyAsync(ctx->host_slot, src, (size_t)P * 16, cudaMemcpyDeviceToHost, ctx->stream));
    DAB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    unsigned char tmp[DAB_MAX_RANKS * 8];
    size_t es = dab_dtype_size(rdt);
    for (int i = 0; i < P; ++i) memcpy(tmp + (size_t)i * es, (const char*)ctx->host_slot + (size_t)i * 16, es);
    unsigned char res[8] = {0};
    st = dab_combine_ordered(rdt, op, tmp, (size_t)P, res);
    if (st != DAB_OK) return dab_fail(ctx, st, "%s", dab_last_error(nullptr));
    memset(out_host, 0, 8);
    memcpy(out_host, res, es);
    return DAB_OK;
}

}  // namespace

extern "C" {

// Base._mapreduce(f, op, ::IndexCartesian, d::DArray), reference src/mapreduce.jl:29-35, for ONE chunk per rank:
//   results = asyncmap(procs(d)) do p; remotecall_fetch(mapreduce(f, op, localpart(d))) end     -> kernel + allgather
//   reduce(op, results)                                                                        -> ordered left fold
int32_t dab_mapreduce_all(dab_ctx* ctx, int32_t dtype, int32_t op, int32_t map, const void* map_param, const void* x, size_t n,
                          void* out_host) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, out_host, DAB_ERR_ARG, "dab_mapreduce_all: null out");
    int32_t rdt;
    if (op == DAB_EXTREMA) return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "dab_mapreduce_all: extrema combines through dab_reduce + dab_allgather");
    if (dab_reduce_result_dtype(dtype, op, map, &rdt) != DAB_OK) return dab_fail(ctx, DAB_ERR_ARG, "bad dtype/op");
    return mapreduce_all_combine(ctx, op, rdt, n, out_host,
                                 [&](void* slot) { return dab_reduce(ctx, dtype, op, map, map_param, x, n, slot); });
}

// y .= a.*x .+ b then sum(y) (any of SUM PROD MAX MIN) of one chunk per rank: dab_mapreduce_all with dab_affine_reduce as the chunk
// reduce, so the step reads x, writes y and never reads y back when the kernel fuses.
int32_t dab_affine_mapreduce_all(dab_ctx* ctx, int32_t dtype, void* y, const void* x, const void* a, const void* b, size_t n, int32_t op,
                                 void* out_host) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, ((x && y) || n == 0) && a && b, DAB_ERR_ARG, "dab_affine: null pointer");
    DAB_REQUIRE(ctx, out_host, DAB_ERR_ARG, "dab_mapreduce_all: null out");
    int32_t rdt;
    if (op == DAB_EXTREMA) return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "dab_mapreduce_all: extrema combines through dab_reduce + dab_allgather");
    if (dab_reduce_result_dtype(dtype, op, DAB_MAP_ID, &rdt) != DAB_OK) return dab_fail(ctx, DAB_ERR_ARG, "bad dtype/op");
    return mapreduce_all_combine(ctx, op, rdt, n, out_host,
                                 [&](void* slot) { return dab_affine_reduce(ctx, dtype, y, x, a, b, n, op, slot); });
}

// ---- mailboxes for the fused reduce + combine kernel ---------------------------------------------------------
int32_t dab_mailbox_create(dab_ctx* ctx, void* handle64) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, handle64, DAB_ERR_ARG, "dab_mailbox_create: null handle");
    if (!ctx->mailbox) {
        DAB_CUDA(ctx, cudaMalloc(&ctx->mailbox, DAB_MBOX_BYTES));
        DAB_CUDA(ctx, cudaMemset(ctx->mailbox, 0, DAB_MBOX_BYTES));
    }
    cudaIpcMemHandle_t h;
    DAB_CUDA(ctx, cudaIpcGetMemHandle(&h, ctx->mailbox));
    memcpy(handle64, &h, 64);
    return DAB_OK;
}

int32_t dab_mailbox_attach(dab_ctx* ctx, const void* handles, int32_t rank, int32_t nranks) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, handles && nranks >= 1 && nranks <= DAB_MAX_RANKS && rank >= 0 && rank < nranks, DAB_ERR_ARG, "dab_mailbox_attach: bad arguments");
    DAB_REQUIRE(ctx, ctx->mailbox, DAB_ERR_ARG, "dab_mailbox_attach: call dab_mailbox_create first");
    DAB_REQUIRE(ctx, ctx->mbox_ranks == 0, DAB_ERR_ARG, "mailboxes already attached");
    for (int j = 0; j < nranks; ++j) {
        if (j == rank) {
            ctx->peer_mbox_host[j] = ctx->mailbox;
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + (size_t)j * 64, 64);
        DAB_CUDA(ctx, cudaIpcOpenMemHandle(&ctx->peer_mbox_host[j], h, cudaIpcMemLazyEnablePeerAccess));
    }
    DAB_CUDA(ctx, cudaMalloc((void**)&ctx->peer_mbox_dev, sizeof(void*) * DAB_MAX_RANKS));
    DAB_CUDA(ctx, cudaMemcpy(ctx->peer_mbox_dev, ctx->peer_mbox_host, sizeof(void*) * nranks, cudaMemcpyHostToDevice));
    ctx->rank = rank;
    ctx->mbox_ranks = nranks;
    ctx->mbox_seq = 0;
    return DAB_OK;
}

int32_t dab_mailbox_detach(dab_ctx* ctx) {
    if (!ctx) return DAB_OK;
    cudaSetDevice(ctx->device);
    for (int j = 0; j < ctx->mbox_ranks; ++j)
        if (j != ctx->rank && ctx->peer_mbox_host[j]) cudaIpcCloseMemHandle(ctx->peer_mbox_host[j]);
    if (ctx->peer_mbox_dev) cudaFree(ctx->peer_mbox_dev);
    if (ctx->mailbox) cudaFree(ctx->mailbox);
    ctx->peer_mbox_dev = nullptr;
    ctx->mailbox = nullptr;
    ctx->mbox_ranks = 0;
    cudaGetLastError();
    return DAB_OK;
}


int32_t dab_peer_barrier(dab_ctx* ctx) {
    DAB_ENTER(ctx);
    if (ctx->mbox_ranks <= 1) return DAB_OK;   // one worker: stream order is the barrier
    volatile unsigned long long* status = (volatile unsigned long long*)((char*)ctx->host_slot + (DAB_MAX_RANKS + 1) * 16);
    const unsigned long long seq = ++ctx->barrier_seq;
    peer_barrier_kernel<<<1, DAB_MAX_RANKS, 0, ctx->stream>>>(ctx->peer_mbox_dev, ctx->rank, ctx->mbox_ranks, seq,
                                                             (unsigned long long)ctx->opt_combine_timeout_ms * 1000000ull, status);
    DAB_LAUNCHED(ctx);
    return DAB_OK;
}

int32_t dab_accumulate_stack(dab_ctx* ctx, int32_t dtype, void* y, size_t n, const void* beta, const void* alpha, const void* stack, size_t stride,
                             int32_t count) {
    DAB_ENTER(ctx);
    if (n == 0) return DAB_OK;
    DAB_REQUIRE(ctx, y && beta && alpha && (stack || count == 0) && count >= 0, DAB_ERR_ARG, "dab_accumulate_stack: bad argument");
    const int grid = dab_grid_for(ctx, (n + 255) / 256, 8);
#define ACC(T)                                                                                                                       \
    {                                                                                                                                \
        const T b = *(const T*)beta, a = *(const T*)alpha, zero = 0, one = 1;                                                        \
        accumulate_stack_kernel<T><<<grid, 256, 0, ctx->stream>>>((T*)y, n, b, b == zero ? 0 : (b == one ? 1 : 2), a, a == one,     \
                                                                   (const T*)stack, stride, count);                                  \
        DAB_LAUNCHED(ctx);                                                                                                           \
        return DAB_OK;                                                                                                               \
    }
    switch (dtype) {
        case DAB_F32: ACC(float)
        case DAB_F64: ACC(double)
        case DAB_I32: ACC(int32_t)
        case DAB_I64: ACC(long long)
        default: return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "dab_accumulate_stack: dtype %d", dtype);
    }
#undef ACC
}

// ---- peer memory -------------------------------------------------------------------------------------------
int32_t dab_ipc_get_handle(dab_ctx* ctx, const void* dptr, void* handle64) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, dptr && handle64, DAB_ERR_ARG, "dab_ipc_get_handle: null pointer");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaIpcMemHandle_t h;
    DAB_CUDA(ctx, cudaIpcGetMemHandle(&h, const_cast<void*>(dptr)));
    memcpy(handle64, &h, 64);
    return DAB_OK;
}
int32_t dab_ipc_open(dab_ctx* ctx, const void* handle64, void** dptr) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, dptr && handle64, DAB_ERR_ARG, "dab_ipc_open: null pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    DAB_CUDA(ctx, cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
    return DAB_OK;
}
int32_t dab_ipc_close(dab_ctx* ctx, void* dptr) {
    DAB_ENTER(ctx);
    if (dptr) DAB_CUDA(ctx, cudaIpcCloseMemHandle(dptr));
    return DAB_OK;
}
int32_t dab_enable_peer(dab_ctx* ctx, int32_t peer_device) {
    DAB_ENTER(ctx);
    if (peer_device == ctx->device) return DAB_OK;
    int can = 0;
    DAB_CUDA(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, peer_device));
    DAB_REQUIRE(ctx, can, DAB_ERR_UNSUPPORTED, "device %d cannot access peer %d", ctx->device, peer_device);
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return DAB_OK;
    }
    DAB_CUDA(ctx, e);
    return DAB_OK;
}

}  // extern "C"
