// dab_elementwise.cu -- K1-K3: the fused per-localpart broadcast / map! loop, as streaming sm_100a kernels.
//
// Replaces Base.Broadcast.copyto!(localpart(dest), lbc) (reference src/broadcast.jl:80), copy(lbc) (:96) and
// map!(f, localpart(dest), makelocal(src, ...)) (src/mapreduce.jl:8).
//
// Roofline: HBM.  Algorithmic traffic = sizeof(T) * (inputs + 1) bytes / element (8 B/elem for y .= a.*x .+ b).
// Design: every element is touched exactly once, so there is no reuse to stage in shared memory (a TMA-staged ring was
// measured and is slower, see the note on ew1_kernel).  One CTA of 256 threads per 8 KiB tile, 2 independent 16-byte
// evict-first loads in flight per thread before any store, 8 CTAs resident per SM (~9.7 MB in flight chip-wide, vs ~5 MB
// needed by Little's law at 7.7 TB/s x ~0.7 us).  Head/tail elements (unaligned views) are peeled by one extra CTA.
#include <type_traits>

#include "dab_scalar_ops.cuh"

namespace {

constexpr int EW_THREADS = 256;

// One CTA per 256*UNROLL-vector tile ("flat" grid): the hardware block scheduler hands tiles out in address order as CTAs
// retire, so the set of concurrently open DRAM pages stays a compact sliding window.  Measured on B200 (tools/sweep_stream.cu,
// profiles/sweep_r1.txt): 6.94 TB/s for y = a*x+b at 2^30 and 2^31 floats, vs 5.95 TB/s for a persistent grid-stride loop whose
// CTAs drift apart, 6.65 TB/s for a TMA (cp.async.bulk + mbarrier) ring and 6.6 TB/s for cudaMemcpy D2D.
// The extra last CTA handles the remainder vectors and the unaligned head / tail elements.
template <typename T, typename F, int UNROLL>
__global__ void __launch_bounds__(EW_THREADS) ew1_kernel(T* y, const T* x, size_t n, size_t head, F f) {
    constexpr int VPT = 16 / sizeof(T);
    const size_t nvec = (n - head) / VPT;
    const int4* xv = reinterpret_cast<const int4*>(x + head);
    int4* yv = reinterpret_cast<int4*>(y + head);
    constexpr size_t TILE = (size_t)EW_THREADS * UNROLL;
    const size_t ntiles = nvec / TILE;
    const size_t t = blockIdx.x;
    if (t < ntiles) {
        const size_t base = t * TILE + threadIdx.x;
        int4 r[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) r[u] = ld_stream(xv + base + (size_t)u * EW_THREADS);
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            Pack<T> p = as_pack<T>(r[u]);
#pragma unroll
            for (int k = 0; k < VPT; ++k) p.v[k] = f(p.v[k]);
            st_stream(yv + base + (size_t)u * EW_THREADS, as_int4(p));
        }
    } else {  // remainder vectors + unaligned head + tail
        for (size_t i = ntiles * TILE + threadIdx.x; i < nvec; i += EW_THREADS) {
            Pack<T> p = as_pack<T>(ld_stream(xv + i));
#pragma unroll
            for (int k = 0; k < VPT; ++k) p.v[k] = f(p.v[k]);
            st_stream(yv + i, as_int4(p));
        }
        for (size_t i = threadIdx.x; i < head; i += EW_THREADS) y[i] = f(x[i]);
        for (size_t i = head + nvec * VPT + threadIdx.x; i < n; i += EW_THREADS) y[i] = f(x[i]);
    }
}

template <typename T, typename F, int UNROLL>
__global__ void __launch_bounds__(EW_THREADS) ew2_kernel(T* z, const T* x, const T* y, size_t n, size_t head, F f) {
    constexpr int VPT = 16 / sizeof(T);
    const size_t nvec = (n - head) / VPT;
    const int4* xv = reinterpret_cast<const int4*>(x + head);
    const int4* yv = reinterpret_cast<const int4*>(y + head);
    int4* zv = reinterpret_cast<int4*>(z + head);
    constexpr size_t TILE = (size_t)EW_THREADS * UNROLL;
    const size_t ntiles = nvec / TILE;
    const size_t t = blockIdx.x;
    if (t < ntiles) {
        const size_t base = t * TILE + threadIdx.x;
        int4 rx[UNROLL], ry[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            rx[u] = ld_stream(xv + base + (size_t)u * EW_THREADS);
            ry[u] = ld_stream(yv + base + (size_t)u * EW_THREADS);
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            Pack<T> p = as_pack<T>(rx[u]), q = as_pack<T>(ry[u]);
#pragma unroll
            for (int k = 0; k < VPT; ++k) p.v[k] = f(p.v[k], q.v[k]);
            st_stream(zv + base + (size_t)u * EW_THREADS, as_int4(p));
        }
    } else {
        for (size_t i = ntiles * TILE + threadIdx.x; i < nvec; i += EW_THREADS) {
            Pack<T> p = as_pack<T>(ld_stream(xv + i)), q = as_pack<T>(ld_stream(yv + i));
#pragma unroll
            for (int k = 0; k < VPT; ++k) p.v[k] = f(p.v[k], q.v[k]);
            st_stream(zv + i, as_int4(p));
        }
        for (size_t i = threadIdx.x; i < head; i += EW_THREADS) z[i] = f(x[i], y[i]);
        for (size_t i = head + nvec * VPT + threadIdx.x; i < n; i += EW_THREADS) z[i] = f(x[i], y[i]);
    }
}

// pointers whose 16-byte misalignments differ: plain coalesced 4/8-byte accesses
template <typename T, typename F>
__global__ void __launch_bounds__(EW_THREADS) ew1_scalar_kernel(T* y, const T* x, size_t n, F f) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) y[i] = f(x[i]);
}
template <typename T, typename F>
__global__ void __launch_bounds__(EW_THREADS) ew2_scalar_kernel(T* z, const T* x, const T* y, size_t n, F f) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) z[i] = f(x[i], y[i]);
}

// ---- TMA-staged variant (opt-in: dab_set_option(ctx, "ew_tma", 1)) ----------------------------------------------------------------
// The north-star design sketch asks for "TMA-staged tiles into shared memory"; this is that kernel: one elected thread streams
// 32 KiB tiles global -> shared with cp.async.bulk (SASS UBLKCP.S.G) completing on an mbarrier ring (3 stages), all threads apply f
// in place in shared memory, then the elected thread streams the tile shared -> global (UBLKCP.G.S, bulk async-group).  Persistent,
// one CTA per SM.  Measured on B200 (tools/sweep_stream.cu, profiles/sweep_r1*.txt): 6.65-6.68 TB/s vs 6.95 TB/s for the flat LDG
// kernel above -- every element is touched once, so staging buys no reuse and only adds a hop; it is therefore NOT the default.
// Bit-identical results (tests/test_gpu_hotpath.py::test_affine_tma_variant).
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "DAB_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DAB_WAIT_DONE;\n"
        "bra DAB_WAIT_LOOP;\n"
        "DAB_WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)), "l"(gsrc),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

constexpr int TMA_TILE_BYTES = 32768;
constexpr int TMA_STAGES = 3;

template <typename T, typename F>
__global__ void __launch_bounds__(EW_THREADS) ew1_tma_kernel(T* __restrict__ y, const T* __restrict__ x, size_t ntiles, F f) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int VPT = 16 / sizeof(T);
    constexpr int TILE_V = TMA_TILE_BYTES / 16;
    constexpr size_t TILE_ELEMS = TMA_TILE_BYTES / sizeof(T);
    int4* buf = reinterpret_cast<int4*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)TMA_STAGES * TMA_TILE_BYTES);
    const size_t mine = (ntiles > blockIdx.x) ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    if (threadIdx.x == 0) {
        for (int s = 0; s < TMA_STAGES; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int s = 0; s < TMA_STAGES - 1 && (size_t)s < mine; ++s) {
            const size_t tile = blockIdx.x + (size_t)s * gridDim.x;
            mbar_expect_tx(&full[s], TMA_TILE_BYTES);
            bulk_load(buf + (size_t)s * TILE_V, x + tile * TILE_ELEMS, TMA_TILE_BYTES, &full[s]);
        }
    }
    for (size_t it = 0; it < mine; ++it) {
        const int s = (int)(it % TMA_STAGES);
        mbar_wait(&full[s], (uint32_t)((it / TMA_STAGES) & 1));
        int4* p = buf + (size_t)s * TILE_V;
#pragma unroll 4
        for (int i = threadIdx.x; i < TILE_V; i += EW_THREADS) {
            Pack<T> pk = as_pack<T>(p[i]);
#pragma unroll
            for (int k = 0; k < VPT; ++k) pk.v[k] = f(pk.v[k]);
            p[i] = as_int4(pk);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the bulk (async proxy) store
        __syncthreads();
        if (threadIdx.x == 0) {
            const size_t tile = blockIdx.x + it * gridDim.x;
            bulk_store(y + tile * TILE_ELEMS, p, TMA_TILE_BYTES);
            bulk_commit();
            const size_t nxt = it + TMA_STAGES - 1;
            if (nxt < mine) {
                const int sn = (int)(nxt % TMA_STAGES);
                bulk_wait_read<1>();  // the store that last read stage sn (committed one iteration ago) has drained shared memory
                mbar_expect_tx(&full[sn], TMA_TILE_BYTES);
                bulk_load(buf + (size_t)sn * TILE_V, x + (blockIdx.x + nxt * gridDim.x) * TILE_ELEMS, TMA_TILE_BYTES, &full[sn]);
            }
        }
    }
    if (threadIdx.x == 0) bulk_wait_read<0>();
}

template <typename T>
inline size_t head_of(const void* p, size_t n) {
    size_t h = ((16 - ((uintptr_t)p & 15)) & 15) / sizeof(T);
    return h > n ? n : h;
}

template <typename T, typename F>
int32_t launch_ew1(dab_ctx* ctx, T* y, const T* x, size_t n, F f) {
    if (n == 0) return DAB_OK;
    if (ctx->opt_ew_tma && (((uintptr_t)x | (uintptr_t)y) & 15) == 0 && n * sizeof(T) >= (size_t)TMA_TILE_BYTES) {
        // opt-in TMA-staged path for the 16-byte aligned bulk; the ragged tail goes through the regular kernel below
        const size_t tile_elems = TMA_TILE_BYTES / sizeof(T);
        const size_t ntiles = n / tile_elems;
        const size_t smem = (size_t)TMA_STAGES * TMA_TILE_BYTES + 8 * TMA_STAGES;
        // the >48 KiB dynamic shared memory opt-in is a property of the (function, DEVICE) pair: remember it per device, not per process
        static unsigned long long attr_set_mask = 0;   // bit d: done on device d (devices >= 64 simply set it every time)
        if (ctx->device >= 64 || !(attr_set_mask & (1ull << ctx->device))) {
            DAB_CUDA(ctx, cudaFuncSetAttribute(ew1_tma_kernel<T, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            if (ctx->device < 64) attr_set_mask |= 1ull << ctx->device;
        }
        int grid = ctx->sm_count < (int)ntiles ? ctx->sm_count : (int)ntiles;
        ew1_tma_kernel<T, F><<<grid, EW_THREADS, smem, ctx->stream>>>(y, x, ntiles, f);
        DAB_LAUNCHED(ctx);
        const size_t done = ntiles * tile_elems;
        if (done == n) return DAB_OK;
        x += done;
        y += done;
        n -= done;
    }
    if ((((uintptr_t)x) & 15) == (((uintptr_t)y) & 15) && (((uintptr_t)x) % sizeof(T)) == 0) {
        constexpr int UNROLL = 2;
        const size_t head = head_of<T>(x, n);
        const size_t tiles = ((n - head) / (16 / sizeof(T))) / ((size_t)EW_THREADS * UNROLL);
        if (tiles + 1 > 0x7fffffffull) return dab_fail(ctx, DAB_ERR_ARG, "array too large for one launch");
        ew1_kernel<T, F, UNROLL><<<(unsigned)(tiles + 1), EW_THREADS, 0, ctx->stream>>>(y, x, n, head, f);
    } else {
        int grid = dab_persistent_grid(ctx, ew1_scalar_kernel<T, F>, EW_THREADS, (n + EW_THREADS - 1) / EW_THREADS);
        ew1_scalar_kernel<T, F><<<grid, EW_THREADS, 0, ctx->stream>>>(y, x, n, f);
    }
    DAB_LAUNCHED(ctx);
    return DAB_OK;
}

template <typename T, typename F>
int32_t launch_ew2(dab_ctx* ctx, T* z, const T* x, const T* y, size_t n, F f) {
    if (n == 0) return DAB_OK;
    uintptr_t mx = (uintptr_t)x & 15, my = (uintptr_t)y & 15, mz = (uintptr_t)z & 15;
    if (mx == my && mx == mz && (((uintptr_t)x) % sizeof(T)) == 0) {
        constexpr int UNROLL = 2;
        const size_t head = head_of<T>(x, n);
        const size_t tiles = ((n - head) / (16 / sizeof(T))) / ((size_t)EW_THREADS * UNROLL);
        if (tiles + 1 > 0x7fffffffull) return dab_fail(ctx, DAB_ERR_ARG, "array too large for one launch");
        ew2_kernel<T, F, UNROLL><<<(unsigned)(tiles + 1), EW_THREADS, 0, ctx->stream>>>(z, x, y, n, head, f);
    } else {
        int grid = dab_persistent_grid(ctx, ew2_scalar_kernel<T, F>, EW_THREADS, (n + EW_THREADS - 1) / EW_THREADS);
        ew2_scalar_kernel<T, F><<<grid, EW_THREADS, 0, ctx->stream>>>(z, x, y, n, f);
    }
    DAB_LAUNCHED(ctx);
    return DAB_OK;
}

// ---- functors (AffineF, a*x + b, lives in dab_scalar_ops.cuh: the fused broadcast + reduce shares it) ---------------------------
template <typename T, int FN>
struct UnaryF {
    __device__ __forceinline__ T operator()(T x) const {
        if constexpr (FN == DAB_MAP_ID) return x;
        else if constexpr (FN == DAB_MAP_ABS) return jl::abs(x);
        else if constexpr (FN == DAB_MAP_ABS2) return jl::mul(x, x);
        else if constexpr (FN == DAB_MAP_NEG) return jl::neg(x);
        else if constexpr (FN == DAB_MAP_SIGN) return jl::sign(x);
        else if constexpr (std::is_floating_point<T>::value) {
            if constexpr (FN == DAB_MAP_SQRT) return jl::sqrt(x);
            else if constexpr (FN == DAB_MAP_INV) return jl::inv(x);
            else if constexpr (FN == DAB_MAP_FLOOR) return floor(x);
            else if constexpr (FN == DAB_MAP_CEIL) return ceil(x);
            else return x;
        } else return x;  // floor/ceil of an integer is the integer
    }
};

template <typename T, int OP>
struct BinOp {
    __device__ __forceinline__ T operator()(T a, T b) const {
        if constexpr (OP == DAB_ADD) return jl::add(a, b);
        else if constexpr (OP == DAB_SUB) return jl::sub(a, b);
        else if constexpr (OP == DAB_MUL) return jl::mul(a, b);
        else if constexpr (OP == DAB_REM) return jl::rem(a, b);
        else if constexpr (OP == DAB_MOD) return jl::mod(a, b);
        else if constexpr (OP == DAB_BMAX) return jl::max(a, b);
        else if constexpr (OP == DAB_BMIN) return jl::min(a, b);
        else if constexpr (std::is_floating_point<T>::value) {
            if constexpr (OP == DAB_DIV) return jl::div(a, b);
            else return a;
        } else {
            if constexpr (OP == DAB_IDIV) return jl::idiv(a, b);
            else if constexpr (OP == DAB_AND) return a & b;
            else if constexpr (OP == DAB_OR) return a | b;
            else if constexpr (OP == DAB_XOR) return a ^ b;
            else return a;
        }
    }
};

template <typename T, int OP, bool LEFT>
struct BinScalarF {
    T s;
    __device__ __forceinline__ T operator()(T x) const { return LEFT ? BinOp<T, OP>()(s, x) : BinOp<T, OP>()(x, s); }
};

template <typename T>
constexpr bool op_ok(int op) {
    if (std::is_floating_point<T>::value) return op == DAB_ADD || op == DAB_SUB || op == DAB_MUL || op == DAB_DIV || op == DAB_REM ||
                                                 op == DAB_BMAX || op == DAB_BMIN || op == DAB_MOD;
    return op == DAB_ADD || op == DAB_SUB || op == DAB_MUL || op == DAB_REM || op == DAB_BMAX || op == DAB_BMIN || op == DAB_MOD ||
           op == DAB_IDIV || op == DAB_AND || op == DAB_OR || op == DAB_XOR;
}

template <typename T>
int32_t unary_t(dab_ctx* ctx, int32_t fn, T* y, const T* x, size_t n) {
    switch (fn) {
#define C(FN) \
    case FN: return launch_ew1(ctx, y, x, n, UnaryF<T, FN>())
        C(DAB_MAP_ID);
        C(DAB_MAP_ABS);
        C(DAB_MAP_ABS2);
        C(DAB_MAP_NEG);
        C(DAB_MAP_SIGN);
        C(DAB_MAP_FLOOR);
        C(DAB_MAP_CEIL);
#undef C
        case DAB_MAP_SQRT:
            if (std::is_floating_point<T>::value) return launch_ew1(ctx, y, x, n, UnaryF<T, DAB_MAP_SQRT>());
            break;
        case DAB_MAP_INV:
            if (std::is_floating_point<T>::value) return launch_ew1(ctx, y, x, n, UnaryF<T, DAB_MAP_INV>());
            break;
        default: break;
    }
    return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "dab_unary: fn %d not served for this dtype (no host fallback)", fn);
}

template <typename T, int OP>
int32_t binary_dispatch(dab_ctx* ctx, T* z, const T* x, const T* y, const T* s, int mode, size_t n) {
    if (mode == 0) return launch_ew2(ctx, z, x, y, n, BinOp<T, OP>());
    if (mode == 1) return launch_ew1(ctx, z, x, n, BinScalarF<T, OP, false>{*s});
    return launch_ew1(ctx, z, x, n, BinScalarF<T, OP, true>{*s});
}

template <typename T>
int32_t binary_t(dab_ctx* ctx, int32_t op, T* z, const T* x, const T* y, const T* s, int mode, size_t n) {
    if (!op_ok<T>(op)) return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "binary op %d not served for this dtype (no host fallback)", op);
    switch (op) {
#define C(OP) \
    case OP: return binary_dispatch<T, OP>(ctx, z, x, y, s, mode, n)
        C(DAB_ADD);
        C(DAB_SUB);
        C(DAB_MUL);
        C(DAB_DIV);
        C(DAB_REM);
        C(DAB_BMAX);
        C(DAB_BMIN);
        C(DAB_MOD);
        C(DAB_IDIV);
        C(DAB_AND);
        C(DAB_OR);
        C(DAB_XOR);
#undef C
        default: return dab_fail(ctx, DAB_ERR_ARG, "bad binary op %d", op);
    }
}

}  // namespace

extern "C" {

int32_t dab_affine(dab_ctx* ctx, int32_t dtype, void* y, const void* x, const void* a, const void* b, size_t n) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, ((x && y) || n == 0) && a && b, DAB_ERR_ARG, "dab_affine: null pointer");
    switch (dtype) {
        case DAB_F32: return launch_ew1(ctx, (float*)y, (const float*)x, n, AffineF<float>{*(const float*)a, *(const float*)b});
        case DAB_F64: return launch_ew1(ctx, (double*)y, (const double*)x, n, AffineF<double>{*(const double*)a, *(const double*)b});
        case DAB_I32: return launch_ew1(ctx, (int32_t*)y, (const int32_t*)x, n, AffineF<int32_t>{*(const int32_t*)a, *(const int32_t*)b});
        case DAB_I64:
            return launch_ew1(ctx, (long long*)y, (const long long*)x, n, AffineF<long long>{*(const long long*)a, *(const long long*)b});
        default: return dab_fail(ctx, DAB_ERR_ARG, "dab_affine: bad dtype %d", dtype);
    }
}

int32_t dab_unary(dab_ctx* ctx, int32_t dtype, int32_t fn, void* y, const void* x, size_t n) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, (x && y) || n == 0, DAB_ERR_ARG, "dab_unary: null pointer");
    switch (dtype) {
        case DAB_F32: return unary_t(ctx, fn, (float*)y, (const float*)x, n);
        case DAB_F64: return unary_t(ctx, fn, (double*)y, (const double*)x, n);
        case DAB_I32: return unary_t(ctx, fn, (int32_t*)y, (const int32_t*)x, n);
        case DAB_I64: return unary_t(ctx, fn, (long long*)y, (const long long*)x, n);
        default: return dab_fail(ctx, DAB_ERR_ARG, "dab_unary: bad dtype %d", dtype);
    }
}

int32_t dab_binary(dab_ctx* ctx, int32_t dtype, int32_t op, void* z, const void* x, const void* y, size_t n) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, (x && y && z) || n == 0, DAB_ERR_ARG, "dab_binary: null pointer");
    switch (dtype) {
        case DAB_F32: return binary_t<float>(ctx, op, (float*)z, (const float*)x, (const float*)y, nullptr, 0, n);
        case DAB_F64: return binary_t<double>(ctx, op, (double*)z, (const double*)x, (const double*)y, nullptr, 0, n);
        case DAB_I32: return binary_t<int32_t>(ctx, op, (int32_t*)z, (const int32_t*)x, (const int32_t*)y, nullptr, 0, n);
        case DAB_I64: return binary_t<long long>(ctx, op, (long long*)z, (const long long*)x, (const long long*)y, nullptr, 0, n);
        default: return dab_fail(ctx, DAB_ERR_ARG, "dab_binary: bad dtype %d", dtype);
    }
}

int32_t dab_binary_scalar(dab_ctx* ctx, int32_t dtype, int32_t op, void* z, const void* x, const void* s, int32_t scalar_left,
                          size_t n) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, ((x && z) || n == 0) && s, DAB_ERR_ARG, "dab_binary_scalar: null pointer");
    int mode = scalar_left ? 2 : 1;
    switch (dtype) {
        case DAB_F32: return binary_t<float>(ctx, op, (float*)z, (const float*)x, nullptr, (const float*)s, mode, n);
        case DAB_F64: return binary_t<double>(ctx, op, (double*)z, (const double*)x, nullptr, (const double*)s, mode, n);
        case DAB_I32: return binary_t<int32_t>(ctx, op, (int32_t*)z, (const int32_t*)x, nullptr, (const int32_t*)s, mode, n);
        case DAB_I64: return binary_t<long long>(ctx, op, (long long*)z, (const long long*)x, nullptr, (const long long*)s, mode, n);
        default: return dab_fail(ctx, DAB_ERR_ARG, "dab_binary_scalar: bad dtype %d", dtype);
    }
}

}  // extern "C"
