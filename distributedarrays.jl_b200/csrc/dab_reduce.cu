// dab_reduce.cu -- K4 / K7: whole-chunk mapreduce(f, op, localpart(d)) as one streaming sm_100a kernel.
//
// Replaces the per-worker Base.mapreduce / reduce / all / any / count at reference src/mapreduce.jl:23,31,100,109,118
// and the caller-side left fold reduce(op, results) at src/mapreduce.jl:26,34 (dab_combine_ordered).
//
// Roofline: HBM, 4 B/element read (sizeof(T)), output negligible.
// Design: flat grid, one CTA of 256 threads per 32 KiB of input; each thread keeps UNROLL independent 16-byte evict-first loads
// in flight, reduces the 16 values of a tile step with a register tree in the element type, and carries the running
// value in a wide accumulator (fp64 for float sums/products, int64 for integers) -- one F2D + DADD per 16 elements, so the
// FP64 pipe is idle >90 % of the time and the result is far inside the 1e-6 tolerance.  Warp shuffle -> shared-memory
// tree -> one partial per CTA -> the LAST CTA to finish (ticket counter) folds the CTA partials in a fixed order, so the
// result is deterministic for a given (n, grid).  No atomics on data, no second launch.
#include <type_traits>

#include <cmath>

#include "dab_reduce_traits.cuh"

namespace {

constexpr int RD_UNROLL = 4;

// Result slot layout (16 bytes at `out`): [0..8) the result in its result dtype, [8..16) the wide accumulator (fp64 for
// float SUM/PROD -- lets the host see the un-rounded carrier; tests use it).
//
// STORE = true (dab_affine_reduce): the kernel also writes every mapped value to y (evict-first 16-byte stores, before the register
// tree consumes the pack), so `y .= f.(x); reduce(op, y)` is one pass of 8 instead of 12 bytes per Float32 element.  Grid, tiles,
// tree and combine are those of the reduce of y, so with x and y at the same offset mod 16 (same head) the result is bit-identical.
// y may alias x (map!(f, d, d)): each thread loads its packs before it stores them, and neither pointer is declared __restrict__.
// Resident CTAs per SM the kernel is compiled for: 8 (32 registers) for every plain reduce.  The store variant keeps 8 where it still
// fits 32 registers without spilling (Float32 SUM / PROD, ptxas -v) and is given 40 registers (6 CTAs per SM) elsewhere.  Occupancy
// does not change the result; the grid mapping, which decides it, is the same for every instantiation.
template <typename T, typename R, bool STORE>
constexpr int rd_min_blocks() {
    return (!STORE || (sizeof(T) == 4 && (std::is_same<R, SumTraits<T>>::value || std::is_same<R, ProdTraits<T>>::value))) ? 8 : 6;
}

template <typename T, typename Map, typename R, typename Out, bool STORE = false>
__global__ void __launch_bounds__(RD_THREADS, rd_min_blocks<T, R, STORE>()) reduce_kernel(const T* x, T* y, size_t n, size_t head, Map map,
                                                             typename R::A* __restrict__ partials, unsigned int* counter,
                                                             void* out, int finalize_mode, long long n_for_all, int tiles_per_cta,
                                                             FusedComm fc) {
    using A = typename R::A;
    using V = typename Map::V;
    static_assert(!STORE || std::is_same<V, T>::value, "the stored map must keep the element type");
    constexpr int VPT = 16 / sizeof(T);
    __shared__ A smem[RD_THREADS / 32];
    __shared__ bool is_last;

    const size_t nvec = (n - head) / VPT;
    const int4* xv = reinterpret_cast<const int4*>(x + head);
    int4* yv = STORE ? reinterpret_cast<int4*>(y + head) : nullptr;
    constexpr size_t TILE = (size_t)RD_THREADS * RD_UNROLL;
    const size_t ntiles = nvec / TILE;
    A acc = R::identity();
    // "flat" grid: CTA b owns the tiles_per_cta consecutive tiles starting at b*tiles_per_cta (fixed mapping -> deterministic
    // result); the block scheduler issues CTAs in address order, keeping the open DRAM pages a compact window.  Measured on
    // B200 (profiles/sweep_r1.txt): 7.55 TB/s vs 7.2 TB/s for a persistent grid-stride loop.
    size_t t_end = ((size_t)blockIdx.x + 1) * (size_t)tiles_per_cta;
    if (t_end > ntiles) t_end = ntiles;
#pragma unroll 1
    for (size_t t = (size_t)blockIdx.x * (size_t)tiles_per_cta; t < t_end; ++t) {
        const size_t base = t * TILE + threadIdx.x;
        int4 r[RD_UNROLL];
#pragma unroll
        for (int u = 0; u < RD_UNROLL; ++u) r[u] = ld_stream(xv + base + (size_t)u * RD_THREADS);
        V tv[RD_UNROLL];
#pragma unroll
        for (int u = 0; u < RD_UNROLL; ++u) {
            Pack<T> p = as_pack<T>(r[u]);
            V m[VPT];
#pragma unroll
            for (int k = 0; k < VPT; ++k) m[k] = map(p.v[k]);
            if constexpr (STORE) {
                Pack<T> q;
#pragma unroll
                for (int k = 0; k < VPT; ++k) q.v[k] = m[k];
                st_stream(yv + base + (size_t)u * RD_THREADS, as_int4(q));
            }
#pragma unroll
            for (int w = VPT; w > 1; w >>= 1)  // register tree inside one 16-byte vector
#pragma unroll
                for (int k = 0; k < w / 2; ++k) m[k] = R::tile(m[k], m[k + w / 2]);
            tv[u] = m[0];
        }
#pragma unroll
        for (int w = RD_UNROLL; w > 1; w >>= 1)
#pragma unroll
            for (int k = 0; k < w / 2; ++k) tv[k] = R::tile(tv[k], tv[k + w / 2]);
        acc = R::comb(acc, R::lift(tv[0]));
    }
    if (blockIdx.x == gridDim.x - 1) {  // remainder vectors, unaligned head, tail
        for (size_t i = ntiles * TILE + threadIdx.x; i < nvec; i += RD_THREADS) {
            Pack<T> p = as_pack<T>(ld_stream(xv + i));
            V mk[VPT];
#pragma unroll
            for (int k = 0; k < VPT; ++k) mk[k] = map(p.v[k]);
            if constexpr (STORE) {
                Pack<T> q;
#pragma unroll
                for (int k = 0; k < VPT; ++k) q.v[k] = mk[k];
                st_stream(yv + i, as_int4(q));
            }
            V m = mk[0];
#pragma unroll
            for (int k = 1; k < VPT; ++k) m = R::tile(m, mk[k]);
            acc = R::comb(acc, R::lift(m));
        }
        auto elem = [&](size_t i) {
            const V v = map(x[i]);
            if constexpr (STORE) y[i] = v;
            acc = R::comb(acc, R::lift(v));
        };
        for (size_t i = threadIdx.x; i < head; i += RD_THREADS) elem(i);
        for (size_t i = head + nvec * VPT + threadIdx.x; i < n; i += RD_THREADS) elem(i);
    }
    acc = block_reduce<R>(acc, smem);
    // ---- two-level "last one out" combine: deterministic, no second launch, tail latency of a few microseconds.
    //  level 1: CTAs form groups of RD_THREADS; the last CTA of a group to finish folds the group's partials (one per thread);
    //  level 2: the last group to finish folds the <= DAB_MAX_REDUCE_BLOCKS/RD_THREADS group partials and writes the result.
    A* gpartials = partials + DAB_MAX_REDUCE_BLOCKS;
    const unsigned int ngroups = (gridDim.x + RD_THREADS - 1) / RD_THREADS;
    const unsigned int g = blockIdx.x / RD_THREADS;
    const unsigned int gsize = (g == ngroups - 1) ? gridDim.x - g * RD_THREADS : RD_THREADS;
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = acc;
        __threadfence();
        unsigned int ticket = atomicAdd(counter + 1 + g, 1u);
        is_last = (ticket == gsize - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    A v = threadIdx.x < gsize ? partials[(size_t)g * RD_THREADS + threadIdx.x] : R::identity();
    v = block_reduce<R>(v, smem);
    if (threadIdx.x == 0) {
        counter[1 + g] = 0;  // self-reset for the next launch on this stream
        gpartials[g] = v;
        __threadfence();
        unsigned int ticket = atomicAdd(counter, 1u);
        is_last = (ticket == ngroups - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    A fin = R::identity();
    for (unsigned int i = threadIdx.x; i < ngroups; i += RD_THREADS) fin = R::comb(fin, gpartials[i]);
    fin = block_reduce<R>(fin, smem);
    if (threadIdx.x == 0) {
        *counter = 0;
        if constexpr (std::is_arithmetic<A>::value) {
            Out res;
            if (finalize_mode == 1) res = (Out)(fin == (A)n_for_all);  // ALL
            else if (finalize_mode == 2) res = (Out)(fin != (A)0);      // ANY
            else res = (Out)fin;
            memcpy(out, &res, sizeof(Out));
            if (sizeof(Out) < 8) memset((char*)out + sizeof(Out), 0, 8 - sizeof(Out));
            A wide = fin;
            memcpy((char*)out + 8, &wide, sizeof(A));
            if (sizeof(A) < 8) memset((char*)out + 8 + sizeof(A), 0, 8 - sizeof(A));
            if (fc.host_out && fc.nranks <= 1) {
                // single worker: the scalar goes straight into pinned host memory (zero-copy), no D2H memcpy launch
                unsigned long long bits = 0;
                memcpy(&bits, &res, sizeof(Out));
                volatile unsigned long long* h = reinterpret_cast<volatile unsigned long long*>(fc.host_out);
                h[0] = bits;
                h[1] = 0ull;
                __threadfence_system();
            }
        } else {  // extrema: the (min, max) pair fills the slot (8 bytes for 4-byte T, 16 for 8-byte T)
            memset(out, 0, 16);
            memcpy(out, &fin, sizeof(A));
        }
    }
    if constexpr (!std::is_arithmetic<Out>::value) return;
    else {
    if (fc.nranks <= 1) return;
    // ---- fused cross-worker combine over NVLink peer memory (replaces remotecall_fetch + reduce(op, results), reference
    // src/mapreduce.jl:30-34, and an ncclAllGather + D2H copy): thread j of this last CTA PUSHES this rank's chunk result into
    // rank j's mailbox (16-byte payload, system fence, then the sequence flag), then polls its own mailbox slot j until rank j's
    // result for this call has landed; thread 0 folds the P results LEFT TO RIGHT in rank (= procs(d)) order in the result type
    // and writes the scalar straight into pinned host memory.  Two parity banks: a fast rank can be at most one call ahead.
    __shared__ unsigned long long pay[2];
    __shared__ unsigned long long got[DAB_MAX_RANKS];
    __shared__ int timed_out;
    if (threadIdx.x == 0) {
        memcpy(&pay[0], out, 8);
        memcpy(&pay[1], (char*)out + 8, 8);
        timed_out = 0;
    }
    __syncthreads();
    const size_t bank = (size_t)(fc.seq & 1ull) * DAB_MAX_RANKS * DAB_MBOX_SLOT;
    if (threadIdx.x < (unsigned)fc.nranks) {
        volatile unsigned long long* dst =
            reinterpret_cast<volatile unsigned long long*>((char*)fc.peers[threadIdx.x] + bank + (size_t)fc.rank * DAB_MBOX_SLOT);
        dst[0] = pay[0];
        dst[1] = pay[1];
        __threadfence_system();
        dst[2] = fc.seq;
        volatile unsigned long long* src =
            reinterpret_cast<volatile unsigned long long*>((char*)fc.peers[fc.rank] + bank + (size_t)threadIdx.x * DAB_MBOX_SLOT);
        // SPMD ranks are not in lockstep (a first-time NVRTC compile, a large H2D copy or GC can hold one back for seconds), so the
        // bound is generous wall-clock time (default 120 s, dab_set_option "combine_timeout_ms") and only exists so that a DEAD
        // peer surfaces as an error instead of a hung GPU; a timeout leaves the communicator unusable, like a failed collective.
        const unsigned long long t0 = dab_globaltimer_ns();
        unsigned int spins = 0;
        while (src[2] != fc.seq) {
            if ((++spins & 1023u) == 0 && dab_globaltimer_ns() - t0 > fc.timeout_ns) {
                timed_out = 1;
                break;
            }
        }
        __threadfence_system();
        got[threadIdx.x] = src[0];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        Out a;
        memcpy(&a, &got[0], sizeof(Out));
        for (int j = 1; j < fc.nranks; ++j) {
            Out b;
            memcpy(&b, &got[j], sizeof(Out));
            switch (fc.op) {
                case DAB_SUM: case DAB_COUNT: a = jl::add(a, b); break;
                case DAB_PROD: a = jl::mul(a, b); break;
                case DAB_MAX: a = jl::max(a, b); break;
                case DAB_MIN: a = jl::min(a, b); break;
                case DAB_ALL: a = (Out)(a != (Out)0 && b != (Out)0); break;
                default: a = (Out)(a != (Out)0 || b != (Out)0); break;  // ANY
            }
        }
        unsigned long long bits = 0;
        memcpy(&bits, &a, sizeof(Out));
        volatile unsigned long long* h = reinterpret_cast<volatile unsigned long long*>(fc.host_out);
        h[0] = bits;
        h[1] = (unsigned long long)timed_out;
        __threadfence_system();
    }
    }  // arithmetic Out
}

template <typename T, typename Map, typename R, typename Out, bool STORE = false>
int32_t launch_reduce(dab_ctx* ctx, const T* x, size_t n, Map map, void* out, int finalize_mode, T* y = nullptr) {
    constexpr int VPT = 16 / sizeof(T);
    size_t head = ((16 - ((uintptr_t)x & 15)) & 15) / sizeof(T);
    if (head > n) head = n;
    size_t tiles = (n - head) / ((size_t)VPT * RD_THREADS * RD_UNROLL);
    size_t k = 2;  // 32 KiB of input per CTA
    if ((tiles + k - 1) / k > (size_t)DAB_MAX_REDUCE_BLOCKS) k = (tiles + DAB_MAX_REDUCE_BLOCKS - 1) / DAB_MAX_REDUCE_BLOCKS;
    size_t grid = (tiles + k - 1) / k;
    if (grid < 1) grid = 1;
    FusedComm fc;
    memset(&fc, 0, sizeof(fc));
    if (ctx->fuse_op >= 0 && ctx->mbox_ranks > 1) {
        fc.peers = ctx->peer_mbox_dev;
        fc.host_out = ctx->host_slot;
        fc.seq = ++ctx->mbox_seq;
        fc.timeout_ns = (unsigned long long)ctx->opt_combine_timeout_ms * 1000000ull;
        fc.rank = ctx->rank;
        fc.nranks = ctx->mbox_ranks;
        fc.op = ctx->fuse_op;
    } else if (ctx->fuse_op >= 0) {
        fc.host_out = ctx->host_slot;  // one worker: zero-copy scalar to the host, nothing to combine
        fc.nranks = 1;
        fc.op = ctx->fuse_op;
    }
    reduce_kernel<T, Map, R, Out, STORE><<<(unsigned)grid, RD_THREADS, 0, ctx->stream>>>(x, y, n, head, map, (typename R::A*)ctx->block_partials,
                                                                                         ctx->counter, out, finalize_mode, (long long)n, (int)k, fc);
    DAB_LAUNCHED(ctx);
    return DAB_OK;
}

template <typename T>
using ResultOfSum = typename std::conditional<std::is_floating_point<T>::value, T, long long>::type;

template <typename T, int FN>
int32_t reduce_arith(dab_ctx* ctx, int32_t op, const T* x, size_t n, void* out) {
    MapF<T, FN> map{(T)0};
    switch (op) {
        case DAB_SUM: return launch_reduce<T, MapF<T, FN>, SumTraits<T>, ResultOfSum<T>>(ctx, x, n, map, out, 0);
        case DAB_PROD: return launch_reduce<T, MapF<T, FN>, ProdTraits<T>, ResultOfSum<T>>(ctx, x, n, map, out, 0);
        case DAB_MAX: return launch_reduce<T, MapF<T, FN>, MaxTraits<T>, T>(ctx, x, n, map, out, 0);
        case DAB_MIN: return launch_reduce<T, MapF<T, FN>, MinTraits<T>, T>(ctx, x, n, map, out, 0);
        case DAB_EXTREMA:
            if constexpr (FN == DAB_MAP_ID) return launch_reduce<T, ExtMapF<T>, ExtremaTraits<T>, Pair<T>>(ctx, x, n, ExtMapF<T>{(T)0}, out, 0);
            else return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "extrema with a map is not served (no host fallback)");
        default: return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "reduce op %d needs a predicate map (no host fallback)", op);
    }
}

// dab_affine_reduce: the reduce_arith<T, DAB_MAP_ID> switch again, with y .= a.*x .+ b as the map and the stores switched on
template <typename T>
int32_t affine_reduce_t(dab_ctx* ctx, int32_t op, T* y, const T* x, size_t n, T a, T b, void* out) {
    const AffineMap<T> map{AffineF<T>{a, b}};
    switch (op) {
        case DAB_SUM: return launch_reduce<T, AffineMap<T>, SumTraits<T>, T, true>(ctx, x, n, map, out, 0, y);
        case DAB_PROD: return launch_reduce<T, AffineMap<T>, ProdTraits<T>, T, true>(ctx, x, n, map, out, 0, y);
        case DAB_MAX: return launch_reduce<T, AffineMap<T>, MaxTraits<T>, T, true>(ctx, x, n, map, out, 0, y);
        default: return launch_reduce<T, AffineMap<T>, MinTraits<T>, T, true>(ctx, x, n, map, out, 0, y);
    }
}

template <typename T, int FN>
int32_t reduce_pred(dab_ctx* ctx, int32_t op, const T* x, size_t n, const void* param, void* out) {
    PredF<T, FN> map{param ? *(const T*)param : (T)0};
    int mode;
    switch (op) {
        case DAB_ALL: mode = 1; break;
        case DAB_ANY: mode = 2; break;
        case DAB_COUNT:
        case DAB_SUM: mode = 0; break;  // sum of Bools == count
        default: return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "reduce op %d on a predicate map (no host fallback)", op);
    }
    return launch_reduce<T, PredF<T, FN>, CountTraits, long long>(ctx, x, n, map, out, mode);
}

template <typename T>
int32_t reduce_t(dab_ctx* ctx, int32_t op, int32_t map, const void* param, const T* x, size_t n, void* out) {
    switch (map) {
        case DAB_MAP_ID: return reduce_arith<T, DAB_MAP_ID>(ctx, op, x, n, out);
        case DAB_MAP_ABS: return reduce_arith<T, DAB_MAP_ABS>(ctx, op, x, n, out);
        case DAB_MAP_ABS2: return reduce_arith<T, DAB_MAP_ABS2>(ctx, op, x, n, out);
        case DAB_MAP_NEG: return reduce_arith<T, DAB_MAP_NEG>(ctx, op, x, n, out);
#define P(FN) \
    case FN: return reduce_pred<T, FN>(ctx, op, x, n, param, out)
            P(DAB_MAP_EQ);
            P(DAB_MAP_NE);
            P(DAB_MAP_LT);
            P(DAB_MAP_LE);
            P(DAB_MAP_GT);
            P(DAB_MAP_GE);
            P(DAB_MAP_ISNAN);
            P(DAB_MAP_NONZERO);
#undef P
        default: return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "map %d not served by a reduce kernel (no host fallback)", map);
    }
}

int32_t reduce_u8(dab_ctx* ctx, int32_t op, int32_t map, const uint8_t* x, size_t n, void* out) {
    // Bool arrays: all(d) / any(d) / count(d) / sum(d) with the identity predicate; max/min on Bool.
    if (map != DAB_MAP_ID && map != DAB_MAP_NONZERO)
        return dab_fail(ctx, DAB_ERR_UNSUPPORTED, "map %d on Bool not served (no host fallback)", map);
    if (op == DAB_MAX) return launch_reduce<uint8_t, MapF<uint8_t, DAB_MAP_ID>, MaxTraits<uint8_t>, uint8_t>(ctx, x, n, {0}, out, 0);
    if (op == DAB_MIN) return launch_reduce<uint8_t, MapF<uint8_t, DAB_MAP_ID>, MinTraits<uint8_t>, uint8_t>(ctx, x, n, {0}, out, 0);
    return reduce_pred<uint8_t, DAB_MAP_NONZERO>(ctx, op, x, n, nullptr, out);
}

// host-side write of the n == 0 result
int32_t empty_result(dab_ctx* ctx, int32_t dtype, int32_t op, void* out_dev) {
    unsigned char buf[16];
    memset(buf, 0, 16);
    bool flt = dtype == DAB_F32 || dtype == DAB_F64;
    switch (op) {
        case DAB_SUM:
        case DAB_ANY:
        case DAB_COUNT: break;
        case DAB_ALL: {
            long long one = 1;
            memcpy(buf, &one, 8);
            break;
        }
        case DAB_PROD:
            if (dtype == DAB_F32) {
                float one = 1.f;
                memcpy(buf, &one, 4);
            } else if (dtype == DAB_F64) {
                double one = 1.0;
                memcpy(buf, &one, 8);
            } else {
                long long one = 1;
                memcpy(buf, &one, 8);
            }
            if (flt) {
                double one = 1.0;
                memcpy(buf + 8, &one, 8);
            }
            break;
        default: return dab_fail(ctx, DAB_ERR_EMPTY, "reducing over an empty collection is not allowed");
    }
    // stream-ordered small copy from a stack buffer: use the pinned slot's tail to stay async-safe
    memcpy((char*)ctx->host_slot + DAB_MAX_RANKS * 16, buf, 16);
    DAB_CUDA(ctx, cudaMemcpyAsync(out_dev, (char*)ctx->host_slot + DAB_MAX_RANKS * 16, 16, cudaMemcpyHostToDevice, ctx->stream));
    DAB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return DAB_OK;
}

}  // namespace

extern "C" {

int32_t dab_reduce_result_dtype(int32_t dtype, int32_t op, int32_t map, int32_t* out_dtype) {
    if (!out_dtype) return DAB_ERR_ARG;
    const bool pred = map >= DAB_MAP_EQ;  // predicate maps yield Bool: sum/count/all/any -> Int64
    switch (op) {
        case DAB_SUM:
        case DAB_PROD:
            *out_dtype = (!pred && (dtype == DAB_F32 || dtype == DAB_F64)) ? dtype : DAB_I64;
            return DAB_OK;
        case DAB_MAX:
        case DAB_MIN:
        case DAB_EXTREMA: *out_dtype = dtype; return DAB_OK;
        case DAB_ALL:
        case DAB_ANY:
        case DAB_COUNT: *out_dtype = DAB_I64; return DAB_OK;
        default: return DAB_ERR_ARG;
    }
}

// out_dev: 16 bytes (result + wide accumulator)
int32_t dab_reduce(dab_ctx* ctx, int32_t dtype, int32_t op, int32_t map, const void* map_param, const void* x, size_t n,
                   void* out_dev) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, out_dev && (x || n == 0), DAB_ERR_ARG, "dab_reduce: null pointer");
    DAB_REQUIRE(ctx, op >= DAB_SUM && op <= DAB_EXTREMA, DAB_ERR_ARG, "dab_reduce: bad op %d", op);
    if (n == 0) return empty_result(ctx, dtype, op, out_dev);
    // predicate maps turn the value into a Bool: only SUM/ALL/ANY/COUNT make sense
    switch (dtype) {
        case DAB_F32: return reduce_t<float>(ctx, op, map, map_param, (const float*)x, n, out_dev);
        case DAB_F64: return reduce_t<double>(ctx, op, map, map_param, (const double*)x, n, out_dev);
        case DAB_I32: return reduce_t<int32_t>(ctx, op, map, map_param, (const int32_t*)x, n, out_dev);
        case DAB_I64: return reduce_t<long long>(ctx, op, map, map_param, (const long long*)x, n, out_dev);
        case DAB_U8: return reduce_u8(ctx, op, map, (const uint8_t*)x, n, out_dev);
        default: return dab_fail(ctx, DAB_ERR_ARG, "dab_reduce: bad dtype %d", dtype);
    }
}

// y .= a.*x .+ b, then dab_reduce(op, identity map) of y into out_dev -- in ONE pass when a kernel serves it: Float32 / Float64, op SUM
// PROD MAX MIN, n > 0, and x and y at the same offset mod 16 (the reduce's head peel, hence its grid, follows the pointer's alignment;
// only then is the fused result bit-identical to reducing y afterwards).  Any other case runs the two launches it replaces.
int32_t dab_affine_reduce(dab_ctx* ctx, int32_t dtype, void* y, const void* x, const void* a, const void* b, size_t n, int32_t op,
                          void* out_dev) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, ((x && y) || n == 0) && a && b, DAB_ERR_ARG, "dab_affine: null pointer");
    DAB_REQUIRE(ctx, out_dev, DAB_ERR_ARG, "dab_reduce: null pointer");
    DAB_REQUIRE(ctx, op >= DAB_SUM && op <= DAB_EXTREMA, DAB_ERR_ARG, "dab_reduce: bad op %d", op);
    const size_t es = dab_dtype_size(dtype);
    const bool fused = (dtype == DAB_F32 || dtype == DAB_F64) && (op == DAB_SUM || op == DAB_PROD || op == DAB_MAX || op == DAB_MIN) &&
                       n > 0 && ((uintptr_t)x & 15) == ((uintptr_t)y & 15) && (uintptr_t)x % es == 0;
    if (!fused) {
        int32_t st = dab_affine(ctx, dtype, y, x, a, b, n);
        if (st != DAB_OK) return st;
        return dab_reduce(ctx, dtype, op, DAB_MAP_ID, nullptr, y, n, out_dev);
    }
    if (dtype == DAB_F32)
        return affine_reduce_t<float>(ctx, op, (float*)y, (const float*)x, n, *(const float*)a, *(const float*)b, out_dev);
    return affine_reduce_t<double>(ctx, op, (double*)y, (const double*)x, n, *(const double*)a, *(const double*)b, out_dev);
}

int32_t dab_reduce_host(dab_ctx* ctx, int32_t dtype, int32_t op, int32_t map, const void* map_param, const void* x, size_t n,
                        void* out_host) {
    DAB_ENTER(ctx);
    DAB_REQUIRE(ctx, out_host, DAB_ERR_ARG, "dab_reduce_host: null out");
    int32_t st = dab_reduce(ctx, dtype, op, map, map_param, x, n, ctx->result_slot);
    if (st != DAB_OK) return st;
    DAB_CUDA(ctx, cudaMemcpyAsync(ctx->host_slot, ctx->result_slot, 16, cudaMemcpyDeviceToHost, ctx->stream));
    DAB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(out_host, ctx->host_slot, 16);
    return DAB_OK;
}

// reduce(op, results) on the caller: plain left fold in procs(d) order, in the result dtype (src/mapreduce.jl:34).
int32_t dab_combine_ordered(int32_t rdt, int32_t op, const void* partials, size_t p, void* out) {
    if (!partials || !out) return dab_fail(nullptr, DAB_ERR_ARG, "dab_combine_ordered: null pointer");
    if (p == 0) return dab_fail(nullptr, DAB_ERR_EMPTY, "reducing over an empty collection is not allowed");
#define FOLD(T, EXPR)                          \
    {                                          \
        const T* v = (const T*)partials;       \
        T a = v[0];                            \
        for (size_t i = 1; i < p; ++i) {       \
            T b = v[i];                        \
            a = (EXPR);                        \
        }                                      \
        *(T*)out = a;                          \
        return DAB_OK;                         \
    }
    auto fmax_jl = [](auto a, auto b) {
        using T = decltype(a);
        if (a != a || b != b) return (T)NAN;
        if (a == b) return std::signbit(a) ? b : a;
        return a > b ? a : b;
    };
    auto fmin_jl = [](auto a, auto b) {
        using T = decltype(a);
        if (a != a || b != b) return (T)NAN;
        if (a == b) return std::signbit(a) ? a : b;
        return a < b ? a : b;
    };
    switch (rdt) {
        case DAB_F32:
            switch (op) {
                case DAB_SUM: {
                    // volatile: keep each partial sum rounded to fp32 (no x87 / contraction surprises)
                    const float* v = (const float*)partials;
                    volatile float a = v[0];
                    for (size_t i = 1; i < p; ++i) a = a + v[i];
                    *(float*)out = a;
                    return DAB_OK;
                }
                case DAB_PROD: {
                    const float* v = (const float*)partials;
                    volatile float a = v[0];
                    for (size_t i = 1; i < p; ++i) a = a * v[i];
                    *(float*)out = a;
                    return DAB_OK;
                }
                case DAB_MAX: FOLD(float, fmax_jl(a, b))
                case DAB_MIN: FOLD(float, fmin_jl(a, b))
                default: break;
            }
            break;
        case DAB_F64:
            switch (op) {
                case DAB_SUM: FOLD(double, a + b)
                case DAB_PROD: FOLD(double, a * b)
                case DAB_MAX: FOLD(double, fmax_jl(a, b))
                case DAB_MIN: FOLD(double, fmin_jl(a, b))
                default: break;
            }
            break;
        case DAB_I64:
            switch (op) {
                case DAB_SUM:
                case DAB_COUNT: FOLD(long long, (long long)((unsigned long long)a + (unsigned long long)b))
                case DAB_PROD: FOLD(long long, (long long)((unsigned long long)a * (unsigned long long)b))
                case DAB_MAX: FOLD(long long, a > b ? a : b)
                case DAB_MIN: FOLD(long long, a < b ? a : b)
                case DAB_ALL: FOLD(long long, (long long)(a && b))
                case DAB_ANY: FOLD(long long, (long long)(a || b))
                default: break;
            }
            break;
        case DAB_I32:
            switch (op) {
                case DAB_MAX: FOLD(int32_t, a > b ? a : b)
                case DAB_MIN: FOLD(int32_t, a < b ? a : b)
                default: break;
            }
            break;
        case DAB_U8:
            switch (op) {
                case DAB_MAX: FOLD(uint8_t, a > b ? a : b)
                case DAB_MIN: FOLD(uint8_t, a < b ? a : b)
                default: break;
            }
            break;
        default: break;
    }
#undef FOLD
    return dab_fail(nullptr, DAB_ERR_UNSUPPORTED, "dab_combine_ordered: dtype %d op %d", rdt, op);
}

}  // extern "C"
