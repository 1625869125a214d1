// dab_reduce_traits.cuh -- reduction traits, map functors and block-level reduction shared by dab_reduce.cu / dab_reducedim.cu
#pragma once
#include <type_traits>

#include "dab_scalar_ops.cuh"

namespace {

constexpr int RD_THREADS = 256;

// ---------------------------------------------------------------------------------------------------------------
// Reduce "traits": V = value type after the map, A = accumulator carried across tiles / threads / CTAs.
//   lift(V) -> A, comb(A, A) -> A (associative up to rounding), tile(V, V) -> V combine inside a tile step.
// ---------------------------------------------------------------------------------------------------------------
template <typename V>
struct SumTraits {
    using A = typename std::conditional<std::is_floating_point<V>::value, double, long long>::type;
    __device__ static __forceinline__ A identity() { return (A)0; }
    __device__ static __forceinline__ V tile(V a, V b) { return jl::add(a, b); }
    __device__ static __forceinline__ A lift(V v) { return (A)v; }
    __device__ static __forceinline__ A comb(A a, A b) { return jl::add(a, b); }
};
template <typename V>
struct ProdTraits {
    using A = typename std::conditional<std::is_floating_point<V>::value, double, long long>::type;
    __device__ static __forceinline__ A identity() { return (A)1; }
    __device__ static __forceinline__ V tile(V a, V b) { return jl::mul(a, b); }
    __device__ static __forceinline__ A lift(V v) { return (A)v; }
    __device__ static __forceinline__ A comb(A a, A b) { return jl::mul(a, b); }
};
template <typename V>
__device__ __forceinline__ V lowest_of() {
    if constexpr (std::is_same<V, float>::value) return -__int_as_float(0x7f800000);
    else if constexpr (std::is_same<V, double>::value) return -__longlong_as_double(0x7ff0000000000000ll);
    else if constexpr (std::is_same<V, int32_t>::value) return (int32_t)0x80000000;
    else if constexpr (std::is_same<V, uint8_t>::value) return (uint8_t)0;
    else return (long long)0x8000000000000000ll;
}
template <typename V>
__device__ __forceinline__ V highest_of() {
    if constexpr (std::is_same<V, float>::value) return __int_as_float(0x7f800000);
    else if constexpr (std::is_same<V, double>::value) return __longlong_as_double(0x7ff0000000000000ll);
    else if constexpr (std::is_same<V, int32_t>::value) return (int32_t)0x7fffffff;
    else if constexpr (std::is_same<V, uint8_t>::value) return (uint8_t)0xff;
    else return (long long)0x7fffffffffffffffll;
}
template <typename V>
struct MaxTraits {  // Julia max: NaN-propagating, +0.0 > -0.0; -Inf is a true identity under those rules
    using A = V;
    __device__ static __forceinline__ A identity() { return lowest_of<V>(); }
    __device__ static __forceinline__ V tile(V a, V b) { return jl::max(a, b); }
    __device__ static __forceinline__ A lift(V v) { return v; }
    __device__ static __forceinline__ A comb(A a, A b) { return jl::max(a, b); }
};
template <typename V>
struct MinTraits {
    using A = V;
    __device__ static __forceinline__ A identity() { return highest_of<V>(); }
    __device__ static __forceinline__ V tile(V a, V b) { return jl::min(a, b); }
    __device__ static __forceinline__ A lift(V v) { return v; }
    __device__ static __forceinline__ A comb(A a, A b) { return jl::min(a, b); }
};
// extrema(localpart) in ONE pass (reference src/mapreduce.jl:124-131): the accumulator is the (min, max) pair
template <typename T>
struct Pair {
    T lo, hi;
};
template <typename T>
struct ExtremaTraits {
    using A = Pair<T>;
    __device__ static __forceinline__ A identity() { return A{highest_of<T>(), lowest_of<T>()}; }
    __device__ static __forceinline__ A tile(A a, A b) { return A{jl::min(a.lo, b.lo), jl::max(a.hi, b.hi)}; }
    __device__ static __forceinline__ A lift(A v) { return v; }
    __device__ static __forceinline__ A comb(A a, A b) { return tile(a, b); }
};
template <typename T>
struct ExtMapF {
    using V = Pair<T>;
    T p;
    __device__ __forceinline__ V operator()(T x) const { return V{x, x}; }
};
struct CountTraits {  // V = int (0/1) ; all / any / count all reduce to "number of trues"
    using A = long long;
    __device__ static __forceinline__ A identity() { return 0; }
    __device__ static __forceinline__ int tile(int a, int b) { return a + b; }
    __device__ static __forceinline__ A lift(int v) { return (A)v; }
    __device__ static __forceinline__ A comb(A a, A b) { return a + b; }
};

// ---- map functors: T -> V -----------------------------------------------------------------------
template <typename T, int FN>
struct MapF {
    using V = T;
    T p;
    __device__ __forceinline__ V operator()(T x) const {
        if constexpr (FN == DAB_MAP_ABS) return jl::abs(x);
        else if constexpr (FN == DAB_MAP_ABS2) return jl::mul(x, x);
        else if constexpr (FN == DAB_MAP_NEG) return jl::neg(x);
        else return x;
    }
};
// y .= a.*x .+ b fused into the reduction of y (dab_affine_reduce): the mapped value is the broadcast's own AffineF, so the values the
// kernel stores and reduces are bit for bit what dab_affine writes and the identity-map reduce of y then reads.
template <typename T>
struct AffineMap {
    using V = T;
    AffineF<T> f;
    __device__ __forceinline__ V operator()(T x) const { return f(x); }
};
template <typename T, int FN>
struct PredF {
    using V = int;
    T p;
    __device__ __forceinline__ V operator()(T x) const {
        if constexpr (FN == DAB_MAP_EQ) return x == p;
        else if constexpr (FN == DAB_MAP_NE) return x != p;
        else if constexpr (FN == DAB_MAP_LT) return x < p;
        else if constexpr (FN == DAB_MAP_LE) return x <= p;
        else if constexpr (FN == DAB_MAP_GT) return x > p;
        else if constexpr (FN == DAB_MAP_GE) return x >= p;
        else if constexpr (FN == DAB_MAP_ISNAN) return x != x;
        else return x != (T)0;  // NONZERO / identity on Bool
    }
};

// ---- shuffles for 4- and 8-byte accumulators -------------------------------------------------------
template <typename A>
__device__ __forceinline__ A shfl_down(A v, int d) {
    if constexpr (sizeof(A) == 16) {
        int w[4];
        memcpy(w, &v, 16);
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = __shfl_down_sync(0xffffffffu, w[k], d);
        A r;
        memcpy(&r, w, 16);
        return r;
    } else if constexpr (sizeof(A) == 8) {
        long long x;
        memcpy(&x, &v, 8);
        int lo = __shfl_down_sync(0xffffffffu, (int)(x & 0xffffffffll), d);
        int hi = __shfl_down_sync(0xffffffffu, (int)(x >> 32), d);
        x = ((long long)hi << 32) | (unsigned int)lo;
        A r;
        memcpy(&r, &x, 8);
        return r;
    } else if constexpr (sizeof(A) == 4) {
        int x;
        memcpy(&x, &v, 4);
        x = __shfl_down_sync(0xffffffffu, x, d);
        A r;
        memcpy(&r, &x, 4);
        return r;
    } else {
        int x = (int)v;
        x = __shfl_down_sync(0xffffffffu, x, d);
        return (A)x;
    }
}

template <typename R>
__device__ __forceinline__ typename R::A block_reduce(typename R::A acc, typename R::A* smem) {
    using A = typename R::A;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc = R::comb(acc, shfl_down<A>(acc, d));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();  // smem may still be read from a previous call
    if (lane == 0) smem[warp] = acc;
    __syncthreads();
    if (warp == 0) {
        acc = lane < (RD_THREADS / 32) ? smem[lane] : R::identity();
#pragma unroll
        for (int d = 4; d > 0; d >>= 1) acc = R::comb(acc, shfl_down<A>(acc, d));
    }
    return acc;  // valid in thread 0
}


}  // namespace
