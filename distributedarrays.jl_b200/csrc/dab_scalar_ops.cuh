// dab_scalar_ops.cuh -- per-element semantics of Julia Base on the hot path (SURVEY Appendix A.2/A.4):
// IEEE round-to-nearest per operation, NO FMA contraction, NaN-propagating max/min with +0.0 > -0.0,
// rem = C fmod (sign of dividend), mod = floored.  The library is additionally built with -fmad=false.
#pragma once
#include "dab_common.cuh"

namespace jl {

// ---- arithmetic, one rounding each ------------------------------------------------------
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ int32_t add(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }
__device__ __forceinline__ int32_t sub(int32_t a, int32_t b) { return (int32_t)((uint32_t)a - (uint32_t)b); }
__device__ __forceinline__ int32_t mul(int32_t a, int32_t b) { return (int32_t)((uint32_t)a * (uint32_t)b); }
__device__ __forceinline__ long long add(long long a, long long b) { return (long long)((unsigned long long)a + (unsigned long long)b); }
__device__ __forceinline__ long long sub(long long a, long long b) { return (long long)((unsigned long long)a - (unsigned long long)b); }
__device__ __forceinline__ long long mul(long long a, long long b) { return (long long)((unsigned long long)a * (unsigned long long)b); }

__device__ __forceinline__ uint8_t add(uint8_t a, uint8_t b) { return (uint8_t)(a + b); }
__device__ __forceinline__ uint8_t mul(uint8_t a, uint8_t b) { return (uint8_t)(a * b); }

// ---- max / min ----------------------------------------------------------------------------
// PTX max.NaN.f32: NaN if either input is NaN; +0.0 > -0.0 (PTX ISA "max": -0.0 < +0.0).
__device__ __forceinline__ float max(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float min(float a, float b) {
    float r;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ double max(double a, double b) {
    if (a != a || b != b) return __longlong_as_double(0x7ff8000000000000ll);
    if (a == b) return (__double_as_longlong(a) < 0) ? b : a;  // pick +0.0 over -0.0
    return a > b ? a : b;
}
__device__ __forceinline__ double min(double a, double b) {
    if (a != a || b != b) return __longlong_as_double(0x7ff8000000000000ll);
    if (a == b) return (__double_as_longlong(a) < 0) ? a : b;  // pick -0.0 over +0.0
    return a < b ? a : b;
}
__device__ __forceinline__ int32_t max(int32_t a, int32_t b) { return a > b ? a : b; }
__device__ __forceinline__ int32_t min(int32_t a, int32_t b) { return a < b ? a : b; }
__device__ __forceinline__ long long max(long long a, long long b) { return a > b ? a : b; }
__device__ __forceinline__ long long min(long long a, long long b) { return a < b ? a : b; }
__device__ __forceinline__ uint8_t max(uint8_t a, uint8_t b) { return a > b ? a : b; }
__device__ __forceinline__ uint8_t min(uint8_t a, uint8_t b) { return a < b ? a : b; }

// ---- rem / mod / integer division ---------------------------------------------------------
__device__ __forceinline__ float rem(float a, float b) { return fmodf(a, b); }
__device__ __forceinline__ double rem(double a, double b) { return fmod(a, b); }
__device__ __forceinline__ int32_t rem(int32_t a, int32_t b) { return (b == 0 || b == -1) ? 0 : a % b; }
__device__ __forceinline__ long long rem(long long a, long long b) { return (b == 0 || b == -1) ? 0 : a % b; }
template <typename T>
__device__ __forceinline__ T fmod_floor(T x, T y) {  // Julia mod(x::AbstractFloat, y)
    T r = rem(x, y);
    if (r == (T)0) return copysign(r, y);
    if ((r > (T)0) != (y > (T)0)) return add(r, y);
    return r;
}
__device__ __forceinline__ float mod(float a, float b) { return fmod_floor<float>(a, b); }
__device__ __forceinline__ double mod(double a, double b) { return fmod_floor<double>(a, b); }
template <typename T>
__device__ __forceinline__ T imod(T a, T b) {
    if (b == 0) return 0;  // Julia throws DivideError; no exceptions on device: defined as 0
    if (b == -1) return 0;
    T r = a % b;
    return (r != 0 && ((r < 0) != (b < 0))) ? r + b : r;
}
__device__ __forceinline__ int32_t mod(int32_t a, int32_t b) { return imod<int32_t>(a, b); }
__device__ __forceinline__ long long mod(long long a, long long b) { return imod<long long>(a, b); }
template <typename T>
__device__ __forceinline__ T idiv(T a, T b) {
    if (b == 0) return 0;  // DivideError in Julia
    if (b == -1) return (T)(0 - (typename std::make_unsigned<T>::type)a);
    return a / b;
}

// ---- unary ----------------------------------------------------------------------------------
__device__ __forceinline__ float abs(float a) { return fabsf(a); }
__device__ __forceinline__ double abs(double a) { return fabs(a); }
__device__ __forceinline__ int32_t abs(int32_t a) { return a < 0 ? (int32_t)(0u - (uint32_t)a) : a; }
__device__ __forceinline__ long long abs(long long a) { return a < 0 ? (long long)(0ull - (unsigned long long)a) : a; }
__device__ __forceinline__ float neg(float a) { return -a; }
__device__ __forceinline__ double neg(double a) { return -a; }
__device__ __forceinline__ int32_t neg(int32_t a) { return (int32_t)(0u - (uint32_t)a); }
__device__ __forceinline__ long long neg(long long a) { return (long long)(0ull - (unsigned long long)a); }
__device__ __forceinline__ float sqrt(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ double sqrt(double a) { return __dsqrt_rn(a); }
__device__ __forceinline__ float inv(float a) { return __fdiv_rn(1.0f, a); }
__device__ __forceinline__ double inv(double a) { return __ddiv_rn(1.0, a); }
template <typename T>
__device__ __forceinline__ T sign(T a) {  // Julia sign: keeps +-0 and NaN
    return a > (T)0 ? (T)1 : (a < (T)0 ? (T)(-1) : a);
}

}  // namespace jl

namespace {

// y = a*x + b, two roundings (Julia never contracts; src/broadcast.jl:80 runs Base's loop).  The one definition behind the broadcast
// kernel (dab_elementwise.cu) and the fused broadcast + reduce (AffineMap, dab_reduce.cu): the fused y and its reduction are therefore
// bit-identical to the broadcast followed by the reduce.
template <typename T>
struct AffineF {
    T a, b;
    __device__ __forceinline__ T operator()(T x) const { return jl::add(jl::mul(a, x), b); }
};

}  // namespace
