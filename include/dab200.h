/*
 * dab200.h -- C ABI of libdab200.so: the B200 (sm_100a) backend for the DArray
 *             map!/broadcast + mapreduce hot path of DistributedArrays.jl.
 *
 * The reference (DistributedArrays.jl v0.6.9) is pure Julia and has NO FFI / plugin
 * interface; this boundary is created at the two seams the reference already has
 * (SURVEY.md section 8b):
 *   1. the chunk-type seam  DArray{T,N,A}  (src/darray.jl:25)  -- a Julia chunk type
 *      B200Array{T,N} overloads the Base generics the hot path calls on localpart(d)
 *      and forwards them with ccall to the entry points below;
 *   2. the combine seam     reduce(op, results) (src/mapreduce.jl:34),
 *      mapreducedim_between! (src/mapreduce.jl:71-81), chunk()/setindex! slab fetch
 *      (src/darray.jl:458,798-820) -- replaced by the comm / peer entry points.
 * Every entry point cites the reference call site(s) it replaces.  Citations are relative
 * to the reference tree.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes.  Device pointers are raw CUDA device addresses
 *     (what a Julia B200Array would hold in a Ptr{Cvoid} field); host pointers are ordinary.
 *   - every function returns an int32_t status (DAB_OK == 0).  No C++ exception or sticky
 *     CUDA error crosses the ABI; dab_last_error(ctx) gives the text.
 *   - a dab_ctx is bound to ONE device and owns ONE stream.  The reference runs one
 *     single-threaded Julia process per worker (src/mapreduce.jl:6-10): one ctx per
 *     worker process.  All compute entry points are ASYNCHRONOUS on the ctx stream
 *     (== remotecall); dab_sync and the *_host variants are the sync points
 *     (== remotecall_wait / remotecall_fetch).  A ctx must not be used from two threads
 *     at once; different ctxs are independent.
 *   - arrays are column-major (Julia), element counts are size_t (8 GiB chunk = 2^31 floats).
 *   - floating-point elementwise arithmetic is IEEE round-to-nearest per operation and is
 *     NEVER contracted into FMA (Julia semantics, SURVEY Appendix A.4).
 */
#ifndef DAB200_H
#define DAB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAB_ABI_VERSION 1

typedef struct dab_ctx dab_ctx;

/* ---- status codes ------------------------------------------------------------------ */
enum {
    DAB_OK = 0,
    DAB_ERR_CUDA = 1,         /* a CUDA runtime call failed (text in dab_last_error)            */
    DAB_ERR_ARG = 2,          /* ArgumentError: bad enum / null pointer / bad dims              */
    DAB_ERR_EMPTY = 3,        /* "reducing over an empty collection is not allowed" (max/min)   */
    DAB_ERR_DIM_MISMATCH = 4, /* DimensionMismatch (src/broadcast.jl:66, src/darray.jl:564)      */
    DAB_ERR_NCCL = 5,         /* NCCL missing or a NCCL call failed                             */
    DAB_ERR_UNSUPPORTED = 6,  /* op/dtype combination not served by a kernel: NO host fallback   */
    DAB_ERR_NVRTC = 7,        /* runtime compilation of a fused broadcast expression failed      */
    DAB_ERR_NOMEM = 8
};

/* ---- element types ----------------------------------------------------------------- */
enum { DAB_F32 = 0, DAB_F64 = 1, DAB_I32 = 2, DAB_I64 = 3, DAB_U8 = 4 /* Bool */,
       DAB_I128 = 5 /* Int128: ONLY as the value type of dab_mapreduce_expr (f widens, e.g. x -> Int128(x)^2; test/darray.jl:286-294);
                       there are no arrays of it.  Its result fills the whole 16-byte slot (two's complement, little endian). */ };

/* ---- reduce operators  (op argument of Base.mapreduce; src/mapreduce.jl:31) ----------- */
enum {
    DAB_SUM = 0,   /* Base.add_sum : Int32 widens to Int64, floats stay (result dtype: f32/f64/i64) */
    DAB_PROD = 1,  /* Base.mul_prod: same widening                                               */
    DAB_MAX = 2,   /* Julia max: NaN-propagating, +0.0 > -0.0                                    */
    DAB_MIN = 3,   /* Julia min                                                                  */
    DAB_ALL = 4,   /* Base._all  (src/mapreduce.jl:97-104)  result int64 0/1                     */
    DAB_ANY = 5,   /* Base._any  (src/mapreduce.jl:106-113) result int64 0/1                     */
    DAB_COUNT = 6, /* Base.count (src/mapreduce.jl:115-122) result int64                         */
    DAB_EXTREMA = 7 /* Base.extrema (src/mapreduce.jl:124-131) in ONE pass: the result slot holds (min, max) as two T (dab_reduce
                       only, MAP_ID only; the cross-worker fold takes min of mins / max of maxes)            */
};

/* ---- map functions f of mapreduce(f, op, A) / unary broadcast ------------------------ */
enum {
    DAB_MAP_ID = 0,
    DAB_MAP_ABS = 1,
    DAB_MAP_ABS2 = 2,
    DAB_MAP_NEG = 3,
    DAB_MAP_SQRT = 4,  /* correctly rounded */
    DAB_MAP_INV = 5,   /* 1/x correctly rounded (float only) */
    DAB_MAP_FLOOR = 6,
    DAB_MAP_CEIL = 7,
    DAB_MAP_SIGN = 8,
    /* predicates against a scalar parameter p (x -> x OP p), for all/any/count; result Bool */
    DAB_MAP_EQ = 16, DAB_MAP_NE = 17, DAB_MAP_LT = 18, DAB_MAP_LE = 19, DAB_MAP_GT = 20, DAB_MAP_GE = 21,
    DAB_MAP_ISNAN = 22, DAB_MAP_NONZERO = 23 /* identity on Bool/number -> (x != 0) */
};

/* ---- binary broadcast operators ------------------------------------------------------ */
enum {
    DAB_ADD = 0, DAB_SUB = 1, DAB_MUL = 2, DAB_DIV = 3 /* float: IEEE div; int: unsupported (Julia / gives Float64) */,
    DAB_REM = 4  /* Julia rem / % : C fmod semantics (sign of dividend); ints: truncated remainder */,
    DAB_BMAX = 5, DAB_BMIN = 6,
    DAB_MOD = 7  /* Julia mod: floored */,
    DAB_IDIV = 8 /* Julia div: truncated integer quotient (ints only) */,
    DAB_AND = 9, DAB_OR = 10, DAB_XOR = 11 /* ints only */
};

/* ==== lifecycle ======================================================================= */
int32_t dab_abi_version(void);
/* number of visible CUDA devices (0 and DAB_ERR_CUDA when there is no driver). */
int32_t dab_device_count(int32_t* count);
/* One context per worker process/device.  Replaces the implicit per-process state of a Julia
 * worker (REGISTRY, src/core.jl:1-52): creates the stream and the reduction scratch. */
int32_t dab_init(int32_t device, dab_ctx** ctx);
int32_t dab_shutdown(dab_ctx* ctx);
const char* dab_last_error(const dab_ctx* ctx); /* ctx may be NULL: last error of dab_init */
const char* dab_status_string(int32_t status);
/* remotecall_wait: block until everything queued on the ctx stream is done. */
int32_t dab_sync(dab_ctx* ctx);
int32_t dab_device_info(dab_ctx* ctx, int32_t* device, int32_t* sm_count, size_t* free_bytes, size_t* total_bytes);
/* the ctx's cudaStream_t (as void*), so a host runtime can order its own work after ours. */
int32_t dab_stream(dab_ctx* ctx, void** stream);
/* tuning switches; "combine_timeout_ms" = wall-clock bound of the fused combine's wait for a peer; "ew_tma" = 1 routes aligned unary elementwise launches through the TMA-staged (cp.async.bulk + mbarrier
 * ring) kernel instead of the default flat LDG/STG kernel -- identical results, measured slower (DESIGN.md section 3). */
int32_t dab_set_option(dab_ctx* ctx, const char* key, int64_t value);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches claim). */
int32_t dab_launch_count(dab_ctx* ctx, uint64_t* launches);

/* ==== device-side timing (CUDA events on the ctx stream) ================================ */
int32_t dab_event_create(dab_ctx* ctx, void** event);
int32_t dab_event_record(dab_ctx* ctx, void* event);
int32_t dab_event_elapsed_ms(dab_ctx* ctx, void* start, void* stop, float* ms); /* syncs on stop */
int32_t dab_event_destroy(dab_ctx* ctx, void* event);

/* ==== buffers: a localpart lives in one GPU's HBM ======================================
 * Replaces Array{T}(undef, ...) on a worker (src/darray.jl:62,174,222-225).  The caller owns
 * the pointer and must dab_free it (a Julia B200Array attaches a finalizer, mirroring
 * src/darray.jl:47-49). */
int32_t dab_alloc(dab_ctx* ctx, size_t nbytes, void** dptr);
int32_t dab_free(dab_ctx* ctx, void* dptr);
/* stream-ordered temporaries (cudaMallocAsync pool; ~1 us, no synchronisation; not IPC-exportable) */
int32_t dab_alloc_async(dab_ctx* ctx, size_t nbytes, void** dptr);
int32_t dab_free_async(dab_ctx* ctx, void* dptr);
int32_t dab_host_alloc(dab_ctx* ctx, size_t nbytes, void** hptr); /* pinned staging */
int32_t dab_host_free(dab_ctx* ctx, void* hptr);
/* distribute(A) / Array(d) per chunk (src/darray.jl:544-555, 574-582): async on the ctx stream.  dab_h2d from PINNED memory is one
 * cudaMemcpyAsync; from large pageable memory it is pipelined through two pinned staging buffers (host threads fill one while the copy
 * engine drains the other) and returns once the source has been consumed, so the caller's array may be reused immediately. */
int32_t dab_h2d(dab_ctx* ctx, void* dptr, const void* hptr, size_t nbytes);
int32_t dab_d2h(dab_ctx* ctx, void* hptr, const void* dptr, size_t nbytes);
int32_t dab_d2d(dab_ctx* ctx, void* dst, const void* src, size_t nbytes);
/* 2-D strided host<->device copy of a column-major box: `cols` columns of `rows*elem` bytes
 * (distribute's A[idxs...] slicing, src/darray.jl:551).  Pitches are in bytes. */
int32_t dab_h2d_2d(dab_ctx* ctx, void* dptr, size_t dpitch, const void* hptr, size_t hpitch, size_t row_bytes, size_t cols);
int32_t dab_d2h_2d(dab_ctx* ctx, void* hptr, size_t hpitch, const void* dptr, size_t dpitch, size_t row_bytes, size_t cols);
/* fill!(localpart(A), x)  (src/darray.jl:822-827).  value points to one element of dtype. */
int32_t dab_fill(dab_ctx* ctx, int32_t dtype, void* x, size_t n, const void* value);
/* rand!(localpart(A)) (src/darray.jl:829-834) with a counter-based generator so the CPU oracle
 * can regenerate any element: x[i] = (hash32(seed, global_offset+i) >> 8) * 2^-24  in [0,1)
 * (distribution of Julia's rand(Float32)).  dtype F32 or F64. */
int32_t dab_rand_u01(dab_ctx* ctx, int32_t dtype, void* x, size_t n, uint64_t seed, uint64_t global_offset);

/* ==== elementwise kernels K1-K3 (HBM-bound, 8 B/element) ===============================
 * Replace the Base loop run on each localpart by
 *   copyto!(localpart(dest), lbc)            src/broadcast.jl:80   (y .= a .* x .+ b)
 *   copy(lbc)                                src/broadcast.jl:96   (map / allocating broadcast)
 *   map!(f, localpart(dest), makelocal(...)) src/mapreduce.jl:8    (map!(x->2x+1, d, d))
 * y may alias x exactly (in place).  a, b, s point to one host scalar of dtype. */
int32_t dab_affine(dab_ctx* ctx, int32_t dtype, void* y, const void* x, const void* a, const void* b, size_t n);
/* y = fn(x), fn from the DAB_MAP_* enum (non-predicate entries). */
int32_t dab_unary(dab_ctx* ctx, int32_t dtype, int32_t fn, void* y, const void* x, size_t n);
/* z = x OP y  (same-shape DArray .op DArray; also map_localparts binary ops src/mapreduce.jl:134-189). */
int32_t dab_binary(dab_ctx* ctx, int32_t dtype, int32_t op, void* z, const void* x, const void* y, size_t n);
/* z = x OP s (scalar_left == 0) or z = s OP x (scalar_left != 0). */
int32_t dab_binary_scalar(dab_ctx* ctx, int32_t dtype, int32_t op, void* z, const void* x, const void* s,
                          int32_t scalar_left, size_t n);
/* General fused broadcast  dest .= f.(args...)  for an arbitrary expression tree, compiled at run
 * time with NVRTC for sm_100a (what Julia's JIT does for a Broadcasted, src/broadcast.jl:65-85).
 * `expr` is C source for ONE element in terms of a0..a{nargs-1} (already converted to their
 * dtypes) and must yield a value of out_dtype, e.g. "a0 - a1 * sinf(a2)".  Each arg k is either
 * a device array (arg_ptrs[k] != NULL) indexed through arg_strides[k*4 .. k*4+3] (0 for an extruded
 * / size-1 dim, src/broadcast.jl:112-113) over the destination box shape[0..3] (column-major,
 * unused dims = 1), or a scalar passed by value through arg_scalars[k] (8 bytes each).
 * Compiled kernels are cached per (expr, dtypes, arg kinds). */
int32_t dab_broadcast_expr(dab_ctx* ctx, const char* expr, int32_t out_dtype, void* out, const size_t shape[4],
                           const size_t out_strides[4], int32_t nargs, const int32_t* arg_dtypes,
                           const void* const* arg_ptrs, const size_t* arg_strides, const uint64_t* arg_scalars);

/* Diagnostic, needs no GPU: generate + NVRTC-compile the kernels dab_broadcast_expr would use for this expression and
 * report the sm_100a cubin size (arg_is_array[k] != 0: array argument, else by-value scalar). */
int32_t dab_jit_compile_check(const char* expr, int32_t out_dtype, int32_t nargs, const int32_t* arg_dtypes,
                              const int32_t* arg_is_array, size_t* cubin_bytes);

/* Fused map + reduce of an arbitrary traced expression over one localpart, ONE pass over HBM:  mapreduce(f, op, args...)
 * (reference src/mapreduce.jl:31 with a general closure f; dot(x, y) = mapreduce(*, +, x, y); d == a via all(x .== y)).
 * expr / args as in dab_broadcast_expr but all array arguments are dense with n elements (linear indexing); val_dtype is the
 * type of the expression's value.  The 16-byte result slot at out_dev has the layout of dab_reduce (val_dtype DAB_I128, ops SUM / PROD /
 * MAX / MIN: the slot IS the Int128 result; wrap-around arithmetic like Julia's).  NVRTC-compiled, cached. */
int32_t dab_mapreduce_expr(dab_ctx* ctx, const char* expr, int32_t val_dtype, int32_t op, size_t n, int32_t nargs, const int32_t* arg_dtypes,
                           const void* const* arg_ptrs, const uint64_t* arg_scalars, void* out_dev);
int32_t dab_jit_compile_check_reduce(const char* expr, int32_t val_dtype, int32_t op, int32_t nargs, const int32_t* arg_dtypes,
                                     const int32_t* arg_is_array, size_t* cubin_bytes);

/* ==== whole-chunk reductions K4 / K7 (HBM-bound, 4 B/element) ==========================
 * Replace mapreduce(f, op, localpart(d)) / reduce(f, localpart(d)) run per worker at
 * src/mapreduce.jl:23,31 and all/any/count/extrema at :100,109,118,127.
 * The chunk result (ONE value of the result dtype: f32/f64 for float SUM/PROD, int64 for integer
 * SUM/PROD and ALL/ANY/COUNT, T for MAX/MIN) is written to out_dev, which must have room for 16 bytes:
 * [0,8) the result in its result dtype, [8,16) the wide carrier (fp64 for float SUM/PROD, else a copy).
 * Float sums are accumulated in fp32 over <=16-element groups and carried in fp64 (more accurate
 * than Base's pairwise fp32; within 1e-6 rel of it -- SURVEY 8c).  map_param: host scalar of dtype for
 * predicate maps, else NULL.  n == 0: SUM->0, PROD->1, ALL->1, ANY/COUNT->0, MAX/MIN -> DAB_ERR_EMPTY. */
int32_t dab_reduce(dab_ctx* ctx, int32_t dtype, int32_t op, int32_t map, const void* map_param, const void* x, size_t n,
                   void* out_dev);
/* Same, then copies the 16-byte result slot to out_host and syncs (== remotecall_fetch, src/mapreduce.jl:31). */
int32_t dab_reduce_host(dab_ctx* ctx, int32_t dtype, int32_t op, int32_t map, const void* map_param, const void* x,
                        size_t n, void* out_host);
/* y .= a .* x .+ b (dab_affine) followed by dab_reduce(op, DAB_MAP_ID) of y into out_dev, same arguments, same results bit for bit.
 * Float32 / Float64, op SUM / PROD / MAX / MIN, n > 0 and x, y at the same offset mod 16 (y == x included): ONE kernel reads x, writes
 * y and reduces the values it has just computed -- 8 instead of 12 bytes per Float32 element.  Any other case runs the two calls. */
int32_t dab_affine_reduce(dab_ctx* ctx, int32_t dtype, void* y, const void* x, const void* a, const void* b, size_t n, int32_t op,
                          void* out_dev);
/* result dtype of dab_reduce for (dtype, op, map). */
int32_t dab_reduce_result_dtype(int32_t dtype, int32_t op, int32_t map, int32_t* out_dtype);
/* Caller-side combine  reduce(op, results)  (src/mapreduce.jl:26,34): P < 16 so a plain LEFT FOLD in
 * procs(d) order, in the result dtype (Float32 partials fold in Float32).  Host arrays. */
int32_t dab_combine_ordered(int32_t result_dtype, int32_t op, const void* partials_host, size_t p, void* out_host);

/* ==== dimensional reduction K5 / K6 =====================================================
 * Replaces mapreduce(f, op, localpart(A), dims=region) (src/mapreduce.jl:64, phase 1) and
 * Base.mapreducedim!(f, op, localpart(R), B) (src/mapreduce.jl:77, phase 2) on the chunk collapsed to
 * the column-major shape (inner, reduce, outer): out[i + inner*o] (op)= x[i + inner*(r + reduce*o)].
 * accumulate == 0: out is overwritten with the reduction (SUM/PROD seeded with 0/1, MAX/MIN with
 * the first element); accumulate != 0: the reduction is combined ONTO the existing out
 * (how init= and the between-phase enter, SURVEY Appendix A.3).  Output dtype follows
 * dab_reduce_result_dtype. */
int32_t dab_reducedim(dab_ctx* ctx, int32_t dtype, int32_t op, int32_t map, const void* x, size_t inner, size_t reduce,
                      size_t outer, void* out, int32_t accumulate);

/* ==== slab / halo copy K8 ===============================================================
 * Replaces the owner-side  localpart(d)[idxs...]  + serialise + TCP + a[idxs...] = ...  of
 * setindex!(::Array, ::SubDArray, ...) (src/darray.jl:798-820), chunk() (:458) and the non-local
 * branch of makelocal (:361-366).  Copies a box of `extent` elements (up to 4 dims, column-major)
 * from src (array shape src_shape, box origin src_off, 0-based) to dst.  src may be a pointer into
 * ANOTHER GPU's memory (peer-enabled in-process, or opened with dab_ipc_open): the copy kernel
 * then pulls over NVLink with 16-byte loads -- one-sided, like the reference's pull-style read. */
int32_t dab_copy_box(dab_ctx* ctx, int32_t elem_bytes, void* dst, const size_t dst_shape[4], const size_t dst_off[4],
                     const void* src, const size_t src_shape[4], const size_t src_off[4], const size_t extent[4]);

/* Strided and vector-indexed views: the piece of Array(d[I...]) held by one chunk when some index is a StepRange or a Vector{Int}
 * (src/darray.jl:661, 798-820; indexin_mask / restrict_indices :706-781).  ndim <= 8.  Coordinate t of dimension k contributes
 * t * dst_strides[k] (resp. src_strides[k], may be negative) ELEMENTS to the destination (source) offset, or, when dst_index[k]
 * (src_index[k]) is non-NULL, the value table[k][t] of a device array of int64 element offsets.  dst / src point at the element of
 * coordinate 0; src may be a peer mapping.  dst_index / src_index may be NULL (all affine). */
int32_t dab_gather_box(dab_ctx* ctx, int32_t elem_bytes, int32_t ndim, void* dst, const long long* dst_strides, const void* const* dst_index,
                       const void* src, const long long* src_strides, const void* const* src_index, const size_t* extent);

/* ==== Level-2 linear algebra K9 (widening row f4; HBM-bound) ==============================
 * r = op(A) * x on ONE column-major chunk A (m x n, leading dimension m): trans = 0 -> r[m] = A x[n];
 * trans = 1 -> r[n] = A' x[m].  Replaces  localpart(A)*convert(localtype(x), xj)  (src/linalg.jl:95-97)
 * and  localpart(A)'*...  (:141) inside mul!(y::DVector, A::DMatrix, x, a, b); the tile results are then
 * combined into y by the caller exactly as the reference does (scale y by b, add a*R[i,j] in j order,
 * :101-117).  Float products accumulate in fp64 and round once; Int32/Int64 wrap.  dtypes: F32 F64 I32 I64. */
int32_t dab_gemv(dab_ctx* ctx, int32_t dtype, int32_t trans, const void* A, size_t m, size_t n, const void* x, void* r);

/* ==== Level-3 tile product K12 (widening row f4; the one contraction on the path: tensor-core roofline) =====================
 * R[m x n] (ldc) = op(A) * B on column-major operands of ONE worker: transA = 0 -> A is m x k (lda); transA = 1 -> op(A) = A^T with A
 * stored k x m (lda); B is k x n (ldb).  Replaces  localpart(A) * convert(localtype(B), Bjk)  and the transpose / adjoint forms of
 * _matmatmul! (src/linalg.jl:218-226); the caller scales C by beta and adds alpha * R per tile exactly as the reference (:232-252).
 * Float32 with 16-byte aligned bases and leading dimensions: TMA-fed tcgen05 (3xTF32 error-compensated, TMEM accumulators drained
 * every "gemm_kc" k for fp32 round-to-nearest accumulation); otherwise and for Float64 / Int32 / Int64: shared-memory tiled FMA kernel
 * (integers wrap like Julia's).  n == 1 with a dense A (lda == its row count) IS a matrix-vector product and is served by K9
 * (dab_gemv: one read of A at the HBM roofline).  R is overwritten. */
int32_t dab_gemm(dab_ctx* ctx, int32_t dtype, int32_t transA, size_t m, size_t n, size_t k, const void* A, size_t lda, const void* B,
                 size_t ldb, void* C, size_t ldc);

/* dst[j + i*dst_ld] = src[i + j*src_ld] for i < rows, j < cols (both column-major): the per-piece body of
 * copy(::Transpose/Adjoint{T,<:DArray{T,2}}) (src/linalg.jl:1-17: transpose!(lp, Array(D[reverse(I)...]))).
 * src may be a PEER pointer: rows are pulled coalesced over NVLink and written coalesced locally through a
 * shared-memory tile, so the fetched block is never materialised untransposed.  elem_bytes in {1,2,4,8,16}. */
int32_t dab_transpose_box(dab_ctx* ctx, int32_t elem_bytes, void* dst, size_t dst_ld, const void* src, size_t src_ld, size_t rows,
                          size_t cols);

/* ==== sort K11 (widening row f4; HBM-bound integer work) ===================================
 * out = sort(in) for one chunk: the  sort(lp; kwargs...)  of sample_n_setup_ref (src/sort.jl:8) and the
 * sort!(lp_sorting)  of scatter_n_sort_localparts (:61).  Ascending in Julia's isless order (-0.0 < 0.0,
 * NaNs last, bit patterns preserved).  LSD radix sort, 8-bit digits; passes whose digit is constant over
 * the chunk are skipped.  tmp: scratch of n elements, distinct from in/out (may be NULL when n <= 1024 and
 * in != out); in == out sorts in place.  Asynchronous on the ctx stream (histograms, pass selection and buffer
 * ping-pong are planned on the device).  dtypes: F32 F64 I32 I64. */
int32_t dab_sort(dab_ctx* ctx, int32_t dtype, const void* in, void* out, void* tmp, size_t n);

/* vals_out = vals reordered by the STABLE ascending order of keys: the  sort(lp; by = f)  /  sort!(lp_sorting; by = f)  of the
 * samplesort with a key function (src/sort.jl:8, 22, 61; `by` is accepted at :111) once the caller has evaluated keys = f.(lp)
 * (dab_broadcast_expr).  Key order is Julia's isless (-0.0 < 0.0; NaN keys last and equal to each other), elements with equal keys
 * keep their input order (Julia's default algorithm for a keyed sort is stable).  A 32-bit radix key and the element's position are
 * packed into one Int64 word per element and sorted by dab_sort (two rounds, least-significant half first, for 64-bit keys); the
 * low halves of the sorted words are the permutation applied to vals.  key dtypes F32 F64 I32 I64; val_bytes 4 or 8; n < 2^32;
 * vals_out must not alias vals.  scratch: device memory of at least dab_sort_by_key_scratch_bytes() bytes, 16-byte aligned.
 * Asynchronous on the ctx stream. */
int32_t dab_sort_by_key(dab_ctx* ctx, int32_t key_dtype, const void* keys, int32_t val_bytes, const void* vals, void* vals_out,
                        void* scratch, size_t scratch_bytes, size_t n);
int32_t dab_sort_by_key_scratch_bytes(int32_t key_dtype, size_t n, size_t* bytes);

/* Split points of a sorted chunk for the boundaries of the samplesort (src/sort.jl:28-40): for each of the
 * nb (<= 256) host values bounds[i] (dtype elements), counts_host[i] = the number of leading elements the
 * reference's scan would pass before the first x > bounds[i] had it started at element 1 -- the count of
 * non-NaN elements <= bounds[i], or n when nothing exceeds the bound (NaNs compare false and stay).
 * Synchronous (returns with counts_host filled). */
int32_t dab_sorted_split(dab_ctx* ctx, int32_t dtype, const void* sorted, size_t n, const void* bounds_host, int32_t nb,
                         unsigned long long* counts_host);

/* ==== cross-worker combine: NCCL over NVLink (replaces Distributed.remotecall_fetch on
 *      this path only; src/mapreduce.jl:30-34, 72-80; src/darray.jl:809-815) ============== */
/* 128-byte ncclUniqueId; rank 0 creates it, the host runtime ships it to the other workers. */
int32_t dab_comm_unique_id(void* id128);
int32_t dab_comm_init_rank(dab_ctx* ctx, const void* id128, int32_t rank, int32_t nranks);
int32_t dab_comm_destroy(dab_ctx* ctx);
/* asyncmap(procs(d)) do p; remotecall_fetch(...) end  -> every rank gets all P partials (device). */
int32_t dab_allgather(dab_ctx* ctx, const void* send_dev, void* recv_dev, size_t nbytes_per_rank);
int32_t dab_allreduce(dab_ctx* ctx, int32_t dtype, int32_t op, const void* send_dev, void* recv_dev, size_t count);
/* point-to-point slab / partial-vector transfer inside a group (mapreducedim_between!, halo). */
int32_t dab_group_start(dab_ctx* ctx);
int32_t dab_group_end(dab_ctx* ctx);
int32_t dab_send(dab_ctx* ctx, const void* send_dev, size_t nbytes, int32_t peer);
int32_t dab_recv(dab_ctx* ctx, void* recv_dev, size_t nbytes, int32_t peer);
/* sum(d) in one call: chunk reduce (dab_reduce) -> allgather of the P chunk results -> ordered left
 * fold (dab_combine_ordered) -> host scalar.  Exactly src/mapreduce.jl:29-35. */
int32_t dab_mapreduce_all(dab_ctx* ctx, int32_t dtype, int32_t op, int32_t map, const void* map_param, const void* x,
                          size_t n, void* out_host);
/* y .= a .* x .+ b (dab_affine) followed by dab_mapreduce_all(op, DAB_MAP_ID) of y: the chunk reduce is dab_affine_reduce (one
 * kernel when it fuses), the cross-worker combine is that of dab_mapreduce_all (fused peer combine, or the NCCL all-gather). */
int32_t dab_affine_mapreduce_all(dab_ctx* ctx, int32_t dtype, void* y, const void* x, const void* a, const void* b, size_t n, int32_t op,
                                 void* out_host);

/* Fused reduce + combine over NVLink peer memory.  After every rank has created its mailbox (dab_mailbox_create returns the
 * 64-byte CUDA IPC handle), exchanged the handles through the host runtime and attached them (handles = nranks * 64 bytes, in
 * rank order), dab_mapreduce_all runs as ONE kernel: the last CTA of the chunk reduction pushes the chunk result into every
 * peer's mailbox with peer stores, waits for the P results, folds them left to right in rank order and writes the scalar into
 * pinned host memory -- no NCCL call, no D2H copy.  A rank that never calls makes the others time out (wall clock, default 120 s, dab_set_option "combine_timeout_ms") with DAB_ERR_NCCL
 * instead of hanging the GPU.  All ranks must call dab_mapreduce_all in the same order (as with any collective). */
int32_t dab_mailbox_create(dab_ctx* ctx, void* handle64);
int32_t dab_mailbox_attach(dab_ctx* ctx, const void* handles, int32_t rank, int32_t nranks);
int32_t dab_mailbox_detach(dab_ctx* ctx);

/* Device-side barrier across the ranks, ordered on the ctx stream (needs the mailboxes above; a no-op for one rank): kernels queued
 * after it start only when every rank's kernels queued before ITS call have completed.  The fence around one-sided peer reads / writes
 * (the remotecall_wait of the reference) without a host synchronisation or an NCCL launch; a peer that never arrives surfaces as
 * DAB_ERR_NCCL at the next dab_sync after "combine_timeout_ms". */
int32_t dab_peer_barrier(dab_ctx* ctx);
/* y = beta*y (fill!(0) when *beta == 0, untouched when 1), then y += alpha * stack[j*stride .. +n) for j = 0..count-1 in order, every
 * multiply and add rounded separately: rmul!/fill! + add!(localpart(y), R[i,j], alpha) of mul! (src/linalg.jl:101-117, 62-76; also the
 * between-phase of a sum over slabs) in one launch.  alpha, beta: host scalars of dtype (F32 F64 I32 I64). */
int32_t dab_accumulate_stack(dab_ctx* ctx, int32_t dtype, void* y, size_t n, const void* beta, const void* alpha, const void* stack,
                             size_t stride, int32_t count);

/* ==== peer memory (one process per GPU): CUDA IPC handles, shipped by the host runtime ==== */
int32_t dab_ipc_get_handle(dab_ctx* ctx, const void* dptr, void* handle64);
int32_t dab_ipc_open(dab_ctx* ctx, const void* handle64, void** dptr);
int32_t dab_ipc_close(dab_ctx* ctx, void* dptr);
/* in-process multi-GPU: enable peer access from ctx's device to `peer_device`. */
int32_t dab_enable_peer(dab_ctx* ctx, int32_t peer_device);

#ifdef __cplusplus
}
#endif
#endif /* DAB200_H */
