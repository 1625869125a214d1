"""ctypes binding of ``csrc/libdab200.so`` -- the executable stand-in for Julia's ``ccall`` layer.

Every signature below mirrors ``include/dab200.h`` one to one.  There is NO fallback: if the shared library is
missing this module raises at first use, and every non-zero status becomes a Python exception that mirrors the
Julia exception the reference would throw at that site (ArgumentError / DimensionMismatch / ErrorException).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "csrc", "libdab200.so")

# ---- enums (include/dab200.h) ----------------------------------------------------------------------------
OK, ERR_CUDA, ERR_ARG, ERR_EMPTY, ERR_DIM_MISMATCH, ERR_NCCL, ERR_UNSUPPORTED, ERR_NVRTC, ERR_NOMEM = range(9)
F32, F64, I32, I64, U8, I128 = range(6)     # I128: value type of dab_mapreduce_expr only
SUM, PROD, MAX, MIN, ALL, ANY, COUNT, EXTREMA = range(8)
MAP_ID, MAP_ABS, MAP_ABS2, MAP_NEG, MAP_SQRT, MAP_INV, MAP_FLOOR, MAP_CEIL, MAP_SIGN = range(9)
MAP_EQ, MAP_NE, MAP_LT, MAP_LE, MAP_GT, MAP_GE, MAP_ISNAN, MAP_NONZERO = range(16, 24)
ADD, SUB, MUL, DIV, REM, BMAX, BMIN, MOD, IDIV, AND, OR, XOR = range(12)


class DabError(RuntimeError):
    """ErrorException: a CUDA / NCCL / NVRTC failure or an op no kernel serves (never a silent host fallback)."""

    def __init__(self, status: int, msg: str):
        super().__init__(f"[dab status {status}] {msg}")
        self.status = status


class ArgumentError(DabError, ValueError):
    """Julia ``ArgumentError`` (e.g. ``sum(d, dims=0)``, reducing an empty collection with max/min)."""


class DimensionMismatch(DabError, ValueError):
    """Julia ``DimensionMismatch`` (reference src/broadcast.jl:66, src/darray.jl:564)."""


class UnsupportedError(DabError, NotImplementedError):
    """The op/dtype is not served by a kernel.  The analogue of ``allowscalar(false)`` (reference
    src/darray.jl:638-640): we raise instead of silently computing on the host."""


_EXC = {ERR_ARG: ArgumentError, ERR_EMPTY: ArgumentError, ERR_DIM_MISMATCH: DimensionMismatch, ERR_UNSUPPORTED: UnsupportedError}

_vp, _sz, _i32, _u64 = C.c_void_p, C.c_size_t, C.c_int32, C.c_uint64
_pvp = C.POINTER(C.c_void_p)
_SZ4 = C.c_size_t * 4

# name -> (restype, argtypes); status-returning unless restype given
_SIGS = {
    "dab_abi_version": (_i32, []),
    "dab_device_count": (_i32, [C.POINTER(_i32)]),
    "dab_init": (_i32, [_i32, _pvp]),
    "dab_shutdown": (_i32, [_vp]),
    "dab_last_error": (C.c_char_p, [_vp]),
    "dab_status_string": (C.c_char_p, [_i32]),
    "dab_sync": (_i32, [_vp]),
    "dab_device_info": (_i32, [_vp, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_sz), C.POINTER(_sz)]),
    "dab_stream": (_i32, [_vp, _pvp]),
    "dab_set_option": (_i32, [_vp, C.c_char_p, C.c_int64]),
    "dab_launch_count": (_i32, [_vp, C.POINTER(_u64)]),
    "dab_event_create": (_i32, [_vp, _pvp]),
    "dab_event_record": (_i32, [_vp, _vp]),
    "dab_event_elapsed_ms": (_i32, [_vp, _vp, _vp, C.POINTER(C.c_float)]),
    "dab_event_destroy": (_i32, [_vp, _vp]),
    "dab_alloc": (_i32, [_vp, _sz, _pvp]),
    "dab_free": (_i32, [_vp, _vp]),
    "dab_alloc_async": (_i32, [_vp, _sz, _pvp]),
    "dab_free_async": (_i32, [_vp, _vp]),
    "dab_host_alloc": (_i32, [_vp, _sz, _pvp]),
    "dab_host_free": (_i32, [_vp, _vp]),
    "dab_h2d": (_i32, [_vp, _vp, _vp, _sz]),
    "dab_d2h": (_i32, [_vp, _vp, _vp, _sz]),
    "dab_d2d": (_i32, [_vp, _vp, _vp, _sz]),
    "dab_h2d_2d": (_i32, [_vp, _vp, _sz, _vp, _sz, _sz, _sz]),
    "dab_d2h_2d": (_i32, [_vp, _vp, _sz, _vp, _sz, _sz, _sz]),
    "dab_fill": (_i32, [_vp, _i32, _vp, _sz, _vp]),
    "dab_rand_u01": (_i32, [_vp, _i32, _vp, _sz, _u64, _u64]),
    "dab_affine": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _sz]),
    "dab_unary": (_i32, [_vp, _i32, _i32, _vp, _vp, _sz]),
    "dab_binary": (_i32, [_vp, _i32, _i32, _vp, _vp, _vp, _sz]),
    "dab_binary_scalar": (_i32, [_vp, _i32, _i32, _vp, _vp, _vp, _i32, _sz]),
    "dab_broadcast_expr": (_i32, [_vp, C.c_char_p, _i32, _vp, C.POINTER(_sz), C.POINTER(_sz), _i32, C.POINTER(_i32), _pvp,
                                  C.POINTER(_sz), C.POINTER(_u64)]),
    "dab_jit_compile_check": (_i32, [C.c_char_p, _i32, _i32, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_sz)]),
    "dab_mapreduce_expr": (_i32, [_vp, C.c_char_p, _i32, _i32, _sz, _i32, C.POINTER(_i32), _pvp, C.POINTER(_u64), _vp]),
    "dab_jit_compile_check_reduce": (_i32, [C.c_char_p, _i32, _i32, _i32, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_sz)]),
    "dab_reduce": (_i32, [_vp, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
    "dab_reduce_host": (_i32, [_vp, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
    "dab_affine_reduce": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "dab_reduce_result_dtype": (_i32, [_i32, _i32, _i32, C.POINTER(_i32)]),
    "dab_combine_ordered": (_i32, [_i32, _i32, _vp, _sz, _vp]),
    "dab_reducedim": (_i32, [_vp, _i32, _i32, _i32, _vp, _sz, _sz, _sz, _vp, _i32]),
    "dab_copy_box": (_i32, [_vp, _i32, _vp, C.POINTER(_sz), C.POINTER(_sz), _vp, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_sz)]),
    "dab_gather_box": (_i32, [_vp, _i32, _i32, _vp, C.POINTER(C.c_longlong), _pvp, _vp, C.POINTER(C.c_longlong), _pvp, C.POINTER(_sz)]),
    "dab_gemv": (_i32, [_vp, _i32, _i32, _vp, _sz, _sz, _vp, _vp]),
    "dab_gemm": (_i32, [_vp, _i32, _i32, _sz, _sz, _sz, _vp, _sz, _vp, _sz, _vp, _sz]),
    "dab_transpose_box": (_i32, [_vp, _i32, _vp, _sz, _vp, _sz, _sz, _sz]),
    "dab_sort": (_i32, [_vp, _i32, _vp, _vp, _vp, _sz]),
    "dab_sorted_split": (_i32, [_vp, _i32, _vp, _sz, _vp, _i32, C.POINTER(C.c_ulonglong)]),
    "dab_sort_by_key": (_i32, [_vp, _i32, _vp, _i32, _vp, _vp, _vp, _sz, _sz]),
    "dab_sort_by_key_scratch_bytes": (_i32, [_i32, _sz, C.POINTER(_sz)]),
    "dab_comm_unique_id": (_i32, [_vp]),
    "dab_comm_init_rank": (_i32, [_vp, _vp, _i32, _i32]),
    "dab_comm_destroy": (_i32, [_vp]),
    "dab_allgather": (_i32, [_vp, _vp, _vp, _sz]),
    "dab_allreduce": (_i32, [_vp, _i32, _i32, _vp, _vp, _sz]),
    "dab_group_start": (_i32, [_vp]),
    "dab_group_end": (_i32, [_vp]),
    "dab_send": (_i32, [_vp, _vp, _sz, _i32]),
    "dab_recv": (_i32, [_vp, _vp, _sz, _i32]),
    "dab_mapreduce_all": (_i32, [_vp, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
    "dab_affine_mapreduce_all": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "dab_mailbox_create": (_i32, [_vp, _vp]),
    "dab_mailbox_attach": (_i32, [_vp, _vp, _i32, _i32]),
    "dab_mailbox_detach": (_i32, [_vp]),
    "dab_peer_barrier": (_i32, [_vp]),
    "dab_accumulate_stack": (_i32, [_vp, _i32, _vp, _sz, _vp, _vp, _vp, _sz, _i32]),
    "dab_ipc_get_handle": (_i32, [_vp, _vp, _vp]),
    "dab_ipc_open": (_i32, [_vp, _vp, _pvp]),
    "dab_ipc_close": (_i32, [_vp, _vp]),
    "dab_enable_peer": (_i32, [_vp, _i32]),
}

EXPORTS = tuple(_SIGS)  # every symbol include/dab200.h declares
_NO_STATUS = {"dab_abi_version", "dab_last_error", "dab_status_string"}

_lib = None


def lib() -> C.CDLL:
    """Load libdab200.so (once).  Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} is missing: the sm_100a CUDA extension has not been built "
                "(run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C distributedarrays.jl_b200/csrc`). "
                "There is no CPU fallback for the DArray hot path.")
        L = C.CDLL(SO_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        if L.dab_abi_version() != 1:
            raise RuntimeError("libdab200.so ABI version mismatch")
        _lib = L
    return _lib


def check(status: int, ctx=None) -> None:
    if status == OK:
        return
    L = lib()
    msg = L.dab_last_error(ctx) or b""
    text = msg.decode("utf-8", "replace") or (L.dab_status_string(status) or b"").decode()
    raise _EXC.get(status, DabError)(status, text)


# Contexts that hold a deferred launch (``Runtime.defer_affine``), keyed by the context's address.  Every C-ABI call on such a context
# launches the deferred op first, so the stream sees the calls in the order they were made.
_DEFERRED = {}


def ctx_key(ctx):
    return ctx.value if isinstance(ctx, C.c_void_p) else ctx


FUSED_STEP = ("dab_affine_reduce", "dab_affine_mapreduce_all")


def serves_fused_step() -> bool:
    """Whether the loaded binding has the fused broadcast + reduce entry points.  libdab200.so always has them (``lib()`` refuses a
    library that lacks a declared symbol); a stand-in object that implements only the unfused C ABI does not, and the runtime then
    launches every broadcast at once instead of deferring it."""
    L = lib()
    return all(hasattr(L, name) for name in FUSED_STEP)


def call(name: str, ctx, *args):
    """Call ``name(ctx, *args)`` and raise on a non-zero status.  A launch deferred on ``ctx`` is made first; an error it returns is
    raised here."""
    if _DEFERRED:
        owner = _DEFERRED.get(ctx_key(ctx))
        if owner is not None:
            owner.flush()
    check(getattr(lib(), name)(ctx, *args), ctx)


def sz4(v) -> C.Array:
    v = list(v) + [1] * (4 - len(v))
    return _SZ4(*v)
