"""Distributed reductions: the reference's ``src/mapreduce.jl:17-131`` on B200.

  * ``reduce`` / ``mapreduce`` / ``sum`` / ``prod`` / ``maximum`` / ``minimum``  -- ``Base._mapreduce(f, op, ::IndexCartesian,
    d::DArray)`` (reference src/mapreduce.jl:29-35): ONE streaming kernel per localpart, the P chunk results are gathered on
    every rank (NCCL all-gather over NVLink instead of ``remotecall_fetch``), then folded LEFT TO RIGHT in ``procs(d)`` order
    in the result type -- exactly ``reduce(op, results)`` (:34).
  * ``mapreduce(...; dims)`` -- ``reducedim_initarray`` (:42-51), ``mapreducedim_within`` (:54-66),
    ``mapreducedim_between!`` (:71-81), ``mapreducedim!`` (:83-94): every worker reduces its chunk along ``region``; the
    owners of R (grid index 1 along the reduced dims, :44) receive the partial slabs of their fibre (grouped NCCL
    send/recv) and accumulate them, in grid order, onto R.
  * ``all`` / ``any`` / ``count`` / ``extrema`` (:97-131).
"""
from __future__ import annotations

import builtins
import ctypes as C
import operator
from typing import Callable, Dict, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._broadcast import Expr, broadcast, tag_of, trace, _NPT
from ._darray import B200Array, DArray, dab_dtype, np_dtype
from .layout import Layout, collapse_for_region, ravel, shape_of, unravel

_OPS = {"+": _lib.SUM, "add": _lib.SUM, "sum": _lib.SUM, "*": _lib.PROD, "mul": _lib.PROD, "prod": _lib.PROD, "max": _lib.MAX,
        "min": _lib.MIN}
_OPF = {operator.add: _lib.SUM, operator.mul: _lib.PROD, builtins.max: _lib.MAX, builtins.min: _lib.MIN, np.add: _lib.SUM,
        np.multiply: _lib.PROD, np.maximum: _lib.MAX, np.minimum: _lib.MIN}


def _op_code(op) -> int:
    if isinstance(op, str) and op in _OPS:
        return _OPS[op]
    if op in _OPF:
        return _OPF[op]
    raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, f"reduction operator {op!r} is not served by a kernel (no host fallback)")


_CMPMAP = {"eq": _lib.MAP_EQ, "ne": _lib.MAP_NE, "lt": _lib.MAP_LT, "le": _lib.MAP_LE, "gt": _lib.MAP_GT, "ge": _lib.MAP_GE}
_FLIP = {"lt": "gt", "le": "ge", "gt": "lt", "ge": "le", "eq": "eq", "ne": "ne"}


def classify_map(f: Optional[Callable], dtype) -> Tuple[Optional[int], Optional[np.ndarray], Optional[Expr]]:
    """f -> (DAB_MAP_* code, predicate parameter, traced expr).  code is None when f needs the general (two-pass) path."""
    if f is None:
        return _lib.MAP_ID, None, None
    tag = tag_of(dtype)
    e = trace(f, [tag])
    if e.op == "arg":
        return _lib.MAP_ID, None, e
    if e.jt == tag and len(e.args) == 1 and e.args[0].op == "arg":
        code = {"abs": _lib.MAP_ABS, "abs2": _lib.MAP_ABS2, "neg": _lib.MAP_NEG}.get(e.op)
        if code is not None:
            return code, None, e
    if e.op == "mul" and e.jt == tag and builtins.all(a.op == "arg" for a in e.args):  # x*x == abs2 for reals
        return _lib.MAP_ABS2, None, e
    if e.op in _CMPMAP:
        l, r = e.args

        def unpromote(side, const):
            """``x > 0.5`` with x::Float32 promotes x to Float64 (Julia); when the Float64 constant is exactly representable in
            x's type the comparison is equivalent in that type, and the predicate kernel can run on the raw chunk."""
            if side.op == "convert" and side.args[0].op == "arg" and side.args[0].jt == tag and const.op == "const":
                c = const.val
                if tag == "f32" and const.jt == "f64" and float(np.float32(c)) == c:
                    return side.args[0], Expr("const", (), tag, c)
                if tag in ("i32", "i64") and const.jt in ("i64",) and side.jt == "i64":
                    return side.args[0], Expr("const", (), tag, c) if -2**31 <= c < 2**31 or tag == "i64" else (side, const)
            return side, const

        l, r = unpromote(l, r)
        r, l = unpromote(r, l)
        if l.op == "arg" and r.op == "const" and l.jt == tag:
            return _CMPMAP[e.op], np.asarray(r.val, dtype=np.dtype(dtype)), e
        if r.op == "arg" and l.op == "const" and r.jt == tag:
            return _CMPMAP[_FLIP[e.op]], np.asarray(l.val, dtype=np.dtype(dtype)), e
    if e.op == "isnan" and e.args[0].op == "arg":
        return _lib.MAP_ISNAN, None, e
    return None, None, e


def _result_dtype(dtype, op: int, mapc: int) -> np.dtype:
    out = C.c_int32()
    _lib.check(_lib.lib().dab_reduce_result_dtype(dab_dtype(dtype), op, mapc, C.byref(out)))
    return np.dtype(np.int64) if out.value == _lib.I64 else np_dtype(out.value)


# ---- whole-array reductions ------------------------------------------------------------------------------------------------


def _gather_slots(d: DArray, launch: Callable[[int, B200Array, int], None]) -> np.ndarray:
    """Run ``launch(pid, chunk, slot_ptr)`` (one reduce kernel writing a 16-byte result slot) for every local chunk, then make
    the slots of ALL workers visible on every rank: bytes, 16 per worker, in worker order."""
    rt = d.rt
    wpr = rt.workers_per_rank
    slots = B200Array.empty(rt, (16 * wpr,), np.uint8, temp=True)
    try:
        for pid, ch in d.chunks.items():
            launch(pid, ch, slots.ptr + 16 * ((pid - 1) % wpr))
        if rt.world > 1:
            allslots = B200Array.empty(rt, (16 * wpr * rt.world,), np.uint8, temp=True)
            _lib.call("dab_allgather", rt.ctx, C.c_void_p(slots.ptr), C.c_void_p(allslots.ptr), 16 * wpr)
            host = allslots.to_numpy()
            allslots.free()
        else:
            host = slots.to_numpy()
    finally:
        rt.sync()
        slots.free()
    return host.view(np.uint8)


def _fold(host: np.ndarray, pids: Sequence[int], rdt: np.dtype, op: int):
    """``reduce(op, results)`` (src/mapreduce.jl:34): left fold in procs(d) order, in the result type."""
    vals = np.empty(len(pids), dtype=rdt)
    for i, pid in enumerate(pids):
        vals[i] = host[16 * (pid - 1):16 * (pid - 1) + rdt.itemsize].view(rdt)[0]
    out = np.zeros(1, dtype=rdt)
    rcode = _lib.I64 if rdt == np.dtype(np.int64) else dab_dtype(rdt)
    _lib.check(_lib.lib().dab_combine_ordered(rcode, op, C.c_void_p(vals.ctypes.data), len(pids), C.c_void_p(out.ctypes.data)))
    return out[0], vals


def _int128(b: bytes) -> int:
    return int.from_bytes(b, "little", signed=True)


def wrap128(v: int) -> int:
    """Two's-complement wrap-around of Int128 machine arithmetic."""
    v &= (1 << 128) - 1
    return v - (1 << 128) if v >> 127 else v


def fold128(vals: Sequence[int], op: int) -> int:
    """``reduce(op, results)`` (src/mapreduce.jl:34) for Int128 chunk results: left fold in procs(d) order, wrapping like Julia."""
    acc = vals[0]
    for v in vals[1:]:
        acc = wrap128(acc + v) if op == _lib.SUM else wrap128(acc * v) if op == _lib.PROD else (max(acc, v) if op == _lib.MAX else min(acc, v))
    return acc


def _check_nonempty(d: DArray, opc: int):
    if opc in (_lib.MAX, _lib.MIN):
        for pid in d.layout.pids:
            if int(np.prod(shape_of(d.layout.localindices(pid)))) == 0:
                raise _lib.ArgumentError(_lib.ERR_EMPTY, "reducing over an empty collection is not allowed")


def _empty_slot(rt, opc: int, rdt: np.dtype, slot_ptr: int):
    """An empty localpart contributes the identity (Base: sum -> 0, prod -> 1, all -> true, any/count -> 0)."""
    v = np.zeros(2, dtype=np.uint64)
    one = {_lib.PROD: 1, _lib.ALL: 1}.get(opc, 0)
    v.view(np.uint8)[:rdt.itemsize] = np.asarray([one], dtype=rdt).view(np.uint8)
    _lib.call("dab_h2d", rt.ctx, C.c_void_p(slot_ptr), C.c_void_p(v.ctypes.data), 16)
    rt.sync()


def _mapreduce_expr(expr: Expr, opc: int, d: DArray, others: Sequence, return_partials: bool = False):
    """General ``mapreduce(f, op, d, others...)``: f is an arbitrary traced expression over 1..8 arguments.  ONE fused NVRTC
    kernel per localpart (``dab_mapreduce_expr``), no temporary f.(d) array; combine as in ``_mapreduce_all``."""
    from ._broadcast import _NPT as NPT, _localise, _prepare_remote_reads, codegen
    rt = d.rt
    args = [d] + list(others)
    for a in others:
        if isinstance(a, DArray) and a.dims != d.dims:
            raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"mapreduce arguments differ in size: {d.dims} vs {a.dims}")
        if isinstance(a, np.ndarray) and a.ndim > 0 and tuple(a.shape) != d.dims:
            raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"mapreduce arguments differ in size: {d.dims} vs {a.shape}")
    if len(args) > 8:
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "more than 8 mapreduce arguments are not served")
    _check_nonempty(d, opc)
    val_tag = expr.jt
    wide = val_tag == "i128"                     # Int128 VALUES (f widens its argument): the 16-byte slot is the result
    if wide and opc not in (_lib.SUM, _lib.PROD, _lib.MAX, _lib.MIN):
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "Int128 values are reduced with + * max min only")
    val_code = _lib.I128 if wide else dab_dtype(NPT[val_tag])
    if val_tag == "bool" and opc == _lib.SUM:
        opc_k = _lib.COUNT                       # sum of Bools == count (Int64)
    else:
        opc_k = opc
    if wide:
        rdt = np.dtype((np.void, 16))            # raw slot bytes; decoded to Python ints below
    else:
        rdt = np.dtype(np.int64) if val_tag in ("bool", "i32", "i64") and opc in (_lib.SUM, _lib.PROD, _lib.ALL, _lib.ANY, _lib.COUNT) else NPT[val_tag]
    src = codegen(expr).encode()
    from ._broadcast import _finish_remote_reads
    remote = _prepare_remote_reads(d.layout, rt, [a for a in others if isinstance(a, DArray)])
    temps = []

    def launch(pid, ch, slot_ptr):
        if ch.size == 0:
            return _empty_slot(rt, opc, np.dtype(np.int64) if wide else rdt, slot_ptr)   # 0 / 1 zero-extended = the Int128 identity
        I = d.layout.localindices(pid)
        largs = [_localise(rt, a, I, pid) for a in args]
        n = len(largs)
        dts = (C.c_int32 * n)(*[dab_dtype(NPT[la.tag]) for la in largs])
        ptrs = (C.c_void_p * n)(*[la.arr.ptr if la.arr is not None else None for la in largs])
        scal = (C.c_uint64 * n)()
        for k, la in enumerate(largs):
            if la.arr is None:
                scal[k] = int.from_bytes(np.asarray(la.scalar, dtype=NPT[la.tag]).tobytes().ljust(8, b"\0"), "little")
            elif la.temp:
                temps.append(la.arr)
        _lib.call("dab_mapreduce_expr", rt.ctx, src, val_code, opc_k, ch.size, n, dts, ptrs, scal, C.c_void_p(slot_ptr))

    try:
        host = _gather_slots(d, launch)
    finally:
        for t in temps:
            t.free()
        _finish_remote_reads(rt, remote)
    if wide:
        vals = [_int128(host[16 * (pid - 1):16 * pid].tobytes()) for pid in d.layout.pids]
        res = fold128(vals, opc)
        return (res, vals) if return_partials else res
    res, vals = _fold(host, d.layout.pids, rdt, opc if opc != _lib.COUNT else _lib.SUM)
    return (res, vals) if return_partials else res


_FUSED_OPS = (_lib.SUM, _lib.PROD, _lib.MAX, _lib.MIN)    # the reductions dab_affine_reduce serves


def _mapreduce_all(f, op, d: DArray, return_partials: bool = False, others: Sequence = ()):
    opc = op if isinstance(op, int) else _op_code(op)
    if others:
        expr = trace(f, [tag_of(d.dtype)] + [_arg_tag_of(a) for a in others])
        return _mapreduce_expr(expr, opc, d, others, return_partials)
    mapc, param, expr = classify_map(f, d.dtype)
    if mapc is None:
        return _mapreduce_expr(expr, opc, d, (), return_partials)   # general closure: one fused NVRTC kernel per chunk
    _check_nonempty(d, opc)
    rt = d.rt
    pp = C.c_void_p(param.ctypes.data) if param is not None else None
    rdt = _result_dtype(d.dtype, opc, mapc)
    code = dab_dtype(d.dtype)
    fusable = mapc == _lib.MAP_ID and opc in _FUSED_OPS and code in (_lib.F32, _lib.F64) and rt.pending is not None

    def take_pending(ch):
        """The deferred ``y .= a.*x .+ b`` when it writes exactly this chunk: the reduce then runs fused with it."""
        return rt.take_pending(code, ch.ptr, ch.size) if fusable else None

    if rt.workers_per_rank == 1 and d.layout.pids == rt.workers() and not return_partials:
        # production mapping, one chunk per GPU: reduce kernel + cross-worker combine + ordered fold in ONE C-ABI call
        ch = d.chunks[rt.myid()]
        out = np.zeros(2, dtype=np.uint64)
        p = take_pending(ch)
        if p is not None:
            _lib.call("dab_affine_mapreduce_all", rt.ctx, code, C.c_void_p(p.y), C.c_void_p(p.x), C.c_void_p(p.a.ctypes.data),
                      C.c_void_p(p.b.ctypes.data), p.n, opc, C.c_void_p(out.ctypes.data))
        else:
            _lib.call("dab_mapreduce_all", rt.ctx, code, opc, mapc, pp, C.c_void_p(ch.ptr), ch.size, C.c_void_p(out.ctypes.data))
        return out.view(np.uint8)[:rdt.itemsize].view(rdt)[0]
    # the deferred broadcast can only have written one local chunk: take it out now (the slot allocation below is a C-ABI call, which
    # would launch it) and run that chunk's reduce fused with it.  The reduces of the other chunks neither read nor write its x or y.
    p = next((q for q in map(take_pending, d.chunks.values()) if q is not None), None) if fusable else None

    def launch(pid, ch, slot):
        nonlocal p
        if p is not None and (p.y, p.n) == (ch.ptr, ch.size):
            q, p = p, None
            _lib.call("dab_affine_reduce", rt.ctx, code, C.c_void_p(q.y), C.c_void_p(q.x), C.c_void_p(q.a.ctypes.data),
                      C.c_void_p(q.b.ctypes.data), q.n, opc, C.c_void_p(slot))
        else:
            _lib.call("dab_reduce", rt.ctx, code, opc, mapc, pp, C.c_void_p(ch.ptr), ch.size, C.c_void_p(slot))

    try:
        host = _gather_slots(d, launch)
    finally:
        if p is not None:                                   # not reached (an error came first): it stays the pending op
            rt.defer_affine(p.dtype, p.y, p.x, p.a, p.b, p.n)
    res, vals = _fold(host, d.layout.pids, rdt, opc)
    return (res, vals) if return_partials else res


def _arg_tag_of(a) -> str:
    from ._broadcast import _arg_tag
    return _arg_tag(a)


def reduce(op, d: DArray, dims=None, init=None):
    """``reduce(f, d::DArray)`` (reference src/mapreduce.jl:17-27); with ``dims`` the dimensional form."""
    return mapreduce(None, op, d, dims=dims, init=init)


def mapreduce(f: Optional[Callable], op, d: DArray, *ds, dims=None, init=None, _partials: bool = False):
    """``mapreduce(f, op, d::DArray, ds...[; dims, init])`` (reference src/mapreduce.jl:29-35 and :42-94).  With extra arguments
    (same-size DArrays / arrays / scalars) ``f`` takes one value per argument: ``mapreduce(*, +, x, y)`` is ``dot(x, y)``.
    A ``SubDArray`` is reduced through ``DArray(d)`` exactly as the reference does (src/mapreduce.jl:36)."""
    from ._darray import SubDArray
    if isinstance(d, SubDArray):
        tmp = d.to_darray()
        try:
            return mapreduce(f, op, tmp, *ds, dims=dims, init=init, _partials=_partials)
        finally:
            if dims is None:
                tmp.close()
    if dims is None:
        if init is not None:
            raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "mapreduce(f, op, d; init) without dims falls back to scalar iteration in the reference; not served")
        return _mapreduce_all(f, op, d, _partials, ds)
    if ds:
        # Base: mapreduce(f, op, A, B...; dims) = reduce(op, map(f, A, B...); dims) -- map gives a DArray (src/mapreduce.jl:3), reduce
        # with dims the dimensional form (:42-94); the temporary is released once R has been launched
        tmp = broadcast(f, d, *ds)
        try:
            return mapreducedim(None, op, tmp, dims, init)
        finally:
            tmp.close()
    return mapreducedim(f, op, d, dims, init)


def sum(d: DArray, f: Optional[Callable] = None, dims=None):  # noqa: A001 - mirrors Base.sum
    return mapreduce(f, "+", d, dims=dims)


def prod(d: DArray, f: Optional[Callable] = None, dims=None):
    return mapreduce(f, "*", d, dims=dims)


def maximum(d: DArray, f: Optional[Callable] = None, dims=None):
    return mapreduce(f, "max", d, dims=dims)


def minimum(d: DArray, f: Optional[Callable] = None, dims=None):
    return mapreduce(f, "min", d, dims=dims)


def _pred_reduce(opc: int, d: DArray, f: Optional[Callable]):
    from ._darray import SubDArray
    if isinstance(d, SubDArray):
        tmp = d.to_darray()
        try:
            return _pred_reduce(opc, tmp, f)
        finally:
            tmp.close()
    if f is None:
        if d.dtype != np.dtype(np.bool_):
            raise TypeError("TypeError: non-boolean used in boolean context")
        return _mapreduce_all(None, opc, d)
    mapc, param, e = classify_map(f, d.dtype)
    if e is not None and e.jt != "bool":
        raise TypeError("TypeError: non-boolean used in boolean context")
    return _mapreduce_all(f, opc, d)


def _count_dims(d: DArray, f: Optional[Callable], dims) -> Tuple[DArray, int]:
    """``count(f, d; dims)`` as a DArray of Int64 plus the number of elements behind each entry.  Base sends the dimensional forms of
    all / any / count through ``mapreduce(f, op, A; dims)``, i.e. through the reference's ``mapreducedim!`` (src/mapreduce.jl:83-94); here
    the predicate is mapped to 0 / 1 in one elementwise launch and summed by the dimensional reduction kernels."""
    from ._broadcast import ifelse
    from ._darray import SubDArray
    if isinstance(d, SubDArray):
        tmp = d.to_darray()
        try:
            return _count_dims(tmp, f, dims)
        finally:
            tmp.close()
    if f is None and d.dtype != np.dtype(np.bool_):
        raise TypeError("TypeError: non-boolean used in boolean context")
    pred = (lambda x: x) if f is None else f
    e = trace(pred, [tag_of(d.dtype)])
    if e.jt != "bool":
        raise TypeError("TypeError: non-boolean used in boolean context")
    ones = broadcast(lambda x: ifelse(pred(x), 1, 0), d)
    try:
        r = mapreducedim(None, "+", ones, dims)
    finally:
        ones.close()
    region = _normalise_region(dims, d.ndim)
    return r, int(np.prod([d.dims[k - 1] for k in region if k <= d.ndim], dtype=np.int64))


def all(d: DArray, f: Optional[Callable] = None, dims=None):  # noqa: A001
    """``Base._all(f, A::DArray, ::Colon)`` (reference src/mapreduce.jl:97-104); with ``dims`` a Bool DArray (``all(f, d; dims)``)."""
    if dims is None:
        return bool(_pred_reduce(_lib.ALL, d, f))
    r, extent = _count_dims(d, f, dims)
    try:
        return broadcast(lambda c: c == extent, r)
    finally:
        r.close()


def any(d: DArray, f: Optional[Callable] = None, dims=None):  # noqa: A001
    """reference src/mapreduce.jl:106-113; with ``dims`` a Bool DArray."""
    if dims is None:
        return bool(_pred_reduce(_lib.ANY, d, f))
    r, _ = _count_dims(d, f, dims)
    try:
        return broadcast(lambda c: c > 0, r)
    finally:
        r.close()


def count(d: DArray, f: Optional[Callable] = None, dims=None):
    """reference src/mapreduce.jl:115-122; with ``dims`` an Int64 DArray."""
    if dims is None:
        return int(_pred_reduce(_lib.COUNT, d, f))
    return _count_dims(d, f, dims)[0]


def nnz(d: DArray) -> int:
    """``nnz(A::DArray)`` (reference ext/SparseArraysExt.jl:7-12: the per-worker ``nnz(localpart)`` summed).  Chunks are dense here, so the
    stored-entry count of the reference's sparse chunks becomes the number of nonzero elements -- one predicate count per localpart."""
    return count(d, lambda x: x != 0)


def extrema(d: DArray):
    """``extrema(d)`` (reference src/mapreduce.jl:124-131): per-chunk (min, max) in ONE pass over the chunk, then the fold
    ``(t, s) -> (min(t[1], s[1]), max(t[2], s[2]))`` over the workers in procs order."""
    from ._darray import SubDArray
    if isinstance(d, SubDArray):
        tmp = d.to_darray()
        try:
            return extrema(tmp)
        finally:
            tmp.close()
    if d.dtype == np.dtype(np.bool_):
        return (_mapreduce_all(None, _lib.MIN, d), _mapreduce_all(None, _lib.MAX, d))
    _check_nonempty(d, _lib.MAX)
    rt, code, es = d.rt, dab_dtype(d.dtype), d.dtype.itemsize
    host = _gather_slots(d, lambda pid, ch, slot: _lib.call("dab_reduce", rt.ctx, code, _lib.EXTREMA, _lib.MAP_ID, None, C.c_void_p(ch.ptr), ch.size,
                                                            C.c_void_p(slot)))
    lo = np.array([host[16 * (p - 1):16 * (p - 1) + es].view(d.dtype)[0] for p in d.layout.pids], dtype=d.dtype)
    hi = np.array([host[16 * (p - 1) + es:16 * (p - 1) + 2 * es].view(d.dtype)[0] for p in d.layout.pids], dtype=d.dtype)
    out = np.zeros(2, dtype=d.dtype)
    L = _lib.lib()
    _lib.check(L.dab_combine_ordered(code, _lib.MIN, C.c_void_p(lo.ctypes.data), lo.size, C.c_void_p(out[0:1].ctypes.data)))
    _lib.check(L.dab_combine_ordered(code, _lib.MAX, C.c_void_p(hi.ctypes.data), hi.size, C.c_void_p(out[1:2].ctypes.data)))
    return (out[0], out[1])


# ---- dimensional reduction ------------------------------------------------------------------------------------------------------


def _normalise_region(dims, ndim: int) -> Tuple[int, ...]:
    if isinstance(dims, (int, np.integer)):
        dims = (int(dims),)
    dims = tuple(int(x) for x in dims)
    for x in dims:
        if x <= 0:  # Base.check_reducedims / reduced_indices: "region dimension(s) must be >= 1"
            raise _lib.ArgumentError(_lib.ERR_ARG, f"ArgumentError: region dimension(s) must be ≥ 1, got {x}")
    return tuple(sorted(set(dims)))


def reduce_chunk_dims(rt, ch: B200Array, region_in: Sequence[int], op: int, mapc: int, out_dtype: np.dtype) -> B200Array:
    """``mapreduce(f, op, localpart(A), dims=region)`` (reference src/mapreduce.jl:64) on one chunk.
    Every maximal run of reduced dims is one (inner, reduce, outer) kernel pass, last run first."""
    shape = list(ch.shape)
    runs = collapse_for_region(shape, set(region_in))
    cur, cur_dtype, cur_map, owned = ch, ch.dtype, mapc, False
    # positions of runs: process reduced runs from the last to the first so `inner` stays the untouched prefix
    ext = [e for _, e in runs]
    for ri in range(len(runs) - 1, -1, -1):
        if not runs[ri][0]:
            continue
        inner = int(np.prod(ext[:ri])) if ri else 1
        red = ext[ri]
        outer = int(np.prod(ext[ri + 1:])) if ri + 1 < len(ext) else 1
        nxt = B200Array.empty(rt, (inner * outer,), out_dtype, temp=True)
        _lib.call("dab_reducedim", rt.ctx, dab_dtype(cur_dtype), op, cur_map, C.c_void_p(cur.ptr), inner, red, outer, C.c_void_p(nxt.ptr), 0)
        if owned:
            cur.free()  # stream-ordered: no host sync needed
        cur, cur_dtype, cur_map, owned = nxt, out_dtype, _lib.MAP_ID, True
        ext[ri] = 1
    rshape = tuple(1 if (k + 1) in region_in else s for k, s in enumerate(ch.shape))
    if not owned:  # nothing reduced (cannot happen when region_in is non-empty)
        return ch
    cur.shape = rshape
    return cur


def plan_reducedim(L: Layout, reg_in: Sequence[int]):
    """Pure layout logic of the dimensional reduction (reference src/mapreduce.jl:42-81).

    Returns ``(Rlayout, fibres)``: the layout of the result R -- ``pids[1:1 along region, : elsewhere]`` (:44), region dims
    collapsed to index 1:1 with cuts [1, 2] (:59-62) -- and, per chunk of R, the 0-based chunk numbers of A whose partial slabs
    are accumulated onto it, in column-major grid order along the reduced dims (the order ``Bfull`` is laid out in, :74-77)."""
    N = len(L.dims)
    Rgrid = tuple(1 if (k + 1) in reg_in else g for k, g in enumerate(L.grid))
    Rpids, Rindices, fibres = [], [], []
    for rl in range(int(np.prod(Rgrid))):
        rc = unravel(rl, Rgrid)
        owner_lin = ravel(rc, L.grid)
        Rpids.append(L.pids[owner_lin])
        Rindices.append(tuple((1, 1) if (k + 1) in reg_in else L.indices[owner_lin][k] for k in range(N)))
        sub = [L.grid[k] if (k + 1) in reg_in else 1 for k in range(N)]
        members = []
        for ml in range(int(np.prod(sub))):
            mc = unravel(ml, sub)
            members.append(ravel(tuple(mc[k] if (k + 1) in reg_in else rc[k] for k in range(N)), L.grid))
        fibres.append(members)
    Rdims = tuple(1 if (k + 1) in reg_in else s for k, s in enumerate(L.dims))
    Rcuts = [[1, 2] if (k + 1) in reg_in else list(L.cuts[k]) for k in range(N)]
    return Layout(Rdims, Rgrid, Rpids, Rindices, Rcuts), fibres


def exchange_plan(L: Layout, Rlayout: Layout, fibres, rank_of: Callable[[int], int], my_rank: int):
    """Who sends which partial slab to whom in ``mapreducedim_between!`` (reference src/mapreduce.jl:71-81), from the point of
    view of ``my_rank``.  Pure function of the layouts; every rank computes the same global plan, so the sends of one rank are
    exactly the receives of its peers (tests/test_dist_gloo.py executes it over gloo).

      owned : R chunk numbers whose owner lives on my rank
      local : (R chunk, slot in the fibre, member pid)            -- member partial already on my rank: device copy
      recvs : (R chunk, slot, member pid, source rank)            -- grouped ncclRecv, in this order
      sends : (member pid, destination rank, R chunk)             -- grouped ncclSend, in this order
    """
    owned, local, recvs, sends = [], [], [], []
    for rl, members in enumerate(fibres):
        owner = Rlayout.pids[rl]
        orank = rank_of(owner)
        if orank == my_rank:
            owned.append(rl)
        for slot, m in enumerate(members):
            mp = L.pids[m]
            mrank = rank_of(mp)
            if orank == my_rank and mrank == my_rank:
                local.append((rl, slot, mp))
            elif orank == my_rank:
                recvs.append((rl, slot, mp, mrank))
            elif mrank == my_rank:
                sends.append((mp, orank, rl))
    return {"owned": owned, "local": local, "recvs": recvs, "sends": sends}


def mapreducedim(f: Optional[Callable], op, d: DArray, dims, init=None) -> DArray:
    """``mapreduce(f, op, d; dims[, init])`` -> DArray R (reference src/mapreduce.jl:42-94)."""
    rt = d.rt
    opc = _op_code(op)
    N = d.ndim
    region = _normalise_region(dims, N)
    reg_in = tuple(r for r in region if r <= N)
    mapc, param, expr = classify_map(f, d.dtype)
    if param is not None or (expr is not None and expr.jt == "bool"):
        if opc == _lib.SUM and init is None:
            return _count_dims(d, f, dims)[0]                    # sum(pred, d; dims): Bools add up as Int (Base.add_sum)
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "Bool-valued maps with dims are served for + only (count / any / all build on it)")
    src, tmp = d, None
    if mapc is None:
        from ._broadcast import LocalArg, run_local
        from ._darray import darray_like
        out_dt = _NPT[expr.jt]
        tmp = darray_like(lambda I: B200Array.empty(rt, shape_of(I), out_dt), d, dtype=out_dt)
        for pid, out in tmp.chunks.items():
            run_local(rt, expr, out, [LocalArg(d.chunks[pid], None, tag_of(d.dtype))])
        src, mapc = tmp, _lib.MAP_ID
    rdt = _result_dtype(src.dtype, opc, mapc)
    L = src.layout
    try:
        if not reg_in or d.size == 0:
            # ``isempty(region) -> copyto!(R, A)`` (src/mapreduce.jl:89-91; f and init are NOT applied there) and
            # ``isempty(A) -> copy(R)`` (:85-87)
            from ._darray import darray_like
            R = darray_like(lambda I: B200Array.empty(rt, shape_of(I), rdt), d, dtype=rdt)
            for pid, out in R.chunks.items():
                if out.size:
                    if d.dtype == rdt:
                        _lib.call("dab_d2d", rt.ctx, C.c_void_p(out.ptr), C.c_void_p(d.chunks[pid].ptr), out.nbytes)
                    else:
                        from ._broadcast import LocalArg, run_local, Expr as _E
                        run_local(rt, _E("arg", (), tag_of(d.dtype), 0), out, [LocalArg(d.chunks[pid], None, tag_of(d.dtype))])
            return R
        Rlayout, fibres = plan_reducedim(L, reg_in)
        Rpids, Rindices = Rlayout.pids, Rlayout.indices
        # ---- phase 1: mapreducedim_within (src/mapreduce.jl:54-66)
        partial: Dict[int, B200Array] = {}
        for pid, ch in src.chunks.items():
            partial[pid] = reduce_chunk_dims(rt, ch, reg_in, opc, mapc, rdt)
        # ---- phase 2: mapreducedim_between! (src/mapreduce.jl:71-81): the partial slabs of a fibre are gathered on the owner of the R
        # chunk, in grid order.  Multi-rank: one-sided puts over NVLink into the owner's exchange arena + a device-side barrier (no NCCL
        # launch, no host sync); slabs too large for the arena, or DAB_FUSED_COMBINE=0, take the grouped ncclSend/ncclRecv path.
        Rchunks: Dict[int, B200Array] = {}
        isz = rdt.itemsize

        def stack_table(rank):
            off, tab = 0, {}
            for rl, members in enumerate(fibres):
                if rt.rank_of(Rpids[rl]) == rank:
                    plen = int(np.prod(shape_of(Rindices[rl])))
                    tab[rl] = (off, plen, len(members))
                    off += (plen * len(members) * isz + 255) & ~255
            return tab, off

        tables = {r: stack_table(r) for r in {rt.rank_of(p) for p in Rpids}}
        use_arena = rt.world > 1 and max(t[1] for t in tables.values()) <= rt.arena()["bank_bytes"]
        my_tab, my_bytes = tables.get(rt.rank, ({}, 0))
        priv = None
        if use_arena:
            bank = rt.arena_next_bank()
            peers = rt.arena()["peers"]
            my_base = peers[rt.rank] + bank
        else:
            priv = B200Array.empty(rt, (max(my_bytes, 16),), np.uint8, temp=True)
            my_base = priv.ptr
        xp = exchange_plan(L, Rlayout, fibres, rt.rank_of, rt.rank)
        for rl, slot, mp in xp["local"]:
            off, plen, _ = my_tab[rl]
            if plen:
                _lib.call("dab_d2d", rt.ctx, C.c_void_p(my_base + off + slot * plen * isz), C.c_void_p(partial[mp].ptr), plen * isz)
        if use_arena:
            for mp, peer, rl in xp["sends"]:
                off, plen, _ = tables[peer][0][rl]
                slot = fibres[rl].index(L.pids.index(mp))
                if plen:
                    _lib.call("dab_d2d", rt.ctx, C.c_void_p(peers[peer] + bank + off + slot * plen * isz), C.c_void_p(partial[mp].ptr), plen * isz)
            rt.device_barrier()
        else:
            sends = [(partial[mp].ptr, partial[mp].size * isz, peer) for mp, peer, _ in xp["sends"]]
            recvs = [(my_base + my_tab[rl][0] + slot * my_tab[rl][1] * isz, my_tab[rl][1] * isz, peer) for rl, slot, _, peer in xp["recvs"]]
            if sends or recvs:
                _lib.call("dab_group_start", rt.ctx)
                for ptr, nb, peer in sends:
                    _lib.call("dab_send", rt.ctx, C.c_void_p(ptr), nb, peer)
                for ptr, nb, peer in recvs:
                    _lib.call("dab_recv", rt.ctx, C.c_void_p(ptr), nb, peer)
                _lib.call("dab_group_end", rt.ctx)
        for rl, (off, plen, nm) in my_tab.items():
            owner = Rpids[rl]
            Rch = B200Array.empty(rt, shape_of(Rindices[rl]), rdt)
            acc = 0
            if init is not None:
                v = np.asarray(init, dtype=rdt)
                _lib.call("dab_fill", rt.ctx, dab_dtype(rdt) if rdt != np.dtype(np.int64) else _lib.I64, C.c_void_p(Rch.ptr), Rch.size,
                          C.c_void_p(v.ctypes.data))
                acc = 1
            # Base.mapreducedim!(identity, op, localpart(R), Bfull): accumulate the nm partial slabs, in grid order, onto R
            _lib.call("dab_reducedim", rt.ctx, dab_dtype(rdt), opc, _lib.MAP_ID, C.c_void_p(my_base + off), plen, nm, 1, C.c_void_p(Rch.ptr), acc)
            Rchunks[owner] = Rch
        if priv is not None:
            priv.free()
        for p in partial.values():
            p.free()
        return DArray(Rlayout, rdt, Rchunks, rt)
    finally:
        if tmp is not None:
            tmp.close()


# ---- Level-1 linear algebra and friends built from the same kernels (reference src/linalg.jl:24-59, ext/StatisticsExt.jl:6) ----------


def dot(x: DArray, y: DArray):
    """``dot(x, y)`` (reference src/linalg.jl:34-46): per-chunk dot products, summed over the chunks -- one fused pass, 8 B/element."""
    if x.dims != y.dims:
        raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"dot: {x.dims} vs {y.dims}")
    return _mapreduce_all(lambda a, b: a * b, _lib.SUM, x, False, (y,))


def norm(x: DArray, p=2):
    """``norm(x, p)`` (reference src/linalg.jl:48-59: per-worker ``norm(localpart(x), p)``, then ``norm(results, p)`` on the caller).
    p = 2, 1, Inf, -Inf and 0 (LinearAlgebra's special cases: Euclidean, sum of magnitudes, largest / smallest magnitude, number of
    nonzeros) and any other real p as ``(sum(abs(x)^p))^(1/p)`` in one fused pass (LinearAlgebra's ``normp`` additionally rescales by the
    largest magnitude against overflow; not done here)."""
    if p == 2:
        return np.sqrt(_mapreduce_all(abs2_fn, _lib.SUM, x))
    if p == 1:
        return _mapreduce_all(abs, _lib.SUM, x)
    if p in (np.inf, float("inf")):
        return _mapreduce_all(abs, _lib.MAX, x)
    if p in (-np.inf, float("-inf")):
        return _mapreduce_all(abs, _lib.MIN, x)
    if p == 0:
        return float(_mapreduce_all(lambda v: v != 0, _lib.COUNT, x))      # norm(x, 0) is a float in Julia
    if isinstance(p, (int, float, np.integer, np.floating)) and not isinstance(p, (bool, np.bool_)):
        pf = float(p)
        s = float(_mapreduce_all(lambda v: (abs(v) * 1.0) ** pf, _lib.SUM, x))   # powers and their sum in Float64 whatever the eltype
        r = s ** (1.0 / pf)
        return np.float32(r) if x.dtype == np.dtype(np.float32) else r            # norm of a Float32 array is a Float32
    raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, f"norm with p={p} is not served")


def abs2_fn(v):
    return v * v


def axpy_(a, x: DArray, y: DArray) -> DArray:
    """``axpy!(a, x, y)``: y .= a .* x .+ y (reference src/linalg.jl:24-32)."""
    from ._broadcast import broadcast_into
    if x.dims != y.dims:
        raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"axpy!: {x.dims} vs {y.dims}")
    s = np.asarray(a, dtype=x.dtype)[()]
    return broadcast_into(y, lambda u, v: s * u + v, x, y)


def rmul_(x: DArray, a) -> DArray:
    """``rmul!(x, a)``: x .= x .* a (reference src/linalg.jl:169-176)."""
    from ._broadcast import broadcast_into
    s = np.asarray(a, dtype=x.dtype)[()]
    return broadcast_into(x, lambda u: u * s, x)


def isequal(d: DArray, other) -> bool:
    """``d == a`` (reference src/darray.jl:403-414): sizes equal and every localpart equal to the matching slice -- one fused
    ``all(x .== y)`` pass per chunk."""
    from ._darray import SubDArray
    if isinstance(d, SubDArray) or isinstance(other, SubDArray):
        a = d.to_darray() if isinstance(d, SubDArray) else d
        b = other.to_darray() if isinstance(other, SubDArray) else other
        if not isinstance(a, DArray):
            a, b = b, a
        try:
            return isequal(a, b)
        finally:
            for t, o in ((a, d), (b, other)):
                if isinstance(o, SubDArray):
                    t.close()
    shape = other.dims if isinstance(other, DArray) else tuple(np.shape(other))
    if tuple(shape) != tuple(d.dims):
        return False
    if d.size == 0:
        return True
    if not isinstance(other, DArray):
        other = np.asarray(other)
    return bool(_mapreduce_all(lambda a, b: a == b, _lib.ALL, d, False, (other,)))


def mean(d: DArray, dims=None, f: Optional[Callable] = None):
    """``mean(d[; dims])`` (reference ext/StatisticsExt.jl:6: ``sum(f, A, dims) ./ prod(size(A)[dims])``)."""
    if dims is None:
        return mapreduce(f, "+", d) / d.size
    from ._broadcast import broadcast
    region = _normalise_region(dims, d.ndim)
    cnt = int(np.prod([d.dims[r - 1] for r in region if r <= d.ndim])) if region else 1
    S = mapreducedim(f, "+", d, dims)
    out_t = np.float64 if S.dtype.kind in "iub" or S.dtype == np.float64 else np.float32
    c = out_t(cnt)
    R = broadcast(lambda s: s / c, S)
    S.close()
    return R
