"""dab_affine_reduce / dab_affine_mapreduce_all against the two calls they replace (dab_affine, then dab_reduce / dab_mapreduce_all of y):
y bit for bit and the whole 16-byte result slot, wide carrier included.  The fused kernel shares the broadcast's functor and the reduce's
grid, tree and combine, so nothing here is compared at a tolerance."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F32, F64 = np.float32, np.float64
OPS = ["SUM", "PROD", "MAX", "MIN"]


def _lib():
    from darray_b200 import _lib as L
    return L


def _dev(dab, rt, host, extra=0):
    """Device copy of `host` (plus `extra` spare elements in front, for offset views); returns (owner, element offset 0 pointer)."""
    arr = dab.B200Array.empty(rt, (host.size + 2,), host.dtype)
    if host.size:
        _lib().call("dab_h2d", rt.ctx, C.c_void_p(arr.ptr + extra * host.itemsize), C.c_void_p(host.ctypes.data), host.nbytes)
    return arr


def _read(rt, ptr, n, dtype):
    out = np.empty(n, dtype=dtype)
    if n:
        _lib().call("dab_d2h", rt.ctx, C.c_void_p(out.ctypes.data), C.c_void_p(ptr), out.nbytes)
    rt.sync()
    return out


def _coefs(dtype, op):
    # PROD: factors in [1, 1 + 1e-6] keep the product of 2^24 values finite; otherwise the bench's y = 1.5 x + 0.25
    return (np.asarray(1e-6, dtype), np.asarray(1.0, dtype)) if op == "PROD" else (np.asarray(1.5, dtype), np.asarray(0.25, dtype))


def _pair(dab, rt, dtype, op, host, xoff=0, yoff=0, in_place=False, a=None, b=None):
    """Run unfused and fused on the same input; return (y_unfused, slot_unfused, y_fused, slot_fused)."""
    L = _lib()
    code = L.F32 if dtype == F32 else L.F64
    opc = getattr(L, op)
    if a is None:
        a, b = _coefs(dtype, op)
    n = host.size
    es = np.dtype(dtype).itemsize
    res = []
    for fused in (False, True):
        xs = _dev(dab, rt, host, xoff)
        xp = xs.ptr + xoff * es
        ys = xs if in_place else dab.B200Array.empty(rt, (n + 2,), dtype)
        yp = xp if in_place else ys.ptr + yoff * es
        slot = dab.B200Array.empty(rt, (16,), np.uint8)
        args = (C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), n)
        if fused:
            L.call("dab_affine_reduce", rt.ctx, code, C.c_void_p(yp), C.c_void_p(xp), *args, opc, C.c_void_p(slot.ptr))
        else:
            L.call("dab_affine", rt.ctx, code, C.c_void_p(yp), C.c_void_p(xp), *args)
            L.call("dab_reduce", rt.ctx, code, opc, L.MAP_ID, None, C.c_void_p(yp), n, C.c_void_p(slot.ptr))
        res += [_read(rt, yp, n, dtype), _read(rt, slot.ptr, 16, np.uint8)]
        for arr in {id(xs): xs, id(ys): ys, id(slot): slot}.values():
            arr.free()
    return res


def _same(res):
    yu, su, yf, sf = res
    assert yu.tobytes() == yf.tobytes(), "y differs"
    assert su.tobytes() == sf.tobytes(), (su, sf)


def _input(n, dtype, seed):
    return np.random.default_rng(seed).random(n).astype(dtype)


@pytest.mark.parametrize("n", [1, 3, 4095, (1 << 20) + 3, 1 << 24])
@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dtype", [F32, F64])
def test_fused_equals_unfused(dab, rt1, dtype, op, n):
    _same(_pair(dab, rt1, dtype, op, _input(n, dtype, n)))


@pytest.mark.parametrize("layout", ["both_offset", "offsets_differ", "in_place"])
@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dtype", [F32, F64])
def test_fused_offsets_and_aliasing(dab, rt1, dtype, op, layout):
    """x and y both one element (4 B for Float32, 8 B for Float64) past a 16-byte boundary (fused, with a head peel); only y offset (the
    entry point runs the two launches); y is x (map!(f, d, d))."""
    n = (1 << 20) + 5
    host = _input(n, dtype, 99)
    if layout == "both_offset":
        res = _pair(dab, rt1, dtype, op, host, xoff=1, yoff=1)
    elif layout == "offsets_differ":
        res = _pair(dab, rt1, dtype, op, host, xoff=0, yoff=1)
    else:
        res = _pair(dab, rt1, dtype, op, host, in_place=True)
    _same(res)


@pytest.mark.parametrize("case", ["signed_zeros", "nan"])
@pytest.mark.parametrize("op", ["MAX", "MIN"])
@pytest.mark.parametrize("dtype", [F32, F64])
def test_fused_max_min_nan_and_signed_zeros(dab, rt1, dtype, op, case):
    """a = 1, b = -0.0 keeps every value (and the sign of zero): Julia's max / min order (+0.0 > -0.0, NaN wins) inside the fused tree."""
    n = 100003
    rng = np.random.default_rng(5)
    host = np.where(rng.random(n) < 0.5, dtype(0.0), dtype(-0.0)).astype(dtype)
    if case == "nan":
        host[rng.integers(0, n, 3)] = np.nan
    a, b = np.asarray(1.0, dtype), np.asarray(-0.0, dtype)
    res = _pair(dab, rt1, dtype, op, host, a=a, b=b)
    _same(res)
    got = res[3][:np.dtype(dtype).itemsize].view(dtype)[0]
    if case == "nan":
        assert np.isnan(got)
    else:
        assert got == 0 and np.signbit(got) == (op == "MIN")


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dtype", [F32, F64])
def test_affine_mapreduce_all_equals_unfused(dab, rt1, dtype, op):
    L = _lib()
    code = L.F32 if dtype == F32 else L.F64
    n = (1 << 22) + 7
    host = _input(n, dtype, 17)
    a, b = _coefs(dtype, op)
    outs = []
    for fused in (False, True):
        xs, ys = _dev(dab, rt1, host), dab.B200Array.empty(rt1, (n,), dtype)
        out = np.zeros(2, dtype=np.uint64)
        args = (C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), n)
        if fused:
            L.call("dab_affine_mapreduce_all", rt1.ctx, code, C.c_void_p(ys.ptr), C.c_void_p(xs.ptr), *args, getattr(L, op), C.c_void_p(out.ctypes.data))
        else:
            L.call("dab_affine", rt1.ctx, code, C.c_void_p(ys.ptr), C.c_void_p(xs.ptr), *args)
            L.call("dab_mapreduce_all", rt1.ctx, code, getattr(L, op), L.MAP_ID, None, C.c_void_p(ys.ptr), n, C.c_void_p(out.ctypes.data))
        outs.append((_read(rt1, ys.ptr, n, dtype).tobytes(), out.tobytes()))
        xs.free()
        ys.free()
    assert outs[0] == outs[1]


def test_fused_full_size(dab, rt1):
    """The bench's chunk: 2^30 Float32 (4 GiB), y = 1.5 x + 0.25, SUM."""
    n = 1 << 30
    if rt1.device_info()["free_bytes"] < (17 << 30):
        pytest.skip("not enough free HBM")
    L = _lib()
    x = dab.drand((n,), dtype=F32, seed=4321)
    xp = dab.localpart(x).ptr
    a, b = _coefs(F32, "SUM")
    ys, slots = [], []
    for fused in (False, True):
        y = dab.B200Array.empty(rt1, (n,), F32)
        slot = dab.B200Array.empty(rt1, (16,), np.uint8)
        args = (C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), n)
        if fused:
            L.call("dab_affine_reduce", rt1.ctx, L.F32, C.c_void_p(y.ptr), C.c_void_p(xp), *args, L.SUM, C.c_void_p(slot.ptr))
        else:
            L.call("dab_affine", rt1.ctx, L.F32, C.c_void_p(y.ptr), C.c_void_p(xp), *args)
            L.call("dab_reduce", rt1.ctx, L.F32, L.SUM, L.MAP_ID, None, C.c_void_p(y.ptr), n, C.c_void_p(slot.ptr))
        ys.append(y)
        slots.append(_read(rt1, slot.ptr, 16, np.uint8).tobytes())
        slot.free()
    assert slots[0] == slots[1]
    for off in range(0, n, 1 << 27):                                  # compare y in 512 MiB pieces
        m = min(1 << 27, n - off)
        assert _read(rt1, ys[0].ptr + 4 * off, m, F32).tobytes() == _read(rt1, ys[1].ptr + 4 * off, m, F32).tobytes()
    for y in ys:
        y.free()
    x.close()


@pytest.mark.parametrize("red", ["sum", "prod", "maximum", "minimum"])
@pytest.mark.parametrize("rtname", ["rt1", "rt2"])
def test_api_broadcast_then_reduce_equals_eager(dab, request, rtname, red):
    """broadcast_into then sum through the public API (fused: the broadcast is deferred into the reduce) against the same calls with the
    broadcast launched at once."""
    rt = request.getfixturevalue(rtname)
    n = (1 << 22) + 3
    a, b = (F32(1e-6), F32(1.0)) if red == "prod" else (F32(1.5), F32(0.25))
    x = dab.drand((n,), dtype=F32, seed=77)
    fn = getattr(dab, red)
    got = []
    for eager in (False, True):
        y = dab.similar(x)
        l0 = rt.launches()
        dab.broadcast_into(y, lambda v: a * v + b, x)
        if eager:
            rt.flush()
        s = fn(y)
        launches = rt.launches() - l0
        got.append((np.asarray(s).tobytes(), dab.to_array(y).tobytes()))
        assert launches == (2 * rt.workers_per_rank if eager else 2 * rt.workers_per_rank - 1), launches
        y.close()
    assert got[0] == got[1]
    x.close()
