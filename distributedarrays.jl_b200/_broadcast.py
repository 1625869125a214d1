"""Distributed broadcast and map / map!: the reference's ``src/broadcast.jl`` and ``src/mapreduce.jl:3-12`` on B200.

The reference receives a Julia closure and lets Julia's JIT fuse the whole expression tree into one loop per localpart
(``copyto!(localpart(dest), lbc)``, src/broadcast.jl:80).  A closure cannot cross a C ABI, so here the Python callable
is *traced* once with symbolic scalars (operator overloading) into an expression tree with Julia's promotion rules, and
the tree is lowered to ONE kernel launch per localpart:

  * ``a*x + b`` (any spelling, e.g. ``2x+1``)        -> ``dab_affine``        (hand-written float4 streaming kernel)
  * a single unary / binary op                        -> ``dab_unary`` / ``dab_binary`` / ``dab_binary_scalar``
  * anything else (nested, N-ary, extruded size-1 dims, mixed element types)
                                                      -> ``dab_broadcast_expr`` (NVRTC-compiled fused kernel, sm_100a)

Semantics kept from the reference: axes check and ``DimensionMismatch`` (src/broadcast.jl:66); plain arrays are
distributed (``bcdistribute``, :124-137); per destination chunk every argument is cut with ``_bcview`` (:103-120; size-1
dims stay ``1:1`` = extrusion) and localised with ``makelocal`` (:140-152), which is zero-copy when the layouts match
and a halo fetch otherwise; allocating broadcast / ``map`` build the result with the DEFAULT layout for its size
(``DArray(map(length, axes(bc)))``, :93; src/darray.jl:174).  Arithmetic is IEEE per operation, never FMA-contracted.
"""
from __future__ import annotations

import ctypes as C
import struct
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from builtins import any as builtins_any

from . import _lib
from ._darray import B200Array, DArray, dab_dtype, darray, makelocal
from .layout import shape_of
from .runtime import runtime

# Julia-type tags and the promotion lattice
_RANK = {"bool": 0, "i32": 1, "i64": 2, "i128": 3, "f32": 4, "f64": 5}


class _TagTypes(dict):
    """Julia type tag -> array element type.  ``i128`` (Int128) exists only as a VALUE type inside ``mapreduce`` (``f`` widens its
    argument, test/darray.jl:286-294): there are no Int128 arrays, so every place that needs an element type for it refuses."""

    def __missing__(self, tag):
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, f"values of type {tag} have no array element type on the B200 backend "
                                    "(Int128 is served as the value type of mapreduce(f, op, d) only)")


_NPT = _TagTypes({"bool": np.dtype(np.bool_), "i32": np.dtype(np.int32), "i64": np.dtype(np.int64), "f32": np.dtype(np.float32),
                  "f64": np.dtype(np.float64)})
_TAG = {v: k for k, v in _NPT.items()}
_CT = {"bool": "bool", "i32": "int", "i64": "long long", "i128": "i128", "f32": "float", "f64": "double"}


def tag_of(dtype) -> str:
    dt = np.dtype(dtype)
    if dt not in _TAG:
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, f"element type {dt} not served by the B200 backend")
    return _TAG[dt]


def promote(a: str, b: str) -> str:
    """``promote_type`` for the supported types (Int32+Float32 -> Float32, Float32+Float64 -> Float64, ...)."""
    if a == b:
        return a
    if "f" in a[0] + b[0]:  # any float wins over ints/Bool (Int64 + Float32 -> Float32); Float64 only if one IS Float64
        fl = [t for t in (a, b) if t[0] == "f"]
        return "f64" if "f64" in fl else "f32"
    return a if _RANK[a] >= _RANK[b] else b


class Expr:
    """Symbolic scalar.  ``op``: 'arg' | 'const' | unary name | binary name; ``jt``: Julia type tag of the value."""

    __slots__ = ("op", "args", "jt", "val", "weak")
    # NumPy scalars must defer to our reflected operators (np.float32(1.5) * x has to stay a Float32 constant; without this
    # NumPy would coerce itself to a Python float -- a Float64 literal in Julia terms -- before calling __rmul__).
    __array_ufunc__ = None

    def __init__(self, op, args=(), jt="f64", val=None, weak=False):
        self.op, self.args, self.jt, self.val, self.weak = op, tuple(args), jt, val, weak

    # -- construction helpers
    @staticmethod
    def wrap(v) -> "Expr":
        if isinstance(v, Expr):
            return v
        if isinstance(v, (bool, np.bool_)):
            return Expr("const", (), "bool", bool(v))
        if isinstance(v, (int, np.integer)):
            if isinstance(v, np.int32):
                return Expr("const", (), "i32", int(v))
            return Expr("const", (), "i64", int(v))  # Julia literal 1 is Int64
        if isinstance(v, np.float32):
            return Expr("const", (), "f32", float(v))
        if isinstance(v, (float, np.floating)):
            return Expr("const", (), "f64", float(v))  # Julia literal 1.5 is Float64
        raise TypeError(f"cannot use {type(v).__name__} inside a broadcast kernel")

    def _bin(self, op, other, swap=False):
        o = Expr.wrap(other)
        a, b = (o, self) if swap else (self, o)
        return binop(op, a, b)

    __add__ = lambda s, o: s._bin("add", o)
    __radd__ = lambda s, o: s._bin("add", o, True)
    __sub__ = lambda s, o: s._bin("sub", o)
    __rsub__ = lambda s, o: s._bin("sub", o, True)
    __mul__ = lambda s, o: s._bin("mul", o)
    __rmul__ = lambda s, o: s._bin("mul", o, True)
    __truediv__ = lambda s, o: s._bin("div", o)
    __rtruediv__ = lambda s, o: s._bin("div", o, True)
    __mod__ = lambda s, o: s._bin("rem", o)        # Julia's % is rem (sign of dividend), not Python's floored %
    __rmod__ = lambda s, o: s._bin("rem", o, True)
    __floordiv__ = lambda s, o: s._bin("idiv", o)  # Julia div (truncated)
    __rfloordiv__ = lambda s, o: s._bin("idiv", o, True)
    __and__ = lambda s, o: s._bin("and", o)
    __or__ = lambda s, o: s._bin("or", o)
    __xor__ = lambda s, o: s._bin("xor", o)
    __lshift__ = lambda s, o: shiftop("x_shl", s, Expr.wrap(o))
    __rlshift__ = lambda s, o: shiftop("x_shl", Expr.wrap(o), s)
    __rshift__ = lambda s, o: shiftop("x_shr", s, Expr.wrap(o))
    __rrshift__ = lambda s, o: shiftop("x_shr", Expr.wrap(o), s)
    __lt__ = lambda s, o: s._bin("lt", o)
    __le__ = lambda s, o: s._bin("le", o)
    __gt__ = lambda s, o: s._bin("gt", o)
    __ge__ = lambda s, o: s._bin("ge", o)
    __eq__ = lambda s, o: s._bin("eq", o)  # type: ignore[assignment]
    __ne__ = lambda s, o: s._bin("ne", o)  # type: ignore[assignment]
    __hash__ = None  # type: ignore[assignment]

    def __neg__(self):
        return unop("neg", self)

    def __pos__(self):
        return self

    def __abs__(self):
        return unop("abs", self)

    def __pow__(self, p):
        if isinstance(p, (int, np.integer)) and not isinstance(p, (bool, np.bool_)) and 1 <= int(p) <= 3:  # Base.literal_pow: x^2 == x*x, x^3 == x*x*x
            r = self
            for _ in range(int(p) - 1):
                r = binop("mul", r, self)
            return r
        pe = Expr.wrap(p)
        if promote(self.jt, pe.jt)[0] != "f":
            # Julia's integer ^ is power_by_squaring and throws DomainError for negative exponents: no kernel serves it
            raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "integer ^ integer is not served by the B200 backend")
        return binop("pow", self, pe)

    def __bool__(self):
        raise TypeError("data-dependent Python control flow cannot be traced; use dab.ifelse(cond, a, b)")

    def key(self) -> str:
        if self.op == "arg":
            return f"a{self.val}:{self.jt}"
        if self.op == "const":
            return f"c{self.jt}:{self.val!r}"
        return f"{self.op}:{self.jt}(" + ",".join(a.key() for a in self.args) + ")"


_FLOAT_ONLY = {"sqrt", "inv", "sin", "cos", "tan", "exp", "exp2", "log", "log2", "log10", "tanh", "sinh", "cosh", "atan", "asin",
               "acos", "expm1", "log1p", "cbrt",
               # libdevice-backed extension block (kPreludeExt in dab_jit.cu; spelled jl_x_* in the generated source)
               "x_asinh", "x_acosh", "x_atanh", "x_exp10", "x_sinpi", "x_cospi", "x_erf", "x_erfc", "x_erfinv", "x_erfcinv", "x_erfcx",
               "x_gamma", "x_loggamma"}
_CMP = {"lt", "le", "gt", "ge", "eq", "ne"}


def binop(op: str, a: Expr, b: Expr) -> Expr:
    jt = promote(a.jt, b.jt)
    if op == "div" and jt[0] != "f":
        jt = "f64"  # Int / Int -> Float64
    if op in ("and", "or", "xor") and jt[0] == "f":
        raise TypeError(f"MethodError: no method matching {op}(::Float, ::Float)")
    if op == "idiv" and jt[0] == "f":
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "div on floats is not served")
    a, b = convert(a, jt), convert(b, jt)
    if op in _CMP:
        return Expr(op, (a, b), "bool")
    if jt == "bool" and op in ("add", "sub", "mul"):
        a, b, jt = convert(a, "i64"), convert(b, "i64"), "i64"
    return Expr(op, (a, b), jt)


def shiftop(op: str, a: Expr, n: Expr) -> Expr:
    """``a << n`` / ``a >> n`` (test/darray.jl:863-867).  Unlike the arithmetic operators the operands are NOT promoted to a common
    type: the result has the type of ``a`` (Bool counts as Int) and ``n`` is a bit count (Int64 here)."""
    if a.jt[0] == "f" or n.jt[0] == "f":
        raise TypeError(f"MethodError: no method matching {'<<' if op == 'x_shl' else '>>'}(::{a.jt}, ::{n.jt})")
    if a.jt == "i128" or n.jt == "i128":
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "shifts of Int128 values are not served")
    if a.jt == "bool":
        a = convert(a, "i64")
    return Expr(op, (a, convert(n, "i64")), a.jt)


def unop(op: str, a: Expr) -> Expr:
    if op in _FLOAT_ONLY and a.jt[0] != "f":
        a = convert(a, "f64")  # sqrt(::Int) -> Float64
    if op in ("isnan", "isinf", "isfinite"):
        return Expr(op, (a,), "bool")
    if op in ("x_trunc", "x_round") and a.jt == "bool":
        a = convert(a, "i64")
    if a.jt == "bool" and op in ("neg", "abs", "abs2"):
        a = convert(a, "i64")
    return Expr(op, (a,), a.jt)


def convert(a: Expr, jt: str) -> Expr:
    if a.jt == jt:
        return a
    if a.op == "const":
        v = a.val
        if jt == "f32":
            v = float(np.float32(v))
        elif jt == "f64":
            v = float(v)
        elif jt in ("i32", "i64", "i128"):
            v = int(v)
        else:
            v = bool(v)
        return Expr("const", (), jt, v)
    return Expr("convert", (a,), jt)


def Int128(x) -> Expr:
    """``Int128(x)`` inside a map function: the value continues in 128-bit wrap-around integer arithmetic
    (``mapreduce(x -> Int128(x)^2 + 2*Int128(x) - 1, *, d)`` -- the exactness test of test/darray.jl:286-294)."""
    return convert(Expr.wrap(x), "i128")


def widen(x) -> Expr:
    """Julia's ``widen``: Int32 -> Int64, Int64 -> Int128, Float32 -> Float64."""
    e = Expr.wrap(x)
    to = {"bool": "i64", "i32": "i64", "i64": "i128", "f32": "f64"}.get(e.jt)
    if to is None:
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, f"widen({e.jt}) is not served")
    return convert(e, to)


def uses_tag(e: Expr, tag: str) -> bool:
    return e.jt == tag or builtins_any(uses_tag(a, tag) for a in e.args)


def ifelse(c, a, b) -> Expr:
    c, a, b = Expr.wrap(c), Expr.wrap(a), Expr.wrap(b)
    jt = promote(a.jt, b.jt)
    return Expr("ifelse", (convert(c, "bool"), convert(a, jt), convert(b, jt)), jt)


def _mk_unary(name):
    def f(x):
        if isinstance(x, Expr):
            return unop(name, x)
        raise TypeError(f"dab.{name} is for use inside broadcast/map kernels")

    f.__name__ = name
    return f


abs2 = _mk_unary("abs2")
sqrt = _mk_unary("sqrt")
inv = _mk_unary("inv")
floor = _mk_unary("floor")
ceil = _mk_unary("ceil")
sign = _mk_unary("sign")
sin = _mk_unary("sin")
cos = _mk_unary("cos")
tan = _mk_unary("tan")
exp = _mk_unary("exp")
log = _mk_unary("log")
tanh = _mk_unary("tanh")
isnan = _mk_unary("isnan")
isinf = _mk_unary("isinf")
isfinite = _mk_unary("isfinite")
# the rest of the real-valued functions of the reference's "scalar math" test (test/darray.jl:775-797) that have a device kernel:
# already in the prelude ...
exp2, log2, log10, sinh, cosh = (_mk_unary(n) for n in ("exp2", "log2", "log10", "sinh", "cosh"))
atan, asin, acos, expm1, log1p, cbrt = (_mk_unary(n) for n in ("atan", "asin", "acos", "expm1", "log1p", "cbrt"))


# ... from libdevice through the extension block (public name without the x_) ...
def _mk_ext(name):
    f = _mk_unary("x_" + name)
    f.__name__ = name
    return f


asinh, acosh, atanh, exp10, sinpi, cospi = (_mk_ext(n) for n in ("asinh", "acosh", "atanh", "exp10", "sinpi", "cospi"))
erf, erfc, erfinv, erfcinv, erfcx, gamma, loggamma = (_mk_ext(n) for n in ("erf", "erfc", "erfinv", "erfcinv", "erfcx", "gamma", "loggamma"))
trunc, round_ = _mk_ext("trunc"), _mk_ext("round")           # round: to nearest, ties to even (Julia's default RoundNearest)


# ... and the ones Julia itself defines by composition (base/special/trig.jl: ``sec(z) = inv(cos(z))``, ``asec(y) = acos(inv(y))``, ...;
# base/math.jl: ``deg2rad(z) = z * (oftype(z, pi) / 180)``, ``rad2deg(z) = z * (180 / oftype(z, pi))``), composed the same way here
def _mk_inv_of(name, inner):
    def f(x):
        return unop("inv", inner(x))
    f.__name__ = name
    return f


def _mk_of_inv(name, outer):
    def f(x):
        if not isinstance(x, Expr):
            raise TypeError(f"dab.{name} is for use inside broadcast/map kernels")
        return outer(unop("inv", x))
    f.__name__ = name
    return f


sec, csc, cot = _mk_inv_of("sec", cos), _mk_inv_of("csc", sin), _mk_inv_of("cot", tan)
sech, csch, coth = _mk_inv_of("sech", cosh), _mk_inv_of("csch", sinh), _mk_inv_of("coth", tanh)
asec, acsc, acot = _mk_of_inv("asec", acos), _mk_of_inv("acsc", asin), _mk_of_inv("acot", atan)
asech, acsch, acoth = _mk_of_inv("asech", acosh), _mk_of_inv("acsch", asinh), _mk_of_inv("acoth", atanh)


def _float_of(x: Expr) -> Expr:
    return x if x.jt[0] == "f" else convert(x, "f64")


def deg2rad(x):
    x = _float_of(Expr.wrap(x))
    t = _NPT[x.jt].type
    return binop("mul", x, Expr("const", (), x.jt, float(t(np.pi) / t(180))))


def rad2deg(x):
    x = _float_of(Expr.wrap(x))
    t = _NPT[x.jt].type
    return binop("mul", x, Expr("const", (), x.jt, float(t(180) / t(np.pi))))


def jl_max(a, b):
    return binop("max", Expr.wrap(a), Expr.wrap(b))


def jl_min(a, b):
    return binop("min", Expr.wrap(a), Expr.wrap(b))


def mod(a, b):
    return binop("mod", Expr.wrap(a), Expr.wrap(b))


def rem(a, b):
    return binop("rem", Expr.wrap(a), Expr.wrap(b))


def trace(f: Callable, arg_tags: Sequence[str]) -> Expr:
    syms = [Expr("arg", (), t, k) for k, t in enumerate(arg_tags)]
    return Expr.wrap(f(*syms))


# ---- code generation for dab_broadcast_expr ----------------------------------------------------------------------------
_FN2 = {"add": "jl_add", "sub": "jl_sub", "mul": "jl_mul", "div": "jl_div", "rem": "jl_rem", "mod": "jl_mod", "idiv": "jl_idiv",
        "max": "jl_max", "min": "jl_min", "pow": "jl_pow", "and": "jl_and", "or": "jl_or", "xor": "jl_xor", "lt": "jl_lt", "le": "jl_le",
        "gt": "jl_gt", "ge": "jl_ge", "eq": "jl_eq", "ne": "jl_ne", "x_shl": "jl_x_shl", "x_shr": "jl_x_shr"}


def _lit(jt: str, v) -> str:
    if jt == "f32":
        return "__int_as_float((int)0x%08x)" % struct.unpack("<I", struct.pack("<f", float(v)))[0]
    if jt == "f64":
        return "__longlong_as_double((long long)0x%016xULL)" % struct.unpack("<Q", struct.pack("<d", float(v)))[0]
    if jt == "i32":
        return "((int)%d)" % int(v)
    if jt == "i64":
        return "((long long)%dLL)" % int(v)
    if jt == "i128":
        v = int(v) % (1 << 128)                                  # two's complement words; a literal cannot be wider than 64 bits in C
        return "((i128)(((u128)0x%016xULL << 64) | (u128)0x%016xULL))" % (v >> 64, v & ((1 << 64) - 1))
    return "true" if v else "false"


def codegen(e: Expr) -> str:
    if e.op == "arg":
        return f"a{e.val}"
    if e.op == "const":
        return _lit(e.jt, e.val)
    if e.op == "convert":
        return f"(({_CT[e.jt]})({codegen(e.args[0])}))"
    if e.op == "ifelse":
        return f"(({codegen(e.args[0])}) ? ({codegen(e.args[1])}) : ({codegen(e.args[2])}))"
    if e.op in _FN2:
        return f"{_FN2[e.op]}({codegen(e.args[0])}, {codegen(e.args[1])})"
    return f"jl_{e.op}({codegen(e.args[0])})"


# ---- pattern matching onto the hand-written kernels -----------------------------------------------------------------------
_UN = {"abs": _lib.MAP_ABS, "abs2": _lib.MAP_ABS2, "neg": _lib.MAP_NEG, "sqrt": _lib.MAP_SQRT, "inv": _lib.MAP_INV,
       "floor": _lib.MAP_FLOOR, "ceil": _lib.MAP_CEIL, "sign": _lib.MAP_SIGN}
_BIN = {"add": _lib.ADD, "sub": _lib.SUB, "mul": _lib.MUL, "div": _lib.DIV, "rem": _lib.REM, "max": _lib.BMAX, "min": _lib.BMIN,
        "mod": _lib.MOD, "idiv": _lib.IDIV, "and": _lib.AND, "or": _lib.OR, "xor": _lib.XOR}


def _is_arg(e: Expr, k=None):
    return e.op == "arg" and (k is None or e.val == k)


def match_affine(e: Expr):
    """e == a*x + b with x = arg 0 and constants a, b of x's type -> (a, b).  ``x + b``, ``a*x``, ``b + x*a`` included."""
    def lin(t):  # t == a*x ?
        if _is_arg(t, 0):
            return 1
        if t.op == "mul":
            l, r = t.args
            if l.op == "const" and _is_arg(r, 0):
                return l.val
            if r.op == "const" and _is_arg(l, 0):
                return r.val
        return None

    if e.op == "add":
        l, r = e.args
        if r.op == "const" and lin(l) is not None:
            return lin(l), r.val
        if l.op == "const" and lin(r) is not None:
            return lin(r), l.val
    return None


def _pad4(v, fill=1):
    v = list(v)
    if len(v) > 4:
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "broadcast whose dimensions do not collapse to 4 groups (see collapse_dims) is not served")
    return v + [fill] * (4 - len(v))


def collapse_dims(out_shape, arg_shapes):
    """Merge neighbouring dimensions of a broadcast that every array argument treats alike -- dense in both, or extruded (size 1,
    src/broadcast.jl:112-113) in both -- and drop the dimensions of extent 1.  A dense column-major argument addresses a merged group
    exactly as it addressed the separate dimensions (the stride of dim d+1 is stride(d) * extent(d)), so the kernel sees fewer
    dimensions and the same elements: ``(2,3,4,5,6) .+ (2,3,1,1,6)`` becomes ``(6,20,6) .+ (6,1,6)``, and any number of same-shape
    arguments becomes 1-D.  Returns (collapsed out shape, [collapsed shape per argument])."""
    nd = len(out_shape)
    shapes = [tuple(int(v) for v in sh) + (1,) * (nd - len(sh)) for sh in arg_shapes]
    groups: List[Tuple[int, List[int]]] = []
    for d in range(nd):
        o = int(out_shape[d])
        ext = [sh[d] for sh in shapes]
        for e, sh in zip(ext, arg_shapes):
            if e != o and e != 1:
                raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"arrays could not be broadcast: {tuple(sh)} vs {tuple(out_shape)}")
        if o == 1:
            continue
        if groups:
            po, pext = groups[-1]
            if all((pe == po and e == o) or (pe == 1 and e == 1) for pe, e in zip(pext, ext)):
                groups[-1] = (po * o, [pe * e for pe, e in zip(pext, ext)])
                continue
        groups.append((o, ext))
    if not groups:
        groups = [(1, [1] * len(shapes))]
    return tuple(g[0] for g in groups), [tuple(g[1][k] for g in groups) for k in range(len(shapes))]


def _dense_strides(shape):
    s, out = 1, []
    for d in shape:
        out.append(s)
        s *= int(d)
    return out


class LocalArg:
    """A broadcast argument localised for one destination chunk: device array (+ shape) or a host scalar."""

    def __init__(self, arr: Optional[B200Array] = None, scalar=None, tag: str = "f64", temp: bool = False):
        self.arr, self.scalar, self.tag, self.temp = arr, scalar, tag, temp


def run_local(rt, expr: Expr, out: B200Array, largs: List[LocalArg]):
    """Launch ONE kernel computing ``out .= expr(largs...)`` on this rank's GPU."""
    n = out.size
    if n == 0:
        return
    out_tag = tag_of(out.dtype)
    full = [a for a in largs if a.arr is not None]
    same = all(a.arr.shape == out.shape or a.arr.size == n and _squeeze(a.arr.shape) == _squeeze(out.shape) for a in full)
    ctx = rt.ctx
    code = dab_dtype(out.dtype)
    rt.last_kernel = "fixed"
    # ---- hand-written kernels when the tree is one of the fixed shapes
    if same and expr.jt == out_tag and out_tag != "bool":
        x0 = largs[0] if largs and largs[0].arr is not None and largs[0].tag == out_tag else None
        if x0 is not None and all(_only_arg0(expr)):
            ab = match_affine(expr)
            if ab is not None:
                a = np.asarray(ab[0], dtype=out.dtype)
                b = np.asarray(ab[1], dtype=out.dtype)
                # deferred: a reduction of `out` issued next runs fused with it (runtime.Runtime.defer_affine); any other call launches it
                rt.defer_affine(code, out.ptr, x0.arr.ptr, a, b, n)
                rt.last_kernel = "dab_affine"
                return
            if expr.op in _UN and _is_arg(expr.args[0], 0):
                _lib.call("dab_unary", ctx, code, _UN[expr.op], C.c_void_p(out.ptr), C.c_void_p(x0.arr.ptr), n)
                return
            if _is_arg(expr, 0):
                _lib.call("dab_unary", ctx, code, _lib.MAP_ID, C.c_void_p(out.ptr), C.c_void_p(x0.arr.ptr), n)
                return
        if expr.op in _BIN and len(expr.args) == 2 and not (expr.op == "div" and out_tag[0] != "f"):
            l, r = expr.args
            la = largs[l.val] if l.op == "arg" else None
            ra = largs[r.val] if r.op == "arg" else None

            def arr_ok(e, a):
                return e.op == "arg" and a is not None and a.arr is not None and a.tag == out_tag

            def sc_val(e, a):
                if e.op == "const" and e.jt == out_tag:
                    return e.val
                if e.op == "arg" and a is not None and a.arr is None and a.tag == out_tag:
                    return a.scalar
                return None

            if arr_ok(l, la) and arr_ok(r, ra):
                _lib.call("dab_binary", ctx, code, _BIN[expr.op], C.c_void_p(out.ptr), C.c_void_p(la.arr.ptr), C.c_void_p(ra.arr.ptr), n)
                return
            if arr_ok(l, la) and sc_val(r, ra) is not None:
                s = np.asarray(sc_val(r, ra), dtype=out.dtype)
                _lib.call("dab_binary_scalar", ctx, code, _BIN[expr.op], C.c_void_p(out.ptr), C.c_void_p(la.arr.ptr), C.c_void_p(s.ctypes.data), 0, n)
                return
            if arr_ok(r, ra) and sc_val(l, la) is not None:
                s = np.asarray(sc_val(l, la), dtype=out.dtype)
                _lib.call("dab_binary_scalar", ctx, code, _BIN[expr.op], C.c_void_p(out.ptr), C.c_void_p(ra.arr.ptr), C.c_void_p(s.ctypes.data), 1, n)
                return
    if expr.op == "const" and expr.jt == out_tag:
        v = np.asarray(expr.val, dtype=out.dtype)
        _lib.call("dab_fill", ctx, code, C.c_void_p(out.ptr), n, C.c_void_p(v.ctypes.data))
        return
    # ---- general fused kernel (NVRTC)
    rt.last_kernel = "dab_broadcast_expr"
    if uses_tag(expr, "i128"):
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "Int128 values are served inside mapreduce(f, op, d) only, not in a broadcast")
    if expr.jt[0] == "f" and out_tag[0] != "f":
        # dest .= f.(...) with an integer/Bool destination and float values: Julia converts exactly or throws InexactError per
        # element; a C cast would silently truncate
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, f"broadcast of {expr.jt} values into a {out_tag} destination (InexactError semantics) is not served")
    src = codegen(convert(expr, out_tag)).encode()
    oshape_nd, ashapes = tuple(out.shape), {k: tuple(a.arr.shape) for k, a in enumerate(largs) if a.arr is not None}
    if len(oshape_nd) > 4 or any(len(sh) > 4 for sh in ashapes.values()):
        # the kernel walks a 4-D box: more dimensions are served when they collapse to <= 4 groups (always for same-shape arguments)
        keys = sorted(ashapes)
        oshape_nd, coll = collapse_dims(oshape_nd, [ashapes[k] for k in keys])
        ashapes = dict(zip(keys, coll))
    oshape = _pad4(oshape_nd)
    nargs = len(largs)
    if nargs > 8:
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, "more than 8 broadcast arguments are not served")
    dts = (C.c_int32 * max(nargs, 1))()
    ptrs = (C.c_void_p * max(nargs, 1))()
    strides = (C.c_size_t * (4 * max(nargs, 1)))()
    scal = (C.c_uint64 * max(nargs, 1))()
    for k, a in enumerate(largs):
        dts[k] = dab_dtype(_NPT[a.tag])
        if a.arr is not None:
            ptrs[k] = a.arr.ptr
            ash = _pad4(ashapes[k])
            dense = _dense_strides(ash)
            for d in range(4):
                if ash[d] == oshape[d]:
                    strides[4 * k + d] = dense[d]
                elif ash[d] == 1:
                    strides[4 * k + d] = 0  # extruded dim (src/broadcast.jl:112-113)
                else:
                    raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"arrays could not be broadcast: {a.arr.shape} vs {out.shape}")
        else:
            ptrs[k] = None
            scal[k] = struct.unpack("<Q", np.asarray(a.scalar, dtype=_NPT[a.tag]).tobytes().ljust(8, b"\0"))[0]
    _lib.call("dab_broadcast_expr", ctx, src, code, C.c_void_p(out.ptr), _lib.sz4(oshape), _lib.sz4(_dense_strides(oshape)), nargs, dts,
              ptrs, strides, scal)


def _squeeze(shape):
    return tuple(s for s in shape if s != 1)


def _only_arg0(e: Expr):
    """Yields True for every leaf that is arg 0 or a constant."""
    if e.op == "arg":
        yield e.val == 0
    elif e.op != "const":
        for a in e.args:
            yield from _only_arg0(a)


# ---- the distributed drivers ----------------------------------------------------------------------------------------------


def _bc_shape(shapes: Sequence[Tuple[int, ...]]) -> Tuple[int, ...]:
    """Julia broadcast shape: dims aligned from the FIRST dim, missing trailing dims count as 1."""
    nd = max((len(s) for s in shapes), default=0)
    out = []
    for k in range(nd):
        ext = 1
        for s in shapes:
            v = s[k] if k < len(s) else 1
            if v != 1:
                if ext != 1 and ext != v:
                    raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"arrays could not be broadcast to a common size: {shapes}")
                ext = v
        out.append(ext)
    return tuple(out)


def _arg_tag(a) -> str:
    if isinstance(a, (DArray,)):
        return tag_of(a.dtype)
    if isinstance(a, np.ndarray) and a.ndim > 0:
        return tag_of(a.dtype)
    return Expr.wrap(a.item() if isinstance(a, np.ndarray) else a).jt


def _bcview(arg_dims: Sequence[int], I) -> Tuple:
    """``_bcview(axes(x), idxs)`` (src/broadcast.jl:103-120): size-1 dims stay 1:1, others take the chunk's range."""
    out = []
    for k, s in enumerate(arg_dims):
        if s == 1:
            out.append((1, 1))
        elif k < len(I):
            lo, hi = I[k]
            if not (1 <= lo and hi <= s):
                raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, "broadcast view could not be constructed")
            out.append((lo, hi))
        else:
            out.append((1, s))
    return tuple(out)


def _localise(rt, a, I, pid) -> LocalArg:
    """``bclocal`` (src/broadcast.jl:140-152)."""
    if isinstance(a, DArray):
        view = _bcview(a.dims, I)
        arr = makelocal(a, view, pid)
        return LocalArg(arr, None, tag_of(a.dtype), temp=arr is not a.chunks.get(pid))
    if isinstance(a, np.ndarray) and a.ndim > 0:
        view = _bcview(a.shape, I)
        sl = a[tuple(slice(lo - 1, hi) for lo, hi in view)]
        return LocalArg(B200Array.from_numpy(rt, sl), None, tag_of(a.dtype), temp=True)
    e = Expr.wrap(a.item() if isinstance(a, np.ndarray) else a)
    return LocalArg(None, e.val, e.jt)


def _prepare_remote_reads(dest_layout, rt, args):
    """Collective: when a DArray argument's layout differs from the destination's, some rank will have to halo-fetch non-owned
    data (makelocal's non-local branch, reference src/darray.jl:361-366).  Every rank takes the same decision from the layouts
    alone, shares the CUDA-IPC handles and fences the producers' streams before the one-sided peer reads."""
    if rt.world == 1:
        return False
    need = [a for a in args if isinstance(a, DArray) and not (a.layout.pids == dest_layout.pids and a.layout.indices == dest_layout.indices)]
    for a in need:
        if a._handles is None:
            a.share()
    if need:
        rt.barrier()
    return bool(need)


def _finish_remote_reads(rt, had_remote: bool):
    """Collective counterpart of ``_prepare_remote_reads``: the owners of the chunks that were read one-sidedly may not overwrite
    or free them before EVERY reader's copy kernel has finished (freed blocks go straight back to the allocator cache).  The
    reference's ``remotecall_fetch`` is synchronous for the same reason.  Stream sync + host barrier, as copy_transposed / mul!."""
    if had_remote:
        rt.sync()
        rt.barrier()


def _materialise_views(args):
    """SubDArray arguments (``a .= 3 .+ abs2.(view(d, ...))``) enter a broadcast as ``DArray(view)`` (reference src/darray.jl:603-609):
    a halo read into a fresh DArray with the default layout, released when the broadcast has been launched."""
    from ._darray import SubDArray
    out, temps = [], []
    for a in args:
        if isinstance(a, SubDArray):
            a = a.to_darray()
            temps.append(a)
        out.append(a)
    return out, temps


def broadcast_into(dest: DArray, f: Callable, *args) -> DArray:
    """``dest .= f.(args...)``: ``Base.copyto!(dest::DArray, bc::Broadcasted{Nothing})`` (reference src/broadcast.jl:65-85)."""
    args, _views = _materialise_views(args)
    try:
        return _broadcast_into(dest, f, *args)
    finally:
        for v in _views:
            v.close()


def _broadcast_into(dest: DArray, f: Callable, *args) -> DArray:
    shapes = [a.dims if isinstance(a, DArray) else (a.shape if isinstance(a, np.ndarray) else ()) for a in args]
    # materialize!(dest, bc) instantiates the Broadcasted with axes(dest): every argument must be broadcastable TO dest's axes
    # (each of its dims is 1 or equals dest's; missing trailing dims count as 1), else DimensionMismatch (src/broadcast.jl:66)
    for shp in shapes:
        for k, s in enumerate(shp):
            want = dest.dims[k] if k < len(dest.dims) else 1
            if s != 1 and s != want:
                raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"destination axes {dest.dims} are not compatible with source axes {tuple(shp)}")
    expr = trace(f, [_arg_tag(a) for a in args])
    rt = dest.rt
    remote = _prepare_remote_reads(dest.layout, rt, args)
    for pid, out in dest.chunks.items():
        I = dest.layout.localindices(pid)
        largs = [_localise(rt, a, I, pid) for a in args]
        run_local(rt, expr, out, largs)
        for la in largs:
            if la.temp and la.arr is not None:
                la.arr.free()                                  # stream-ordered: the block is only reused by later launches
    _finish_remote_reads(rt, remote)
    return dest


def broadcast(f: Callable, *args, rt=None) -> DArray:
    """``f.(args...)`` allocating: ``Base.copy(bc::Broadcasted{<:DArrayStyle})`` (reference src/broadcast.jl:91-98).
    The result gets the DEFAULT layout for its size, not the arguments' (src/darray.jl:174)."""
    args, _views = _materialise_views(args)
    try:
        return _broadcast(f, *args, rt=rt)
    finally:
        for v in _views:
            v.close()


def _broadcast(f: Callable, *args, rt=None) -> DArray:
    rt = rt or next((a.rt for a in args if isinstance(a, DArray)), None) or runtime()
    shapes = [a.dims if isinstance(a, DArray) else (a.shape if isinstance(a, np.ndarray) else ()) for a in args]
    dims = _bc_shape(shapes)
    expr = trace(f, [_arg_tag(a) for a in args])
    out_dt = _NPT[expr.jt]
    dest = darray(lambda I: B200Array.empty(rt, shape_of(I), out_dt), dims, dtype=out_dt, rt=rt)
    remote = _prepare_remote_reads(dest.layout, rt, args)
    for pid, out in dest.chunks.items():
        I = dest.layout.localindices(pid)
        largs = [_localise(rt, a, I, pid) for a in args]
        run_local(rt, expr, out, largs)
        for la in largs:
            if la.temp and la.arr is not None:
                la.arr.free()                                  # stream-ordered: the block is only reused by later launches
    _finish_remote_reads(rt, remote)
    return dest


def copy(d: DArray) -> DArray:
    """``copy(d::DArray)`` / ``deepcopy(d)`` (reference src/darray.jl:689-697; ``copy`` is Base's generic ``copyto!(similar(d), d)``): a new
    DArray on ``procs(d)`` with its own localparts (test/darray.jl:84-131: writing into the copy never shows in the original).  One
    identity broadcast per localpart -- a device-to-device stream at the HBM roofline; a ``dist`` that ``similar`` does not inherit is
    bridged by the halo fetch like any mixed-layout broadcast."""
    from ._darray import similar
    return _broadcast_into(similar(d), lambda x: x, d)


deepcopy = copy          # a localpart is one dense device array: there is nothing shallow to share


def drandn(dims, procs=None, dist=None, dtype=np.float64, seed: int = 1234, rt=None) -> DArray:
    """``drandn(dims, ...)`` (reference src/darray.jl:526-532): standard-normal entries.  Box-Muller over two counter-based uniform streams
    (``drand`` with seeds ``seed`` and ``seed + 1``; layout-independent like ``drand``), fused into one elementwise kernel:
    ``sqrt(-2 log(1 - u1)) * cos(2 pi u2)`` with ``1 - u1`` in (0, 1] so the logarithm is finite."""
    from ._darray import drand
    dt = np.dtype(dtype)
    if dt.kind != "f":
        raise _lib.UnsupportedError(_lib.ERR_UNSUPPORTED, f"drandn of eltype {dt}")
    u1 = drand(dims, procs, dist, dtype=dt, seed=seed, rt=rt)
    u2 = drand(dims, procs, dist, dtype=dt, seed=seed + 1, rt=rt)
    two, one, twopi = dt.type(2), dt.type(1), dt.type(2 * np.pi)
    _broadcast_into(u1, lambda a, b: sqrt(-two * log(one - a)) * cos(twopi * b), u1, u2)
    u2.close()
    return u1


def map_(f: Callable, d0: DArray, *ds) -> DArray:
    """``map(f, d0::DArray, ds...) = broadcast(f, d0, ds...)`` (reference src/mapreduce.jl:3)."""
    return broadcast(f, d0, *ds)


def map_inplace(f: Callable, dest: DArray, src: DArray) -> DArray:
    """``map!(f, dest::DArray, src::DArray)`` (reference src/mapreduce.jl:5-12): per worker
    ``map!(f, localpart(dest), makelocal(src, localindices(dest)...))``."""
    expr = trace(f, [tag_of(src.dtype)])
    rt = dest.rt
    remote = _prepare_remote_reads(dest.layout, rt, [src])
    for pid, out in dest.chunks.items():
        I = dest.layout.localindices(pid)
        arr = makelocal(src, I, pid)
        temp = arr is not src.chunks.get(pid)
        run_local(rt, expr, out, [LocalArg(arr, None, tag_of(src.dtype))])
        if temp:
            arr.free()
    _finish_remote_reads(rt, remote)
    return dest


map_bang = map_inplace


def map_localparts(f: Callable, A, B=None) -> DArray:
    """``map_localparts(f, d1, d2)`` and the binary operators built on it -- ``+ - div mod rem & | xor`` between two DArrays or
    a DArray and an Array of the same element type (reference src/mapreduce.jl:137-189).  The result keeps the layout of the
    (first) DArray argument (``DArray(d1) do I ... end``, :138-140), NOT the default layout an allocating broadcast would pick; a
    second DArray with different cuts is first brought to that layout (``samedist``, :172-178) -- here by the halo fetch inside
    the fused kernel launch.  ``f`` acts elementwise (traced like any broadcast function)."""
    lead = A if isinstance(A, DArray) else B
    if not isinstance(lead, DArray):
        raise TypeError("map_localparts needs at least one DArray")
    args = (A,) if B is None else (A, B)
    for a in args:
        shp = a.dims if isinstance(a, DArray) else tuple(np.shape(a))
        if tuple(shp) != tuple(lead.dims):
            raise _lib.DimensionMismatch(_lib.ERR_DIM_MISMATCH, f"DimensionMismatch: {lead.dims} vs {shp}")   # samedist, :173
        dt = a.dtype if isinstance(a, (DArray, np.ndarray)) else np.asarray(a).dtype
        if np.dtype(dt) != lead.dtype:
            raise TypeError(f"MethodError: no method matching op(::DArray{{{lead.dtype}}}, ::{type(a).__name__}{{{np.dtype(dt)}}}) "
                            "(the reference defines these operators for equal element types only)")
    expr = trace(f, [_arg_tag(a) for a in args])
    rt = lead.rt
    out_dt = _NPT[expr.jt]
    from ._darray import darray_like
    dest = darray_like(lambda I: B200Array.empty(rt, shape_of(I), out_dt), lead, dtype=out_dt)
    remote = _prepare_remote_reads(dest.layout, rt, args)
    for pid, out in dest.chunks.items():
        I = dest.layout.localindices(pid)
        largs = [_localise(rt, a, I, pid) for a in args]
        run_local(rt, expr, out, largs)
        for la in largs:
            if la.temp and la.arr is not None:
                la.arr.free()                                  # stream-ordered: the block is only reused by later launches
    _finish_remote_reads(rt, remote)
    return dest
