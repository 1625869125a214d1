"""GPU parity tests for what the LAST session of round 2 added after the round's GPU budget was spent:

  * ``sort(d; by = f)``: ``dab_sort_by_key`` (dab_sortby.cu) and the keyed samplesort of ``_sort.py`` (reference src/sort.jl:8, 22, 32,
    61, 77, 111);
  * ``dab_gemm`` with a one-column B routed to K9 (``dab_gemv``) -- host-side dispatch only, both kernels are GPU-tested on their own;
  * Int128 as the value type of ``mapreduce`` (``dab.Int128`` / ``dab.widen``; the reference's exactness test test/darray.jl:286-294);
  * the rest of the reference's "scalar math" vocabulary that has a device kernel (test/darray.jl:775-797): libdevice-backed functions in
    a conditional prelude block, and the functions Julia defines by composition;
  * ``<<`` / ``>>`` on integer DArrays (test/darray.jl:863-867);
  * ``reshape(A::DVector, dims)`` (one vector-indexed view per new localpart, the gather kernel of round 2);
  * ``copy`` / ``deepcopy`` of a DArray and ``drandn`` (host-side compositions of the broadcast kernels);
  * ``all`` / ``any`` / ``count`` with ``dims`` (host-side compositions: predicate -> 0 / 1, dimensional sum, compare);
  * ``norm(x, p)`` for p = 0, -Inf and general p (host-side compositions of the fused map + reduce);
  * general broadcasts over more than 4 dimensions (``collapse_dims`` in ``_broadcast.py``; reference src/broadcast.jl is N-d).

Also verified on CPU: the sort-by-key composition (key|position words, two rounds for 64-bit keys, gather) step by step in
``tests/hostmem_abi.py`` against a stable ``isless`` argsort, the whole host flow of ``_sort.py`` against the oracle
(``tests/test_cpu_sort.py``), and that the collapsed box of ``collapse_dims`` addresses exactly the elements NumPy's broadcasting reads
(``tests/test_cpu_host.py``), that the Int128 reduce kernels compile with NVRTC for sm_100a and that the host side (slot decoding,
wrap-around fold) is exact (``tests/test_cpu_jit_reduce.py``).  What only a B200 can verify: the two small sort-by-key kernels, their
ctypes bindings, and the N-d broadcast through the real NVRTC kernel.  The module runs LAST (file name), and inside it host-side
compositions of GPU-tested kernels come first, new NVRTC device code (extension prelude, Int128 carriers) next, the two hand-written
sort-by-key kernels last -- a fault in newer code cannot take the evidence for the rest with it."""
import ctypes as C

import numpy as np
import pytest

from oracle import darray_oracle as orc

INT128_BIG_N = (1 << 22) + 5                    # the CPU dry run of these tests (tests/test_cpu_host.py) shrinks the big sizes
SORT_BY_KEY_SIZES = (1, 2, 33, 1024, 1025, 4097, 100003, (1 << 20) + 17)

pytestmark = pytest.mark.gpu


def test_broadcast_more_than_4_dims(dab, rt8):
    """General (NVRTC) broadcasts over 5-D / 6-D arrays: same-shape arguments collapse to one dimension, extruded arguments to at
    most 4 groups; bit-exact against NumPy in the same precision."""
    rng = np.random.default_rng(91)
    A = rng.standard_normal((6, 5, 4, 3, 4)).astype(np.float32)
    B = rng.standard_normal((6, 5, 4, 3, 4)).astype(np.float32)
    a, b = dab.distribute(A), dab.distribute(B)
    r = dab.broadcast(lambda x, y: x - y * x, a, b)                             # nested tree: the fused general kernel
    assert rt8.last_kernel == "dab_broadcast_expr"
    assert np.array_equal(dab.to_array(r), A - B * A)
    M = rng.standard_normal((6, 5, 1, 1, 4)).astype(np.float32)                 # extruded middle dims, plain array -> distributed
    r2 = dab.broadcast(lambda x, m: x - m * x, a, M)
    assert np.array_equal(dab.to_array(r2), A - M * A)
    dest = dab.similar(a)
    dab.broadcast_into(dest, lambda x, y: dab.sqrt(dab.abs2(x) + dab.abs2(y)), a, b)
    assert np.array_equal(dab.to_array(dest), np.sqrt(A * A + B * B))
    Cc = rng.integers(-50, 50, (6, 5, 4, 3, 4, 5)).astype(np.int64)
    e = dab.distribute(Cc, procs=list(range(1, 9)), dist=(2, 1, 2, 1, 2, 1))
    r3 = dab.broadcast(lambda x: x * x + 2 * x - 1, e)                          # result has the default layout: operands are halo-fetched
    assert np.array_equal(dab.to_array(r3), Cc * Cc + 2 * Cc - 1)
    V = rng.integers(-5, 5, (6, 1, 4, 1, 4, 1)).astype(np.int64)                # alternating extrusion: 6 groups, does not collapse
    with pytest.raises(dab.UnsupportedError):
        dab.broadcast(lambda x, v: x * v + v, e, V)


@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.int32, np.int64])
@pytest.mark.parametrize("transA", [False, True])
def test_gemm_single_column_goes_through_gemv(dab, rt1, dtype, transA):
    """``A * b`` with a one-column ``b`` (n == 1, dense A): served by K9 -- fp64 / wrap-around carriers, so Float32 is within one
    rounding of the fp64 product and integers are exact; the same call with a padded leading dimension stays on K12."""
    from test_gpu_gemm import check_float, gemm
    rng = np.random.default_rng(101)
    for m, k in [(4096, 2048), (1000, 37), (1, 1), (37, 4099)]:
        shape = (k, m) if transA else (m, k)
        if np.dtype(dtype).kind == "f":
            A, B = rng.standard_normal(shape).astype(dtype), rng.standard_normal((k, 1)).astype(dtype)
            n0 = rt1.launches()
            R = gemm(dab, rt1, A, B, transA)
            assert R.shape == (m, 1) and rt1.launches() > n0
            check_float(R, A, B, transA, 1.2e-7 if dtype == np.float32 else 1e-15 * max(k, 8))
            ra = A.shape[0]
            Rp = gemm(dab, rt1, A, B, transA, lda=(ra + 3) // 4 * 4 + 4)        # padded lda: not a dense chunk -> the tile kernels
            check_float(Rp, A, B, transA, 2e-6 if dtype == np.float32 else 1e-15 * max(k, 8))
        else:
            hi = 2 ** 20 if dtype == np.int32 else 2 ** 40
            A, B = rng.integers(-hi, hi, shape).astype(dtype), rng.integers(-hi, hi, (k, 1)).astype(dtype)
            with np.errstate(over="ignore"):
                want = (A.T if transA else A) @ B
            assert np.array_equal(gemm(dab, rt1, A, B, transA), want)


def test_norm_other_p(dab, rt8):
    """``norm(x, p)`` (src/linalg.jl:48-59) beyond p = 1, 2, Inf: -Inf, 0 and a general p, against NumPy in Float64."""
    rng = np.random.default_rng(48)
    for T in (np.float64, np.float32, np.int64):
        a = (rng.standard_normal(10007) * 3).astype(T)
        a[::97] = 0
        d = dab.distribute(a)
        a64 = a.astype(np.float64)
        assert float(dab.norm(d, 0)) == float(np.count_nonzero(a))
        assert float(dab.norm(d, -np.inf)) == float(np.abs(a64).min()) and float(dab.norm(d, np.inf)) == float(np.abs(a64).max())
        for p in (3, 2.5, 0.5):
            got = dab.norm(d, p)
            want = float((np.abs(a64) ** p).sum() ** (1.0 / p))
            assert abs(float(got) - want) <= (2e-6 if T == np.float32 else 1e-12) * want, (T, p)
            assert isinstance(got, np.float32) == (T == np.float32)


def test_copy_deepcopy_drandn(dab, rt8):
    """test/darray.jl:84-131: a copy equals the original and owns its localparts; ``drandn`` (src/darray.jl:526-532) gives finite
    standard-normal entries that do not depend on the layout."""
    D = dab.drand((200, 200), procs=[1, 2])
    A = dab.to_array(D)
    for cp in (dab.copy, dab.deepcopy):
        DC = cp(D)
        assert dab.isequal(D, DC) and list(DC.layout.pids) == list(D.layout.pids)
        dab.fill_(DC, 0.0)                                                       # writing into the copy ...
        assert np.array_equal(dab.to_array(D), A) and not dab.isequal(D, DC)     # ... never shows in the original
        DC.close()
    E = dab.distribute(A, procs=[1, 2, 3, 4], dist=[1, 4])                       # a dist that similar() does not inherit
    EC = dab.copy(E)
    assert np.array_equal(dab.to_array(EC), A)
    for T in (np.float64, np.float32):
        n1 = dab.to_array(dab.drandn((300, 400), dtype=T))
        n2 = dab.to_array(dab.drandn((300, 400), procs=[1, 2, 3], dist=[3, 1], dtype=T))
        assert n1.dtype == np.dtype(T) and np.array_equal(n1, n2) and np.all(np.isfinite(n1))
        assert abs(float(n1.mean())) < 0.02 and abs(float(n1.std()) - 1.0) < 0.02 and float(np.abs(n1).max()) > 3.0
        assert not np.array_equal(n1, dab.to_array(dab.drandn((300, 400), dtype=T, seed=99)))
    v = dab.drandn((20,))
    assert abs(float(dab.norm(v)) - float(np.linalg.norm(dab.to_array(v)))) < 1e-7   # test/darray.jl:946-957
    # test/darray.jl:225-234 "test copy!": copyto!(D2, D1) with D2 built from irregular chunks (3 + 7 rows), D1 = dzeros; on the devices
    rng = np.random.default_rng(225)
    D1 = dab.dzeros((10, 10))
    D2 = dab.darray_from_chunks([rng.standard_normal((3, 10)), rng.standard_normal((7, 10))], (2, 1))
    assert dab.copyto(D2, D1) is D2 and dab.isequal(D1, D2) and np.array_equal(dab.to_array(D2), np.zeros((10, 10)))
    R = rng.standard_normal((10, 10))
    dab.copyto(D2, dab.distribute(R)[0:10, 0:10])                                 # a SubDArray source
    assert np.array_equal(dab.to_array(D2), R) and D2.layout.indices[0][0] == (1, 3)
    with pytest.raises(dab.DimensionMismatch):
        dab.copyto(D2, dab.dzeros((10, 9)))


def test_multi_argument_mapreduce_with_dims(dab, rt8):
    """``mapreduce(f, op, A, B; dims)`` = ``reduce(op, map(f, A, B); dims)`` (Base) on DArrays."""
    rng = np.random.default_rng(3)
    A, B = rng.integers(-9, 9, (60, 70)).astype(np.int64), rng.integers(-9, 9, (60, 70)).astype(np.int64)
    a, b = dab.distribute(A), dab.distribute(B)
    for dims, axis in ((1, 0), (2, 1), ((1, 2), (0, 1))):
        r = dab.mapreduce(lambda x, y: x * y + 1, "+", a, b, dims=dims)
        assert np.array_equal(dab.to_array(r), (A * B + 1).sum(axis=axis, keepdims=True))
    r = dab.mapreduce(lambda x, y: x - y, "max", a, 3, dims=2)                  # a scalar argument
    assert np.array_equal(dab.to_array(r), (A - 3).max(axis=1, keepdims=True))


def test_reshape_dvector(dab, rt8):
    """``reshape(A::DVector, d::Dims)`` (src/darray.jl:612-636; test/darray.jl:150-165): column-major relabelling into a new DArray with the
    default layout; ``DimensionMismatch`` unless the sizes agree; ``nnz``."""
    rng = np.random.default_rng(612)
    for n, dims in ((40000, (100, 400)), (40000, (200, 200)), (360, (3, 4, 5, 6)), (17 * 9, (17, 9)), (64, (64,)), (64, (1, 64))):
        a = rng.standard_normal(n)
        d = dab.distribute(a)
        r = dab.reshape(d, dims)
        assert r.dims == dims and np.array_equal(dab.to_array(r), a.reshape(dims, order="F")), dims
        assert list(r.layout.indices) == list(dab.similar(r).layout.indices)
    with pytest.raises(dab.DimensionMismatch):
        dab.reshape(d, (100, 100))
    with pytest.raises(dab.UnsupportedError):
        dab.reshape(r, (64,))                                                   # only a one-dimensional DArray, as in the reference
    ii = rng.integers(-3, 3, 600).astype(np.int32)
    di = dab.distribute(ii)
    assert np.array_equal(dab.to_array(dab.reshape(di, (20, 30))), ii.reshape((20, 30), order="F"))
    assert dab.nnz(di) == int(np.count_nonzero(ii))


def test_predicates_with_dims(dab, rt8):
    """``count(f, d; dims)`` -> Int64 DArray, ``any`` / ``all(f, d; dims)`` -> Bool DArray (Base routes them through mapreduce(...; dims), i.e.
    the reference's mapreducedim!, src/mapreduce.jl:83-94), for every kind of region; Bool arrays without a predicate; the whole-array forms
    are unchanged."""
    rng = np.random.default_rng(1)
    A = rng.integers(-5, 5, (30, 22, 6)).astype(np.int64)
    a = dab.distribute(A)
    for dims, axis in ((1, 0), (2, 1), ((1, 3), (0, 2)), ((1, 2, 3), (0, 1, 2))):
        c = dab.count(a, lambda x: x > 2, dims=dims)
        assert c.dtype == np.int64 and np.array_equal(dab.to_array(c), (A > 2).sum(axis=axis, keepdims=True)), dims
        assert np.array_equal(dab.to_array(dab.any(a, lambda x: x > 3, dims=dims)), (A > 3).any(axis=axis, keepdims=True))
        r = dab.to_array(dab.all(a, lambda x: x > -5, dims=dims))
        assert r.dtype == np.bool_ and np.array_equal(r, (A > -5).all(axis=axis, keepdims=True))
    B = A > 0
    b = dab.distribute(B)
    assert np.array_equal(dab.to_array(dab.count(b, dims=2)), B.sum(axis=1, keepdims=True))
    assert np.array_equal(dab.to_array(dab.all(b, dims=(1, 2))), B.all(axis=(0, 1), keepdims=True))
    with pytest.raises(TypeError):
        dab.count(a, dims=1)                                                    # non-boolean used in boolean context
    assert dab.count(a, lambda x: x > 2) == int((A > 2).sum()) and dab.all(b) == bool(B.all())


def test_reference_scalar_math_vocabulary(dab, rt8):
    """test/darray.jl:775-797 (``f.(a) == f.(b)`` for a = drand(20, 20)): here ``f.(d)`` on the device against NumPy / SciPy in the same
    precision.  Transcendental kernels are libdevice's (1-2 ulp for the elementary functions, up to ~10 ulp documented for tgamma / erfinv /
    erfc in double), so the comparison is at 6 ulp, 16 ulp for the special functions; the functions that are exact by construction (trunc, round, isinf, isfinite, deg2rad, rad2deg as one multiplication) are bit-exact."""
    import scipy.special as sp
    rng = np.random.default_rng(775)
    for T in (np.float64, np.float32):
        A = rng.random((20, 20)).astype(T)
        B = A + T(1)
        d, d1 = dab.distribute(A), dab.distribute(B)
        one, pi = T(1), T(np.pi)
        cases = [("acos", A, np.arccos), ("asin", A, np.arcsin), ("atan", A, np.arctan), ("asinh", A, np.arcsinh), ("atanh", A, np.arctanh),
                 ("acosh", B, np.arccosh), ("cbrt", A, np.cbrt), ("cosh", A, np.cosh), ("sinh", A, np.sinh), ("exp2", A, np.exp2),
                 ("exp10", A, lambda v: np.power(T(10), v)), ("expm1", A, np.expm1), ("log10", B, np.log10), ("log2", B, np.log2),
                 ("log1p", A, np.log1p),
                 # reference without cancellation: 1 - v and 0.5 - v are exact here, so the small results near v = 1 (v = 0.5) keep full precision
                 ("sinpi", A, lambda v: np.sin(np.pi * np.where(v > 0.5, 1.0 - v.astype(np.float64), v.astype(np.float64)))),
                 ("cospi", A, lambda v: np.where(v > 0.25, np.sin(np.pi * (0.5 - v.astype(np.float64))), np.cos(np.pi * v.astype(np.float64)))),
                 ("erf", A, sp.erf), ("erfc", A, sp.erfc), ("erfcx", A, sp.erfcx), ("erfinv", A * T(0.99), sp.erfinv),
                 ("erfcinv", B * T(0.5), sp.erfcinv), ("gamma", B, sp.gamma), ("loggamma", B + T(1.5), sp.gammaln),
                 ("sec", A, lambda v: one / np.cos(v)), ("csc", B, lambda v: one / np.sin(v)), ("cot", B, lambda v: one / np.tan(v)),
                 ("sech", A, lambda v: one / np.cosh(v)), ("csch", B, lambda v: one / np.sinh(v)), ("coth", B, lambda v: one / np.tanh(v)),
                 ("asec", B, lambda v: np.arccos(one / v)), ("acsc", B, lambda v: np.arcsin(one / v)), ("acot", B, lambda v: np.arctan(one / v)),
                 ("asech", B * T(0.4), lambda v: np.arccosh(one / v)), ("acsch", B, lambda v: np.arcsinh(one / v)),
                 ("acoth", B + one, lambda v: np.arctanh(one / v))]
        srcs = {}
        for nm, H, ref in cases:
            if id(H) not in srcs:
                srcs[id(H)] = dab.distribute(np.ascontiguousarray(H))
            f = getattr(dab, nm)
            got = dab.to_array(dab.map_(lambda x: f(x), srcs[id(H)]))
            want = np.asarray(ref(H)).astype(T)
            assert got.dtype == np.dtype(T)
            ulp = np.spacing(np.abs(want).astype(T))
            tol = 16 if nm in ("erfc", "erfcx", "erfinv", "erfcinv", "gamma", "loggamma", "sinpi", "cospi") else 6
            assert np.all(np.abs(got.astype(np.float64) - want.astype(np.float64)) <= tol * ulp.astype(np.float64)), (nm, T)
        # exact ones
        S = ((A - T(0.5)) * T(10)).astype(T)
        S[0, :4] = [np.inf, -np.inf, np.nan, T(2.5)]
        ds = dab.distribute(S)
        for nm, ref in (("trunc", np.trunc), ("round_", np.rint)):
            f = getattr(dab, nm)
            assert np.array_equal(dab.to_array(dab.map_(lambda x: f(x), ds)), ref(S), equal_nan=True), nm
        assert np.array_equal(dab.to_array(dab.map_(lambda x: dab.isinf(x), ds)), np.isinf(S))
        assert np.array_equal(dab.to_array(dab.map_(lambda x: dab.isfinite(x), ds)), np.isfinite(S))
        assert np.array_equal(dab.to_array(dab.map_(lambda x: dab.deg2rad(x), d)), A * (pi / T(180)))
        assert np.array_equal(dab.to_array(dab.map_(lambda x: dab.rad2deg(x), d)), A * (T(180) / pi))
        assert abs(float(dab.sum(d1, lambda x: dab.log2(x))) - float(np.log2(B.astype(np.float64)).sum())) <= 1e-5 * B.size   # inside a fused mapreduce


def test_reference_shift_ops(dab, rt8):
    """test/darray.jl:863-867: ``f.(a, 2) == f.(b, 2)``, ``f.(2, a) == f.(2, b)``, ``f.(a, a) == f.(b, b)`` for f in (<<, >>) on
    ``a = dones(Int, 20, 20)``; plus counts that are negative or past the width, Int32 values, against the Julia-semantics model."""
    import hostmem_abi as hm
    a = dab.dones((20, 20), dtype=np.int64)
    ones = np.ones((20, 20), dtype=np.int64)
    assert np.array_equal(dab.to_array(dab.map_(lambda x: x << 2, a)), ones << 2)
    assert np.array_equal(dab.to_array(dab.map_(lambda x: 2 << x, a)), 2 << ones)
    assert np.array_equal(dab.to_array(dab.broadcast(lambda x, y: x << y, a, a)), ones << ones)
    assert np.array_equal(dab.to_array(dab.map_(lambda x: x >> 2, a)), ones >> 2)
    assert np.array_equal(dab.to_array(dab.map_(lambda x: 2 >> x, a)), 2 >> ones)
    assert np.array_equal(dab.to_array(dab.broadcast(lambda x, y: x >> y, a, a)), ones >> ones)
    rng = np.random.default_rng(863)
    for T, bits in ((np.int64, 64), (np.int32, 32)):
        X = rng.integers(np.iinfo(T).min, np.iinfo(T).max, (37, 11), dtype=T)
        N = rng.integers(-80, 80, (37, 11)).astype(np.int64)
        dx, dn = dab.distribute(X), dab.distribute(N)
        for left, f in ((True, lambda x, n: x << n), (False, lambda x, n: x >> n)):
            got = dab.to_array(dab.broadcast(f, dx, dn))
            want = np.vectorize(lambda x, n: hm.jl_shift(int(x), int(n), bits, left), otypes=[T])(X, N)
            assert got.dtype == np.dtype(T) and np.array_equal(got, want), (T, left)


def test_reference_int128_mapreduce_is_exact(dab, rt8):
    """test/darray.jl:286-294 as written: 25 random vectors of 1:5, length 2..30, f Int128-valued, ``mapreduce(f, opt, DA)`` EXACTLY equal
    to the local result (here: Python's exact integers wrapped to 128 bits; the products overflow Int64 by far)."""
    rng = np.random.default_rng(286)
    fs = [(lambda x: dab.Int128(2 * x), lambda v: 2 * v), (lambda x: dab.Int128(x) ** 2, lambda v: v * v),
          (lambda x: dab.Int128(x) ** 2 + 2 * dab.Int128(x) - 1, lambda v: v * v + 2 * v - 1)]
    for _ in range(25):
        a = rng.integers(1, 6, int(rng.integers(2, 31))).astype(np.int64)
        if a.size < 8:
            a = np.resize(a, 8)                                                 # rt8: at least one element per worker, like the reference's 4 procs
        d = dab.distribute(a)
        od = orc.distribute(a, nworkers=8)
        for tf, pf in fs:
            for op in ("+", "*"):
                got = dab.mapreduce(tf, op, d)
                assert isinstance(got, int) and got == orc.darray_mapreduce_int128(pf, op, od), (a, op)
        d.close()
    # a long vector: many CTAs, the 16-byte shuffles and partials of the Int128 carrier; the sum passes 2^64
    n = INT128_BIG_N
    a = rng.integers(-2 ** 62, 2 ** 62, n).astype(np.int64)
    d = dab.distribute(a)
    want = sum(int(v) * 8 for v in a)
    assert dab.mapreduce(lambda x: dab.widen(x) * 8, "+", d) == want and abs(want) >= 0
    assert dab.mapreduce(lambda x: dab.widen(x) * (2 ** 40), "max", d) == int(a.max()) * 2 ** 40
    assert dab.mapreduce(lambda x: dab.widen(x) * (2 ** 40), "min", d) == int(a.min()) * 2 ** 40
    with pytest.raises(dab.UnsupportedError):
        dab.map_(lambda x: dab.Int128(x), d)                                    # no arrays of Int128


def _sort_by_key(dab, rt, keys, vals):
    from darray_b200 import _lib
    n = keys.size
    dk, dv = dab.B200Array.from_numpy(rt, keys), dab.B200Array.from_numpy(rt, vals)
    out = dab.B200Array.empty(rt, (n,), vals.dtype)
    need = C.c_size_t()
    _lib.check(_lib.lib().dab_sort_by_key_scratch_bytes(dab.dab_dtype(keys.dtype), n, C.byref(need)))
    scratch = dab.B200Array.empty(rt, (need.value,), np.uint8)
    _lib.call("dab_sort_by_key", rt.ctx, dab.dab_dtype(keys.dtype), C.c_void_p(dk.ptr), vals.itemsize, C.c_void_p(dv.ptr), C.c_void_p(out.ptr),
              C.c_void_p(scratch.ptr), need.value, n)
    got = out.to_numpy()
    assert np.array_equal(dk.to_numpy().view(np.uint8), keys.view(np.uint8)) and np.array_equal(dv.to_numpy(), vals)   # inputs are never written
    for b in (dk, dv, out, scratch):
        b.free()
    return got


@pytest.mark.parametrize("KT", [np.float32, np.float64, np.int32, np.int64])
def test_sort_by_key_kernel(dab, rt1, KT):
    rng = np.random.default_rng(71)
    for n in SORT_BY_KEY_SIZES:
        if np.dtype(KT).kind == "f":
            keys = np.round(rng.standard_normal(n) * 10.0 ** rng.integers(-3, 3, n), 2).astype(KT)        # many ties
            if n > 64:
                keys[rng.integers(0, n, n // 16)] = rng.choice(np.array([np.nan, -np.nan, 0.0, -0.0, np.inf, -np.inf], dtype=KT), n // 16)
                raw = keys.view(np.uint32 if KT == np.float32 else np.uint64)                           # NaN payloads: still ONE key
                raw[5] = raw.dtype.type(0x7FC00123 if KT == np.float32 else 0x7FF8000000000123)
                raw[9] = raw.dtype.type(0xFFC00001 if KT == np.float32 else 0xFFF8000000000001)
        else:
            keys = rng.integers(np.iinfo(KT).min, np.iinfo(KT).max, n, dtype=KT)
            keys[rng.integers(0, n, max(1, n // 2))] = KT(7)
            if n > 64:
                keys[:4] = [np.iinfo(KT).min, np.iinfo(KT).max, -1, 0]
        perm = orc.jl_sortperm_stable(keys)
        for VT in (np.float32, np.int64):
            vals = np.arange(n).astype(VT)                                      # the value IS the input position: checks stability exactly
            assert np.array_equal(_sort_by_key(dab, rt1, keys, vals), vals[perm]), (KT, VT, n)


def _by_cases(dab, T):
    cases = [(lambda x: abs(x), lambda v: np.abs(v)), (lambda x: x, lambda v: v), (lambda x: -x, lambda v: -v)]
    if np.dtype(T).kind == "i":
        cases += [(lambda x: dab.rem(x, 7), lambda v: np.fmod(v, np.dtype(T).type(7))), (lambda x: x * 0.5, lambda v: v * 0.5),
                  (lambda x: x > 3, lambda v: (v > 3).astype(np.int32))]
    else:
        cases += [(lambda x: dab.floor(x * 4), lambda v: np.floor(v * np.dtype(T).type(4))),
                  (lambda x: dab.ifelse(x > 0.5, x, 1 - x), lambda v: np.where(v > np.dtype(T).type(0.5), v, np.dtype(T).type(1) - v))]
    return cases


@pytest.mark.parametrize("T", [np.int64, np.float64, np.float32, np.int32])
def test_darray_sort_by(dab, rt8, T):
    """Result, boundaries, result layout and per-worker chunks equal the oracle's -- including the reference's behaviour of shipping
    nothing behind the last split point when ``by(typemax(T))`` is not the largest key (see ``orc.darray_sort``)."""
    rng = np.random.default_rng(81)
    for n in (8, 1000, 200003):
        a = rng.integers(-50, 50, n).astype(T) if np.dtype(T).kind == "i" else rng.random(n).astype(T)
        d = dab.distribute(a)
        od = orc.distribute(a, nworkers=8)
        smp = a[rng.integers(0, n, min(n, 64))]
        lohi = (T(-60), T(60)) if np.dtype(T).kind == "i" else (T(0), T(1))
        for sample in (True, False, lohi, smp):
            for tby, nby in _by_cases(dab, T):
                try:
                    o2, ob = orc.darray_sort(od, sample, by=nby)
                except ValueError:
                    with pytest.raises(dab.ArgumentError):
                        dab.sort_with_boundaries(d, sample, tby)
                    continue
                d2, b = dab.sort_with_boundaries(d, sample, tby)
                assert np.array_equal(b, ob, equal_nan=True)
                assert list(d2.layout.pids) == o2.pids and list(d2.layout.indices) == o2.indices
                for pid, ch in d2.chunks.items():
                    assert np.array_equal(ch.to_numpy().view(np.uint8), o2.chunks[o2.pids.index(pid)].view(np.uint8)), (n, tby)
                d2.close()
        d.close()
