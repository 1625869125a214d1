"""CPU-only tests (run with -m "not gpu"): the C-ABI library loads and exports every declared symbol, host-side logic of the
product (layout math, tracer / promotion / lowering, ordered combine, NVRTC code generation) and the C oracle vs the NumPy
oracle.  No kernel is launched here.
"""
import ctypes as C
import os
import sys
import re

import numpy as np
import pytest

from oracle import core as ocore
from oracle import darray_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ C ABI
def test_library_exports_every_declared_symbol(dab):
    from darray_b200 import _lib

    hdr = open(os.path.join(ROOT, "include", "dab200.h")).read()
    declared = set(re.findall(r"\b(dab_[a-z0-9_]+)\s*\(", hdr)) - {"dab_ctx"}
    L = _lib.lib()
    for name in sorted(declared):
        assert hasattr(L, name), f"libdab200.so does not export {name}"
    assert declared == set(_lib.EXPORTS), (declared ^ set(_lib.EXPORTS))
    assert L.dab_abi_version() == 1
    assert L.dab_status_string(_lib.ERR_EMPTY).decode().startswith("ArgumentError")


def test_no_gpu_means_loud_failure_not_fallback(dab):
    """Without a GPU the product must raise, never compute on the host."""
    from darray_b200 import _lib

    n = C.c_int32(-1)
    st = _lib.lib().dab_device_count(C.byref(n))
    if st == _lib.OK and n.value > 0:
        pytest.skip("a GPU is visible")
    with pytest.raises(_lib.DabError):
        dab.Runtime(use_dist=False)


def test_combine_ordered_is_a_left_fold_in_the_result_type(dab):
    """dab_combine_ordered == reduce(op, results) (reference src/mapreduce.jl:34): host-only entry point."""
    from darray_b200 import _lib

    L = _lib.lib()
    v = np.array([1e8, 1.0, -1e8, 1.0, 3.0], dtype=np.float32)
    out = np.zeros(1, dtype=np.float32)
    _lib.check(L.dab_combine_ordered(_lib.F32, _lib.SUM, C.c_void_p(v.ctypes.data), v.size, C.c_void_p(out.ctypes.data)))
    fold = v[0]
    for x in v[1:]:
        fold = np.float32(fold + x)
    assert out[0] == fold == ocore.lib().orc_fold_sum_f32(v.ctypes.data_as(C.POINTER(C.c_float)), v.size)
    for op, vals, want in [(_lib.MAX, [1.0, np.nan, 3.0], np.nan), (_lib.MAX, [-0.0, 0.0], 0.0), (_lib.MIN, [0.0, -0.0], -0.0),
                           (_lib.MIN, [2.0, -1.0, 5.0], -1.0), (_lib.PROD, [2.0, 3.0, 0.5], 3.0)]:
        a = np.array(vals, dtype=np.float32)
        _lib.check(L.dab_combine_ordered(_lib.F32, op, C.c_void_p(a.ctypes.data), a.size, C.c_void_p(out.ctypes.data)))
        assert (np.isnan(out[0]) and np.isnan(want)) or (out[0] == want and np.signbit(out[0]) == np.signbit(np.float32(want)))
    iv = np.array([2**62, 2**62, 5], dtype=np.int64)
    io = np.zeros(1, dtype=np.int64)
    _lib.check(L.dab_combine_ordered(_lib.I64, _lib.SUM, C.c_void_p(iv.ctypes.data), 3, C.c_void_p(io.ctypes.data)))
    assert io[0] == np.int64(-2**63 + 5)  # wraps like Julia Int64
    assert L.dab_combine_ordered(_lib.F32, _lib.SUM, C.c_void_p(v.ctypes.data), 0, C.c_void_p(out.ctypes.data)) == _lib.ERR_EMPTY
    dt = C.c_int32()
    for (d, op, m, want) in [(_lib.F32, _lib.SUM, _lib.MAP_ID, _lib.F32), (_lib.I32, _lib.SUM, _lib.MAP_ID, _lib.I64),
                             (_lib.I32, _lib.MAX, _lib.MAP_ID, _lib.I32), (_lib.F64, _lib.COUNT, _lib.MAP_GT, _lib.I64),
                             (_lib.F32, _lib.SUM, _lib.MAP_GT, _lib.I64), (_lib.F64, _lib.PROD, _lib.MAP_ABS, _lib.F64)]:
        assert L.dab_reduce_result_dtype(d, op, m, C.byref(dt)) == 0 and dt.value == want


# ------------------------------------------------------------------------------------------------ layout (product) vs oracle
def test_layout_matches_oracle_exhaustively(dab):
    rng = np.random.default_rng(0)
    cases = [((50,), 4), ((3,), 2), ((1024, 1024), 2), ((1 << 33,), 8), ((65536, 65536), 8), ((73, 73), 2), ((20, 20, 20), 8), ((7, 1), 8), ((1, 9), 8),
             ((2, 3, 5, 4), 8), ((100, 100), 6), ((5, 5), 7), ((2, 2), 8), ((1,), 3)]
    for _ in range(200):
        nd = int(rng.integers(1, 5))
        cases.append((tuple(int(x) for x in rng.integers(1, 40, nd)), int(rng.integers(1, 17))))
    for dims, nw in cases:
        procs = list(range(1, orc.default_nprocs(dims, nw) + 1))
        assert dab.layout.default_procs(dims, list(range(1, nw + 1))) == procs
        lay, od = dab.make_layout(dims, procs), orc.make_layout(dims, procs)
        assert lay.grid == tuple(od.grid) and lay.pids == od.pids and lay.indices == od.indices and lay.cuts == od.cuts, (dims, nw)
        assert dab.defaultdist(dims, len(procs)) == tuple(orc.defaultdist_grid(dims, len(procs)))
    assert dab.cuts_for(50, 4) == [1, 14, 27, 39, 51]                    # reference test/darray.jl:66
    with pytest.raises(ValueError):
        dab.make_layout((4, 4), [])
    lay = dab.make_layout((200, 200), [1, 2])
    assert lay.locate(1, 101) == (1, 2) and lay.locate(200, 100) == (1, 1)
    with pytest.raises(ValueError):
        lay.locate(1, 201)
    l2 = dab.layout.layout_from_chunk_shapes([(3, 10), (7, 10)], (2, 1), [1, 2])
    o2 = orc.from_chunks([np.zeros((3, 10)), np.zeros((7, 10))], (2, 1), [1, 2])
    assert l2.dims == o2.dims and l2.indices == o2.indices and l2.cuts == o2.cuts


def test_slab_plan_matches_oracle(dab):
    rng = np.random.default_rng(1)
    for _ in range(100):
        nd = int(rng.integers(1, 4))
        dims = tuple(int(x) for x in rng.integers(2, 30, nd))
        procs = list(range(1, orc.default_nprocs(dims, 8) + 1))
        lay, od = dab.make_layout(dims, procs), orc.make_layout(dims, procs)
        J = []
        for s in dims:
            lo = int(rng.integers(1, s + 1))
            J.append((lo, int(rng.integers(lo, s + 1))))
        got = [(p.chunk, p.src, p.dst, p.whole_chunk) for p in dab.slab_plan(lay, J)]
        assert got == [tuple(x) for x in orc.slab_plan(od, J)]


def test_collapse_for_region(dab):
    c = dab.layout.collapse_for_region
    assert c((32768, 16384), {1}) == [(True, 32768), (False, 16384)]
    assert c((4, 5, 6), {1, 2}) == [(True, 20), (False, 6)]
    assert c((4, 5, 6), {1, 3}) == [(True, 4), (False, 5), (True, 6)]
    assert c((4, 5, 6), {2}) == [(False, 4), (True, 5), (False, 6)]


# ------------------------------------------------------------------------------------------------ tracer / promotion / lowering
def test_tracer_promotion_follows_julia():
    from darray_b200 import abs2, ifelse, sqrt
    from darray_b200._broadcast import codegen, convert, match_affine, trace

    f32 = np.float32
    e = trace(lambda x: 2 * x + 1, ["f32"])                                   # map!(x->2x+1): Int literals adopt Float32
    assert e.jt == "f32" and match_affine(e) == (2.0, 1.0)
    assert match_affine(trace(lambda x: f32(1.5) * x + f32(0.25), ["f32"])) == (1.5, 0.25)
    assert match_affine(trace(lambda x: f32(0.25) + x * f32(1.5), ["f32"])) == (1.5, 0.25)
    assert match_affine(trace(lambda x: x + 3, ["i64"])) == (1, 3)
    assert trace(lambda x: 1.5 * x, ["f32"]).jt == "f64"                       # Float64 literal * Float32 -> Float64
    assert trace(lambda x: f32(1.5) * x, ["f32"]).jt == "f32"
    assert trace(lambda x: x + 1, ["i32"]).jt == "i64"                         # Int32 + (Int64 literal) -> Int64
    assert trace(lambda x: x / 2, ["i64"]).jt == "f64"                         # Int / Int -> Float64
    assert trace(lambda x: x > 1.0, ["f64"]).jt == "bool"
    assert trace(lambda x, y: x * y, ["f32", "f64"]).jt == "f64"
    assert trace(lambda x: sqrt(x), ["i64"]).jt == "f64"
    assert trace(lambda x: x ** 2, ["i64"]).key() == "mul:i64(a0:i64,a0:i64)"   # literal_pow
    assert trace(lambda x: 1, ["f64"]).op == "const"                           # map(x->1, D)
    src = codegen(convert(trace(lambda a, m, c: a - m * abs2(c), ["f64", "f64", "f64"]), "f64"))
    assert src == "jl_sub(a0, jl_mul(a1, jl_abs2(a2)))"
    assert "?" in codegen(trace(lambda x, y: ifelse(x < y, x, y), ["f32", "f32"]))
    with pytest.raises(TypeError):
        trace(lambda x: x if x > 0 else -x, ["f32"])                            # data-dependent Python control flow


def test_classify_map_for_reductions():
    from darray_b200 import _lib, abs2
    from darray_b200._mapreduce import classify_map

    assert classify_map(None, np.float32)[0] == _lib.MAP_ID
    assert classify_map(lambda x: x, np.float32)[0] == _lib.MAP_ID
    assert classify_map(abs, np.int64)[0] == _lib.MAP_ABS
    assert classify_map(abs2, np.float32)[0] == _lib.MAP_ABS2
    assert classify_map(lambda t: t * t, np.float64)[0] == _lib.MAP_ABS2
    code, p, _ = classify_map(lambda x: x > 1.0, np.float64)
    assert code == _lib.MAP_GT and p == 1.0
    code, p, _ = classify_map(lambda x: 2.0 == x, np.float64)
    assert code == _lib.MAP_EQ and p == 2.0
    code, p, _ = classify_map(lambda x: 3 < x, np.int64)
    assert code == _lib.MAP_GT and p == 3
    assert classify_map(lambda x: 2 * x, np.int64)[0] is None                 # general f -> fused map kernel + identity reduce


def test_nvrtc_codegen_compiles_for_sm100a(dab):
    """The exact source dab_broadcast_expr would JIT, compiled with NVRTC for sm_100a on this CPU-only box."""
    from darray_b200 import _lib, abs2, ifelse, jl_max, mod, sin, sqrt
    from darray_b200._broadcast import codegen, convert, trace

    L = _lib.lib()
    code = {"f32": 0, "f64": 1, "i32": 2, "i64": 3, "bool": 4}
    cases = [(lambda a, m, c: a - m * sin(c), ["f64", "f64", "f64"], "f64"), (lambda z: 3 + abs2(z), ["f64"], "f64"),
             (lambda x, y: x % y, ["f32", "f32"], "f32"), (lambda x: x > 1.0, ["f64"], "bool"), (lambda x: 2 * x * x - 1, ["i64"], "i64"),
             (lambda x, y: ifelse(x < y, jl_max(x, y), sqrt(x)), ["f32", "f32"], "f32"), (lambda x, y: mod(x, y) // 3, ["i32", "i32"], "i64"),
             (lambda x, s: x * s + 1, ["f32", "f64"], "f64")]
    for f, tags, out in cases:
        e = trace(f, tags)
        src = codegen(convert(e, out)).encode()
        n = len(tags)
        dts = (C.c_int32 * n)(*[code[t] for t in tags])
        arr = (C.c_int32 * n)(*([1] * (n - 1) + [0 if n > 1 else 1]))
        sz = C.c_size_t()
        st = L.dab_jit_compile_check(src, code[out], n, dts, arr, C.byref(sz))
        assert st == 0, L.dab_last_error(None)
        assert sz.value > 1000
    sz = C.c_size_t()
    bad = L.dab_jit_compile_check(b"a0 +* 1", 0, 1, (C.c_int32 * 1)(0), (C.c_int32 * 1)(1), C.byref(sz))
    assert bad == _lib.ERR_NVRTC and b"error" in L.dab_last_error(None)


# ------------------------------------------------------------------------------------------------ C oracle == NumPy oracle
@pytest.mark.parametrize("n", [1, 2, 15, 16, 17, 33, 34, 1023, 1024, 1025, 1026, 2049, 5000, 100003])
def test_c_oracle_matches_numpy_model_bit_for_bit(n):
    x = ocore.rand_u01_f32(1234, 7, n)
    assert np.array_equal(x, orc.rand_u01(1234, 7, n))
    assert ocore.rand_ksum(1234, 7, n) == orc.rand_u01_ksum(1234, 7, n) == ocore.ksum_f32(x)
    for simd in [(8, 4), (1, 1), (4, 2)]:
        assert ocore.sum_f32(x, *simd) == orc.julia_mapreduce(None, "+", x, simd=simd)
    x64 = x.astype(np.float64) * 1.1
    assert ocore.sum_f64(x64) == orc.julia_mapreduce(None, "+", x64)
    assert np.array_equal(ocore.affine_f32(x, 1.5, 0.25), orc.affine_unfused(1.5, x, 0.25))
    y = x - np.float32(0.5)
    if n > 3:
        y[n // 2] = -0.0
    assert ocore.max_f32(y) == orc.julia_mapreduce(None, "max", y) and ocore.min_f32(y) == orc.julia_mapreduce(None, "min", y)


def test_c_oracle_sumdim_matches_numpy_model():
    for inner, red, outer in [(1, 5000, 7), (1, 20, 9), (1, 12, 3), (6, 33, 4), (16, 4, 1)]:
        x = orc.rand_u01(3, 0, inner * red * outer)
        got = ocore.sumdim_f32(x, inner, red, outer)
        A = x.reshape((inner, red, outer), order="F")
        want = orc.julia_mapreducedim(None, "+", A, [2]).ravel(order="F")
        assert np.array_equal(got, want), (inner, red, outer)
    with pytest.raises(ValueError):
        ocore.max_f32(np.zeros(0, dtype=np.float32))


def test_workers_run_cpu_baseline_smoke():
    best, mean, res = ocore.workers_run(3, 2, 1 << 16, 1234, 1.5, 0.25, 1, 2)
    assert best > 0 and mean >= best
    # two map! passes were warm-up + 2 timed = 3 applications of a*x+b in place, then the sum of the last state
    x0 = orc.rand_u01(1234, 0, 1 << 16)
    x1 = orc.rand_u01(1234, 1 << 16, 1 << 16)
    for _ in range(3):
        x0, x1 = orc.affine_unfused(1.5, x0, 0.25), orc.affine_unfused(1.5, x1, 0.25)
    want = np.float32(ocore.sum_f32(x0) + ocore.sum_f32(x1))
    assert res == want


# ------------------------------------------------------------------------------------------------ committed golden fixtures
def test_golden_fixtures(dab):
    import json

    g = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))
    assert orc.defaultdist_cuts(50, 4) == g["reference_literals"]["defaultdist_50_4"]["value"] == dab.cuts_for(50, 4)
    assert repr(float(orc.julia_mapreduce(None, "+", np.full((100, 100), 1.1)))) == g["reference_literals"]["sum_fill_1p1_100x100_local"]["value"]
    for key, bits in g["rand_u01_f32_bits"].items():
        seed, start = [int(x[len(p):]) for x, p in zip(key.split("_"), ("seed", "start"))]
        assert [int(v) for v in orc.rand_u01(seed, start, 16).view(np.uint32)] == bits
        assert [int(v) for v in ocore.rand_u01_f32(seed, start, 16).view(np.uint32)] == bits
    assert ocore.rand_ksum(1234, 0, 65536) == g["rand_u01_ksum"]["seed1234_start0_n65536"]
    for key, lay in g["layouts"].items():
        dims, npids = key.split("_np")
        dims = tuple(int(x) for x in dims.split("x"))
        assert list(dab.defaultdist(dims, int(npids))) == lay["grid"]
        assert [dab.cuts_for(d, c) for d, c in zip(dims, lay["grid"])] == lay["cuts"]


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` must print ONE JSON line with the contract keys, using only the CPU."""
    import json
    import subprocess
    import sys

    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"], capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in j, k
    assert j["impl"] == "reference" and j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1 and j["value"] > 0
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["value"] == j["value"]


def test_bench_parity_fold_check_detects_a_swapped_order():
    """bench.py's `fold` check compares sum(y) with the Float32 LEFT fold of the chunk results in procs(d) order (reference
    src/mapreduce.jl:34): a fold in another order must not pass for chunk results of the bench's magnitude."""
    import importlib.util
    import os

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(0)
    differs = 0
    for _ in range(50):
        vals = (rng.random(8) * 1e6 + 2.68e8).astype(np.float32)          # 8 chunk sums of 2^30 values of mean 0.25..1.75
        a = bench.left_fold_f32(list(vals))
        b = bench.left_fold_f32(list(vals[::-1]))
        want = np.float32(0)
        acc = np.float32(vals[0])
        for v in vals[1:]:
            acc = np.float32(acc + v)
        assert a.tobytes() == acc.tobytes()
        differs += a.tobytes() != b.tobytes()
    assert differs > 10                                                    # the order is visible in Float32
    assert bench.rel_err(1.0 + 2e-6, 1.0) > bench.REL_TOL > bench.rel_err(1.0 + 5e-7, 1.0)


def test_collapse_dims_addresses_the_same_elements():
    """``collapse_dims`` (broadcast over more than 4 dimensions): walking the collapsed box with dense / zero strides must read exactly
    the elements NumPy's broadcasting reads."""
    from darray_b200 import _broadcast as bc
    from darray_b200 import _lib

    def walk(out_shape, arg_shapes, arrays):
        oc, ac = bc.collapse_dims(out_shape, arg_shapes)
        assert len(oc) <= 4, (out_shape, arg_shapes, oc)
        o4 = list(oc) + [1] * (4 - len(oc))
        n = int(np.prod(o4))
        idx = np.unravel_index(np.arange(n), o4, order="F")
        res = []
        for sh, a in zip(ac, arrays):
            s4 = list(sh) + [1] * (4 - len(sh))
            dense = bc._dense_strides(s4)
            strides = [dense[d] if s4[d] == o4[d] else 0 for d in range(4)]
            assert all(s4[d] in (o4[d], 1) for d in range(4))
            off = sum(idx[d] * strides[d] for d in range(4))
            res.append(a.reshape(-1, order="F")[off])
        return n, res

    rng = np.random.default_rng(3)
    cases = [((2, 3, 4, 5, 6), [(2, 3, 4, 5, 6), (2, 3, 1, 1, 6)]),
             ((2, 3, 4, 5, 6), [(2, 3, 4, 5, 6), (2, 3, 4, 5, 6), (1, 1, 1, 1, 1)]),
             ((6, 5, 4, 3, 4, 5), [(6, 5, 4, 3, 4, 5), (6, 1, 4, 3, 1, 1), (1, 5, 1, 1, 1, 1)]),
             ((3, 1, 2, 1, 4, 1, 5), [(3, 1, 2, 1, 4, 1, 5), (3, 1, 1, 1, 4)]),
             ((1, 1, 1, 1, 1), [(1, 1, 1, 1, 1)]),
             ((4, 3, 2, 2, 3), [(4, 1, 2, 1, 3), (1, 3, 1, 2, 1)])]
    for out_shape, arg_shapes in cases[:5]:
        arrays = [rng.standard_normal(sh) for sh in arg_shapes]
        n, res = walk(out_shape, arg_shapes, arrays)
        assert n == int(np.prod(out_shape))
        for sh, a, r in zip(arg_shapes, arrays, res):
            full = tuple(sh) + (1,) * (len(out_shape) - len(sh))
            want = np.broadcast_to(a.reshape(full), out_shape).reshape(-1, order="F")
            assert np.array_equal(r, want), (out_shape, sh)
    assert bc.collapse_dims((2, 3, 4, 5, 6), [(2, 3, 4, 5, 6)] * 3)[0] == (720,)
    assert bc.collapse_dims((2, 3, 4, 5, 6), [(2, 3, 4, 5, 6), (2, 3, 1, 1, 6)]) == ((6, 20, 6), [(6, 20, 6), (6, 1, 6)])
    oc, _ = bc.collapse_dims(*cases[5])                       # alternating extrusion patterns do not merge: 5 groups stay
    assert len(oc) == 5
    with pytest.raises(_lib.DimensionMismatch):
        bc.collapse_dims((2, 3, 4, 5, 6), [(2, 3, 4, 5, 7)])


def test_last_session_gpu_tests_dry_run_on_the_host_memory_abi(hostmem, dab):
    """The GPU tests of tests/test_gpu_zz_last_session.py that the host-memory ABI emulation can carry (all but the dab_gemm dispatch) are
    executed here, on CPU, exactly as written (same functions, a runtime on the emulation in place of the rt fixtures): the host runtime
    above the ABI -- tracer, run_local's routing and stride tables, collapse_dims, layouts, halo plans, the sort / Int128 / copy / norm
    flows -- runs for real, only the kernels are NumPy.  Whatever fails on the B200 later is then in a kernel or a binding, not in a typo,
    a shape or a wrong NumPy twin of the TEST, nor in the host logic."""
    import test_gpu_zz_last_session as z
    rt = dab.init(workers_per_rank=8, use_dist=False)
    z.test_broadcast_more_than_4_dims(dab, rt)                # the REAL run_local: collapse_dims + stride tables against the emulated 4-D box walk
    z.test_norm_other_p(dab, rt)
    z.test_copy_deepcopy_drandn(dab, rt)
    z.test_multi_argument_mapreduce_with_dims(dab, rt)
    z.test_predicates_with_dims(dab, rt)
    z.test_reshape_dvector(dab, rt)
    z.test_reference_shift_ops(dab, rt)
    z.test_reference_scalar_math_vocabulary(dab, rt)
    for T in (np.int64, np.float32):
        z.test_darray_sort_by(dab, rt, T)
    big, z.INT128_BIG_N = z.INT128_BIG_N, (1 << 12) + 5          # the emulator folds Python integers one by one
    try:
        z.test_reference_int128_mapreduce_is_exact(dab, rt)
    finally:
        z.INT128_BIG_N = big
    rt1 = dab.init(workers_per_rank=1, use_dist=False)
    sizes, z.SORT_BY_KEY_SIZES = z.SORT_BY_KEY_SIZES, (1, 2, 33, 1025, 4097)
    try:
        for KT in (np.float32, np.float64, np.int32, np.int64):
            z.test_sort_by_key_kernel(dab, rt1, KT)
    finally:
        z.SORT_BY_KEY_SIZES = sizes
    assert hostmem.launches > 1000, hostmem.launches          # the tests really drove the emulated entry points


def test_gpu_test_modules_against_the_host_memory_abi():
    """Host-runtime regression net: the ``-m gpu`` modules (hot path, widening, views, linalg host flows, sort, the last-session module)
    executed in a subprocess with ``DAB_HOSTMEM=1`` -- the C ABI emulated over host memory (tests/hostmem_abi.py), everything above it
    real.  Left out: the full-size tests (GiB-sized arrays), the tests that only make sense on the device (TMA variant, pinned H2D rates,
    the GEMM kernel module, multi-GPU).  A failure here is a regression in the HOST logic; the kernels are the ``-m gpu`` tier's job."""
    import subprocess
    env = dict(os.environ, DAB_HOSTMEM="1")
    mods = ["tests/test_gpu_hotpath.py", "tests/test_gpu_widen.py", "tests/test_gpu_views.py", "tests/test_gpu_linalg.py", "tests/test_gpu_sort.py",
            "tests/test_gpu_zz_last_session.py"]
    r = subprocess.run([sys.executable, "-m", "pytest", *mods, "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "--timeout", "600",
                        "-k", "not full_size and not tma_variant and not pinned_large and not bandwidth_shape and not transpose_large"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = "\n".join((r.stdout + r.stderr).splitlines()[-25:])
    assert r.returncode == 0, tail
    import re
    m = re.search(r"(\d+) passed", r.stdout)
    assert m and int(m.group(1)) >= 200, tail


def test_bench_host_logic_against_the_host_memory_abi():
    """bench.py end to end (N = 1, 2^16 elements, no extras, no CPU leg) with the C ABI emulated over host memory: the JSON line is complete
    and the in-run parity block -- exact sums, ordered fold, maximum, bit-exact windows -- comes out true.  Checks the HOST side of the
    driver-run artifact after changes to shared host code; the numbers themselves mean nothing here."""
    import json
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_on_hostmem.py"), "bench.py", "--log2n", "16", "--steps", "2", "--warmup", "3",
                        "--no-cpu", "--no-extras"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config",
                "roofline", "e2e", "gpu_launches", "clocks", "parity"):
        assert key in line, key
    assert line["parity"]["ok"] is True, line["parity"]
    assert line["n_gpus"] == 1 and line["steps"] == 2 and line["e2e"]["h2d_bytes_per_step"] == 4 * (1 << 16) and line["gpu_launches"] > 0


@pytest.mark.parametrize("log2n", [16, 23])
def test_bench_dump_outputs_against_the_host_memory_abi(tmp_path, log2n):
    """``bench.py --dump-outputs DIR`` (C ABI emulated over host memory): y.npy holds y = fl(fl(a*x)+b) bit-exact -- all of it at 2^16
    elements, the seeded windows at 2^23 -- sum.npy the printed sum, and a second run with the same arguments writes the same files."""
    import importlib.util
    import json
    import subprocess
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = 1 << log2n
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_on_hostmem.py"), "bench.py", "--log2n", str(log2n), "--steps", "1",
                            "--warmup", "3", "--no-cpu", "--no-extras", "--no-parity", "--dump-outputs", str(out)],
                           cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert sorted(p.name for p in out.iterdir()) == ["sum.npy", "y.npy"]
        y, s = np.load(out / "y.npy"), np.load(out / "sum.npy")
        assert y.dtype == np.float32 and s.dtype == np.float32 and s.shape == (1,) and float(s[0]) == line["sum"]
        assert y.nbytes + s.nbytes <= 64 << 20
        offs = bench.dump_offsets(n, 1)
        if offs is None:
            want = ocore.affine_f32(ocore.rand_u01_f32(bench.SEED, 0, n), bench.A_COEF, bench.B_COEF)
        else:
            assert y.size == bench.DUMP_ELEMS < n
            want = np.concatenate([ocore.affine_f32(ocore.rand_u01_f32(bench.SEED, int(o), bench.WINDOW), bench.A_COEF, bench.B_COEF) for o in offs])
        assert np.array_equal(y.view(np.uint32), want.view(np.uint32))
        dumps.append((y, s))
    assert all(np.array_equal(u.view(np.uint32), v.view(np.uint32)) for u, v in zip(*dumps))


def test_smoke_host_logic_against_the_host_memory_abi():
    """``__graft_entry__.smoke()`` (what the driver runs on the B200 before the bench) with the C ABI emulated over host memory: its host side
    -- layouts vs the oracle, map!, broadcast, sum / maximum, sum(dims=1), the halo read, A*B, the strided view, sort -- runs through."""
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_on_hostmem.py"), "__graft_entry__.py", "smoke"], cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "smoke ok" in r.stdout, (r.stdout + r.stderr)[-2000:]


def test_nd_broadcast_random_shapes_on_the_host_memory_abi(hostmem, dab):
    """General broadcasts over 5..7 dimensions with random extents and random extrusion patterns, through the REAL run_local (collapse_dims,
    stride tables) and the emulated strided box walk, against NumPy's broadcasting; patterns that do not collapse to 4 groups must raise."""
    rng = np.random.default_rng(55)
    dab.init(workers_per_rank=4, use_dist=False)
    served = refused = 0
    for trial in range(60):
        nd = int(rng.integers(5, 8))
        shape = tuple(int(v) for v in rng.integers(1, 5, nd))
        if int(np.prod(shape)) < 4:
            continue
        A = rng.integers(-9, 9, shape).astype(np.int64)
        ext = rng.random(nd) < 0.35
        mshape = tuple(1 if e else s for e, s in zip(ext, shape))
        M = rng.integers(-9, 9, mshape).astype(np.int64)
        a = dab.distribute(A)
        try:
            r = dab.broadcast(lambda x, m: x * m - m, a, M)
        except dab.UnsupportedError:
            refused += 1
            continue                                            # per-chunk shapes decide; a refusal is an exception, never silent
        assert np.array_equal(dab.to_array(r), A * M - M), (shape, mshape)
        served += 1
        r.close()
        a.close()
    assert served >= 30, (served, refused)
