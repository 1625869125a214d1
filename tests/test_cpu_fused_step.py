"""The deferred broadcast (runtime.Runtime.defer_affine) on the host-memory emulation of the C ABI: ``y .= a.*x .+ b`` followed by a
reduction of y runs as one fused call, and every other call in between launches the broadcast first.  Each sequence of API calls below
is run twice, with the deferral and with every broadcast launched at once (eager), and must give the same bytes in every array and scalar
it reads back.  Says nothing about the CUDA kernels (tests/test_gpu_fused_reduce.py compares those bit for bit)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 4099
A, B = np.float32(1.5), np.float32(0.25)


def f(v):
    return A * v + B


def g(v):
    return np.float32(-2.0) * v + np.float32(3.0)


def install_fused(fake):
    """Give the host-memory emulation (tests/hostmem_abi.py) the fused entry points: dab_affine, then the identity-map reduce of y --
    counted as ONE launch when libdab200.so fuses them (Float32 / Float64, SUM PROD MAX MIN, n > 0, x and y at the same offset mod 16),
    else as the two launches it replaces.  Without them the runtime launches every broadcast at once."""
    import hostmem_abi as hm

    def affine_reduce(ctx, dtype, y, x, a, b, n, op, out):
        before = fake.launches
        fake.dab_affine(ctx, dtype, y, x, a, b, n)
        st = fake._reduce(dtype, op, 0, None, y, n, out)
        if int(dtype) in (hm.F32, hm.F64) and int(op) in (0, 1, 2, 3) and int(n) > 0 and hm._addr(x) % 16 == hm._addr(y) % 16:
            fake.launches = before + 1
        return st

    fake.dab_affine_reduce = fake.dab_affine_mapreduce_all = affine_reduce
    return fake


@pytest.fixture()
def fused(hostmem):
    return install_fused(hostmem)


def _d2h(dab, rt, arr, off, n):
    out = np.empty(n, dtype=arr.dtype)
    dab._lib.call("dab_d2h", rt.ctx, C.c_void_p(out.ctypes.data), C.c_void_p(arr.ptr + off * arr.dtype.itemsize), n * arr.dtype.itemsize)
    rt.sync()
    return out


def _bytes(v):
    return np.asarray(v).tobytes()


def _trigger_localpart(dab, rt, x, y):
    return [dab.localpart(y).to_numpy(), dab.sum(y)]


def _trigger_d2h_window(dab, rt, x, y):
    return [_d2h(dab, rt, dab.localpart(y), 7, 100), dab.sum(y)]


def _trigger_copyto_x(dab, rt, x, y):
    dab.copyto(x, np.full(x.dims, 0.5, dtype=x.dtype))
    return [dab.sum(y), dab.to_array(y), dab.to_array(x)]


def _trigger_close_x(dab, rt, x, y):
    x.close()
    return [dab.sum(y), dab.to_array(y)]


def _trigger_two_broadcasts(dab, rt, x, y):
    dab.broadcast_into(y, g, x)
    return [dab.sum(y), dab.to_array(y)]


def _trigger_broadcast_in_place(dab, rt, x, y):
    dab.broadcast_into(y, g, y)
    return [dab.sum(y), dab.to_array(y)]


def _trigger_sync(dab, rt, x, y):
    rt.sync()
    return [dab.sum(y)]


def _trigger_record(dab, rt, x, y):
    e = rt.event()
    rt.record(e)
    rt.event_destroy(e)
    return [dab.sum(y)]


def _trigger_maximum(dab, rt, x, y):
    return [dab.maximum(y), dab.sum(y)]


def _trigger_extrema(dab, rt, x, y):
    return [np.asarray(dab.extrema(y)), dab.sum(y)]


def _trigger_sum_x(dab, rt, x, y):
    return [dab.sum(x), dab.sum(y)]


def _trigger_sum_abs(dab, rt, x, y):
    return [dab.mapreduce(abs, "+", y), dab.sum(y)]


def _trigger_view(dab, rt, x, y):
    return [dab.sum(y[3:N - 5]), dab.sum(y)]


TRIGGERS = [_trigger_localpart, _trigger_d2h_window, _trigger_copyto_x, _trigger_close_x, _trigger_two_broadcasts, _trigger_broadcast_in_place,
            _trigger_sync, _trigger_record, _trigger_maximum, _trigger_extrema, _trigger_sum_x, _trigger_sum_abs, _trigger_view]


def _run(dab, wpr, trigger, eager):
    rtm = sys.modules["darray_b200.runtime"]
    mp = pytest.MonkeyPatch()
    if eager:
        defer = rtm.Runtime.defer_affine

        def defer_then_flush(self, *a):
            defer(self, *a)
            self.flush()

        mp.setattr(rtm.Runtime, "defer_affine", defer_then_flush)
    rt = dab.init(workers_per_rank=wpr, use_dist=False)
    try:
        x = dab.drand((N,), dtype=np.float32, seed=11)
        y = dab.similar(x)
        dab.broadcast_into(y, f, x)
        assert rt.last_kernel == "dab_affine"
        out = trigger(dab, rt, x, y) + [dab.to_array(y)]
        assert rt.pending is None
        return [_bytes(v) for v in out]
    finally:
        mp.undo()
        dab.d_closeall()
        rt.shutdown()


@pytest.mark.parametrize("wpr", [1, 2])
@pytest.mark.parametrize("trigger", TRIGGERS, ids=lambda t: t.__name__[len("_trigger_"):])
def test_flush_triggers_match_eager(fused, dab, trigger, wpr):
    deferred = _run(dab, wpr, trigger, False)
    eager = _run(dab, wpr, trigger, True)
    assert deferred == eager


@pytest.mark.parametrize("wpr", [1, 2])
@pytest.mark.parametrize("red", ["sum", "prod", "maximum", "minimum"])
def test_fused_step_is_one_launch(fused, dab, wpr, red):
    rt = dab.init(workers_per_rank=wpr, use_dist=False)
    x = dab.drand((N,), dtype=np.float32, seed=3)
    y = dab.similar(x)
    fn = getattr(dab, red)
    want = fn(dab.distribute(f(dab.to_array(x))))
    l0 = rt.launches()
    dab.broadcast_into(y, f, x)
    assert rt.pending is not None                                      # the last chunk's broadcast is deferred (launches() would launch it)
    s = fn(y)
    assert rt.launches() - l0 == 2 * wpr - 1 and rt.pending is None    # ... and runs fused with that chunk's reduce
    assert _bytes(s) == _bytes(want)
    l0 = rt.launches()
    dab.broadcast_into(y, f, x)
    rt.sync()
    fn(y)
    assert rt.launches() - l0 == 2 * wpr                               # flushed by the sync: broadcast and reduce launched apart


def test_unfused_cases_launch_twice(fused, dab):
    rt = dab.init(workers_per_rank=1, use_dist=False)
    x = dab.drand((N,), dtype=np.float32, seed=5)
    y = dab.similar(x)
    for red in (lambda: dab.sum(x), lambda: dab.mapreduce(abs, "+", y), lambda: dab.extrema(y)):
        l0 = rt.launches()
        dab.broadcast_into(y, f, x)
        red()
        assert rt.launches() - l0 == 2 and rt.pending is None
    xi = dab.distribute(np.arange(N, dtype=np.int64))
    yi = dab.similar(xi)
    l0 = rt.launches()
    dab.broadcast_into(yi, lambda v: 3 * v + 1, xi)
    assert int(dab.sum(yi)) == int(np.sum(3 * np.arange(N, dtype=np.int64) + 1))
    assert rt.launches() - l0 == 2                                     # Int64: not fused


def test_every_broadcast_is_launched(fused, dab):
    """A pending broadcast is never dropped, even when the next one overwrites the same y."""
    rt = dab.init(workers_per_rank=1, use_dist=False)
    x = dab.drand((N,), dtype=np.float32, seed=6)
    y = dab.similar(x)
    l0 = rt.launches()
    for _ in range(5):
        dab.broadcast_into(y, f, x)
    e = rt.event()
    rt.record(e)
    assert rt.launches() - l0 == 5 and rt.pending is None
    rt.event_destroy(e)


def test_no_deferral_without_the_fused_entry_points(hostmem, dab):
    """A binding that has only the unfused calls: the broadcast is launched when it is traced, as before the fused step existed."""
    rt = dab.init(workers_per_rank=1, use_dist=False)
    x = dab.drand((N,), dtype=np.float32, seed=8)
    y = dab.similar(x)
    l0 = hostmem.launches
    dab.broadcast_into(y, f, x)
    assert rt.pending is None and hostmem.launches - l0 == 1
    assert _bytes(dab.sum(y)) == _bytes(dab.sum(dab.distribute(f(dab.to_array(x)))))


def test_error_of_a_deferred_launch_surfaces_from_the_flushing_call(fused, dab):
    rt = dab.init(workers_per_rank=1, use_dist=False)
    x = dab.drand((N,), dtype=np.float32, seed=7)
    y = dab.similar(x)
    dab.broadcast_into(y, f, x)                                        # recorded, not launched: no error yet
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(fused, "dab_affine", lambda *a: dab._lib.ERR_CUDA)
        with pytest.raises(dab.DabError):
            rt.sync()
    assert rt.pending is None
    rt.sync()


# bench.py on the host-memory emulation with the fused entry points installed (what tests/run_on_hostmem.py does, plus install_fused)
_BENCH_RUNNER = r"""
import os, runpy, sys
ROOT = sys.argv[1]
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import darray_b200, hostmem_abi, test_cpu_fused_step
lib_mod, bc_mod = sys.modules["darray_b200._lib"], sys.modules["darray_b200._broadcast"]
fake = test_cpu_fused_step.install_fused(hostmem_abi.HostMemABI())
lib_mod._lib = fake
real_codegen = bc_mod.codegen
def recording_codegen(e):
    src = real_codegen(e)
    fake.exprs[src.encode()] = e
    return src
bc_mod.codegen = recording_codegen
sys.argv = ["bench.py"] + sys.argv[2:]
runpy.run_path(os.path.join(ROOT, "bench.py"), run_name="__main__")
"""


def test_bench_fused_sum_matches_the_unfused_parity_sum():
    """bench.py at 2^16 on the emulation: parity still ok, the line's sum (the fused timed step) equals sum_y of the parity block (taken
    after an unfused broadcast), and a step costs one launch."""
    r = subprocess.run([sys.executable, "-c", _BENCH_RUNNER, ROOT, "--log2n", "16", "--steps", "3", "--warmup", "3", "--no-cpu", "--no-extras"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["parity"]["ok"] is True, line["parity"]
    assert np.float32(line["sum"]).tobytes() == np.float32(line["parity"]["checks"]["sum_y"]["got"]).tobytes()
    assert line["gpu_launches"] == 3 + 2                               # the timed steps and the two warm-up steps of timed(): one launch each
