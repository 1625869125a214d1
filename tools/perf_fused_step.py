#!/usr/bin/env python
"""The bench step's chunk work through the C ABI, in one process: `y .= a.*x .+ b` then the whole-chunk sum of y, as the pair
dab_affine + dab_mapreduce_all (12 B/element in Float32: read x, write y, read y) against the fused dab_affine_mapreduce_all
(8 B/element: read x, write y).  CUDA events around REPS calls, warm-up first, ROUNDS rounds alternating the two sequences; the
median round is reported.  Inputs are >= 4 GiB, far larger than the 126 MB L2.  Also checks that both give the same y and sum bits.

    python tools/perf_fused_step.py [--reps 20] [--rounds 3]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = [(30, "f32"), (31, "f32"), (29, "f64")]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as ex:  # noqa: BLE001
        return f"unknown ({ex!r})"


def peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        for k in ("hbm_gbs", "hbm_gbps", "hbm_gb_s"):
            if k in j:
                return float(j[k])
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import numpy as np

    import darray_b200 as dab
    from darray_b200 import _lib as L

    rt = dab.init(workers_per_rank=1, use_dist=False)
    pk = peak()
    print(f"card: {card()}   (name, power limit, max SM clock)")
    print(f"measured HBM peak (MEASURED_PEAKS.json): {pk if pk else 'not available'} GB/s")
    print(f"{args.reps} calls per timed round, {args.rounds} rounds alternating pair / fused, median round reported")
    print(f"{'size':>10} {'dtype':>5} {'sequence':>34} {'ms/call':>9} {'B/elem':>6} {'GB/s':>8} {'frac':>6} {'rounds ms':>28}")
    for log2n, tag in SIZES:
        dt = np.float32 if tag == "f32" else np.float64
        code = L.F32 if tag == "f32" else L.F64
        es = np.dtype(dt).itemsize
        n = 1 << log2n
        x = dab.drand((n,), dtype=dt, seed=1234)
        y = dab.similar(x)
        xp, yp = C.c_void_p(dab.localpart(x).ptr), C.c_void_p(dab.localpart(y).ptr)
        a, b = np.asarray(1.5, dt), np.asarray(0.25, dt)
        ab = (C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data))
        out = np.zeros(2, dtype=np.uint64)
        op = C.c_void_p(out.ctypes.data)

        def pair():
            L.call("dab_affine", rt.ctx, code, yp, xp, *ab, n)
            L.call("dab_mapreduce_all", rt.ctx, code, L.SUM, L.MAP_ID, None, yp, n, op)

        def fused():
            L.call("dab_affine_mapreduce_all", rt.ctx, code, yp, xp, *ab, n, L.SUM, op)

        res = {}
        for name, fn in (("pair", pair), ("fused", fused)):
            fn()
            res[name] = (out.tobytes(), dab.localpart(y).to_numpy()[:: max(1, n >> 20)].tobytes())
        same = res["pair"] == res["fused"]
        times = {"pair": [], "fused": []}
        e0, e1 = rt.event(), rt.event()
        for _ in range(args.rounds):
            for name, fn in (("pair", pair), ("fused", fused)):
                for _ in range(args.warmup):
                    fn()
                rt.sync()
                rt.record(e0)
                for _ in range(args.reps):
                    fn()
                rt.record(e1)
                rt.sync()
                times[name].append(rt.elapsed_ms(e0, e1) / args.reps)
        rt.event_destroy(e0)
        rt.event_destroy(e1)
        for name, label, bpe in (("pair", "dab_affine + dab_mapreduce_all", 3 * es), ("fused", "dab_affine_mapreduce_all", 2 * es)):
            ms = statistics.median(times[name])
            gbs = bpe * n / (ms * 1e-3) / 1e9
            frac = f"{gbs / pk:.3f}" if pk else "n/a"
            print(f"{'2^%d' % log2n:>10} {tag:>5} {label:>34} {ms:9.4f} {bpe:6d} {gbs:8.0f} {frac:>6} {' '.join(f'{t:.4f}' for t in times[name]):>28}")
        print(f"{'':>10} {'':>5} {'fused / pair time':>34} {statistics.median(times['fused']) / statistics.median(times['pair']):9.3f}   "
              f"same y (sampled) and sum bits: {same}")
        x.close()
        y.close()
    dab.d_closeall()
    rt.shutdown()


if __name__ == "__main__":
    main()
