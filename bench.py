#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: GB/s (and % of the HBM roofline) for map!/broadcast and sum on a Float32 DArray.

A "step" is one pass of the hot path over one resident batch:   y .= a .* x .+ b   (8 B/element)  then   s = sum(y)
(4 B/element, incl. the cross-worker combine and the scalar on the host).  Workload at N GPUs: BASELINE configs[1]/[2], a 1-D
Float32 DArray of N * 2^30 elements, one 2^30-element (4 GiB) localpart per GPU (weak scaling, defaultdist grid (N,)).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--log2n 30]            # our arm (one process per GPU under torchrun)
  python bench.py --impl reference ...                                         # the reference's CPU path (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                                       # also write the last timed step's y (sampled) and sum(y)

Prints ONE JSON line (rank 0).  value = whole-job algorithmic GB/s with inputs resident in HBM; e2e = same metric through the
public API with HOST (pinned) input each step; roofline = the dominant kernel (the broadcast) against the measured HBM peak;
cpu_baseline = the oracle port timed on this box's host cores (bounded sample).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

A_COEF, B_COEF = 1.5, 0.25
SEED = 1234


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            for k in ("hbm_gbs", "hbm_gbps", "hbm_gb_s"):
                if k in j:
                    return float(j[k]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def traffic_from_capture(kernel, log2n):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/ncu_traffic.json: a list of
    {kernel, log2n, dram_bytes, source_sha16, capture}); None unless the entry was captured from the current kernel source."""
    import hashlib
    try:
        ent = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        src = os.path.join(ROOT, "distributedarrays.jl_b200", "csrc", "dab_elementwise.cu")
        sha = hashlib.sha256(open(src, "rb").read()).hexdigest()[:16]
        for e in ent:
            if e.get("kernel") == kernel and int(e.get("log2n", -1)) == int(log2n) and e.get("source_sha16") == sha:
                return float(e["dram_bytes"])
    except Exception:
        pass
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.path = device, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def cpu_leg(log2n_per_worker, steps, warmup, workers=None):
    """The reference's CPU-process path: P single-threaded workers (one per host core), each running Base's loops on its own
    chunk -- map!(x->a*x+b, d, d) then sum(d) + the caller-side left fold (oracle/oracle_core.c).  Compute only: the reference's
    remotecall / serialisation overhead is NOT reproduced (that flatters the reference)."""
    from oracle import core as ocore

    cores = ocore.num_procs()          # loads the liboracle_core.so that build() made; never recompiles into the tree
    n_per = 1 << log2n_per_worker
    tried = {}
    if workers:
        P = workers
    else:
        # "all the host threads it can use": the online core count over-states what a container may use (CPU quotas, SMT,
        # NUMA), and more workers than usable cores makes the reference SLOWER (measured: 128 workers 64 GB/s, 8 workers
        # 130 GB/s on the same box).  Give the reference its best worker count: quick scan, then the timed run at the best P.
        cand, p = [], cores
        while p >= 4:
            cand.append(p)
            p //= 2
        for p in cand or [cores]:
            _, m, _ = ocore.workers_run(3, p, n_per, SEED, A_COEF, B_COEF, 1, 2)   # same chunk size as the timed run (>> LLC)
            tried[p] = 12.0 * n_per * p / m / 1e9
        P = max(tried, key=tried.get)
    best, mean, res = ocore.workers_run(3, P, n_per, SEED, A_COEF, B_COEF, max(1, warmup), max(1, steps))
    gbs = 12.0 * n_per * P / mean / 1e9
    return {"value": gbs, "unit": "GB/s", "cores": P, "kind": "port",
            "sample": f"{P} workers x 2^{log2n_per_worker} Float32 (in-place map! a*x+b, then pairwise-1024 sum + left fold), "
                      f"{steps} timed passes, mean {mean * 1e3:.2f} ms/pass, best {best * 1e3:.2f} ms; host cores online: {cores}; "
                      f"worker-count scan GB/s: { {k: round(v, 1) for k, v in tried.items()} }",
            "ms_per_step": mean * 1e3, "result": float(res)}


# ---- in-run parity (checker = oracle/, outside every timed region) ----------------------------------------------------------------
REL_TOL = 1e-6          # BASELINE north_star: "outputs within 1e-6 rel of reference"
N_WINDOWS, WINDOW = 64, 4096
N_COLS = 64


def left_fold_f32(vals):
    """``reduce(+, results)`` on the caller (reference src/mapreduce.jl:34): left fold in procs(d) order, in Float32."""
    import numpy as np
    acc = np.float32(vals[0])
    for v in vals[1:]:
        acc = np.float32(acc + np.float32(v))
    return acc


def rel_err(got, exact):
    return abs(float(got) - float(exact)) / max(abs(float(exact)), 1e-300)


def _d2h_window(dab, rt, chunk, off, n):
    import ctypes as C

    import numpy as np
    out = np.empty(n, dtype=chunk.dtype)
    dab._lib.call("dab_d2h", rt.ctx, C.c_void_p(out.ctypes.data), C.c_void_p(chunk.ptr + off * chunk.dtype.itemsize), n * chunk.dtype.itemsize)
    rt.sync()
    return out


def _sum_of(dab, rt, arr, n):
    """sum of a raw device array through the C ABI (dab_reduce_host)."""
    import ctypes as C

    import numpy as np
    out = np.zeros(2, dtype=np.uint64)
    dab._lib.call("dab_reduce_host", rt.ctx, dab._lib.F32, dab._lib.SUM, dab._lib.MAP_ID, None, C.c_void_p(arr.ptr), n, C.c_void_p(out.ctypes.data))
    return out.view(np.float32)[0]


def parity_hot_path(dab, rt, x, y, n_per, world):
    """Checks of the timed step's outputs against exact ground truth (every rank takes part; rank 0 reports).

    sum_x / sum_y : Float32 result vs the EXACT sum (uint64 accumulation of the 2^-24 / 2^-25 grid values over all N*2^log2n
                    elements, regenerated index-wise by the oracle) at 1e-6 rel;  per_chunk: every localpart's partial likewise
    fold          : sum(y) == left fold, in Float32, of the P chunk results in procs(d) order (src/mapreduce.jl:34) -- bit-exact
    maximum_y     : bit-exact vs the oracle's max over all elements
    windows_y     : N_WINDOWS random WINDOW-element windows of y per rank, bit-exact vs fl(fl(a*x)+b) (two roundings, no FMA)
    """
    import numpy as np
    from oracle import core as ocore

    rank = rt.rank
    threads = max(1, ocore.num_usable_procs() // max(1, min(world, 8)))
    st = ocore.rand_stats(SEED, rank * n_per, n_per, A_COEF, B_COEF, 25, threads)
    allst = rt.allgather_object(st)
    ksum = sum(t["ksum"] for t in allst)
    ysum = sum(t["ysum"] for t in allst)
    inexact = sum(t["inexact"] for t in allst)
    exact_x, exact_y = ksum * 2.0 ** -24, ysum * 2.0 ** -25          # < 2^60: the products are exact in fp64 up to one rounding
    ymax = max(np.float32(t["ymax"]) for t in allst)
    checks = {}
    sx = dab.sum(x)
    sy = dab.sum(y)
    checks["sum_x"] = {"got": float(sx), "exact": exact_x, "rel_err": rel_err(sx, exact_x), "tol": REL_TOL}
    checks["sum_y"] = {"got": float(sy), "exact": exact_y, "rel_err": rel_err(sy, exact_y), "tol": REL_TOL, "grid_inexact_elems": inexact}
    for c in (checks["sum_x"], checks["sum_y"]):
        c["ok"] = c["rel_err"] <= c["tol"]
    checks["sum_y"]["ok"] = checks["sum_y"]["ok"] and inexact == 0
    res, vals = dab.mapreduce(None, "+", y, _partials=True)           # chunk results through dab_reduce + all-gather (not the fused path)
    fold = left_fold_f32(list(vals))
    worst = max(rel_err(v, t["ysum"] * 2.0 ** -25) for v, t in zip(vals, allst))
    checks["fold"] = {"ok": bool(np.float32(sy).tobytes() == fold.tobytes() and np.float32(res).tobytes() == fold.tobytes()),
                      "sum": float(sy), "left_fold_of_chunk_results": float(fold), "tol": "bit-exact", "order": "procs(d)",
                      "per_chunk_worst_rel_err": worst, "per_chunk_ok": worst <= REL_TOL}
    checks["fold"]["ok"] = checks["fold"]["ok"] and checks["fold"]["per_chunk_ok"]
    my = dab.maximum(y)
    checks["maximum_y"] = {"ok": bool(np.float32(my).tobytes() == np.float32(ymax).tobytes()), "got": float(my), "exact": float(ymax), "tol": "bit-exact"}
    rng = np.random.default_rng(SEED + 77 + rank)
    ch = dab.localpart(y)
    offs = [0, n_per - WINDOW] + [int(o) for o in rng.integers(0, n_per - WINDOW, N_WINDOWS - 2)]
    bad = 0
    for off in offs:
        got = _d2h_window(dab, rt, ch, off, WINDOW)
        want = ocore.affine_f32(ocore.rand_u01_f32(SEED, rank * n_per + off, WINDOW), A_COEF, B_COEF)
        bad += int(not np.array_equal(got.view(np.uint32), want.view(np.uint32)))
    bad_all = sum(rt.allgather_object(bad))
    checks["windows_y"] = {"ok": bad_all == 0, "windows_per_rank": len(offs), "window_elems": WINDOW, "mismatching_windows": bad_all, "tol": "bit-exact"}
    return checks


def parity_sum_dims1(dab, rt, A, R, seed):
    """sum(A, dims=1) on the drand matrix: owners of R must be grid row 1 of A (reference src/mapreduce.jl:44) and N_COLS sampled
    columns per owner must match the EXACT column sums (a column of a column-major global array is a contiguous run of generator
    indices, so its exact sum is one ksum) at 1e-6 rel."""
    import numpy as np
    from oracle import core as ocore

    g0 = A.layout.grid[0]
    owners_ok = list(R.layout.pids) == [A.layout.pids[j * g0] for j in range(A.layout.grid[1])] and R.dims == (1, A.dims[1])
    rows = A.dims[0]
    rng = np.random.default_rng(seed + rt.rank)
    worst, n = 0.0, 0
    for pid, ch in R.chunks.items():
        lo, hi = R.layout.localindices(pid)[1]
        host = ch.to_numpy().reshape(-1)
        cols = sorted({lo - 1, hi - 1} | {int(c) for c in rng.integers(lo - 1, hi, N_COLS - 2)})
        for c in cols:
            exact = ocore.rand_ksum(seed, c * rows, rows) * 2.0 ** -24
            worst = max(worst, rel_err(host[c - (lo - 1)], exact))
            n += 1
    allw = rt.allgather_object((worst, n))
    worst, n = max(w for w, _ in allw), sum(k for _, k in allw)
    return {"ok": bool(owners_ok and worst <= REL_TOL and n > 0), "owners_are_grid_row_1": bool(owners_ok), "columns_checked": n,
            "worst_rel_err": worst, "tol": REL_TOL}


def parity_halo(dab, rt, dst, seed, rows_total, r0, c0):
    """The halo slab (rows r0.., columns c0.. of the global drand matrix, 0-based) bit-exact on N_COLS sampled columns."""
    import numpy as np
    from oracle import core as ocore

    nr, nc = dst.shape
    rng = np.random.default_rng(seed + 991 + rt.rank)
    cols = sorted({0, nc - 1} | {int(c) for c in rng.integers(0, nc, N_COLS - 2)})
    bad = 0
    for j in cols:
        got = _d2h_window(dab, rt, dst, j * nr, nr)
        want = ocore.rand_u01_f32(seed, (c0 + j) * rows_total + r0, nr)
        bad += int(not np.array_equal(got.view(np.uint32), want.view(np.uint32)))
    bad_all = sum(rt.allgather_object(bad))
    return {"ok": bad_all == 0, "columns_per_rank": len(cols), "mismatching_columns": bad_all, "tol": "bit-exact"}


DUMP_ELEMS = 1 << 22    # y values written by --dump-outputs over all ranks: 16 MiB of Float32


def dump_offsets(n_per, world):
    """Start offsets (within a localpart) of the WINDOW-element windows of y that --dump-outputs writes; None: the whole localpart."""
    import numpy as np

    per_rank = DUMP_ELEMS // world
    if n_per <= per_rank:
        return None
    return np.sort(np.random.default_rng(SEED + 5).choice(n_per // WINDOW, per_rank // WINDOW, replace=False)) * WINDOW


def dump_outputs(dab, rt, y, s, n_per, world, out_dir):
    """What the timed step hands its caller, written after its last step: ``y.npy`` (Float32; the whole of y when it holds at most
    DUMP_ELEMS elements, else the windows of every localpart at dump_offsets(), concatenated in rank order) and ``sum.npy`` (the
    Float32 sum(y)).  Same arguments -> same inputs and same sample, so two builds can be compared file by file."""
    import numpy as np

    ch = dab.localpart(y)
    offs = dump_offsets(n_per, world)
    if offs is None:
        part = ch.to_numpy().reshape(-1)
    else:
        part = np.concatenate([_d2h_window(dab, rt, ch, int(off), WINDOW) for off in offs])
    parts = rt.allgather_object(part)
    if rt.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "y.npy"), np.concatenate(parts).astype(np.float32))
        np.save(os.path.join(out_dir, "sum.npy"), np.array([s], dtype=np.float32))



def main():
    sys.dont_write_bytecode = True     # the benchmark leaves the tree as build() left it (no __pycache__ of the modules it imports)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=30, help="log2 of the elements per GPU (default 2^30 = 4 GiB chunk)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (y, sum(y)) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(3, args.warmup)
    n_per = 1 << args.log2n
    workload = (f"C2/C3: 1-D Float32 DArray, {world} x 2^{args.log2n} elements ({4 * n_per / 2**30:.0f} GiB localpart per GPU); "
                f"step = y .= {A_COEF}f0 .* x .+ {B_COEF}f0 then sum(y)")

    if args.impl == "reference":
        if rank != 0:
            return
        c = cpu_leg(24, args.steps, warmup)
        line = {"impl": "reference", "metric": "GB/s for map! and sum on Float32 DArray", "value": c["value"], "unit": "GB/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup, "ms_per_step": c["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload, "reference_arm": "CPU restatement of the reference's per-worker Base loops (Julia is not "
                           "installable here; oracle/oracle_core.c), one single-threaded worker per host core, bounded sample"},
                "cpu_baseline": {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": c["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return

    import numpy as np

    import darray_b200 as dab

    rt = dab.init(workers_per_rank=1)
    a, b = np.float32(A_COEF), np.float32(B_COEF)
    N = n_per * world
    x = dab.drand((N,), dtype=np.float32, seed=SEED)       # generated on device, reproducible on the CPU oracle
    y = dab.similar(x)
    f = lambda v: a * v + b  # noqa: E731  (traced once -> dab_affine)

    def step():
        dab.broadcast_into(y, f, x)
        return dab.sum(y)

    def fence():
        rt.sync()
        if rt.dist is not None:
            rt.dist.barrier()

    def timed(fn, k, warm=2):
        for _ in range(warm):   # first launches pay CUDA's lazy kernel loading and pool growth: never inside a timed region
            fn()
        e0, e1 = rt.event(), rt.event()
        fence()
        rt.device_barrier()     # the ranks leave the host barrier tens of microseconds apart: start the timed region aligned on the DEVICES
        rt.record(e0)
        r = None
        for _ in range(k):
            r = fn()
        rt.record(e1)
        ms = rt.elapsed_ms(e0, e1)
        fence()
        rt.event_destroy(e0)
        rt.event_destroy(e1)
        return ms, r

    def max_over_ranks(v):
        if rt.dist is None:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64)
        rt.dist.all_reduce(t, op=rt.dist.ReduceOp.MAX)
        return float(t.item())

    # clocks: the sampler starts BEFORE the warm-up (nvidia-smi needs ~100 ms to deliver its first sample; the K timed steps alone last
    # ~20 ms) and stops after the per-kernel timings, so every sample is taken while this process keeps the GPU busy.  The warm-up
    # first runs 160 untimed steps (~0.3 s): a freshly created context starts from an idle power state, and the first
    # few tens of milliseconds of work run at ramping SM / memory clocks (seen once as a 2.04 ms instead of a 1.86 ms step).
    clocks = ClockSampler(rt.device)
    if rank == 0:
        clocks.start()
    for _ in range(160):     # ~0.3 s; a FIXED count: the step contains a collective, every rank must make the same number of calls
        s = step()
    for _ in range(warmup):
        s = step()
    l0 = rt.launches()
    ms, s = timed(step, args.steps)
    launches = rt.launches() - l0
    if args.dump_outputs:
        dump_outputs(dab, rt, y, s, n_per, world, args.dump_outputs)
    ms = max_over_ranks(ms)
    value = 12.0 * N * args.steps / (ms * 1e-3) / 1e9

    # ---- per-kernel timings (same resident data; inputs 4 GiB >> 126 MB L2, so no flush needed)
    ms_bc, _ = timed(lambda: dab.broadcast_into(y, f, x), args.steps)
    bc_entry = rt.last_kernel  # which C-ABI entry point served the broadcast (dab_affine = the hand-written kernel)
    ms_sum, _ = timed(lambda: dab.sum(y), args.steps)
    ms_max, _ = timed(lambda: dab.maximum(y), args.steps)
    ms_bc, ms_sum, ms_max = max_over_ranks(ms_bc), max_over_ranks(ms_sum), max_over_ranks(ms_max)
    clk = clocks.stop() if rank == 0 else None
    peak, peak_kind = measured_peak()
    bc_gbs = 8.0 * n_per * args.steps / (ms_bc * 1e-3) / 1e9          # per GPU: the kernel's own HBM rate
    sum_gbs = 4.0 * n_per * args.steps / (ms_sum * 1e-3) / 1e9
    max_gbs = 4.0 * n_per * args.steps / (ms_max * 1e-3) / 1e9

    # ---- parity inside the bench run, outside the timed regions: exact ground truth from the oracle (checker only)
    parity = {"checks": {}}
    if not args.no_parity:
        try:
            parity["checks"].update(parity_hot_path(dab, rt, x, y, n_per, world))
        except Exception as ex:
            parity["checks"]["hot_path"] = {"ok": False, "error": repr(ex)[:300]}

    # ---- e2e: the same step through the public API with HOST input every step (pinned), scalar result back on the host
    e2e = None
    try:
        from darray_b200 import pinned_empty
        hx = pinned_empty(rt, (n_per,), np.float32)
        hx[:] = 0.5
        hx[::4096] = 0.25
        e2e_steps = max(1, args.e2e_steps)

        def e2e_step():
            if world == 1:
                dab.copyto(x, hx)                                          # copyto!(x::DArray, host::Array): H2D of the step's input
            else:
                dab.localpart(x).copy_from_host(hx, sync=False)            # copyto!(localpart(x), host chunk) on every worker
            dab.broadcast_into(y, f, x)
            return dab.sum(y)

        for _ in range(2):
            e2e_step()
        ms_e, _ = timed(e2e_step, e2e_steps)
        ms_e = max_over_ranks(ms_e)
        # the bound of this leg: the step moves 4 B/element over PCIe and is credited 12 B/element, so e2e <= 3 x the H2D rate; measured
        # beside it: the pinned H2D rate alone and the pipelined pageable path (dab_h2d staging) on 1 GiB
        lp = dab.localpart(x)
        ms_c, _ = timed(lambda: lp.copy_from_host(hx, sync=False), 2, warm=1)
        ms_c = max_over_ranks(ms_c)
        n_pg = min(1 << 28, n_per)                                         # 1 GiB of pageable memory (the whole chunk when it is smaller)
        pg = np.empty(n_pg, dtype=np.float32)
        pg[:] = 0.5
        lpv = dab.B200Array(rt, lp.ptr, (n_pg,), np.float32, own=False)
        ms_p, _ = timed(lambda: lpv.copy_from_host(pg, sync=False), 2, warm=1)
        ms_p = max_over_ranks(ms_p)
        del pg
        h2d = 4.0 * n_per * 2 / (ms_c * 1e-3) / 1e9
        e2e = {"value": 12.0 * N * e2e_steps / (ms_e * 1e-3) / 1e9, "unit": "GB/s", "h2d_bytes_per_step": 4 * N,
               "d2h_bytes_per_step": 16 * world, "ms_per_step": ms_e / e2e_steps,
               "path": "copyto!(x::DArray, host Array) [pinned H2D] -> y .= a.*x .+ b -> sum(y) -> host scalar",
               "h2d_pinned_GBs_per_gpu": h2d, "h2d_pageable_pipelined_GBs_per_gpu": 4.0 * n_pg * 2 / (ms_p * 1e-3) / 1e9,
               "bound": f"PCIe-bound: 4 of the 12 credited bytes/element cross the host link, so e2e <= 3 x H2D = {3 * h2d * world:.0f} GB/s at "
                        f"{world} GPU(s); the device part of the step is {ms / args.steps:.2f} ms of the {ms_e / e2e_steps:.1f} ms. A CPU worker pool "
                        "streams the same step from host DRAM (no link to cross), which is why one GPU cannot win this leg however fast its kernels are"}
    except Exception as ex:  # never lose the main line because of the e2e leg
        e2e = {"value": None, "unit": "GB/s", "error": repr(ex)[:200]}

    # ---- extras (not part of `value`): the TMA-staged variant of the broadcast kernel, BASELINE configs 4 and 5 at this N
    extras = {}
    if not args.no_extras:
        try:
            rt.set_option("ew_tma", 1)
            ms_t, _ = timed(lambda: dab.broadcast_into(y, f, x), args.steps)
            rt.set_option("ew_tma", 0)
            ms_t = max_over_ranks(ms_t)
            extras["broadcast_tma_variant"] = {"GBs_per_gpu": 8.0 * n_per * args.steps / (ms_t * 1e-3) / 1e9,
                                               "what": "same y .= a.*x .+ b through the opt-in cp.async.bulk + mbarrier shared-memory ring "
                                                       "(dab_set_option ew_tma=1); the default flat LDG/STG kernel is `kernels.broadcast_GBs_per_gpu`"}
        except Exception as ex:
            extras["broadcast_tma_variant"] = {"error": repr(ex)[:200]}
            try:
                rt.set_option("ew_tma", 0)
            except Exception:
                pass
        try:
            g = dab.defaultdist((65536, 65536), world)                   # (2,4) at N=8
            dimsA = (32768 * g[0], 16384 * g[1])                         # 32768 x 16384 Float32 (2 GiB) per GPU; exactly 65536^2 at N=8
            A = dab.drand(dimsA, dtype=np.float32, seed=SEED + 1)
            reps = 10
            ms_d, _ = timed(lambda: dab.sum(A, dims=1).close(), reps)    # within-chunk kernel + between-phase exchange + R allocation
            ms_d = max_over_ranks(ms_d)
            extras["sum_dims1"] = {"GBs": 4.0 * dimsA[0] * dimsA[1] * reps / (ms_d * 1e-3) / 1e9, "dims": list(dimsA), "grid": list(g),
                                   "ms": ms_d / reps, "bytes_per_elem": 4,
                                   "what": "sum(A, dims=1): per-chunk column reduction + partial slabs PUT into the fibre owners' exchange arena over NVLink "
                                           "+ device-side barrier + ordered accumulate (no NCCL launch, no host sync)"}
            if not args.no_parity:
                R = dab.sum(A, dims=1)
                parity["checks"]["sum_dims1"] = parity_sum_dims1(dab, rt, A, R, SEED + 1)
                R.close()
            if world > 1:
                A.share()
                rt.barrier()
                nxt = A.layout.pids[(A.layout.pids.index(rt.myid()) + 1) % world]
                I = A.layout.localindices(nxt)
                sub = A[I[0][0] - 1:I[0][1], I[1][0] - 1:I[1][0] - 1 + 2048]   # 32768 x 2048 Float32 = 256 MiB inside the neighbour's chunk
                dst = dab.B200Array.empty(rt, (32768, 2048), np.float32)
                sub.copy_to(dst)
                ms_h, _ = timed(lambda: sub.copy_to(dst), reps)
                ms_h = max_over_ranks(ms_h)
                extras["halo_getindex"] = {"GBs_per_reader": 4.0 * 32768 * 2048 * reps / (ms_h * 1e-3) / 1e9, "slab_bytes": 4 * 32768 * 2048,
                                           "peak_GBs": 770.0, "what": "every rank pulls a 256 MiB slab of its right neighbour's chunk over NVLink (CUDA-IPC peer loads)"}
                extras["halo_getindex"]["frac_of_peak"] = extras["halo_getindex"]["GBs_per_reader"] / 770.0
                if not args.no_parity:
                    parity["checks"]["halo_getindex"] = parity_halo(dab, rt, dst, SEED + 1, dimsA[0], I[0][0] - 1, I[1][0] - 1)
                dst.free()
            # Level-2 widening (K9): y = A*x and y = A'*x on the same matrix, through the public API (tile products, exchange of the
            # tile results to y's owners, ordered accumulate); x is a DVector so no host copy sits inside the timed region
            xv = dab.dfill(1.0, (dimsA[1],), dtype=np.float32)
            xt = dab.dfill(1.0, (dimsA[0],), dtype=np.float32)
            for key, W, v in (("matvec_A_x", A, xv), ("matvec_At_x", A.T, xt)):
                ms_m, _ = timed(lambda: (W @ v).close(), reps)
                ms_m = max_over_ranks(ms_m)
                extras[key] = {"GBs": 4.0 * dimsA[0] * dimsA[1] * reps / (ms_m * 1e-3) / 1e9, "ms": ms_m / reps, "bytes_per_elem": 4,
                               "what": "mul!(y, A, x) on the sum_dims1 matrix: x blocks halo-fetched (peer loads), dab_gemv per chunk (fp64 carriers), tile "
                                       "results PUT into the y owners' exchange arena over NVLink, device-side barriers, one fused beta-scale + ordered add!"}
            xv.close()
            xt.close()
            # Level-3 widening (K12): C = A*B through the public API (tile products on the tcgen05 3xTF32 kernel, B blocks halo-fetched,
            # tile results shipped to the owners of C, ordered add!); useful flops = 2*m*n*k, the tensor core executes 3x that in TF32
            try:
                nB = 2048
                Bm = dab.drand((dimsA[1], nB), dtype=np.float32, seed=SEED + 2)
                ms_g, _ = timed(lambda: (A @ Bm).close(), 3)
                ms_g = max_over_ranks(ms_g)
                fl = 2.0 * dimsA[0] * dimsA[1] * nB * 3
                tf = fl / (ms_g * 1e-3) / 1e12
                pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops") if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else None
                extras["matmat_A_B"] = {"useful_TFLOPs": tf, "tf32_mma_TFLOPs": 3 * tf, "ms": ms_g / 3, "dims": [dimsA[0], dimsA[1], nB],
                                        "frac_of_tf32_peak": (3 * tf / (world * pk / 2)) if pk else None,
                                        "what": "A*B (mul!(C, A, B)): dab_gemm tiles = TMA + tcgen05.mma kind::tf32 with TMEM accumulators, 3xTF32 "
                                                "error-compensated; tf32 peak taken as measured bf16 peak / 2"}
                if not args.no_parity:
                    Cm = A @ Bm
                    from oracle import core as ocore
                    lc = dab.localpart(Cm)
                    worst, rows = 0.0, 64
                    if lc.size:
                        Ic = Cm.layout.localindices(rt.myid())
                        r0 = Ic[0][0] - 1
                        arow = np.empty((rows, dimsA[1]))
                        for kk in range(dimsA[1]):                             # A[r0:r0+64, :] regenerated from the counter-based generator
                            arow[:, kk] = ocore.rand_u01_f32(SEED + 1, kk * dimsA[0] + r0, rows)
                        for jc in (Ic[1][0] - 1, Ic[1][1] - 1):                # first and last column of this rank's chunk of C
                            want = arow @ ocore.rand_u01_f32(SEED + 2, jc * dimsA[1], dimsA[1]).astype(np.float64)
                            got = _d2h_window(dab, rt, lc, (jc - (Ic[1][0] - 1)) * lc.shape[0], rows)
                            worst = max(worst, float(np.abs(got - want).max() / np.abs(want).min()))
                    allw = max(rt.allgather_object(worst))
                    parity["checks"]["matmat_A_B"] = {"ok": allw <= 2e-6, "worst_rel_err": allw, "tol": 2e-6, "entries_per_rank": 2 * rows,
                                                      "vs": "fp64 product of the regenerated inputs"}
                    Cm.close()
                Bm.close()
            except Exception as ex:
                extras["matmat_A_B"] = {"error": repr(ex)[:300]}
            A.close()
            # sort widening (K11 onesweep): one chunk through the C ABI, and sort(d::DVector) end to end (samplesort incl. the exchange)
            try:
                import ctypes as C
                from darray_b200 import _lib
                ns = 1 << 28
                keys = dab.drand((ns * world,), dtype=np.float32, seed=SEED + 3)
                kin = dab.localpart(keys)
                kout, ktmp = dab.B200Array.empty(rt, (ns,), np.float32), dab.B200Array.empty(rt, (ns,), np.float32)
                ms_s, _ = timed(lambda: _lib.call("dab_sort", rt.ctx, _lib.F32, C.c_void_p(kin.ptr), C.c_void_p(kout.ptr), C.c_void_p(ktmp.ptr), ns), 5)
                ms_s = max_over_ranks(ms_s) / 5
                if not args.no_parity:
                    head = _d2h_window(dab, rt, kout, 0, 1 << 20)
                    s_in, s_out = float(_sum_of(dab, rt, kin, ns)), float(_sum_of(dab, rt, kout, ns))   # this rank's chunk before / after
                    srt_ok = bool(np.all(head[:-1] <= head[1:])) and abs(s_in - s_out) <= 1e-6 * s_in
                    parity["checks"]["sort_chunk"] = {"ok": bool(all(rt.allgather_object(srt_ok))), "what": "first 2^20 keys ascending; sum preserved (1e-6)"}
                kout.free()
                ktmp.free()
                # rand(Float32) keys occupy 3 of the 4 digit positions fully (sign/exponent byte varies little but is not constant)
                extras["sort_chunk_f32_2p28"] = {"ms": ms_s, "Gkeys_s_per_gpu": ns / ms_s / 1e6, "algorithmic_GBs_per_gpu": 4.0 * ns * (1 + 2 * 4) / ms_s / 1e6,
                                                 "frac_of_hbm_peak": 4.0 * ns * (1 + 2 * 4) / ms_s / 1e6 / peak,
                                                 "what": "dab_sort (onesweep LSD radix sort, 8-bit digits) of one 2^28 Float32 chunk per GPU; algorithmic "
                                                         "bytes = 4 B x (1 histogram read + 2 per digit pass x 4 passes)"}
                keys.close()
                dv = dab.drand(((1 << 26) * world,), dtype=np.float32, seed=SEED + 4)
                ms_d, _ = timed(lambda: dab.sort(dv).close(), 3)
                ms_d = max_over_ranks(ms_d) / 3
                extras["sort_dvector_2p26_per_gpu"] = {"ms": ms_d, "Gkeys_s": (1 << 26) * world / ms_d / 1e6,
                                                       "what": "sort(d::DVector; sample=true) end to end: chunk sorts, sampling, split, exchange of the pieces, result DArray"}
                if not args.no_parity:
                    sd = dab.sort(dv)
                    tot = float(dab.sum(sd))
                    okd = abs(tot - float(dab.sum(dv))) <= 1e-6 * tot and len(sd) == len(dv)
                    lp = dab.localpart(sd)
                    if lp.size > 1:
                        w = _d2h_window(dab, rt, lp, 0, min(lp.size, 1 << 20))
                        okd = okd and bool(np.all(w[:-1] <= w[1:]))
                    parity["checks"]["sort_dvector"] = {"ok": bool(all(rt.allgather_object(bool(okd)))), "what": "length and sum preserved; local head ascending"}
                    sd.close()
                dv.close()
            except Exception as ex:
                extras["sort"] = {"error": repr(ex)[:300]}
        except Exception as ex:
            extras["error"] = repr(ex)[:300]

    line = {"metric": "GB/s for map! and sum on Float32 DArray", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "l2": "inputs (4 GiB/GPU) >> 126 MB L2, no flush needed", "grid": list(x.layout.grid),
                       "combine": ("single chunk" if world == 1 else
                                   "fused in the reduce kernel: peer-memory all-gather of the P chunk results over NVLink + ordered left fold"
                                   if rt.fused_combine else "NCCL all-gather of the P chunk results + ordered left fold")},
            "roofline": {"bound": "hbm", "kernel": "ew1_kernel<float, AffineF<float>, 2>", "entry": bc_entry, "achieved": bc_gbs, "peak": peak,
                         "peak_kind": peak_kind, "unit": "GB/s", "frac": bc_gbs / peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of THIS
                         # kernel source at this size (profiles/ncu_traffic.json, written by tools/ncu_summary.py); null when the
                         # capture is missing or older than the kernel source's recorded hash
                         "traffic": traffic_from_capture("ew1_kernel", args.log2n),
                         "algorithmic_bytes_per_launch": 8 * n_per},
            "kernels": {"broadcast_GBs_per_gpu": bc_gbs, "sum_GBs_per_gpu": sum_gbs, "maximum_GBs_per_gpu": max_gbs,
                        "broadcast_frac": bc_gbs / peak, "sum_frac": sum_gbs / peak, "maximum_frac": max_gbs / peak,
                        "ms_broadcast": ms_bc / args.steps, "ms_sum": ms_sum / args.steps},
            "e2e": e2e, "extras": extras, "gpu_launches": launches, "clocks": clk, "parity": parity, "sum": float(s)}
    parity["ok"] = bool(parity["checks"]) and all(c.get("ok") is True for c in parity["checks"].values())
    parity["note"] = ("Float32 reduction ORDER inside a chunk is parity-unpinned (no reference test pins it); sums are checked at 1e-6 rel "
                      "against exact integer ground truth, the cross-chunk fold and everything elementwise / indexed bit-exactly")
    if rank == 0:
        if world == 1 and not args.no_cpu:
            try:
                c = cpu_leg(24, 5, 2)
                line["cpu_baseline"] = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")}
            except Exception as ex:
                line["cpu_baseline"] = {"value": None, "error": repr(ex)[:200]}
        print(json.dumps(line))
    fence()
    dab.d_closeall()
    rt.shutdown()


if __name__ == "__main__":
    main()
