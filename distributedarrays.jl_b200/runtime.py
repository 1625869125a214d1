"""Process / device runtime: the stand-in for Julia's ``Distributed`` worker pool on this path.

One OS process per GPU (launched by ``torchrun``; RANK / LOCAL_RANK / WORLD_SIZE from the environment), exactly like the
reference's one Julia process per worker (test/runtests.jl:10-15).  ``torch.distributed`` is plumbing only: it ships
the 128-byte NCCL id and the CUDA IPC handles between ranks and provides host barriers.  All data-path traffic goes
through ``libdab200.so`` (NCCL / peer loads over NVLink).

One broadcast is deferred per runtime.  ``y .= a .* x .+ b`` (``dab_affine``) is not launched when it is traced: it is recorded as the
runtime's pending op, so that a ``sum(y)`` (``maximum``, ``minimum``, ``prod``) issued next can run both as ONE kernel that reads x,
writes y and reduces the values it has just computed (``dab_affine_mapreduce_all`` / ``dab_affine_reduce``): 8 instead of 12 bytes per
Float32 element, same bits.  Any other C-ABI call on the runtime's context (``_lib.call``: events, ``sync``, copies, frees, NCCL, another
launch) launches the pending op first, so the stream sees every call in program order and nothing is ever skipped.  An error that the
deferred launch returns is raised by the call that launched it.

Workers are numbered 1..P like ``workers()``.  ``P = world_size * workers_per_rank``; worker ``w`` lives on rank
``(w-1) // workers_per_rank``.  ``workers_per_rank > 1`` puts several chunks on one GPU -- used to exercise multi-chunk
layouts (grids, fibres, halo reads) on a single-GPU box; the production mapping is one worker per GPU.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, NamedTuple, Optional

import numpy as np

from . import _lib

_RT: Optional["Runtime"] = None


class PendingAffine(NamedTuple):
    """The deferred ``dab_affine(ctx, dtype, y, x, a, b, n)``; a and b are one-element host arrays of the element type."""
    dtype: int
    y: int
    x: int
    a: np.ndarray
    b: np.ndarray
    n: int


class Runtime:
    def __init__(self, workers_per_rank: int = 1, device: Optional[int] = None, use_dist: Optional[bool] = None):
        L = _lib.lib()
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.workers_per_rank = int(workers_per_rank)
        n = C.c_int32(0)
        _lib.check(L.dab_device_count(C.byref(n)))
        if n.value < 1:
            raise _lib.DabError(_lib.ERR_CUDA, "no CUDA device visible: the DArray hot path has no CPU fallback")
        self.device = int(device) if device is not None else self.local_rank % n.value
        ctx = C.c_void_p()
        _lib.check(L.dab_init(self.device, C.byref(ctx)))
        self.ctx = ctx
        self.dist = None
        self._ipc_cache = {}
        self.last_kernel = None  # which entry point served the last local broadcast launch (diagnostics)
        self.pending: Optional[PendingAffine] = None   # the deferred broadcast (module docstring)
        self.fused_combine = False
        self._arena = None
        if use_dist is None:
            use_dist = self.world > 1
        if use_dist and self.world > 1:
            self._init_dist()

    # ---- torch.distributed plumbing ----------------------------------------------------------------------
    def _init_dist(self):
        import torch
        import torch.distributed as dist

        if not dist.is_initialized():
            torch.cuda.set_device(self.device)
            dist.init_process_group(backend="cpu:gloo,cuda:nccl", rank=self.rank, world_size=self.world)
        self.dist = dist
        ident = np.zeros(128, dtype=np.uint8)
        if self.rank == 0:
            _lib.check(_lib.lib().dab_comm_unique_id(ident.ctypes.data_as(C.c_void_p)))
        box = [ident.tobytes()]
        dist.broadcast_object_list(box, src=0)
        buf = C.create_string_buffer(box[0], 128)
        _lib.call("dab_comm_init_rank", self.ctx, buf, self.rank, self.world)
        # mailboxes for the fused reduce + combine kernel (peer stores over NVLink instead of ncclAllGather + D2H);
        # DAB_FUSED_COMBINE=0 keeps the NCCL path (A/B measurements, debugging)
        if os.environ.get("DAB_FUSED_COMBINE", "1") != "0":
            h = C.create_string_buffer(64)
            _lib.call("dab_mailbox_create", self.ctx, h)
            allh = [None] * self.world
            dist.all_gather_object(allh, h.raw)
            _lib.call("dab_mailbox_attach", self.ctx, C.create_string_buffer(b"".join(allh), 64 * self.world), self.rank, self.world)
            self.fused_combine = True
            dist.barrier()

    def barrier(self):
        """Stream sync + host barrier: the fence before one-sided (peer) reads of other workers' chunks."""
        self.sync()
        if self.dist is not None:
            self.dist.barrier()

    def device_barrier(self):
        """Stream-ordered barrier across the ranks (``dab_peer_barrier``): later launches on this rank's stream start only after every
        rank's earlier launches have completed -- the fence around one-sided peer reads / puts, without a host synchronisation.  Falls
        back to the host barrier when the peer mailboxes are not attached (``DAB_FUSED_COMBINE=0``)."""
        if self.world == 1:
            return
        if self.fused_combine:
            _lib.call("dab_peer_barrier", self.ctx)
        else:
            self.barrier()

    def arena(self, bank_bytes: int = 8 << 20):
        """The exchange arena: two banks of device memory per rank, mapped by every other rank over CUDA IPC (collective on first use).
        Small cross-worker payloads (tile results of ``mul!``, partial slabs of ``mapreducedim_between!``) are PUT straight into the
        consumer's bank with device-to-device copies over NVLink and ordered by ``device_barrier`` -- no NCCL launch, no host sync.
        Banks alternate per exchange, so a producer can fill the next bank while the consumer still reads the previous one."""
        if self._arena is None:
            bank_bytes = int(os.environ.get("DAB_ARENA_KB", bank_bytes >> 10)) << 10   # DAB_ARENA_KB=1 forces the NCCL fallbacks (tests)
            ptr = self.alloc(2 * bank_bytes + 256)
            base = (ptr + 255) & ~255
            if self.world > 1:
                handles = self.allgather_object((self.ipc_handle(ptr), base - ptr))
                peers = [base if r == self.rank else self.ipc_open(h) + off for r, (h, off) in enumerate(handles)]
            else:
                peers = [base]
            self._arena = {"alloc": ptr, "peers": peers, "bank_bytes": bank_bytes, "turn": 0}
        return self._arena

    def arena_next_bank(self) -> int:
        """Byte offset of the bank the next exchange uses (every rank calls this once per exchange, in the same order)."""
        a = self.arena()
        off = (a["turn"] & 1) * a["bank_bytes"]
        a["turn"] += 1
        return off

    def allgather_small(self, arr: Optional[np.ndarray] = None, dev_ptr: int = 0, nbytes: int = 0, dtype=np.uint8) -> List[np.ndarray]:
        """All-gather of one small fixed-size payload per rank WITHOUT a host collective: every rank PUTs its payload (a host array,
        or ``nbytes`` at ``dev_ptr`` on the device) into slot ``rank`` of every peer's exchange-arena bank, a device-side barrier makes
        the puts visible, one D2H copy brings the whole bank to the host.  ~50 us instead of the milliseconds of a pickled
        ``all_gather_object``.  Payloads must have the same size on every rank; falls back to the object gather when they do not fit."""
        if arr is not None:
            arr = np.ascontiguousarray(arr)
            nbytes, dtype = arr.nbytes, arr.dtype
        if self.world == 1:
            if arr is not None:
                return [arr.copy()]
            out = np.empty(nbytes, dtype=np.uint8)
            _lib.call("dab_d2h", self.ctx, C.c_void_p(out.ctypes.data), C.c_void_p(dev_ptr), nbytes)
            self.sync()
            return [out.view(dtype)]
        slot = (nbytes + 255) & ~255
        if not self.fused_combine or slot * self.world > self.arena()["bank_bytes"]:
            if arr is None:
                arr = np.empty(nbytes, dtype=np.uint8)
                _lib.call("dab_d2h", self.ctx, C.c_void_p(arr.ctypes.data), C.c_void_p(dev_ptr), nbytes)
                self.sync()
                arr = arr.view(dtype)
            return self.allgather_object(arr)
        bank = self.arena_next_bank()
        peers = self.arena()["peers"]
        tmp = 0
        if arr is not None:
            tmp = self.alloc_temp(max(nbytes, 16))
            _lib.call("dab_h2d", self.ctx, C.c_void_p(tmp), C.c_void_p(arr.ctypes.data), nbytes)
            self.sync()                                    # arr may be a temporary of the caller
            dev_ptr = tmp
        for r in range(self.world):
            if nbytes:
                _lib.call("dab_d2d", self.ctx, C.c_void_p(peers[r] + bank + self.rank * slot), C.c_void_p(dev_ptr), nbytes)
        self.device_barrier()
        host = np.empty(slot * self.world, dtype=np.uint8)
        _lib.call("dab_d2h", self.ctx, C.c_void_p(host.ctypes.data), C.c_void_p(peers[self.rank] + bank), slot * self.world)
        self.sync()
        if tmp:
            self.free_temp(tmp)
        return [host[r * slot:r * slot + nbytes].view(dtype) for r in range(self.world)]

    def allgather_object(self, obj) -> list:
        if self.dist is None:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    # ---- workers -------------------------------------------------------------------------------------------
    @property
    def nworkers(self) -> int:
        return self.world * self.workers_per_rank

    def workers(self) -> List[int]:
        return list(range(1, self.nworkers + 1))

    def rank_of(self, pid: int) -> int:
        return (pid - 1) // self.workers_per_rank

    def is_local(self, pid: int) -> bool:
        return self.rank_of(pid) == self.rank

    def local_workers(self) -> List[int]:
        return [p for p in self.workers() if self.is_local(p)]

    def myid(self) -> int:
        """The first worker of this rank (the only one when workers_per_rank == 1)."""
        return self.rank * self.workers_per_rank + 1

    # ---- the deferred broadcast ----------------------------------------------------------------------------
    def defer_affine(self, dtype: int, y: int, x: int, a: np.ndarray, b: np.ndarray, n: int):
        """Record ``dab_affine(dtype, y, x, a, b, n)`` as the pending op instead of launching it (an earlier pending op launches first).
        Launched at once when the binding has no fused entry point to hand it to (``_lib.serves_fused_step``)."""
        self.flush()
        self.pending = PendingAffine(dtype, y, x, a, b, n)
        _lib._DEFERRED[_lib.ctx_key(self.ctx)] = self
        if not _lib.serves_fused_step():
            self.flush()

    def flush(self):
        """Launch the pending op, if any."""
        p = self.take_pending()
        if p is not None:
            _lib.check(_lib.lib().dab_affine(self.ctx, p.dtype, C.c_void_p(p.y), C.c_void_p(p.x), C.c_void_p(p.a.ctypes.data),
                                             C.c_void_p(p.b.ctypes.data), p.n), self.ctx)

    def take_pending(self, dtype: Optional[int] = None, y: Optional[int] = None, n: Optional[int] = None) -> Optional[PendingAffine]:
        """Remove and return the pending op -- only if it writes exactly ``n`` elements of ``dtype`` at ``y`` when those are given.
        The caller then owns the launch."""
        p = self.pending
        if p is None or (dtype is not None and (p.dtype, p.y, p.n) != (dtype, y, n)):
            return None
        self.pending = None
        _lib._DEFERRED.pop(_lib.ctx_key(self.ctx), None)
        return p

    # ---- device helpers ------------------------------------------------------------------------------------
    def sync(self):
        _lib.call("dab_sync", self.ctx)

    def alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        _lib.call("dab_alloc", self.ctx, int(nbytes), C.byref(p))
        return int(p.value)

    def free(self, ptr: int):
        if ptr and self.ctx:
            _lib.call("dab_free", self.ctx, C.c_void_p(ptr))

    def alloc_temp(self, nbytes: int) -> int:
        """Stream-ordered temporary (cudaMallocAsync pool): no synchronisation, not IPC-exportable."""
        p = C.c_void_p()
        _lib.call("dab_alloc_async", self.ctx, int(nbytes), C.byref(p))
        return int(p.value)

    def free_temp(self, ptr: int):
        if ptr and self.ctx:
            _lib.call("dab_free_async", self.ctx, C.c_void_p(ptr))

    def set_option(self, key: str, value: int):
        """``dab_set_option``: e.g. ``set_option("ew_tma", 1)`` selects the TMA-staged elementwise kernel (same results)."""
        _lib.call("dab_set_option", self.ctx, key.encode(), int(value))

    def launches(self) -> int:
        n = C.c_uint64(0)
        _lib.call("dab_launch_count", self.ctx, C.byref(n))
        return int(n.value)

    def device_info(self):
        dev, sms, fr, tot = C.c_int32(), C.c_int32(), C.c_size_t(), C.c_size_t()
        _lib.call("dab_device_info", self.ctx, C.byref(dev), C.byref(sms), C.byref(fr), C.byref(tot))
        return {"device": dev.value, "sm_count": sms.value, "free_bytes": fr.value, "total_bytes": tot.value}

    # events on the ctx stream
    def event(self) -> int:
        e = C.c_void_p()
        _lib.call("dab_event_create", self.ctx, C.byref(e))
        return int(e.value)

    def record(self, ev: int):
        _lib.call("dab_event_record", self.ctx, C.c_void_p(ev))

    def elapsed_ms(self, e0: int, e1: int) -> float:
        ms = C.c_float()
        _lib.call("dab_event_elapsed_ms", self.ctx, C.c_void_p(e0), C.c_void_p(e1), C.byref(ms))
        return float(ms.value)

    def event_destroy(self, ev: int):
        _lib.call("dab_event_destroy", self.ctx, C.c_void_p(ev))

    # peer memory
    def ipc_handle(self, ptr: int) -> bytes:
        h = C.create_string_buffer(64)
        _lib.call("dab_ipc_get_handle", self.ctx, C.c_void_p(ptr), h)
        return h.raw

    def ipc_open(self, handle: bytes) -> int:
        if handle in self._ipc_cache:
            return self._ipc_cache[handle]
        p = C.c_void_p()
        _lib.call("dab_ipc_open", self.ctx, C.create_string_buffer(handle, 64), C.byref(p))
        self._ipc_cache[handle] = int(p.value)
        return int(p.value)

    def shutdown(self):
        global _RT
        if self.ctx:
            try:
                self.flush()                               # dab_shutdown below is called directly, not through _lib.call
            except _lib.DabError:
                pass
            for p in self._ipc_cache.values():
                try:
                    _lib.call("dab_ipc_close", self.ctx, C.c_void_p(p))
                except _lib.DabError:
                    pass
            self._ipc_cache.clear()
            if self._arena is not None:
                try:
                    _lib.call("dab_free", self.ctx, C.c_void_p(self._arena["alloc"]))
                except _lib.DabError:
                    pass
                self._arena = None
            _lib.lib().dab_shutdown(self.ctx)
            self.ctx = None
        if self.dist is not None:
            try:
                if self.dist.is_initialized():
                    self.dist.destroy_process_group()
            except Exception:
                pass
            self.dist = None
        if _RT is self:
            _RT = None


def init(workers_per_rank: int = 1, device: Optional[int] = None, use_dist: Optional[bool] = None) -> Runtime:
    """``addprocs`` analogue: create (or re-create) the process-wide runtime."""
    global _RT
    if _RT is not None:
        if _RT.workers_per_rank == workers_per_rank and (device is None or device == _RT.device):
            return _RT
        _RT.shutdown()
    _RT = Runtime(workers_per_rank, device, use_dist)
    return _RT


def runtime() -> Runtime:
    global _RT
    if _RT is None:
        _RT = Runtime()
    return _RT


def nworkers() -> int:
    return runtime().nworkers


def workers() -> List[int]:
    return runtime().workers()


def myid() -> int:
    return runtime().myid()
