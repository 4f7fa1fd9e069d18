"""ctypes binding for libb200coll (coll/lib/libb200coll.so) — the only thing PyTorch is used for here is
launching ranks and holding the synthetic buffers (BASELINE.json north-star: "PyTorch is only the harness").

The library is the transport-installer payload (reference role: gpudirect-rdma/nccl-rdma-installer.yaml:70-77);
this module is what a pod's Python code imports once the device plugin's Allocate has mounted it.
Fails loudly when the shared object is missing on a GPU box — there is no eager/PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from pathlib import Path
from typing import Optional

REPO_ROOT = Path(__file__).resolve().parents[2]
_LIB_CANDIDATES = [
    os.environ.get("B200COLL_LIB", ""),
    str(REPO_ROOT / "coll" / "lib" / "libb200coll.so"),
    "/usr/local/nvidia/lib64/libb200coll.so",   # where Allocate mounts the installer's drop
    "libb200coll.so",
]

SUCCESS = 0
NO_DRIVER = 9
MAX_RANKS = 8

F32, F16, BF16, FP8_E4M3, I8, U8, I32, U32, I64, U64, F64, FP8_E5M2 = range(12)
SUM, AVG, PROD, MIN, MAX = range(5)
OP_ALLREDUCE, OP_ALLGATHER, OP_REDUCESCATTER, OP_ALLTOALL = 0, 1, 2, 3
ALGO_AUTO, ALGO_LL, ALGO_ONESHOT, ALGO_TWOSHOT, ALGO_NVLS, ALGO_COPY, ALGO_LL2 = range(7)
ALGO_NAMES = ["auto", "ll", "oneshot", "twoshot", "nvls", "copy", "ll2"]
DTYPE_SIZE = {F32: 4, F16: 2, BF16: 2, FP8_E4M3: 1, I8: 1, U8: 1, I32: 4, U32: 4, I64: 8, U64: 8, F64: 8, FP8_E5M2: 1}


class UniqueId(C.Structure):
    _fields_ = [("internal", C.c_char * 128)]


class Epilogue(C.Structure):
    _fields_ = [("in_dtype", C.c_int), ("out_dtype", C.c_int), ("scale", C.c_float)]


class Config(C.Structure):
    _fields_ = [("arena_bytes", C.c_size_t), ("enable_nvls", C.c_int), ("max_ctas", C.c_int), ("timeout_ms", C.c_int), ("debug", C.c_int)]


class CommInfo(C.Structure):
    _fields_ = [("rank", C.c_int), ("nranks", C.c_int), ("device", C.c_int), ("nvls", C.c_int), ("p2p_ok", C.c_int),
                ("same_device_loopback", C.c_int), ("arena_bytes", C.c_size_t), ("arena_used", C.c_size_t), ("sm_count", C.c_int),
                ("driver_version", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("calls", C.c_uint64 * 6), ("bytes", C.c_uint64 * 6), ("algo_calls", C.c_uint64 * 7), ("kernel_launches", C.c_uint64),
                ("staged_calls", C.c_uint64), ("p2p_sends", C.c_uint64), ("p2p_recvs", C.c_uint64), ("p2p_bytes", C.c_uint64),
                ("host_calls", C.c_uint64), ("host_bytes", C.c_uint64), ("host_zero_copy", C.c_uint64), ("host_pipelined", C.c_uint64), ("bulk_launches", C.c_uint64), ("generic_launches", C.c_uint64)]


class Fault(C.Structure):
    _fields_ = [("code", C.c_uint32), ("rank", C.c_uint32), ("peer", C.c_uint32), ("block", C.c_uint32), ("expected", C.c_uint32),
                ("observed", C.c_uint32), ("op", C.c_uint32), ("reserved", C.c_uint32)]


class B200CollError(RuntimeError):
    def __init__(self, code: int, what: str, detail: str):
        super().__init__(f"{what}: {detail}" if detail else what)
        self.code = code


_lib: Optional[C.CDLL] = None


def lib_path() -> Optional[str]:
    for cand in _LIB_CANDIDATES[:-1]:
        if cand and os.path.exists(cand):
            return cand
    return None


def load() -> C.CDLL:
    """dlopen the library once and declare prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    last = None
    for cand in _LIB_CANDIDATES:
        if not cand:
            continue
        try:
            _lib = C.CDLL(cand, mode=C.RTLD_GLOBAL)
            break
        except OSError as e:   # keep looking
            last = e
    if _lib is None:
        raise ImportError(f"libb200coll.so not found (run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C coll`): {last}")
    L = _lib
    vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
    L.b200collGetErrorString.restype = C.c_char_p; L.b200collGetErrorString.argtypes = [ci]
    L.b200collGetLastError.restype = C.c_char_p
    L.b200collGetVersion.restype = ci
    L.b200collConfigDefault.argtypes = [C.POINTER(Config)]
    L.b200collGetUniqueId.argtypes = [C.POINTER(UniqueId)]
    L.b200collUniqueIdFromString.argtypes = [C.c_char_p, C.POINTER(UniqueId)]
    L.b200collCommInitRank.argtypes = [C.POINTER(vp), ci, C.POINTER(UniqueId), ci, C.POINTER(Config)]
    L.b200collCommInitAll.argtypes = [C.POINTER(vp), ci, C.POINTER(ci), C.POINTER(Config)]
    L.b200collCommDestroy.argtypes = [vp]
    L.b200collCommSplit.argtypes = [vp, ci, ci, C.POINTER(vp), C.POINTER(Config)]
    L.b200collDebugSplitPlan.argtypes = [ci, ci, C.POINTER(ci), C.POINTER(ci), C.POINTER(ci), C.POINTER(ci)]
    L.b200collCommInfoGet.argtypes = [vp, C.POINTER(CommInfo)]
    L.b200collCommStatsGet.argtypes = [vp, C.POINTER(Stats)]
    L.b200collCommGetAsyncError.argtypes = [vp, C.POINTER(Fault)]
    L.b200collHostBarrier.argtypes = [vp]
    L.b200collMemAlloc.argtypes = [vp, C.POINTER(vp), sz]
    L.b200collMemFree.argtypes = [vp, vp]
    L.b200collIsSymmetric.argtypes = [vp, vp, sz]
    L.b200collSetAllocatorComm.argtypes = [vp]
    L.b200collTorchAlloc.argtypes = [sz, ci, vp]; L.b200collTorchAlloc.restype = vp
    L.b200collTorchFree.argtypes = [vp, sz, ci, vp]; L.b200collTorchFree.restype = None
    L.b200collAllReduce.argtypes = [vp, vp, sz, C.POINTER(Epilogue), ci, vp, vp]
    L.b200collAllGather.argtypes = [vp, vp, sz, C.POINTER(Epilogue), vp, vp]
    L.b200collReduceScatter.argtypes = [vp, vp, sz, C.POINTER(Epilogue), ci, vp, vp]
    L.b200collAllToAll.argtypes = [vp, vp, sz, C.POINTER(Epilogue), vp, vp]
    L.b200collAllToAllv.argtypes = [vp, vp, sz, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(Epilogue), vp, vp]
    L.b200collBroadcast.argtypes = [vp, vp, sz, C.POINTER(Epilogue), ci, vp, vp]
    L.b200collReduce.argtypes = [vp, vp, sz, C.POINTER(Epilogue), ci, ci, vp, vp]
    L.b200collBarrier.argtypes = [vp, vp]
    L.b200collHostAlloc.argtypes = [vp, C.POINTER(vp), sz]
    L.b200collHostFree.argtypes = [vp, vp]
    L.b200collAllReduceHost.argtypes = [vp, vp, sz, C.POINTER(Epilogue), ci, vp, vp]
    L.b200collCommNumaGet.argtypes = [vp, C.POINTER(ci), C.c_char_p, sz]
    L.b200collDebugParseCpuList.argtypes = [C.c_char_p, C.POINTER(ci), ci]
    L.b200collGroupStart.argtypes = []; L.b200collGroupEnd.argtypes = []
    L.b200collSend.argtypes = [vp, sz, ci, vp, vp]
    L.b200collRecv.argtypes = [vp, sz, ci, vp, vp]
    L.b200collTunerPick.argtypes = [ci, sz, ci, ci]; L.b200collTunerPick.restype = ci
    L.b200collCommSetAlgo.argtypes = [vp, ci]
    L.b200collCommGetAlgo.argtypes = [vp]; L.b200collCommGetAlgo.restype = ci
    L.b200collCommSetMaxCtas.argtypes = [vp, ci]
    L.b200collCommSetLaunchShape.argtypes = [vp, ci, ci, ci]
    L.b200collCommSetP2pWindow.argtypes = [vp, sz]
    L.b200collAlgoName.argtypes = [ci]; L.b200collAlgoName.restype = C.c_char_p
    L.b200collTypeSize.argtypes = [ci]; L.b200collTypeSize.restype = sz
    L.b200collSelfCheck.argtypes = [C.c_char_p, sz]
    return L


def _check(rc: int, what: str) -> None:
    if rc != SUCCESS:
        L = load()
        raise B200CollError(rc, f"{what}: {L.b200collGetErrorString(rc).decode()}", L.b200collGetLastError().decode())


class group:
    """`with coll.group(): comm.send(...); comm.recv(...)`: every send / recv issued inside (by this thread, on any communicator)
    becomes one kernel per communicator at exit (ncclGroupStart / ncclGroupEnd). Needed whenever a rank both sends and receives in
    one step: outside a group each call waits for its peer before the next one is launched."""

    def __enter__(self):
        _check(load().b200collGroupStart(), "GroupStart")
        return self

    def __exit__(self, exc_type, exc, tb):
        rc = load().b200collGroupEnd()
        if exc_type is None:
            _check(rc, "GroupEnd")
        return False


def tuner_pick(op: int, nbytes: int, nranks: int, nvls: bool) -> str:
    return ALGO_NAMES[load().b200collTunerPick(op, nbytes, nranks, 1 if nvls else 0)]


def self_check() -> tuple[bool, str]:
    buf = C.create_string_buffer(8192)
    rc = load().b200collSelfCheck(buf, len(buf))
    return rc == SUCCESS, buf.value.decode()


def torch_dtype_code(dtype) -> int:
    import torch
    return {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16, torch.float8_e4m3fn: FP8_E4M3, torch.float8_e5m2: FP8_E5M2, torch.int8: I8, torch.uint8: U8, torch.int32: I32,
            torch.int64: I64, torch.float64: F64, torch.bool: U8}[dtype]


class _CudaArray:
    """Minimal __cuda_array_interface__ carrier so torch can alias arena memory without a copy."""

    def __init__(self, ptr: int, nbytes: int, owner):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}
        self._owner = owner


@dataclass
class SymBuffer:
    ptr: int
    nbytes: int


class Comm:
    """One communicator rank. `Comm.from_env()` under torchrun; `Comm.init_all()` for in-process groups."""

    def __init__(self, handle: int, owner_group=None):
        self._h = C.c_void_p(handle)
        self._group = owner_group
        self._allocs: dict[int, int] = {}
        info = CommInfo()
        _check(load().b200collCommInfoGet(self._h, C.byref(info)), "CommInfoGet")
        self.rank, self.nranks, self.device, self.nvls = info.rank, info.nranks, info.device, bool(info.nvls)
        self.loopback = bool(info.same_device_loopback)
        self.sm_count = info.sm_count

    # ---------------------------------------------------------------- construction
    @staticmethod
    def make_config(arena_mb: Optional[int] = None, nvls: Optional[int] = None, timeout_ms: Optional[int] = None) -> Config:
        cfg = Config()
        load().b200collConfigDefault(C.byref(cfg))
        if arena_mb is not None:
            cfg.arena_bytes = int(arena_mb) << 20
        if nvls is not None:
            cfg.enable_nvls = nvls
        if timeout_ms is not None:
            cfg.timeout_ms = timeout_ms
        return cfg

    @classmethod
    def from_env(cls, arena_mb: Optional[int] = None, tag: str = "0", **kw) -> "Comm":
        """torchrun-style: RANK / WORLD_SIZE / LOCAL_RANK / MASTER_ADDR / MASTER_PORT. The caller has already
        selected its GPU (torch.cuda.set_device(LOCAL_RANK))."""
        rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
        key = f"{os.environ.get('MASTER_ADDR', '127.0.0.1')}:{os.environ.get('MASTER_PORT', '0')}/{os.environ.get('TORCHELASTIC_RUN_ID', '')}/{tag}"
        return cls.init_rank(rank, world, key, arena_mb=arena_mb, **kw)

    @classmethod
    def init_rank(cls, rank: int, nranks: int, key: str, arena_mb: Optional[int] = None, **kw) -> "Comm":
        L = load()
        uid = UniqueId()
        _check(L.b200collUniqueIdFromString(key.encode(), C.byref(uid)), "UniqueIdFromString")
        cfg = cls.make_config(arena_mb, **kw)
        h = C.c_void_p()
        _check(L.b200collCommInitRank(C.byref(h), nranks, C.byref(uid), rank, C.byref(cfg)), "CommInitRank")
        return cls(h.value)

    @classmethod
    def init_all(cls, devices: list[int], arena_mb: Optional[int] = None, **kw) -> list["Comm"]:
        L = load()
        n = len(devices)
        hs = (C.c_void_p * n)()
        devs = (C.c_int * n)(*devices)
        cfg = cls.make_config(arena_mb, **kw)
        _check(L.b200collCommInitAll(hs, n, devs, C.byref(cfg)), "CommInitAll")
        return [cls(hs[i]) for i in range(n)]

    def mem_pool(self):
        """A `torch.cuda.MemPool` whose memory is this communicator's symmetric arena (PyTorch's pluggable-allocator hook calling
        b200collMemAlloc). Tensors created under `torch.cuda.use_mem_pool(pool)` — a model's parameters, DDP's gradient buckets with
        `gradient_as_bucket_view=True` — are then arena tensors: collectives on them skip staging and may use NVLS. Every rank must
        allocate the same sizes in the same order inside the pool (SPMD code does). One pool-backed communicator per process."""
        import torch
        from torch.cuda.memory import CUDAPluggableAllocator
        if getattr(self, "_pool", None) is None:
            _check(load().b200collSetAllocatorComm(self._h), "SetAllocatorComm")
            self._pool_allocator = CUDAPluggableAllocator(lib_path(), "b200collTorchAlloc", "b200collTorchFree")
            self._pool = torch.cuda.MemPool(self._pool_allocator.allocator())
        return self._pool

    def split(self, color: int, key: int = 0, arena_mb: Optional[int] = None, **kw) -> Optional["Comm"]:
        """ncclCommSplit: every rank of this (multi-process) communicator calls it; ranks with the same color >= 0 get a new communicator
        with its own arena, ordered by (key, rank here). A negative color takes part and returns None. Tensor-parallel and data-parallel
        groups of one job are two splits of the world communicator."""
        cfg = self.make_config(arena_mb, **kw) if (arena_mb is not None or kw) else None
        h = C.c_void_p()
        _check(load().b200collCommSplit(self._h, color, key, C.byref(h), C.byref(cfg) if cfg is not None else None), "CommSplit")
        return type(self)(h.value) if h.value else None

    def destroy(self) -> None:
        if self._h:
            load().b200collCommDestroy(self._h)
            self._h = None

    # ---------------------------------------------------------------- memory
    def alloc(self, nbytes: int) -> SymBuffer:
        p = C.c_void_p()
        _check(load().b200collMemAlloc(self._h, C.byref(p), nbytes), "MemAlloc")
        self._allocs[p.value] = nbytes
        return SymBuffer(p.value, nbytes)

    def free(self, buf: SymBuffer) -> None:
        _check(load().b200collMemFree(self._h, C.c_void_p(buf.ptr)), "MemFree")
        self._allocs.pop(buf.ptr, None)

    def empty(self, numel: int, dtype):
        """A torch tensor living in the symmetric arena (zero-copy fast paths, NVLS capable)."""
        import torch
        itemsize = torch.empty((), dtype=dtype).element_size()
        buf = self.alloc(numel * itemsize)
        raw = torch.as_tensor(_CudaArray(buf.ptr, buf.nbytes, self), device=torch.device("cuda", self.device))
        t = raw.view(dtype)[:numel]
        t._b200coll_buf = buf   # keep the allocation discoverable
        return t

    def release(self, tensor) -> None:
        """Give a tensor from `empty()` back to the arena. Explicit on purpose: allocation is a collective contract (same order and
        sizes on every rank keep the offsets identical), so it must not depend on when each rank's garbage collector runs.
        The caller guarantees no collective is still using the tensor."""
        buf = getattr(tensor, "_b200coll_buf", None)
        if buf is None:
            raise ValueError("tensor was not allocated with Comm.empty()")
        self.free(buf)
        tensor._b200coll_buf = None

    def is_symmetric(self, tensor) -> bool:
        return bool(load().b200collIsSymmetric(self._h, C.c_void_p(tensor.data_ptr()), tensor.numel() * tensor.element_size()))

    # ---------------------------------------------------------------- collectives (tensors)
    @staticmethod
    def _stream(stream) -> C.c_void_p:
        import torch
        s = stream if stream is not None else torch.cuda.current_stream()
        return C.c_void_p(s.cuda_stream)

    def _ep(self, src, dst, scale: float) -> Epilogue:
        return Epilogue(torch_dtype_code(src.dtype), torch_dtype_code(dst.dtype), float(scale))

    def all_reduce(self, src, dst=None, scale: float = 1.0, op: int = SUM, stream=None):
        dst = src if dst is None else dst
        ep = self._ep(src, dst, scale)
        _check(load().b200collAllReduce(C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), src.numel(), C.byref(ep), op, self._h, self._stream(stream)), "AllReduce")
        return dst

    def all_reduce_from_host(self, host_in, out, chunk_bytes: int = 32 << 20, scale: float = 1.0, op: int = SUM, stream=None):
        """End-to-end step: `out` (device, ideally from `empty()`) = all-reduce of every rank's pinned host tensor `host_in`.
        The host→device copy is pipelined with the collective: chunk i+1 crosses PCIe on a copy stream while chunk i is reduced out
        of one of two arena staging buffers, so the step costs about the copy time instead of copy + collective. Same call (sizes,
        chunking) on every rank. EXPERIMENTAL: composed from validated pieces (copies, events, `all_reduce`) but not yet timed on hardware."""
        import torch
        assert host_in.device.type == "cpu" and out.is_cuda and host_in.numel() == out.numel() and host_in.is_contiguous() and out.is_contiguous()
        main = stream if stream is not None else torch.cuda.current_stream()
        itemsize = host_in.element_size()
        chunk = max(1, chunk_bytes // itemsize // 64 * 64)
        if not hasattr(self, "_h2d"):
            self._h2d = {"stream": torch.cuda.Stream(), "bufs": {}, "ready": [torch.cuda.Event(), torch.cuda.Event()], "free": [torch.cuda.Event(), torch.cuda.Event()]}
        st = self._h2d
        key = (chunk, host_in.dtype)
        if key not in st["bufs"]:
            st["bufs"][key] = [self.empty(chunk, host_in.dtype), self.empty(chunk, host_in.dtype)]
        bufs, ready, free, copy_stream = st["bufs"][key], st["ready"], st["free"], st["stream"]
        copy_stream.wait_stream(main)                       # staging buffers may still be in use by earlier work on the caller's stream
        n_total, flat_in, flat_out = host_in.numel(), host_in.view(-1), out.view(-1)
        for i, off in enumerate(range(0, n_total, chunk)):
            k, n = i & 1, min(chunk, n_total - off)
            with torch.cuda.stream(copy_stream):
                if i >= 2:
                    copy_stream.wait_event(free[k])         # the collective that read this staging buffer two chunks ago is done
                bufs[k][:n].copy_(flat_in[off:off + n], non_blocking=True)
                ready[k].record(copy_stream)
            main.wait_event(ready[k])
            self.all_reduce(bufs[k][:n], flat_out[off:off + n], scale=scale, op=op, stream=main)
            free[k].record(main)
        return out

    def host_empty(self, numel: int, dtype):
        """A pinned, device-mapped CPU tensor on the NUMA node of this rank's GPU (b200collHostAlloc): the buffer to hand to
        `all_reduce_host`. On a two-socket 8-GPU box this placement is what keeps eight concurrent host<->device copies at link rate."""
        import torch
        itemsize = torch.empty((), dtype=dtype).element_size()
        nbytes = max(1, numel * itemsize)
        p = C.c_void_p()
        _check(load().b200collHostAlloc(self._h, C.byref(p), nbytes), "HostAlloc")
        raw = (C.c_uint8 * nbytes).from_address(p.value)
        t = torch.frombuffer(raw, dtype=torch.uint8).view(dtype)[:numel]
        t._b200coll_host = p.value
        self._host_allocs = getattr(self, "_host_allocs", {})
        self._host_allocs[p.value] = raw
        return t

    def host_release(self, tensor) -> None:
        p = getattr(tensor, "_b200coll_host", None)
        if p is None:
            raise ValueError("tensor was not allocated with Comm.host_empty()")
        _check(load().b200collHostFree(self._h, C.c_void_p(p)), "HostFree")
        self._host_allocs.pop(p, None)
        tensor._b200coll_host = None

    def numa(self) -> tuple[int, str]:
        """(NUMA node of this rank's GPU or -1, its local CPU list as sysfs prints it)."""
        node = C.c_int(-1)
        buf = C.create_string_buffer(256)
        _check(load().b200collCommNumaGet(self._h, C.byref(node), buf, len(buf)), "CommNumaGet")
        return node.value, buf.value.decode()

    def all_reduce_host(self, host_in, host_out=None, scale: float = 1.0, op: int = SUM, stream=None):
        """The end-to-end step as one library call: `host_out` (pinned CPU tensor, default in place) = cast(scale * sum over ranks
        of `host_in`). Asynchronous on `stream`; tiny messages run as one zero-copy kernel over PCIe, large ones are chunked so that
        the copy in, the all-reduce and the copy back overlap (b200collAllReduceHost, coll/src/hostpath.cu). Same call on every rank."""
        host_out = host_in if host_out is None else host_out
        assert host_in.device.type == "cpu" and host_out.device.type == "cpu" and host_in.is_contiguous() and host_out.is_contiguous()
        assert host_in.numel() == host_out.numel()
        ep = self._ep(host_in, host_out, scale)
        _check(load().b200collAllReduceHost(C.c_void_p(host_in.data_ptr()), C.c_void_p(host_out.data_ptr()), host_in.numel(), C.byref(ep), op, self._h,
                                            self._stream(stream)), "AllReduceHost")
        return host_out

    def all_gather(self, src, dst, scale: float = 1.0, stream=None):
        ep = self._ep(src, dst, scale)
        _check(load().b200collAllGather(C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), src.numel(), C.byref(ep), self._h, self._stream(stream)), "AllGather")
        return dst

    def reduce_scatter(self, src, dst, scale: float = 1.0, op: int = SUM, stream=None):
        ep = self._ep(src, dst, scale)
        _check(load().b200collReduceScatter(C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), dst.numel(), C.byref(ep), op, self._h, self._stream(stream)), "ReduceScatter")
        return dst

    def all_to_all(self, src, dst, scale: float = 1.0, stream=None):
        ep = self._ep(src, dst, scale)
        _check(load().b200collAllToAll(C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), src.numel() // self.nranks, C.byref(ep), self._h, self._stream(stream)), "AllToAll")
        return dst

    def all_to_all_v(self, src, dst, row_elems: int, send_rows, send_row_off, recv_row_off_at_peer, scale: float = 1.0, stream=None):
        ep = self._ep(src, dst, scale)
        n = self.nranks
        arr = lambda xs: (C.c_int64 * n)(*[int(x) for x in xs])
        _check(load().b200collAllToAllv(C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), row_elems, arr(send_rows), arr(send_row_off), arr(recv_row_off_at_peer),
                                        C.byref(ep), self._h, self._stream(stream)), "AllToAllv")
        return dst

    def broadcast(self, src, dst=None, root: int = 0, scale: float = 1.0, stream=None):
        """dst on every rank = cast(scale * src of `root`). src is read on the root only (ncclBroadcast)."""
        dst = src if dst is None else dst
        ep = self._ep(src, dst, scale)
        _check(load().b200collBroadcast(C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), dst.numel(), C.byref(ep), root, self._h, self._stream(stream)), "Broadcast")
        return dst

    def reduce(self, src, dst=None, root: int = 0, scale: float = 1.0, op: int = SUM, stream=None):
        """dst on `root` = cast(scale * sum over ranks of src); dst is untouched elsewhere (ncclReduce)."""
        dst = src if dst is None else dst
        ep = self._ep(src, dst, scale)
        _check(load().b200collReduce(C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr()), src.numel(), C.byref(ep), op, root, self._h, self._stream(stream)), "Reduce")
        return dst

    def send(self, src, peer: int, stream=None) -> None:
        """Send the bytes of (contiguous) `src` to rank `peer` (ncclSend). Pairs with the peer's recv of the same size, in call order.
        Outside `group()` the call blocks the stream until the peer's recv runs."""
        _check(load().b200collSend(C.c_void_p(src.data_ptr()), src.numel() * src.element_size(), peer, self._h, self._stream(stream)), "Send")

    def recv(self, dst, peer: int, stream=None):
        """Receive into (contiguous) `dst` from rank `peer` (ncclRecv): written over NVLink in place when dst is an arena tensor, else staged."""
        _check(load().b200collRecv(C.c_void_p(dst.data_ptr()), dst.numel() * dst.element_size(), peer, self._h, self._stream(stream)), "Recv")
        return dst

    def barrier(self, stream=None) -> None:
        _check(load().b200collBarrier(self._h, self._stream(stream)), "Barrier")

    def host_barrier(self) -> None:
        _check(load().b200collHostBarrier(self._h), "HostBarrier")

    # ---------------------------------------------------------------- control / introspection
    def set_algo(self, name: str) -> None:
        _check(load().b200collCommSetAlgo(self._h, ALGO_NAMES.index(name)), "CommSetAlgo")
        self._algo = name

    class _BitExact:
        """Payloads that are not floating point (token ids, masks) must not take the Lamport path: it recognises empty slots by a NaN bit
        pattern and rewrites payload words that collide with it (harmless for floats, fatal for an int64 -1), and it passes data through
        fp32 registers. The barrier-based push kernels forward 16-byte vectors untouched when the epilogue is the identity."""

        def __init__(self, comm):
            self.comm = comm
            self.prev = getattr(comm, "_algo", None) or ALGO_NAMES[load().b200collCommGetAlgo(comm._h)]      # B200COLL_ALGO may have forced one at init

        def __enter__(self):
            self.comm.set_algo("twoshot")
            return self.comm

        def __exit__(self, *exc):
            self.comm.set_algo(self.prev)
            return False

    def bit_exact(self) -> "Comm._BitExact":
        """`with comm.bit_exact(): comm.all_gather(words, out)` — moves arbitrary bits (viewed as fp16 / fp32 words) unchanged."""
        return Comm._BitExact(self)

    def set_max_ctas(self, n: int) -> None:
        _check(load().b200collCommSetMaxCtas(self._h, n), "CommSetMaxCtas")

    def set_p2p_window(self, nbytes: int) -> None:
        """Staging-window size for receives into tensors outside the arena (0 = automatic)."""
        _check(load().b200collCommSetP2pWindow(self._h, nbytes), "CommSetP2pWindow")

    def set_launch_shape(self, kind: str, max_ctas: int = 0, threads: int = 0) -> None:
        _check(load().b200collCommSetLaunchShape(self._h, {"nvls": 0, "p2p": 1, "ll": 2, "nvls_rs": 3, "rooted": 4}[kind], max_ctas, threads), "CommSetLaunchShape")

    def stats(self) -> dict:
        s = Stats()
        _check(load().b200collCommStatsGet(self._h, C.byref(s)), "CommStatsGet")
        return {"calls": list(s.calls), "bytes": list(s.bytes), "algo_calls": dict(zip(ALGO_NAMES, s.algo_calls)),
                "kernel_launches": s.kernel_launches, "staged_calls": s.staged_calls,
                "p2p_sends": s.p2p_sends, "p2p_recvs": s.p2p_recvs, "p2p_bytes": s.p2p_bytes,
                "host_calls": s.host_calls, "host_bytes": s.host_bytes, "host_zero_copy": s.host_zero_copy, "host_pipelined": s.host_pipelined, "bulk_launches": s.bulk_launches, "generic_launches": s.generic_launches}

    def check_async_error(self) -> None:
        f = Fault()
        rc = load().b200collCommGetAsyncError(self._h, C.byref(f))
        if rc != SUCCESS:
            raise B200CollError(rc, "watchdog", f"code={f.code} rank={f.rank} peer={f.peer} block={f.block} expected={f.expected} observed={f.observed} op={f.op}")
