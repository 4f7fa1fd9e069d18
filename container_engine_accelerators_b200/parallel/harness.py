"""nccl-tests-protocol sweep harness shared by bench.py and bench/*_perf.py.

Protocol (reference: gpudirect-tcpx/nccl-config.yaml:61-62 `-b .. -e .. -f 2 -g 1 -w 5 --iters 100`,
gpudirect-rdma/nccl-test-a4x-max-jobset.yaml:141-153): one rank per GPU, per message size `warmup` untimed
launches then `steps` back-to-back launches timed with CUDA events on the launching stream, bracketed by a
cross-rank barrier + device synchronize; time = max over ranks; algbw = bytes/time; busbw = algbw x
{all_reduce: 2(N-1)/N, others: (N-1)/N}; out-of-place and in-place; "Avg bus bandwidth" = mean over every
measured (size, placement). Buffers rotate through a >L2 window (192 MiB > 126 MB) so no timed launch
re-reads lines left in L2 by the previous one.

Two arms, same harness, same buffers sizes, same ctypes-level call overhead:
  ours       libb200coll on symmetric-arena tensors (container_engine_accelerators_b200.ops.coll)
  reference  stock libnccl through its C API (container_engine_accelerators_b200.parallel.nccl_ref)
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

OPS = ("all_reduce", "all_gather", "reduce_scatter", "alltoall", "broadcast", "reduce")   # index = b200collOp_t
P2P_OPS = ("sendrecv", "gather", "scatter")     # nccl-tests sendrecv_perf (a ring step), gather_perf, scatter_perf: groups of send / recv through the point-to-point kernel
ALL_OPS = OPS + P2P_OPS
ROOT = 0   # rooted ops are measured from rank 0, as nccl-tests does by default
FULL_MESSAGE_OPS = ("all_reduce", "broadcast", "reduce", "sendrecv")   # gather / scatter split the message over the ranks like all_gather / reduce_scatter   # count = whole message; the others split it over the ranks
WINDOW = 192 << 20


def bus_factor(op: str, n: int) -> float:
    if n <= 1:
        return 1.0   # nccl-tests prints busbw 0 for one rank; we report algbw there and say so
    if op in ("broadcast", "reduce", "sendrecv"):
        return 1.0   # nccl-tests: rooted ops (and a ring step) move the whole message over one rank's links, busbw = algbw
    return 2.0 * (n - 1) / n if op == "all_reduce" else (n - 1) / n


@dataclass
class Row:
    nbytes: int
    count: int
    algo: str
    oop_us: float = -1.0
    ip_us: float = -1.0
    e2e_us: float = -1.0
    in_bytes: int = 0
    out_bytes: int = 0

    def bw(self, op: str, n: int) -> dict:
        f = bus_factor(op, n)
        ab = lambda us: (self.nbytes / us / 1e3) if us > 0 else 0.0
        return {"oop_algbw": ab(self.oop_us), "ip_algbw": ab(self.ip_us), "oop_busbw": ab(self.oop_us) * f, "ip_busbw": ab(self.ip_us) * f,
                "e2e_busbw": ab(self.e2e_us) * f}


class Dist:
    """CPU-side control plane (gloo): barrier and max-over-ranks. world_size 1 is a no-op."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.pg = None
        if self.world > 1:
            import torch.distributed as dist
            if not dist.is_initialized():
                os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
                os.environ.setdefault("MASTER_PORT", "29500")
                dist.init_process_group("gloo")
            self.pg = dist

    def barrier(self):
        if self.pg:
            self.pg.barrier()

    def max_(self, values):
        import torch
        t = torch.tensor(values, dtype=torch.float64)
        if self.pg:
            self.pg.all_reduce(t, op=self.pg.ReduceOp.MAX)
        return t.tolist()

    def sum_(self, values):
        import torch
        t = torch.tensor(values, dtype=torch.float64)
        if self.pg:
            self.pg.all_reduce(t, op=self.pg.ReduceOp.SUM)
        return t.tolist()

    def bcast_bytes(self, b: bytes | None, n: int) -> bytes:
        import torch
        t = torch.zeros(n, dtype=torch.uint8)
        if self.rank == 0:
            t.copy_(torch.frombuffer(bytearray(b), dtype=torch.uint8))
        if self.pg:
            self.pg.broadcast(t, src=0)
        return bytes(t.numpy().tobytes())

    def close(self):
        if self.pg and self.pg.is_initialized():
            self.pg.destroy_process_group()


class OursBackend:
    name = "b200coll"

    def __init__(self, dist: Dist, capacity_elems: int, dtype, tag: str = "bench"):
        import torch
        from ..ops import coll
        self.coll, self.torch = coll, torch
        itemsize = 2
        arena_mb = (2 * capacity_elems * itemsize >> 20) + 128
        if dist.world > 1:
            self.comm = coll.Comm.from_env(arena_mb=arena_mb, tag=tag)
        else:
            self.comm = coll.Comm.init_all([dist.local_rank], arena_mb=arena_mb)[0]
        self.send = self.comm.empty(capacity_elems, dtype)
        self.recv = self.comm.empty(capacity_elems, dtype)
        self.L = coll.load()
        self.ep = coll.Epilogue(coll.torch_dtype_code(dtype), coll.torch_dtype_code(dtype), 1.0)
        self.h = self.comm._h
        self.nvls = self.comm.nvls
        self.version = f"libb200coll {self.L.b200collGetVersion()} nvls={int(self.nvls)}"

    def algo(self, op: str, nbytes_per_rank: int) -> str:
        if op in P2P_OPS:
            return "p2p"
        opid = OPS.index(op)
        return self.coll.tuner_pick(opid, nbytes_per_rank, self.comm.nranks, self.nvls)

    def launch(self, op: str, send_ptr: int, recv_ptr: int, count: int, stream: int) -> None:
        L, ep = self.L, C.byref(self.ep)
        if op in P2P_OPS:
            n, r, nbytes = self.comm.nranks, self.comm.rank, count * self.send.element_size()
            rc = L.b200collGroupStart()
            if op == "sendrecv":
                rc = rc or L.b200collSend(send_ptr, nbytes, (r + 1) % n, self.h, stream)
                rc = rc or L.b200collRecv(recv_ptr, nbytes, (r - 1) % n, self.h, stream)
            elif op == "gather":
                rc = rc or L.b200collSend(send_ptr, nbytes, ROOT, self.h, stream)
                for p in (range(n) if r == ROOT else ()):
                    rc = rc or L.b200collRecv(recv_ptr + p * nbytes, nbytes, p, self.h, stream)
            else:
                for p in (range(n) if r == ROOT else ()):
                    rc = rc or L.b200collSend(send_ptr + p * nbytes, nbytes, p, self.h, stream)
                rc = rc or L.b200collRecv(recv_ptr, nbytes, ROOT, self.h, stream)
            rc = L.b200collGroupEnd() or rc
        elif op == "all_reduce":
            rc = L.b200collAllReduce(send_ptr, recv_ptr, count, ep, 0, self.h, stream)
        elif op == "all_gather":
            rc = L.b200collAllGather(send_ptr, recv_ptr, count, ep, self.h, stream)
        elif op == "reduce_scatter":
            rc = L.b200collReduceScatter(send_ptr, recv_ptr, count, ep, 0, self.h, stream)
        elif op == "broadcast":
            rc = L.b200collBroadcast(send_ptr, recv_ptr, count, ep, ROOT, self.h, stream)
        elif op == "reduce":
            rc = L.b200collReduce(send_ptr, recv_ptr, count, ep, 0, ROOT, self.h, stream)
        else:
            rc = L.b200collAllToAll(send_ptr, recv_ptr, count, ep, self.h, stream)
        if rc != 0:
            raise RuntimeError(f"b200coll {op}: {L.b200collGetErrorString(rc).decode()}: {L.b200collGetLastError().decode()}")

    def launches(self) -> int:
        return int(self.comm.stats()["kernel_launches"])

    def device_rendezvous(self, stream) -> None:
        """Every rank's stream meets every other rank's on the device (k_barrier): the timed region that follows starts at the same moment
        everywhere, so the microseconds by which ranks leave the host barrier apart are not charged to the first timed call."""
        if self.comm.nranks > 1:
            self.comm.barrier(stream)

    def host_buffers(self, in_elems: int, out_elems: int, dtype):
        # pinned host memory on the NUMA node of this rank's GPU (b200collHostAlloc): part of the library's public API
        return self.comm.host_empty(in_elems, dtype), self.comm.host_empty(out_elems, dtype)

    def e2e_step(self, op: str, h_in, h_out, count: int, dev_off: int, stream) -> None:
        """One end-to-end step through the public API. all_reduce: ONE call, b200collAllReduceHost (zero-copy kernel for tiny messages,
        copy-in | all-reduce | copy-back pipelined over chunks for large ones). Other ops: copy in, collective, copy the whole result back."""
        if op == "all_reduce":
            self.comm.all_reduce_host(h_in, h_out, stream=stream)
            return
        _copy_launch_copy(self, op, h_in, h_out, count, dev_off, stream)

    def check(self) -> None:
        self.comm.check_async_error()

    def close(self):
        self.comm.destroy()


def _copy_launch_copy(backend, op: str, h_in, h_out, count: int, dev_off: int, stream) -> None:
    """What a user of a device-pointer collective API writes: pinned host -> device, the collective, the whole result -> pinned host."""
    s, r = backend.send[dev_off:dev_off + h_in.numel()], backend.recv[dev_off:dev_off + h_out.numel()]
    s.copy_(h_in, non_blocking=True)
    backend.launch(op, s.data_ptr(), r.data_ptr(), count, stream.cuda_stream)
    h_out.copy_(r, non_blocking=True)


class NcclBackend:
    name = "nccl"
    # NCCL's ring / tree kernels round the running sum to bf16 at every hop (measured: its 8-GPU all-reduce, reduce-scatter and reduce
    # miss the 1-ulp-of-the-result bound that an fp32-accumulated reduction meets, by far where the sum cancels), so the reference arm
    # is held to one ulp of the partial sums' magnitude (sum of |inputs|) per rank instead.
    verify_per_hop = True

    def __init__(self, dist: Dist, capacity_elems: int, dtype):
        import torch
        from . import nccl_ref
        self.torch = torch
        # Default: stock NCCL settings (its own tuning for one NVSwitch node). B200_REF_PROFILE=1 applies the reference's multi-node
        # env profile (gpudirect-tcpxo/README.md:71-103; it turns the LL protocol off) — both are measured in profiles/allreduce_sweep.md.
        if os.environ.get("B200_REF_PROFILE", "0") == "1":
            for k, v in nccl_ref.REFERENCE_ENV.items():
                os.environ.setdefault(k, v)
        # NCCL's INFO log is evidence (rank count, algorithm, NVLS): keep it, but on stderr — stdout carries exactly one JSON line.
        if "B200_REF_NCCL_DEBUG" in os.environ:
            os.environ["NCCL_DEBUG"] = os.environ["B200_REF_NCCL_DEBUG"]
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):      # images often preset WARN: the rank count and the algorithm lines need INFO
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT,ENV")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            uid = nccl_ref.NcclComm.new_unique_id() if dist.rank == 0 else None
            uid = dist.bcast_bytes(uid, 128)
            self.comm = nccl_ref.NcclComm(dist.rank, dist.world, uid)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
        self.profile = "reference env profile" if os.environ.get("B200_REF_PROFILE", "0") == "1" else "NCCL defaults"
        self.windows = []
        if os.environ.get("B200_REF_SYM", "0") == "1":
            # NCCL's own fast path for registered memory: ncclMemAlloc + ncclCommWindowRegister(NCCL_WIN_COLL_SYMMETRIC) (2.27+)
            itemsize = torch.empty((), dtype=dtype).element_size()
            self.send = self.comm.sym_tensor(capacity_elems, dtype, itemsize, self.windows)
            self.recv = self.comm.sym_tensor(capacity_elems, dtype, itemsize, self.windows)
            self.profile += ", ncclMemAlloc + symmetric windows"
        else:
            self.send = torch.empty(capacity_elems, dtype=dtype, device="cuda")
            self.recv = torch.empty(capacity_elems, dtype=dtype, device="cuda")
        self.dt = {torch.bfloat16: nccl_ref.NCCL_BFLOAT16, torch.float16: nccl_ref.NCCL_FLOAT16, torch.float32: nccl_ref.NCCL_FLOAT32}[dtype]
        self.itemsize = self.send.element_size()
        self.nvls = None
        self.version = f"NCCL {self.comm.version} ({os.path.basename(self.comm.path)}; {self.profile})"
        self._launches = 0

    def algo(self, op, nbytes):
        return "nccl"

    def launch(self, op: str, send_ptr: int, recv_ptr: int, count: int, stream: int) -> None:
        c = self.comm
        if op == "sendrecv":
            c.send_recv(send_ptr, (c.rank + 1) % c.nranks, recv_ptr, (c.rank - 1) % c.nranks, count, self.dt, stream)
        elif op in ("gather", "scatter"):
            c.gather_scatter(op, send_ptr, recv_ptr, count, self.dt, self.itemsize, ROOT, stream)
        elif op == "all_reduce":
            c.all_reduce(send_ptr, recv_ptr, count, self.dt, stream)
        elif op == "all_gather":
            c.all_gather(send_ptr, recv_ptr, count, self.dt, stream)
        elif op == "reduce_scatter":
            c.reduce_scatter(send_ptr, recv_ptr, count, self.dt, stream)
        elif op == "broadcast":
            c.broadcast(send_ptr, recv_ptr, count, self.dt, ROOT, stream)
        elif op == "reduce":
            c.reduce(send_ptr, recv_ptr, count, self.dt, ROOT, stream)
        else:
            c.all_to_all(send_ptr, recv_ptr, count, self.dt, self.itemsize, stream)
        self._launches += 1

    def launches(self) -> int:
        return 0   # NCCL's kernels are not ours

    def device_rendezvous(self, stream) -> None:
        if self.comm.nranks > 1:      # the same alignment for the NCCL arm: a one-vector all-reduce on a private scratch buffer
            if not hasattr(self, "_sync_buf"):
                self._sync_buf = self.torch.zeros(8, dtype=self.torch.float32, device="cuda")
            self.comm.all_reduce(self._sync_buf.data_ptr(), self._sync_buf.data_ptr(), 8, 7, stream.cuda_stream)      # 7 = ncclFloat32

    def host_buffers(self, in_elems: int, out_elems: int, dtype):
        return self.torch.empty(in_elems, dtype=dtype).pin_memory(), self.torch.empty(out_elems, dtype=dtype).pin_memory()

    def e2e_step(self, op: str, h_in, h_out, count: int, dev_off: int, stream) -> None:
        _copy_launch_copy(self, op, h_in, h_out, count, dev_off, stream)

    def check(self):
        pass

    def close(self):
        for win, p in self.windows:
            self.comm.lib.ncclCommWindowDeregister(self.comm.comm, win)
            self.comm.lib.ncclMemFree(p)
        self.comm.destroy()


def _gen_expected(torch, op, rank, n, count, device):
    """Pseudo-random bf16-representable values in (-4, 4) from an integer hash of (rank, index): every rank can compute every other
    rank's input, and — unlike small multiples of 0.25 — sums of them are NOT exactly representable in bf16, so the accumulate precision
    and the final rounding of a reduction are actually tested."""
    def gen(r, idx):
        h = (idx * 2654435761 + (r + 1) * 40503 + ((idx >> 7) * 977)) & 0xFFFF
        v = (h.to(torch.float32) - 32768.0) / 8192.0
        return v.to(torch.bfloat16).to(torch.float32)
    return gen


def bf16_ulp(torch, x):
    """Spacing of bf16 numbers around |x| (8 significand bits), as fp32."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - 7)


def reduction_ok(torch, got32, want32, out_dtype, nranks: int, max_abs_in: float = 4.0, ulps: float = 1.0, per_hop_mag=None):
    """got32 (the kernel's output widened to fp32) must lie within ONE ulp of the output type around the fp32-accumulated reference:
    a correctly rounded fp32 accumulation lands within half an ulp whatever the summation order; accumulating in bf16 / fp16 (e.g. a
    multimem.ld_reduce without .acc::f32) is off by several ulps on a large share of the elements and fails. The absolute slack covers
    fp32 reassociation when a sum cancels to almost nothing."""
    err = (got32 - want32).abs()
    ulp = bf16_ulp(torch, want32) if out_dtype == torch.bfloat16 else (want32.abs() * 2.0 ** -10 if out_dtype == torch.float16 else want32.abs() * 2.0 ** -22)
    tol = ulps * ulp + nranks * max_abs_in * 2.0 ** -22
    if per_hop_mag is not None:      # an implementation that rounds the running sum to the element type at every hop: one ulp of the partial sums' magnitude per rank
        tol = tol + nranks * bf16_ulp(torch, per_hop_mag)
    return bool((err <= tol).all().item())


VERIFY_COUNTS = {"all_reduce": (1 << 16, (1 << 21) + 8, (1 << 20) + 13)}   # Lamport path; NVLS / two-shot body; a count that leaves a scalar tail


def verify(backend, dist: Dist, op: str, dtype, count: int | None = None) -> bool:
    """Correctness against a plain PyTorch fp32 reference of the same op, on the sizes listed in VERIFY_COUNTS (all_reduce: one per
    algorithm family that the timed sweep uses) with data whose sums are not exact in bf16."""
    import torch
    counts = (count,) if count else VERIFY_COUNTS.get(op, (1 << 16,))
    ok = all(_verify_one(backend, dist, op, dtype, c) for c in counts)
    return dist.sum_([1.0 if ok else 0.0])[0] == dist.world


def _verify_one(backend, dist: Dist, op: str, dtype, count: int) -> bool:
    import torch
    n, rank = dist.world, dist.rank
    dev = backend.send.device
    gen = _gen_expected(torch, op, rank, n, count, dev)
    E = 8
    if op != "all_reduce":
        count = max(E, count // E * E)
    if op in FULL_MESSAGE_OPS:
        in_elems, out_elems = count, count
    elif op in ("all_gather", "gather"):
        in_elems, out_elems = count, count * n
    elif op in ("reduce_scatter", "scatter"):
        in_elems, out_elems = count * n, count
    else:
        in_elems, out_elems = count * n, count * n
    idx = torch.arange(in_elems, device=dev)
    backend.send[:in_elems] = gen(rank, idx).to(dtype)
    backend.recv[:out_elems] = 77.0
    torch.cuda.synchronize(); dist.barrier()
    st = torch.cuda.current_stream().cuda_stream
    backend.launch(op, backend.send.data_ptr(), backend.recv.data_ptr(), count, st)
    torch.cuda.synchronize(); dist.barrier()
    backend.check()
    got = backend.recv[:out_elems].float()
    reduced = False
    mag = None
    if op == "all_reduce":
        want = sum(gen(r, idx) for r in range(n)); reduced = True
        mag = sum(gen(r, idx).abs() for r in range(n))
    elif op == "broadcast":
        want = gen(ROOT, idx)
    elif op == "sendrecv":
        want = gen((rank - 1) % n, idx)
    elif op == "reduce":                                   # only the root's recv is defined
        want = sum(gen(r, idx) for r in range(n)) if rank == ROOT else torch.full_like(got, 77.0)
        reduced = rank == ROOT
        mag = sum(gen(r, idx).abs() for r in range(n))
    elif op == "all_gather" or (op == "gather" and rank == ROOT):
        j = torch.arange(count, device=dev)
        want = torch.cat([gen(r, j) for r in range(n)])
    elif op == "gather":                                   # only the root's recv is defined
        want = torch.full_like(got, 77.0)
    elif op == "scatter":
        want = gen(ROOT, torch.arange(count, device=dev) + rank * count)
    elif op == "reduce_scatter":
        j = torch.arange(count, device=dev) + rank * count
        want = sum(gen(r, j) for r in range(n)); reduced = True
        mag = sum(gen(r, j).abs() for r in range(n))
    else:
        j = torch.arange(count, device=dev) + rank * count
        want = torch.cat([gen(r, j) for r in range(n)])
    if reduced and n > 1:
        return reduction_ok(torch, got, want, dtype, n, per_hop_mag=mag if getattr(backend, "verify_per_hop", False) else None)
    return bool(torch.equal(got, want.to(dtype).float()))


def verify_e2e(backend, dist: Dist, dtype) -> bool:
    """The end-to-end all-reduce (host in, host out) at one size per regime: zero-copy kernel, single chunk, chunked pipeline."""
    import torch
    n, rank = dist.world, dist.rank
    ok = True
    counts = (1 << 14, (1 << 19) + 24, (5 << 20) + 13)
    h_in, h_out = backend.host_buffers(max(counts), max(counts), dtype)
    gen = _gen_expected(torch, "all_reduce", rank, n, 0, "cpu")
    stream = torch.cuda.current_stream()
    for count in counts:
        idx = torch.arange(count)
        h_in[:count] = gen(rank, idx).to(dtype)
        h_out[:count] = 77.0
        torch.cuda.synchronize(); dist.barrier()
        backend.e2e_step("all_reduce", h_in[:count], h_out[:count], count, 0, stream)
        torch.cuda.synchronize(); dist.barrier()
        backend.check()
        want = sum(gen(r, idx) for r in range(n))
        got = h_out[:count].float()
        mag = sum(gen(r, idx).abs() for r in range(n)) if getattr(backend, "verify_per_hop", False) else None
        ok = ok and (reduction_ok(torch, got, want, dtype, n, per_hop_mag=mag) if n > 1 else bool(torch.equal(got, want.to(dtype).float())))
    return dist.sum_([1.0 if ok else 0.0])[0] == dist.world


def fill_inputs(backend, dist: Dist, chunk: int = 1 << 26) -> None:
    """Seeded contents for the whole send buffer (same integer hash as verify()), so that what a sweep computes depends on its
    arguments only. The receive buffer is left as allocated: the out-of-place pass writes it before anything reads it, and the in-place
    pass reads what the out-of-place pass of the same size wrote. Writing it here would also slow the timed copies into it: on a B200,
    sizes of 256 KB - 8 MB (which fit in L2) took 6.3 instead of 4.6 us per launch once the receive buffer had been written before."""
    import torch
    gen = _gen_expected(torch, "all_reduce", dist.rank, dist.world, 0, None)
    buf = backend.send
    for lo in range(0, buf.numel(), chunk):
        hi = min(lo + chunk, buf.numel())
        buf[lo:hi] = gen(dist.rank, torch.arange(lo, hi, device=buf.device)).to(buf.dtype)
    torch.cuda.synchronize()


def sweep(backend, dist: Dist, op: str, dtype, steps: int, warmup: int, min_bytes: int, max_bytes: int, factor: int = 2,
          placements=(0, 1), e2e: bool = False, on_output=None) -> list[Row]:
    """on_output(name, tensor), when given, is called after each timed window (outside it) with what the window's last launch wrote:
    the output in the device receive buffer, or for e2e the whole pinned host result."""
    import torch
    n, rank = dist.world, dist.rank
    itemsize = backend.send.element_size()
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    rows: list[Row] = []
    raw = []   # per (row, placement) local ms
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    host_in = host_out = None
    if e2e:
        # sized for the largest row of the sweep; the rows below use prefixes
        n_max = max_bytes // itemsize
        if op in FULL_MESSAGE_OPS:
            cap_in = cap_out = n_max
        else:
            cap_in = n_max if op not in ("all_gather", "gather") else n_max // n + 64
            cap_out = n_max if op not in ("reduce_scatter", "scatter") else n_max // n + 64
        host_in, host_out = backend.host_buffers(cap_in, cap_out, dtype)
        host_in.fill_(0.25)
        host_out.zero_()
    nbytes = min_bytes
    while nbytes <= max_bytes:
        E = 16 // itemsize
        if op in FULL_MESSAGE_OPS:
            count = nbytes // itemsize
            in_elems = out_elems = count
        else:
            count = nbytes // itemsize // n // E * E
            in_elems = count if op in ("all_gather", "gather") else count * n
            out_elems = count if op in ("reduce_scatter", "scatter") else count * n
        if count == 0:
            nbytes *= factor
            continue
        total = (count if op in FULL_MESSAGE_OPS else count * n) * itemsize
        slot_elems = (max(in_elems, out_elems) * itemsize + 4095) // 4096 * 4096 // itemsize
        slots = max(1, min(64, WINDOW // (slot_elems * itemsize)))
        per_rank_bytes = count * itemsize
        row = Row(total, count, backend.algo(op, per_rank_bytes), in_bytes=in_elems * itemsize)
        sbase, rbase = backend.send.data_ptr(), backend.recv.data_ptr()
        for ip in placements:
            if ip == 1 and (op in ("alltoall",) + P2P_OPS or n == 1):
                continue

            def ptrs(slot: int):
                off = slot * slot_elems * itemsize
                if not ip:
                    return sbase + off, rbase + off
                if op == "all_gather":
                    return rbase + off + rank * count * itemsize, rbase + off
                if op == "reduce_scatter":
                    return rbase + off, rbase + off + rank * count * itemsize
                return rbase + off, rbase + off
            for i in range(warmup):
                s, r = ptrs(i % slots)
                backend.launch(op, s, r, count, st)
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
            backend.device_rendezvous(stream)
            e0.record(stream)
            for i in range(steps):
                s, r = ptrs(i % slots)
                backend.launch(op, s, r, count, st)
            e1.record(stream)
            torch.cuda.synchronize()
            raw.append((len(rows), "ip" if ip else "oop", e0.elapsed_time(e1) / steps))
            if on_output is not None:
                r = ptrs((steps - 1) % slots)[1]
                lo = (r - rbase) // itemsize
                on_output(f"{op}_{'ip' if ip else 'oop'}_{total:010d}B", backend.recv[lo:lo + out_elems])
        if e2e:
            # the user-visible step: this rank's input starts in pinned host memory and the whole result ends there
            h_in, h_out = host_in[:in_elems], host_out[:out_elems]
            row.out_bytes = out_elems * itemsize
            for i in range(min(warmup, 2)):
                backend.e2e_step(op, h_in, h_out, count, 0, stream)
            torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
            backend.device_rendezvous(stream)
            e0.record(stream)
            for i in range(steps):
                backend.e2e_step(op, h_in, h_out, count, (i % slots) * slot_elems, stream)
            e1.record(stream)
            torch.cuda.synchronize()
            raw.append((len(rows), "e2e", e0.elapsed_time(e1) / steps))
            if on_output is not None:
                on_output(f"{op}_e2e_{total:010d}B", h_out)
        rows.append(row)
        nbytes *= factor
    backend.check()
    worst = dist.max_([r[2] for r in raw]) if raw else []
    for (ri, kind, _), ms in zip(raw, worst):
        setattr(rows[ri], f"{kind}_us", ms * 1e3)
    return rows


def summarize(rows: list[Row], op: str, n: int) -> dict:
    vals, e2e_vals, peak = [], [], 0.0
    for r in rows:
        b = r.bw(op, n)
        for k, us in (("oop_busbw", r.oop_us), ("ip_busbw", r.ip_us)):
            if us > 0:
                vals.append(b[k]); peak = max(peak, b[k])
        if r.e2e_us > 0:
            e2e_vals.append(b["e2e_busbw"])
    sweep_ms = sum((r.oop_us if r.oop_us > 0 else 0) + (r.ip_us if r.ip_us > 0 else 0) for r in rows) / 1e3
    return {"avg_busbw": sum(vals) / len(vals) if vals else 0.0, "peak_busbw": peak, "sweep_ms": sweep_ms,
            "avg_e2e_busbw": sum(e2e_vals) / len(e2e_vals) if e2e_vals else None, "measurements": len(vals)}


def format_table(rows: list[Row], op: str, n: int, title: str) -> str:
    out = [f"# {title}", f"#{'size(B)':>13} {'count':>12} {'algo':>8} | {'oop us':>10} {'algbw':>8} {'busbw':>8} | {'ip us':>10} {'algbw':>8} {'busbw':>8}"]
    for r in rows:
        b = r.bw(op, n)
        out.append(f"{r.nbytes:>14} {r.count:>12} {r.algo:>8} | {r.oop_us:>10.2f} {b['oop_algbw']:>8.2f} {b['oop_busbw']:>8.2f} | {r.ip_us:>10.2f} {b['ip_algbw']:>8.2f} {b['ip_busbw']:>8.2f}")
    s = summarize(rows, op, n)
    out.append(f"# Avg bus bandwidth : {s['avg_busbw']:.3f} GB/s   peak {s['peak_busbw']:.2f} GB/s")
    return "\n".join(out)


def rows_json(rows: list[Row], op: str, n: int) -> list[dict]:
    return [{"bytes": r.nbytes, "algo": r.algo, "oop_us": round(r.oop_us, 3), "ip_us": round(r.ip_us, 3), "oop_busbw": round(r.bw(op, n)["oop_busbw"], 2),
             "ip_busbw": round(r.bw(op, n)["ip_busbw"], 2), **({"e2e_us": round(r.e2e_us, 3), "e2e_busbw": round(r.bw(op, n)["e2e_busbw"], 2)} if r.e2e_us > 0 else {})} for r in rows]
