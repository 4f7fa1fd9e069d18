"""`torch.distributed` backend "b200coll": `dist.init_process_group("b200coll")` puts DDP / FSDP / user collectives on libb200coll.

Why: the reference's transports are drop-in for frameworks because frameworks speak NCCL and the installers swap the NCCL under them
(gpudirect-rdma/nccl-rdma-installer.yaml:70-77, LD_LIBRARY_PATH=/usr/local/nvidia/lib64). PyTorch's NCCL process group uses far more
of the NCCL API than nccl-tests does, so for PyTorch the faithful drop-in is a process group, not the symbol shim.

How: a Python subclass of `torch.distributed.ProcessGroup` (c10d dispatches to it through its trampoline, the mechanism PyTorch's own
tests use for Python process groups). CUDA tensors that the library can take as they are — contiguous, 16-byte aligned, fp32 / fp16 /
bf16 / fp8 (e4m3fn, e5m2), sum or avg — go straight to the collective kernels **on the caller's current stream**, so ordering with the surrounding compute
is plain stream order and `Work.wait()` has nothing to wait for (NCCL's side stream + event dance is not needed). Tensors allocated
with `pg.empty()` live in the symmetric arena and take the zero-copy / NVLS paths; any other device tensor is staged by the library.
Point-to-point on CUDA tensors uses the library's grouped send / recv kernel (queued until the first wait, so an isend + irecv pair
is one launch); gather / scatter are one such group around the root. Everything else (CPU tensors, integer reductions, min/max/product,
odd shapes) is executed by an
internal Gloo group over host copies: slow but correct, which keeps DDP's bookkeeping collectives and object broadcasts working.

Status: the fallback and dispatch logic is exercised on CPU (tests/test_process_group.py); the CUDA fast paths reuse the calls the GPU
suite covers through `ops.coll.Comm`, but the process group itself has not run on a GPU box yet (tests/test_process_group.py has the
two-process GPU test, opt-in until it has).
"""
from __future__ import annotations

import os
import uuid
from datetime import timedelta
from typing import Optional

import torch
import torch.distributed as dist

from ..ops import coll

BACKEND_NAME = "b200coll"
_FAST_DTYPES = (torch.float32, torch.float16, torch.bfloat16)
# fp8 reductions: sum / avg on the fused kernels (fp32 accumulation, saturating result), min / max / product on the generic kernel. Not in
# _FAST_DTYPES: all-gather, all-to-all and broadcast of fp8 keep moving raw words (bit-exact, never the Lamport path).
_FP8_DTYPES = (torch.float8_e4m3fn, torch.float8_e5m2)


class _Work(dist._Work):
    """Completed-at-enqueue work handle: the collective is already ordered on the caller's stream."""

    def __init__(self, result, sync_on_wait: bool = False, comm=None):
        super().__init__()
        self._result = result
        self._sync = sync_on_wait
        self._comm = comm               # when set: wait() raises if the library's watchdog has fired (a peer never arrived)
        self._future: Optional[torch.futures.Future] = None

    def wait(self, timeout: Optional[timedelta] = None) -> bool:
        if self._sync and torch.cuda.is_available():
            torch.cuda.current_stream().synchronize()
        if self._comm is not None:
            self._comm.check_async_error()
        return True

    def is_completed(self) -> bool:
        return True

    def is_success(self) -> bool:
        return True

    def result(self):
        return self._result

    def get_future(self) -> torch.futures.Future:
        if self._future is None:
            self._future = torch.futures.Future()
            self._future.set_result(self._result)
        return self._future


class _P2pWork(_Work):
    """Handle of a queued send / recv: waiting launches everything queued so far as one grouped kernel (stream-ordered afterwards)."""

    def __init__(self, pg, result):
        super().__init__(result)
        self._pg = pg

    def wait(self, timeout: Optional[timedelta] = None) -> bool:
        self._pg._flush_p2p()
        return True


def _fast(t: torch.Tensor) -> bool:
    return t.is_cuda and t.is_contiguous() and t.dtype in _FAST_DTYPES and t.data_ptr() % 16 == 0 and t.numel() > 0


def _rs_direct(t: torch.Tensor) -> bool:
    """Reduce-scatter runs on the library directly for the fast dtypes and for fp8 (sum / avg)."""
    return _fast(t) or (t.is_cuda and t.is_contiguous() and t.dtype in _FP8_DTYPES and t.data_ptr() % 16 == 0 and t.numel() > 0)


_GENERIC_DTYPES = (torch.int8, torch.uint8, torch.int32, torch.int64, torch.float64)      # any operator but AVG, on the generic P2P kernel


def _sum_or_avg(op) -> Optional[int]:
    if op == dist.ReduceOp.SUM:
        return coll.SUM
    if op == dist.ReduceOp.AVG:
        return coll.AVG
    return None


def _red_op(op) -> Optional[int]:
    """Every reduction libb200coll implements (sum / avg fused fast paths; min / max / product on the generic kernel).
    Compared with ==, not looked up in a dict: the option structs carry a `ReduceOp` object, which equals the `ReduceOp.SUM`
    constants but does not hash like them."""
    for theirs, ours in ((dist.ReduceOp.SUM, coll.SUM), (dist.ReduceOp.AVG, coll.AVG), (dist.ReduceOp.MIN, coll.MIN), (dist.ReduceOp.MAX, coll.MAX),
                         (dist.ReduceOp.PRODUCT, coll.PROD)):
        if op == theirs:
            return ours
    return None


def _reducible(t: torch.Tensor, op: Optional[int]) -> bool:
    if op is None or not (t.is_cuda and t.is_contiguous() and t.data_ptr() % 16 == 0 and t.numel() > 0):
        return False
    if t.dtype in _FAST_DTYPES or t.dtype in _FP8_DTYPES:
        return True
    return t.dtype in _GENERIC_DTYPES and op != coll.AVG


def alltoallv_layout(split_matrix: list[list[int]], rank: int) -> tuple[list[int], list[int], list[int], int]:
    """Given M[src][dst] = rows src sends to dst, return for `rank`: (send_rows, send_row_off, recv_row_off_at_peer, max_recv_rows).
    Rows from lower-ranked sources land first on every destination (the order all_to_all_single promises)."""
    n = len(split_matrix)
    send_rows = list(split_matrix[rank])
    send_off = [sum(send_rows[:d]) for d in range(n)]
    recv_off_at_peer = [sum(split_matrix[s][d] for s in range(rank)) for d in range(n)]
    max_recv = max(sum(split_matrix[s][d] for s in range(n)) for d in range(n))
    return send_rows, send_off, recv_off_at_peer, max_recv


class B200CollProcessGroup(dist.ProcessGroup):
    def __init__(self, store, rank: int, size: int, timeout: timedelta = timedelta(minutes=10)):
        super().__init__(rank, size)
        self._store, self._rank, self._size, self._timeout = store, rank, size, timeout
        self._comm: Optional[coll.Comm] = None
        self._gloo = None
        self._scratch: dict = {}          # (nbytes class) -> symmetric uint8 tensor, for all-to-all-v receive staging
        self._last_stream = None          # stream and completion event of the previous device collective (see _ordered)
        self._last_event = None
        self._pending: list = []          # queued point-to-point operations: (kind, tensor, peer), launched as one group
        self.fast_calls = 0               # collectives that ran on libb200coll
        self.fallback_calls = 0           # collectives that ran on the Gloo group

    # ------------------------------------------------------------------ plumbing
    def _work(self, result, **kw) -> _Work:
        # every handle checks the communicator's fault record in wait(): a watchdog hit on an earlier collective surfaces as an exception
        return _Work(result, comm=self._comm, **kw)

    def getBackendName(self) -> str:
        return BACKEND_NAME

    @property
    def comm(self) -> coll.Comm:
        """The libb200coll communicator, created on first use on the caller's current CUDA device."""
        if self._comm is None:
            if self._rank == 0:
                self._store.set("b200coll/key", uuid.uuid4().hex)
            key = self._store.get("b200coll/key").decode()
            arena = os.environ.get("B200COLL_ARENA_MB")
            # the process group's timeout (c10d default: 10 min) is the library's watchdog and rendezvous timeout too
            timeout_ms = int(self._timeout.total_seconds() * 1000) if self._timeout is not None else None
            if "B200COLL_TIMEOUT_MS" in os.environ:
                timeout_ms = None             # an explicit environment setting wins (tests use a short one)
            self._comm = coll.Comm.init_rank(self._rank, self._size, f"pg/{key}", arena_mb=int(arena) if arena else None, timeout_ms=timeout_ms)
        return self._comm

    @property
    def gloo(self):
        if self._gloo is None:
            self._gloo = dist.ProcessGroupGloo(dist.PrefixStore("b200coll-gloo", self._store), self._rank, self._size, self._timeout)
        return self._gloo

    def empty(self, numel: int, dtype: torch.dtype) -> torch.Tensor:
        """A tensor in the symmetric arena (same call order and sizes on every rank): zero-copy collectives, NVLS capable."""
        return self.comm.empty(numel, dtype)

    def mem_pool(self):
        """`with torch.cuda.use_mem_pool(pg.mem_pool()): ...` allocates in the symmetric arena (see `Comm.mem_pool`): wrap model and
        DDP construction in it and the gradient all-reduces become zero-copy."""
        return self.comm.mem_pool()

    def shutdown(self) -> None:
        if self._comm is not None:
            self._flush_p2p()
            torch.cuda.synchronize()
            self._scratch.clear()
            self._comm.destroy()
            self._comm = None

    abort = shutdown

    class _ordered:
        """A communicator runs one collective at a time (its barrier epochs and Lamport buffers are per communicator, as NCCL's channels
        are). Calls that stay on one stream are ordered by the stream. When the caller moves to another stream (FSDP all-gathers on its
        unshard stream while reduce-scatters run on the post-backward stream) the new stream first waits for the previous collective."""

        def __init__(self, pg):
            self.pg = pg

        def __enter__(self):
            pg, cur = self.pg, torch.cuda.current_stream()
            if pg._last_stream is not None and pg._last_stream != cur and pg._last_event is not None:
                cur.wait_event(pg._last_event)
            pg._launch_pending()          # queued sends / recvs keep their place in the order of calls
            return cur

        def __exit__(self, *exc):
            pg, cur = self.pg, torch.cuda.current_stream()
            if pg._last_event is None or pg._last_stream != cur:
                pg._last_event = torch.cuda.Event()
            pg._last_event.record(cur)
            pg._last_stream = cur
            return False

    def _via_gloo(self, tensors, run):
        """Run `run(cpu_tensors)` on the Gloo group and copy results back into the (possibly CUDA) originals."""
        self.fallback_calls += 1
        flat = list(tensors)
        host = [t.detach().cpu() if t.is_cuda else t for t in flat]
        work = run(host)
        if work is not None:
            work.wait()
        for t, h in zip(flat, host):
            if t.is_cuda:
                t.copy_(h)
        return host

    # ------------------------------------------------------------------ collectives
    def allreduce(self, tensors, opts=None):
        op = _red_op(opts.reduceOp) if opts is not None else coll.SUM
        if op is not None and all(_reducible(t, op) for t in tensors):
            with self._ordered(self):
                for t in tensors:
                    self.comm.all_reduce(t, op=op)
            self.fast_calls += 1
            return self._work(tensors)
        gopts = dist.AllreduceOptions()
        if opts is not None:
            gopts.reduceOp = opts.reduceOp
        avg = opts is not None and opts.reduceOp == dist.ReduceOp.AVG       # Gloo has no AVG
        if avg:
            gopts.reduceOp = dist.ReduceOp.SUM
        self._via_gloo(tensors, lambda h: self.gloo.allreduce(h, gopts))
        if avg:
            for t in tensors:
                t.div_(self._size)
        return self._work(tensors)

    def allreduce_coalesced(self, tensors, opts=None):
        return self.allreduce(tensors, opts)

    def broadcast(self, tensors, opts=None):
        root = opts.rootRank if opts is not None else 0
        done = []
        for t in tensors:
            words = self._as_words(t)
            if words is None:
                break
            with self._ordered(self):
                self.comm.broadcast(words, root=root)
            done.append(t)
        if len(done) == len(tensors):
            self.fast_calls += 1
            return self._work(tensors)
        gopts = dist.BroadcastOptions()
        gopts.rootRank = root
        def run(host):
            for x in host:
                self.gloo.broadcast([x], gopts).wait()
        self._via_gloo(tensors[len(done):], run)
        return self._work(tensors)

    @staticmethod
    def _as_words(t: torch.Tensor) -> Optional[torch.Tensor]:
        """View any contiguous CUDA tensor as fp16/fp32 words for bit-exact movement (broadcast does not care about the dtype)."""
        if not (t.is_cuda and t.is_contiguous() and t.numel() > 0 and t.data_ptr() % 16 == 0):
            return None
        if t.dtype in _FAST_DTYPES:
            return t.view(-1)
        nbytes = t.numel() * t.element_size()
        raw = t.view(-1).view(torch.uint8)
        if nbytes % 4 == 0:
            return raw.view(torch.float32)
        if nbytes % 2 == 0:
            return raw.view(torch.float16)
        return None

    @classmethod
    def _word_views(cls, *tensors):
        """All-gather and all-to-all only move bits, so any dtype can ride the fp kernels: the same word type for every tensor, or None."""
        views = [cls._as_words(t) for t in tensors]
        if any(v is None for v in views):
            return None
        if len({v.dtype for v in views}) > 1:                  # e.g. one tensor's byte count is only a multiple of 2: use the narrower word
            views = [t.view(-1).view(torch.uint8).view(torch.float16) if (t.numel() * t.element_size()) % 2 == 0 else None for t in tensors]
            if any(v is None for v in views):
                return None
        return views

    def reduce(self, tensors, opts=None):
        root = opts.rootRank if opts is not None else 0
        op = _red_op(opts.reduceOp) if opts is not None else coll.SUM
        if op is not None and all(_reducible(t, op) for t in tensors):
            with self._ordered(self):
                for t in tensors:
                    self.comm.reduce(t, root=root, op=op)
            self.fast_calls += 1
            return self._work(tensors)
        gopts = dist.ReduceOptions()
        gopts.rootRank = root
        if opts is not None:
            gopts.reduceOp = opts.reduceOp
        self._via_gloo(tensors, lambda h: self.gloo.reduce(h, gopts))
        return self._work(tensors)

    def _allgather_base(self, output, input, opts=None):
        if _fast(output) and _fast(input) and output.dtype == input.dtype and (input.numel() * input.element_size()) % 16 == 0 \
                and output.numel() == input.numel() * self._size:
            with self._ordered(self):
                self.comm.all_gather(input.view(-1), output.view(-1))
            self.fast_calls += 1
            return self._work(output)
        words = self._word_views(output, input) if output.dtype == input.dtype and output.numel() == input.numel() * self._size \
            and (input.numel() * input.element_size()) % 16 == 0 else None
        if words is not None:                                   # integer / bool / fp8 payloads (token ids, masks): moved as raw words
            with self._ordered(self), self.comm.bit_exact():
                self.comm.all_gather(words[1], words[0])
            self.fast_calls += 1
            return self._work(output)
        chunks = list(output.view(-1).chunk(self._size))
        self.allgather([chunks], [input.view(-1)])
        return self._work(output)

    def allgather(self, output_tensors, input_tensors, opts=None):
        for outs, inp in zip(output_tensors, input_tensors):
            same = all(o.shape == inp.shape and o.dtype == inp.dtype for o in outs)
            if same and _fast(inp) and all(o.is_cuda for o in outs) and (inp.numel() * inp.element_size()) % 16 == 0:
                flat = torch.empty(inp.numel() * self._size, dtype=inp.dtype, device=inp.device)
                with self._ordered(self):
                    self.comm.all_gather(inp.view(-1), flat)
                for o, piece in zip(outs, flat.chunk(self._size)):
                    o.copy_(piece.view_as(o))
                self.fast_calls += 1
            else:
                self.fallback_calls += 1
                host_in = inp.detach().cpu() if inp.is_cuda else inp
                host_out = [torch.empty_like(o, device="cpu") for o in outs]
                self.gloo.allgather([host_out], [host_in]).wait()
                for o, h in zip(outs, host_out):
                    o.copy_(h)
        return self._work(output_tensors)

    def allgather_into_tensor_coalesced(self, outputs, inputs, opts=None):
        for o, i in zip(outputs, inputs):
            self._allgather_base(o, i, opts)
        return self._work(outputs)

    def _reduce_scatter_base(self, output, input, opts=None):
        op = _sum_or_avg(opts.reduceOp) if opts is not None else coll.SUM
        if op is not None and _rs_direct(output) and _rs_direct(input) and output.dtype == input.dtype and (output.numel() * output.element_size()) % 16 == 0 \
                and input.numel() == output.numel() * self._size:
            with self._ordered(self):
                self.comm.reduce_scatter(input.view(-1), output.view(-1), op=op)
            self.fast_calls += 1
            return self._work(output)
        # generic: all-reduce a copy, keep my slice
        tmp = input.detach().clone().view(-1)
        self.allreduce([tmp], opts)
        output.view(-1).copy_(tmp.chunk(self._size)[self._rank])
        return self._work(output)

    def reduce_scatter(self, output_tensors, input_tensors, opts=None):
        for out, ins in zip(output_tensors, input_tensors):
            flat = torch.cat([i.reshape(-1) for i in ins])
            self._reduce_scatter_base(out, flat, opts)
        return self._work(output_tensors)

    def reduce_scatter_tensor_coalesced(self, outputs, inputs, opts=None):
        for o, i in zip(outputs, inputs):
            self._reduce_scatter_base(o, i, opts)
        return self._work(outputs)

    def alltoall_base(self, output, input, output_split_sizes, input_split_sizes, opts=None):
        n = self._size
        even = not output_split_sizes and not input_split_sizes
        if even and _fast(output) and _fast(input) and output.dtype == input.dtype and output.data_ptr() != input.data_ptr() \
                and input.numel() % n == 0 and (input.numel() // n * input.element_size()) % 16 == 0 and output.numel() == input.numel():
            with self._ordered(self):
                self.comm.all_to_all(input.view(-1), output.view(-1))
            self.fast_calls += 1
            return self._work(output)
        words = self._word_views(output, input) if even and output.dtype == input.dtype and output.data_ptr() != input.data_ptr() and input.numel() % n == 0 \
            and (input.numel() // n * input.element_size()) % 16 == 0 and output.numel() == input.numel() else None
        if words is not None:
            with self._ordered(self), self.comm.bit_exact():
                self.comm.all_to_all(words[1], words[0])
            self.fast_calls += 1
            return self._work(output)
        row_elems = input[0].numel() if input.dim() > 0 and input.shape[0] > 0 else 0
        if not even and row_elems and _fast(input) and output.is_cuda and output.is_contiguous() and output.dtype == input.dtype \
                and (row_elems * input.element_size()) % 16 == 0:
            return self._alltoallv_rows(output, input, list(input_split_sizes), row_elems)
        # Gloo: works on host copies for any layout
        self.fallback_calls += 1
        host_in = input.detach().cpu() if input.is_cuda else input
        host_out = torch.empty_like(output, device="cpu")
        self.gloo.alltoall_base(host_out, host_in, list(output_split_sizes or []), list(input_split_sizes or [])).wait()
        output.copy_(host_out)
        return self._work(output)

    def _alltoallv_rows(self, output, input, in_splits, row_elems):
        """Expert-dispatch shaped all_to_all_single: rows of dim 0 with per-peer counts. The split matrix travels over Gloo (a few
        integers); the payload goes through b200collAllToAllv into a symmetric scratch buffer (peers write into it), then into `output`."""
        n = self._size
        mine = torch.tensor(in_splits, dtype=torch.int64)
        allm = [torch.zeros(n, dtype=torch.int64) for _ in range(n)]
        self.gloo.allgather([allm], [mine]).wait()
        matrix = [m.tolist() for m in allm]
        send_rows, send_off, recv_off_at_peer, max_recv = alltoallv_layout(matrix, self._rank)
        row_bytes = row_elems * input.element_size()
        need = max(1, max_recv) * row_bytes
        cls = 1 << (need - 1).bit_length()                   # same on every rank: max_recv is a global quantity
        scratch = self._scratch.get(cls)
        if scratch is None:
            scratch = self._scratch[cls] = self.comm.empty(cls, torch.uint8)
        recv = scratch[:need].view(input.dtype)
        with self._ordered(self):
            self.comm.all_to_all_v(input.view(-1), recv, row_elems, send_rows, send_off, recv_off_at_peer)
        got_rows = sum(matrix[s][self._rank] for s in range(n))
        output.view(-1)[:got_rows * row_elems].copy_(recv[:got_rows * row_elems])
        self.fast_calls += 1
        return self._work(output)

    def alltoall(self, output_tensors, input_tensors, opts=None):
        same = len({(t.numel(), t.dtype) for t in list(output_tensors) + list(input_tensors)}) == 1
        if same and all(t.is_cuda for t in list(output_tensors) + list(input_tensors)):
            src = torch.cat([t.reshape(-1) for t in input_tensors])
            dst = torch.empty_like(src)
            self.alltoall_base(dst, src, [], [])
            for o, piece in zip(output_tensors, dst.chunk(self._size)):
                o.copy_(piece.view_as(o))
            return self._work(output_tensors)
        self.fallback_calls += 1
        host_in = [t.detach().cpu() if t.is_cuda else t for t in input_tensors]
        host_out = [torch.empty_like(t, device="cpu") for t in output_tensors]
        self.gloo.alltoall(host_out, host_in).wait()
        for o, h in zip(output_tensors, host_out):
            o.copy_(h)
        return self._work(output_tensors)

    def barrier(self, opts=None):
        if torch.cuda.is_available() and self._comm is not None:
            with self._ordered(self):
                self.comm.barrier()
            self.fast_calls += 1
            return self._work(None, sync_on_wait=True)
        self.fallback_calls += 1
        self.gloo.barrier().wait()
        return self._work(None)

    # ------------------------------------------------------------------ things only Gloo does
    def gather(self, output_tensors, input_tensors, opts=None):
        root = opts.rootRank if opts is not None else 0
        if all(t.is_cuda for t in input_tensors) and all(o.is_cuda for outs in output_tensors for o in outs):
            # one group around the root: everybody sends, the root receives from everybody (its own block is a local copy in the library)
            for i, inp in enumerate(input_tensors):
                self._pending.append(("send", inp, root))
                if self._rank == root:
                    self._pending.extend(("recv", o, p) for p, o in enumerate(output_tensors[i]))
            self.fast_calls += 1
            return _P2pWork(self, output_tensors)
        self.fallback_calls += 1
        gopts = dist.GatherOptions(); gopts.rootRank = root
        host_in = [t.detach().cpu() if t.is_cuda else t for t in input_tensors]
        host_out = [[torch.empty_like(o, device="cpu") for o in outs] for outs in output_tensors]
        self.gloo.gather(host_out, host_in, gopts).wait()
        for outs, hs in zip(output_tensors, host_out):
            for o, h in zip(outs, hs):
                o.copy_(h)
        return self._work(output_tensors)

    def scatter(self, output_tensors, input_tensors, opts=None):
        root = opts.rootRank if opts is not None else 0
        if all(o.is_cuda for o in output_tensors) and all(t.is_cuda for ins in input_tensors for t in ins):
            for i, out in enumerate(output_tensors):
                if self._rank == root:
                    self._pending.extend(("send", t, p) for p, t in enumerate(input_tensors[i]))
                self._pending.append(("recv", out, root))
            self.fast_calls += 1
            return _P2pWork(self, output_tensors)
        self.fallback_calls += 1
        gopts = dist.ScatterOptions(); gopts.rootRank = root
        host_out = [torch.empty_like(o, device="cpu") for o in output_tensors]
        host_in = [[t.detach().cpu() if t.is_cuda else t for t in ins] for ins in input_tensors]
        self.gloo.scatter(host_out, host_in, gopts).wait()
        for o, h in zip(output_tensors, host_out):
            o.copy_(h)
        return self._work(output_tensors)

    # ------------------------------------------------------------------ point to point
    # CUDA tensors go through the library's send / recv kernel (tags are ignored, as ProcessGroupNCCL does: messages of a pair match in
    # call order). The decision "library or Gloo" uses only what both sides of a message share (device type), never layout: a tensor
    # that is not contiguous or not 16-byte aligned travels through a temporary. Operations are queued and launched together — as ONE
    # grouped kernel — by the first `wait()` (blocking `dist.send` / `dist.recv` wait at once) or by the next collective, so
    # `isend(right); irecv(left); wait both` cannot deadlock the way two separately launched, stream-blocking kernels would, also
    # through `batch_isend_irecv` (which, for a Python process group, just calls isend / irecv in a loop).
    def send(self, tensors, dst_rank, tag=0):
        if all(t.is_cuda for t in tensors):
            self._pending.extend(("send", t, dst_rank) for t in tensors)
            self.fast_calls += 1
            return _P2pWork(self, tensors)
        self.fallback_calls += 1
        self.gloo.send([t.detach().cpu() if t.is_cuda else t for t in tensors], dst_rank, tag).wait()
        return self._work(tensors)

    def recv(self, tensors, src_rank, tag=0):
        if all(t.is_cuda for t in tensors):
            self._pending.extend(("recv", t, src_rank) for t in tensors)
            self.fast_calls += 1
            return _P2pWork(self, tensors)
        self._via_gloo(tensors, lambda h: self.gloo.recv(h, src_rank, tag))
        return self._work(tensors)

    def _flush_p2p(self) -> None:
        if self._pending:
            with self._ordered(self):       # entering the ordered section launches what is queued
                pass

    def _launch_pending(self) -> None:
        ops, self._pending = self._pending, []
        if not ops:
            return
        comm, copy_out, keep = self.comm, [], []
        direct = lambda t: t.is_contiguous() and t.data_ptr() % 16 == 0
        with coll.group():
            for kind, t, peer in ops:
                if t.numel() == 0:
                    continue
                if kind == "send":
                    if not direct(t):
                        t = t.contiguous().clone()      # clone(): a fresh allocation is aligned
                        keep.append(t)                  # Comm.send only records the pointer; the kernel is launched when the group closes,
                    comm.send(t, peer)                  # so the temporary must stay allocated (and un-reused) until then
                elif direct(t):
                    comm.recv(t, peer)
                else:
                    tmp = torch.empty(t.shape, dtype=t.dtype, device=t.device)
                    comm.recv(tmp, peer)
                    copy_out.append((t, tmp))
        for t, tmp in copy_out:
            t.copy_(tmp)
        del keep                                        # the grouped kernel is enqueued: the caching allocator's stream ordering takes over


def _create(store, rank, size, timeout):
    return B200CollProcessGroup(store, rank, size, timeout)


def register() -> None:
    """Idempotent: make `backend="b200coll"` known to torch.distributed (also runs when this module is imported)."""
    if BACKEND_NAME.upper() not in getattr(dist.Backend, "_plugins", {}):
        dist.Backend.register_backend(BACKEND_NAME, _create, devices=["cpu", "cuda"])


register()
