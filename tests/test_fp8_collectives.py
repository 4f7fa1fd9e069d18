"""FP8 (e4m3 / e5m2) as an input type of libb200coll: the fused fp32-accumulating reductions, the generic min / max / prod kernel,
data movement, the host path, the NCCL shim and the torch.distributed backend.

Numerics contract: every finite e4m3 is a multiple of 2^-9 with |x| <= 448, so a sum over <= 8 ranks is exact in fp32 in any order;
e5m2 (multiples of 2^-16) is exact while partial sums stay below 256, which the quarter-valued fills here do, and so do sums of large
values alone. The result is therefore bit-identical to clamp(sum(x_r.float()) * scale, -max, max).to(fp8) — the clamp is the
kernels' saturating cast (torch's own cast would give NaN / inf on overflow) — on every algorithm without multicast."""
import ctypes as C
import functools
import os
import subprocess

import pytest
import torch
import torch.distributed as dist

from container_engine_accelerators_b200.ops import coll
from container_engine_accelerators_b200.parallel import process_group as pgmod

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP8 = {"e4m3": torch.float8_e4m3fn, "e5m2": torch.float8_e5m2}
FP8_MAX = {torch.float8_e4m3fn: 448.0, torch.float8_e5m2: 57344.0}
NCCL_FP8 = {"e4m3": 10, "e5m2": 11}


def _ref(total: torch.Tensor, dtype) -> torch.Tensor:
    """The fp32 result after the kernels' round-to-nearest, saturating cast to `dtype`."""
    if dtype in FP8_MAX:
        total = total.clamp(-FP8_MAX[dtype], FP8_MAX[dtype])
    return total.to(dtype)


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.view(torch.uint8) if t.element_size() == 1 else t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _same(a: torch.Tensor, b: torch.Tensor) -> bool:
    return a.dtype == b.dtype and torch.equal(_bits(a.contiguous()), _bits(b.contiguous()))


# ------------------------------------------------------------------------------------------------- no GPU
def test_header_declares_e5m2_and_type_sizes(tmp_path, coll_lib):
    src = tmp_path / "probe.c"
    src.write_text(r'''
#include <stdio.h>
#include "b200coll.h"
int main(void) { printf("%d %d %d\n", b200collFloat8e4m3, b200collFloat8e5m2, b200collNumTypes); return 0; }''')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "coll", "include"), str(src), "-o", str(exe)], check=True)
    e4m3, e5m2, ntypes = map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert (e4m3, e5m2, ntypes) == (coll.FP8_E4M3, coll.FP8_E5M2, 12) and e5m2 == 11
    lib = coll.load()
    assert lib.b200collTypeSize(coll.FP8_E4M3) == 1 and lib.b200collTypeSize(coll.FP8_E5M2) == 1 and lib.b200collTypeSize(12) == 0
    assert coll.DTYPE_SIZE[coll.FP8_E5M2] == 1
    assert coll.torch_dtype_code(torch.float8_e4m3fn) == coll.FP8_E4M3 and coll.torch_dtype_code(torch.float8_e5m2) == coll.FP8_E5M2


class _DeviceLike(torch.Tensor):
    """A CPU tensor that answers is_cuda=True, so the process group takes its CUDA branch while the test stays on CPU."""
    is_cuda = property(lambda self: True)

    @staticmethod
    def of(t):
        return torch.Tensor._make_subclass(_DeviceLike, t)


def test_process_group_sends_fp8_reductions_to_the_library(monkeypatch):
    """all_reduce (SUM / AVG / MAX) and reduce_scatter_tensor (SUM / AVG direct, MAX through an all-reduce) of fp8 device tensors
    reach the communicator, never Gloo; fp8 all-gather keeps the bit-exact word path."""
    class _Stream:
        def wait_event(self, e): pass
    class _Event:
        def record(self, s): pass
    stream = _Stream()
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: stream)
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    log = []

    class _Comm:
        nranks = 2
        _algo = "auto"
        def check_async_error(self): pass
        def set_algo(self, name): log.append(("algo", name)); self._algo = name
        def bit_exact(self): return coll.Comm._BitExact(self)
        def all_reduce(self, t, op=coll.SUM): log.append(("all_reduce", t.dtype, op))
        def reduce_scatter(self, src, dst, op=coll.SUM): log.append(("reduce_scatter", src.dtype, op, src.numel(), dst.numel()))
        def all_gather(self, src, dst): log.append(("all_gather", src.dtype, src.numel(), dst.numel()))

    class _NoGloo:
        def __getattr__(self, name): raise AssertionError(f"Gloo used for {name}")
    pg = pgmod.B200CollProcessGroup(store=None, rank=0, size=2)
    pg._comm, pg._gloo = _Comm(), _NoGloo()
    for dtype in FP8.values():
        for name, ours in (("SUM", coll.SUM), ("AVG", coll.AVG), ("MAX", coll.MAX)):
            o = dist.AllreduceOptions(); o.reduceOp = getattr(dist.ReduceOp, name)
            pg.allreduce([_DeviceLike.of(torch.zeros(64, dtype=dtype))], o)
            assert log[-1] == ("all_reduce", dtype, ours), (dtype, name)
            o = dist.ReduceScatterOptions(); o.reduceOp = getattr(dist.ReduceOp, name)
            pg._reduce_scatter_base(_DeviceLike.of(torch.zeros(32, dtype=dtype)), _DeviceLike.of(torch.zeros(64, dtype=dtype)), o)
            assert log[-1] == (("reduce_scatter", dtype, ours, 64, 32) if name != "MAX" else ("all_reduce", dtype, ours)), (dtype, name)
        del log[:]
        pg._allgather_base(_DeviceLike.of(torch.zeros(128, dtype=dtype)), _DeviceLike.of(torch.zeros(64, dtype=dtype)))
        assert log == [("algo", "twoshot"), ("all_gather", torch.float32, 16, 32), ("algo", "auto")]
        del log[:]
    assert pg.fallback_calls == 0 and pg.fast_calls == 2 * (3 * 2 + 1)


# ------------------------------------------------------------------------------------------------- one B200, virtual ranks
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture
def group(torch_cuda, coll_lib, request):
    n = getattr(request, "param", 2)
    coll.load()                          # raises if the .so is missing: GPU tests must never pass on a fallback
    comms = coll.Comm.init_all([0] * n, arena_mb=96)
    streams = [torch.cuda.Stream() for _ in comms]
    yield comms, streams
    torch.cuda.synchronize()
    for c in comms:
        c.destroy()


def _quarters(count, r, dtype, device="cuda"):
    """Multiples of 0.25 in [-2, 2]: exact in e4m3, e5m2, bf16, f16 and f32."""
    return ((((torch.arange(count, device=device) * (2 * r + 3) + r) % 17) - 8) * 0.25).to(dtype)


def _fill(comms, count, dtype, arena=True):
    srcs = []
    for r, c in enumerate(comms):
        t = c.empty(count, dtype) if arena else torch.empty(count, dtype=dtype, device="cuda")
        t.copy_(_quarters(count, r, dtype))
        srcs.append(t)
    torch.cuda.synchronize()
    return srcs


def _run_all(comms, streams, fn):
    for r, c in enumerate(comms):
        fn(r, c, streams[r])
    torch.cuda.synchronize()
    for c in comms:
        c.check_async_error()


def _total(srcs):
    return sum(s.float() for s in srcs)


@gpu
@pytest.mark.parametrize("group", [2, 4], indirect=True)
@pytest.mark.parametrize("name", ["e4m3", "e5m2"])
def test_fp8_all_reduce_every_algorithm_is_exact(torch_cuda, group, name):
    comms, streams = group
    dtype = FP8[name]
    for algo in ("ll", "ll2", "oneshot", "twoshot"):
        for count in (16, 1000, 1 << 15):                        # one vector, a scalar tail, many vectors
            srcs = _fill(comms, count, dtype)
            dsts = [c.empty(count, dtype) for c in comms]
            for c in comms:
                c.set_algo(algo)
            _run_all(comms, streams, lambda r, c, st: c.all_reduce(srcs[r], dsts[r], stream=st))
            want = _ref(_total(srcs), dtype)
            for d in dsts:
                assert _same(d, want), (algo, count)
            for c in comms:
                c.release(srcs[comms.index(c)]); c.release(dsts[comms.index(c)])
    for c in comms:
        assert c.stats()["algo_calls"]["ll2"] == 3 and c.stats()["generic_launches"] == 0


@gpu
@pytest.mark.parametrize("group", [2], indirect=True)
@pytest.mark.parametrize("name", ["e4m3", "e5m2"])
def test_fp8_buffers_outside_the_arena_are_staged(torch_cuda, group, name):
    comms, streams = group
    dtype = FP8[name]
    count = (1 << 20) + 40                                        # 1 MiB: beyond the Lamport paths; 8-element scalar tail
    srcs = _fill(comms, count, dtype, arena=False)
    dsts = [torch.empty(count, dtype=dtype, device="cuda") for _ in comms]
    _run_all(comms, streams, lambda r, c, st: c.all_reduce(srcs[r], dsts[r], stream=st))
    want = _ref(_total(srcs), dtype)
    assert all(_same(d, want) for d in dsts)
    rs = [torch.empty(count // 2 // 16 * 16, dtype=dtype, device="cuda") for _ in comms]
    m = rs[0].numel()
    _run_all(comms, streams, lambda r, c, st: c.reduce_scatter(srcs[r][:2 * m], rs[r], stream=st))
    full = _ref(sum(s[:2 * m].float() for s in srcs), dtype)
    assert all(_same(rs[r], full[r * m:(r + 1) * m]) for r in range(2))
    assert all(c.stats()["staged_calls"] == 2 for c in comms)


@gpu
@pytest.mark.parametrize("group", [4], indirect=True)
def test_fp8_fused_epilogues(torch_cuda, group):
    """Dequantise (e4m3 -> bf16, e5m2 -> f32, scale 0.5), AVG on fp8, and quantise bf16 -> e5m2."""
    comms, streams = group
    n, count = len(comms), 4096 + 8
    cases = [(torch.float8_e4m3fn, torch.bfloat16, 0.5, coll.SUM), (torch.float8_e5m2, torch.float32, 0.5, coll.SUM),
             (torch.float8_e4m3fn, torch.float8_e4m3fn, 1.0, coll.AVG), (torch.float8_e5m2, torch.float8_e5m2, 1.0, coll.AVG),
             (torch.bfloat16, torch.float8_e5m2, 0.25, coll.SUM)]
    for in_dt, out_dt, scale, op in cases:
        srcs = _fill(comms, count, in_dt)
        dsts = [c.empty(count, out_dt) for c in comms]
        algos = ("ll", "ll2", "oneshot", "twoshot") if in_dt == out_dt else ("ll", "oneshot", "twoshot")
        for algo in algos:
            for c in comms:
                c.set_algo(algo)
            _run_all(comms, streams, lambda r, c, st: c.all_reduce(srcs[r], dsts[r], scale=scale, op=op, stream=st))
            want = _ref(_total(srcs) * scale / (n if op == coll.AVG else 1), out_dt)
            for d in dsts:
                assert _same(d, want), (in_dt, out_dt, algo)


@gpu
@pytest.mark.parametrize("group", [2, 4], indirect=True)
@pytest.mark.parametrize("name", ["e4m3", "e5m2"])
def test_fp8_reduce_scatter_reduce_and_data_movement(torch_cuda, group, name):
    comms, streams = group
    n, dtype = len(comms), FP8[name]
    for algo in ("ll", "twoshot"):
        for c in comms:
            c.set_algo(algo)
        m = 2048
        srcs = _fill(comms, n * m, dtype)
        outs = [c.empty(m, dtype) for c in comms]
        _run_all(comms, streams, lambda r, c, st: c.reduce_scatter(srcs[r], outs[r], stream=st))
        full = _ref(_total(srcs), dtype)
        assert all(_same(outs[r], full[r * m:(r + 1) * m]) for r in range(n)), algo
        # dequantising all-gather: per-tensor scale fused into the push
        gat = [c.empty(n * m, torch.bfloat16) for c in comms]
        _run_all(comms, streams, lambda r, c, st: c.all_gather(srcs[r][:m], gat[r], scale=0.5, stream=st))
        want = torch.cat([(s[:m].float() * 0.5).to(torch.bfloat16) for s in srcs])
        assert all(_same(g, want) for g in gat), algo
        # bit-exact movement: all-gather, all-to-all, broadcast on fp8
        g8 = [c.empty(n * m, dtype) for c in comms]
        _run_all(comms, streams, lambda r, c, st: c.all_gather(srcs[r][:m], g8[r], stream=st))
        assert all(_same(g, torch.cat([s[:m] for s in srcs])) for g in g8), algo
        a2a = [c.empty(n * m, dtype) for c in comms]
        _run_all(comms, streams, lambda r, c, st: c.all_to_all(srcs[r], a2a[r], stream=st))
        for r in range(n):
            assert _same(a2a[r], torch.cat([srcs[s][r * m:(r + 1) * m] for s in range(n)])), algo
    count = 1003                                                   # not a whole number of 16-element vectors
    srcs = _fill(comms, count, dtype)
    for root in range(n):
        outs = [c.empty(count, dtype) for c in comms]
        for o in outs:
            o.copy_(torch.full((count,), 3.0, device="cuda").to(dtype))
        torch.cuda.synchronize()
        _run_all(comms, streams, lambda r, c, st: c.broadcast(srcs[r], outs[r], root=root, stream=st))
        assert all(_same(o, srcs[root]) for o in outs), root
        red = [c.empty(count, dtype) for c in comms]
        for o in red:
            o.copy_(torch.full((count,), 3.0, device="cuda").to(dtype))
        torch.cuda.synchronize()
        _run_all(comms, streams, lambda r, c, st: c.reduce(srcs[r], red[r], root=root, stream=st))
        for r in range(n):
            assert _same(red[r], _ref(_total(srcs), dtype) if r == root else torch.full((count,), 3.0, device="cuda").to(dtype)), (root, r)


@gpu
@pytest.mark.parametrize("group", [2, 4], indirect=True)
@pytest.mark.parametrize("name", ["e4m3", "e5m2"])
def test_fp8_sums_saturate_to_the_largest_finite_value(torch_cuda, group, name):
    comms, streams = group
    dtype = FP8[name]
    big = 320.0 if dtype == torch.float8_e4m3fn else 40960.0      # two of them exceed 448 / 57344
    count = 4096 + 8
    sign = torch.where(torch.arange(count, device="cuda") % 2 == 0, 1.0, -1.0)
    for algo in ("ll", "ll2", "oneshot", "twoshot"):
        for c in comms:
            c.set_algo(algo)
        srcs = [c.empty(count, dtype) for c in comms]
        for s in srcs:
            s.copy_((sign * big).to(dtype))
        dsts = [c.empty(count, dtype) for c in comms]
        torch.cuda.synchronize()
        _run_all(comms, streams, lambda r, c, st: c.all_reduce(srcs[r], dsts[r], stream=st))
        want = (sign * FP8_MAX[dtype]).to(dtype)
        assert all(_same(d, want) for d in dsts), algo


@gpu
@pytest.mark.parametrize("group", [2, 4], indirect=True)
@pytest.mark.parametrize("name", ["e4m3", "e5m2"])
def test_fp8_min_max_prod_on_the_generic_kernel(torch_cuda, group, name):
    comms, streams = group
    n, dtype = len(comms), FP8[name]
    for count, arena in ((1000, True), (1000, False)):
        srcs = _fill(comms, count, dtype, arena=arena)
        for op, fold in ((coll.MIN, torch.minimum), (coll.MAX, torch.maximum), (coll.PROD, torch.mul)):
            dsts = [c.empty(count, dtype) if arena else torch.empty(count, dtype=dtype, device="cuda") for c in comms]
            _run_all(comms, streams, lambda r, c, st: c.all_reduce(srcs[r], dsts[r], op=op, stream=st))
            want = _ref(functools.reduce(fold, [s.float() for s in srcs]), dtype)      # rank order, fp32
            assert all(_same(d, want) for d in dsts), (op, arena)
        m = count // n // 16 * 16                                 # reduce-scatter blocks are whole 16-byte vectors
        rs = [torch.empty(m, dtype=dtype, device="cuda") for _ in comms]
        _run_all(comms, streams, lambda r, c, st: c.reduce_scatter(srcs[r][:n * m], rs[r], op=coll.MAX, stream=st))
        full = _ref(functools.reduce(torch.maximum, [s[:n * m].float() for s in srcs]), dtype)
        assert all(_same(rs[r], full[r * m:(r + 1) * m]) for r in range(n))
    assert all(c.stats()["generic_launches"] >= 8 for c in comms)


@gpu
@pytest.mark.parametrize("group", [2], indirect=True)
@pytest.mark.parametrize("name", ["e4m3", "e5m2"])
def test_fp8_all_reduce_host_zero_copy_and_pipelined(torch_cuda, group, name):
    comms, streams = group
    dtype = FP8[name]
    for count in (4096, (9 << 20) + 5):                           # one zero-copy kernel; a chunked pipeline (9 MiB)
        ins = [_quarters(count, r, dtype, device="cpu") for r in range(2)]
        h_in = [c.host_empty(count, dtype) for c in comms]
        h_out = [c.host_empty(count, dtype) for c in comms]
        for r in range(2):
            h_in[r].copy_(ins[r]); h_out[r].fill_(0)
        for r, c in enumerate(comms):
            c.all_reduce_host(h_in[r], h_out[r], stream=streams[r])
        torch.cuda.synchronize()
        want = _ref(_total(ins), dtype)
        assert all(_same(h, want) for h in h_out), count
        for r, c in enumerate(comms):
            c.host_release(h_in[r]); c.host_release(h_out[r])
    st = comms[0].stats()
    assert st["host_zero_copy"] == 1 and st["host_pipelined"] == 1, st
    for c in comms:
        c.check_async_error()


@gpu
def test_fp8_through_the_nccl_shim(torch_cuda, coll_lib):
    """ncclFloat8e4m3 / ncclFloat8e5m2 through libb200coll_nccl.so on plain cudaMalloc buffers: reductions on the fused and generic
    kernels, movement bit for bit."""
    from tests.test_coll_gpu import _NcclShim
    s = _NcclShim()
    L, n = s.L, 2
    SUM, MAX, AVG = 0, 2, 4
    comms = (C.c_void_p * n)()
    s.ck(L.ncclCommInitAll(comms, n, (C.c_int * n)(0, 0)))
    try:
        streams = [torch.cuda.Stream() for _ in range(n)]
        st = [C.c_void_p(x.cuda_stream) for x in streams]
        p = lambda t: C.c_void_p(t.data_ptr())

        def every(fn):
            for r in range(n):
                s.ck(fn(r))
            torch.cuda.synchronize()
            for r in range(n):
                err = C.c_int(-1)
                s.ck(L.ncclCommGetAsyncError(comms[r], C.byref(err)))
                assert err.value == 0

        e4 = torch.float8_e4m3fn
        for count in (1000, 3 << 19):                              # Lamport path, then staged
            src = [_quarters(count, r, e4) for r in range(n)]
            for op, want in ((SUM, _ref(_total(src), e4)), (AVG, _ref(_total(src) / n, e4)),
                             (MAX, torch.maximum(src[0].float(), src[1].float()).to(e4))):
                dst = [torch.empty(count, dtype=e4, device="cuda") for _ in range(n)]
                every(lambda r: L.ncclAllReduce(p(src[r]), p(dst[r]), count, NCCL_FP8["e4m3"], op, comms[r], st[r]))
                assert all(_same(d, want) for d in dst), (count, op)
        e5 = torch.float8_e5m2
        m = 4096
        src = [_quarters(n * m, r, e5) for r in range(n)]
        rs = [torch.empty(m, dtype=e5, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclReduceScatter(p(src[r]), p(rs[r]), m, NCCL_FP8["e5m2"], SUM, comms[r], st[r]))
        full = _ref(_total(src), e5)
        assert all(_same(rs[r], full[r * m:(r + 1) * m]) for r in range(n))
        for name, dtype in FP8.items():
            dt = NCCL_FP8[name]
            # every byte value but NaN (and inf for e5m2) in the payload; the movement ops carry them unchanged
            payload = []
            for r in range(n):
                raw = (torch.arange(2 * m, device="cuda", dtype=torch.int32) * 7 + 37 * r) % 256
                bad = (raw & 0x7F) == 0x7F if name == "e4m3" else (raw & 0x7C) == 0x7C
                payload.append(torch.where(bad, 0, raw).to(torch.uint8).view(dtype))
            gat = [torch.empty(n * 2 * m, dtype=dtype, device="cuda") for _ in range(n)]
            every(lambda r: L.ncclAllGather(p(payload[r]), p(gat[r]), 2 * m, dt, comms[r], st[r]))
            assert all(_same(g, torch.cat(payload)) for g in gat), name
            bc = [x.clone() for x in payload]
            every(lambda r: L.ncclBroadcast(p(bc[r]), p(bc[r]), 2 * m, dt, 1, comms[r], st[r]))
            assert all(_same(b, payload[1]) for b in bc), name
            a2a = [torch.empty(2 * m, dtype=dtype, device="cuda") for _ in range(n)]
            every(lambda r: L.ncclAlltoAll(p(payload[r]), p(a2a[r]), m, dt, comms[r], st[r]))
            for r in range(n):
                assert _same(a2a[r], torch.cat([payload[q][r * m:(r + 1) * m] for q in range(n)])), name
    finally:
        torch.cuda.synchronize()
        for c in comms:
            L.ncclCommDestroy(c)


def _fp8_pair(rank, world):
    torch.cuda.set_device(0)                                      # two ranks share cuda:0 on a one-GPU box
    pg = dist.group.WORLD
    fast, fb = pg.fast_calls, pg.fallback_calls
    x = _quarters(1 << 16, rank, torch.float8_e4m3fn)
    want = _ref(sum(_quarters(1 << 16, r, torch.float8_e4m3fn).float() for r in range(world)), torch.float8_e4m3fn)
    dist.all_reduce(x)
    assert _same(x, want)
    y = _quarters(4096, rank, torch.float8_e4m3fn)
    dist.all_reduce(y, op=dist.ReduceOp.AVG)
    assert _same(y, _ref(sum(_quarters(4096, r, torch.float8_e4m3fn).float() for r in range(world)) / world, torch.float8_e4m3fn))
    src = _quarters(world * 4096, rank, torch.float8_e5m2)
    out = torch.empty(4096, dtype=torch.float8_e5m2, device="cuda")
    dist.reduce_scatter_tensor(out, src)
    full = _ref(sum(_quarters(world * 4096, r, torch.float8_e5m2).float() for r in range(world)), torch.float8_e5m2)
    assert _same(out, full[rank * 4096:(rank + 1) * 4096])
    assert pg.fast_calls == fast + 3 and pg.fallback_calls == fb
    return pg.fast_calls


@gpu
def test_fp8_process_group_two_ranks(torch_cuda):
    from tests.test_process_group import _run
    _run(_fp8_pair, 2)


# ------------------------------------------------------------------------------------------------- >= 2 B200s
@gpu
def test_fp8_multi_gpu_takes_the_p2p_kernels_and_is_exact(torch_cuda, coll_lib):
    """No multicast kernel is built for fp8 inputs: on an NVSwitch system a call the tuner (or --algo nvls) sends to NVLS runs two-shot,
    and the perf tool's check is exact for fp8 sums."""
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    perf = os.path.join(ROOT, "build", "b200coll_perf")
    devs = ",".join(str(i) for i in range(n))
    for dt in ("e4m3", "e5m2"):
        for op in ("all_reduce", "reduce_scatter", "reduce"):
            for algo in ("auto", "nvls"):
                r = subprocess.run([perf, "--devs", devs, "--procs", "--op", op, "--algo", algo, "-d", dt, "-b", "1K", "-e", "64M", "-f", "16", "--iters", "3", "--warmup", "1"],
                                   capture_output=True, text=True, timeout=180, env={**os.environ, "B200COLL_TIMEOUT_MS": "5000"})
                assert r.returncode == 0 and "errors=0" in r.stdout, r.stdout + r.stderr


@gpu
def test_fp8_perf_tool_virtual_ranks_zero_errors(torch_cuda, coll_lib):
    """b200coll_perf -d e4m3|e5m2 and --out-dtype e5m2: the tool's check is exact for fp8 sums on the fp32-accumulating paths."""
    perf = os.path.join(ROOT, "build", "b200coll_perf")
    for args in (["--op", "all_reduce", "-d", "e4m3"], ["--op", "reduce_scatter", "-d", "e5m2"], ["--op", "all_gather", "-d", "e4m3", "--out-dtype", "f32"],
                 ["--op", "all_reduce", "-d", "bf16", "--out-dtype", "e5m2"]):
        r = subprocess.run([perf, "--devs", "0,0,0,0", *args, "-b", "1K", "-e", "1M", "-f", "4", "--iters", "3", "--warmup", "1"], capture_output=True, text=True,
                           timeout=120, env={**os.environ, "B200COLL_TIMEOUT_MS": "5000"})
        assert r.returncode == 0 and "errors=0" in r.stdout, r.stdout + r.stderr
