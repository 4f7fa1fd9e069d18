"""Which algorithm each fused collective runs, and how buffers outside the symmetric arena are staged (GPU, virtual ranks on cuda:0).

Every case checks the output against a plain PyTorch fp32 reference and the exact per-call change of the communicator's counters.
The expected algorithm follows the selection rules written out in `_resolve` below: the forced algorithm or the tuner's pick, moved
to one the call can run. Virtual ranks have no multicast, so a forced `nvls` is checked as the fallback it takes there. The large
size of every op is one staging chunk plus 1024 elements, so a staged call runs its chunk loop twice."""
import ctypes as C

import pytest

pytestmark = pytest.mark.gpu

OPS = ["all_reduce", "all_gather", "reduce_scatter", "all_to_all", "broadcast", "reduce"]
OP_INDEX = {op: i for i, op in enumerate(OPS)}               # b200collOp_t order
ALGOS = ["auto", "ll", "ll2", "oneshot", "twoshot", "nvls", "copy"]
LL_MAX = 512 << 10                                            # Lamport one-shot limit per source (kLLOneShotMaxBytes)
STAGE_HALF = 32 << 20                                         # bytes of one staging half (kStageHalfBytes)
BULK_MIN = 1 << 20                                            # copy-engine path threshold (B200COLL_BULK_MIN_KB default)
SMALL = 48 << 10                                              # elements: 96 KiB of bf16, below the Lamport limit
INVALID_ARGUMENT = 4


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def coll_mod(coll_lib):
    from container_engine_accelerators_b200.ops import coll
    coll.load()          # raises if the .so is missing: GPU tests must never pass on a fallback
    return coll


@pytest.fixture(scope="module", params=[2, 4])
def group(torch_cuda, coll_mod, request):
    comms = coll_mod.Comm.init_all([0] * request.param, arena_mb=192)      # heap after the 89 MiB of control and staging: two 32 MiB buffers
    streams = [torch_cuda.cuda.Stream() for _ in comms]
    yield comms, streams
    torch_cuda.cuda.synchronize()
    for c in comms:
        c.destroy()


def _dtype(torch, name):
    return getattr(torch, name)


def _size(torch, name):
    return torch.empty((), dtype=_dtype(torch, name)).element_size()


def _chunk(op, n, is_, os_):
    """Elements per staging chunk: one staging half over the element size, and over nranks for ops staged as one row per rank."""
    if op in ("all_gather", "all_to_all"):
        return STAGE_HALF // os_ // n // 64 * 64
    if op == "reduce_scatter":
        return STAGE_HALF // is_ // n // 64 * 64
    return STAGE_HALF // max(is_, os_) // 64 * 64


def _resolve(coll, op, nbytes, n, forced, sym_in, sym_out, same_size):
    """The algorithm the library runs (no multicast); None: an all-reduce that no algorithm can run in place, so it is staged."""
    a = forced if forced != "auto" else coll.tuner_pick(OP_INDEX[op], nbytes, n, False)
    if op == "all_reduce":
        feasible = {"ll": nbytes <= LL_MAX, "ll2": same_size and nbytes <= LL_MAX * n, "oneshot": sym_in, "twoshot": sym_in and sym_out}
        if feasible.get(a, False):
            return a
        return next((x for x in ("twoshot", "oneshot", "ll", "ll2") if feasible[x]), None)
    if op in ("all_gather", "reduce_scatter", "all_to_all"):
        a = "ll" if a == "ll2" else a
        if a == "ll" and nbytes <= LL_MAX:
            return "ll"
        return "twoshot" if op == "all_to_all" or a in ("ll", "oneshot", "nvls", "copy") else a
    return "twoshot"


def _expect(coll, op, n, count, forced, arena, is_, os_, identity):
    """(accounted calls as [(bytes, algo)], kernel launches, staged calls, copy-engine launches) of one call on one rank."""
    nbytes = count * is_
    a = _resolve(coll, op, nbytes, n, forced, arena, arena, is_ == os_)
    per_peer = n if op == "all_to_all" else 1
    if a == "ll":
        return [(nbytes * per_peer, "ll")], 1, 0, 0
    bulk = arena and identity and nbytes % 16 == 0 and (
        (op == "all_gather" and nbytes >= BULK_MIN) or (op == "all_to_all" and nbytes * n >= BULK_MIN) or (op == "broadcast" and nbytes >= BULK_MIN))
    if bulk:
        return [(nbytes * per_peer, a)], 1, 0, 1
    if a is not None and (arena or op == "all_reduce"):        # an all-reduce algorithm that was not staged reads the buffers in place
        return [(nbytes * per_peer, a)], 1, 0, 0
    chunk = _chunk(op, n, is_, os_)
    inner = a or "twoshot"                                    # the staged all-reduce runs two-shot between the staging halves
    sizes = [min(chunk, count - done) for done in range(0, count, chunk)]
    return [(m * is_ * per_peer, inner) for m in sizes], len(sizes), 1, 0


def _fill(torch, n, numel, dtype, seed):
    base = torch.arange(numel, device="cuda")
    return [((((base * (2 * r + 3) + r + seed) % 17) - 8).float() * 0.25).to(dtype) for r in range(n)]


def _cast(torch, t, name):
    """fp32 -> `name` with the kernels' round-to-nearest, saturating cast."""
    limit = {"float8_e4m3fn": 448.0, "float8_e5m2": 57344.0}.get(name)
    return (t.clamp(-limit, limit) if limit else t).to(_dtype(torch, name))


def _place(torch, comms, tensors, arena):
    if not arena:
        return tensors
    out = []
    for c, t in zip(comms, tensors):
        a = c.empty(t.numel(), t.dtype)
        a.copy_(t)
        out.append(a)
    return out


def _release(comms, arena, *lists):
    if arena:
        for ts in lists:
            for c, t in zip(comms, ts):
                c.release(t)


def _counters(c):
    s = c.stats()
    return s["calls"], s["bytes"], s["algo_calls"], {k: s[k] for k in ("kernel_launches", "staged_calls", "bulk_launches", "generic_launches")}


def _delta(before, after):
    calls = [b - a for a, b in zip(before[0], after[0])]
    nbytes = [b - a for a, b in zip(before[1], after[1])]
    algos = {k: after[2][k] - before[2][k] for k in after[2]}
    other = {k: after[3][k] - before[3][k] for k in after[3]}
    return calls, nbytes, algos, other


def _run(torch, coll, comms, streams, op, forced, arena, count, in_name="bfloat16", out_name="bfloat16"):
    n = len(comms)
    in_dt, out_dt = _dtype(torch, in_name), _dtype(torch, out_name)
    is_, os_ = _size(torch, in_name), _size(torch, out_name)
    root = n - 1
    in_numel = count * n if op in ("reduce_scatter", "all_to_all") else count
    out_numel = count * n if op in ("all_gather", "all_to_all") else count
    srcs = _place(torch, comms, _fill(torch, n, in_numel, in_dt, OP_INDEX[op]), arena)
    dsts = _place(torch, comms, [torch.full((out_numel,), 3.0, device="cuda").to(out_dt) for _ in range(n)], arena)
    torch.cuda.synchronize()
    for c in comms:
        c.set_algo(forced)
    before = [_counters(c) for c in comms]
    for r, c in enumerate(comms):
        s, d, st = srcs[r], dsts[r], streams[r]
        if op == "all_reduce":
            c.all_reduce(s, d, stream=st)
        elif op == "all_gather":
            c.all_gather(s, d, stream=st)
        elif op == "reduce_scatter":
            c.reduce_scatter(s, d, stream=st)
        elif op == "all_to_all":
            c.all_to_all(s, d, stream=st)
        elif op == "broadcast":
            c.broadcast(s, d, root=root, stream=st)
        else:
            c.reduce(s, d, root=root, stream=st)
    torch.cuda.synchronize()
    for c in comms:
        c.check_async_error()
    after = [_counters(c) for c in comms]

    f = [s.float() for s in srcs]
    total = sum(f)
    for r in range(n):
        if op == "all_reduce":
            want = total
        elif op == "all_gather":
            want = torch.cat(f)
        elif op == "reduce_scatter":
            want = total[r * count:(r + 1) * count]
        elif op == "all_to_all":
            want = torch.cat([f[s][r * count:(r + 1) * count] for s in range(n)])
        elif op == "broadcast":
            want = f[root]
        else:
            want = total if r == root else torch.full((count,), 3.0, device="cuda")
        assert torch.equal(dsts[r].float(), _cast(torch, want, out_name).float()), (op, forced, arena, count, r)

    accounted, launches, staged, bulk = _expect(coll, op, n, count, forced, arena, is_, os_, in_name == out_name)
    calls, nbytes = [0] * 6, [0] * 6
    calls[OP_INDEX[op]], nbytes[OP_INDEX[op]] = len(accounted), sum(b for b, _ in accounted)
    algos = dict.fromkeys(coll.ALGO_NAMES, 0)
    for _, a in accounted:
        algos[a] += 1
    want = (calls, nbytes, algos, {"kernel_launches": launches, "staged_calls": staged, "bulk_launches": bulk, "generic_launches": 0})
    for r in range(n):
        assert _delta(before[r], after[r]) == want, (op, forced, arena, count, r)
    _release(comms, arena, srcs, dsts)


def _large(torch, op, n, in_name="bfloat16", out_name="bfloat16"):
    return _chunk(op, n, _size(torch, in_name), _size(torch, out_name)) + 1024


@pytest.mark.parametrize("size", ["small", "large"])
@pytest.mark.parametrize("arena", [True, False], ids=["arena", "plain"])
@pytest.mark.parametrize("forced", ALGOS)
@pytest.mark.parametrize("op", OPS)
def test_algorithm_and_staging(torch_cuda, coll_mod, group, op, forced, arena, size):
    if forced == "copy" and op in ("all_gather", "reduce_scatter"):
        pytest.skip("test_forced_copy_all_gather_reduce_scatter_counts_twoshot")
    comms, streams = group
    count = SMALL if size == "small" else _large(torch_cuda, op, len(comms))
    _run(torch_cuda, coll_mod, comms, streams, op, forced, arena, count)


@pytest.mark.parametrize("arena", [True, False], ids=["arena", "plain"])
@pytest.mark.parametrize("forced", ["auto", "twoshot"])
@pytest.mark.parametrize("pair", [("bfloat16", "bfloat16"), ("bfloat16", "float32"), ("float8_e4m3fn", "bfloat16"), ("float32", "float8_e5m2")],
                         ids=lambda p: f"{p[0]}-{p[1]}")
@pytest.mark.parametrize("op", OPS)
def test_type_pairs(torch_cuda, coll_mod, group, op, pair, forced, arena):
    comms, streams = group
    _run(torch_cuda, coll_mod, comms, streams, op, forced, arena, _large(torch_cuda, op, len(comms), *pair), *pair)


@pytest.mark.parametrize("size", ["small", "large"])
@pytest.mark.parametrize("arena", [True, False], ids=["arena", "plain"])
def test_generic_int32_max_all_reduce(torch_cuda, coll_mod, group, arena, size):
    torch = torch_cuda
    comms, streams = group
    n = len(comms)
    chunk = STAGE_HALF // 4 // 64 * 64
    count = SMALL if size == "small" else chunk + 1024
    base = torch.arange(count, device="cuda", dtype=torch.int32)
    srcs = _place(torch, comms, [(base * (r + 7)) % 1000003 - 500000 for r in range(n)], arena)
    dsts = _place(torch, comms, [torch.zeros(count, dtype=torch.int32, device="cuda") for _ in range(n)], arena)
    torch.cuda.synchronize()
    before = [_counters(c) for c in comms]
    for r, c in enumerate(comms):
        c.all_reduce(srcs[r], dsts[r], op=coll_mod.MAX, stream=streams[r])
    torch.cuda.synchronize()
    for c in comms:
        c.check_async_error()
    want_out = torch.stack(srcs).amax(0)
    kernels = 1 if arena else -(-count // chunk)
    algos = dict.fromkeys(coll_mod.ALGO_NAMES, 0)
    algos["twoshot"] = 1
    want = ([1, 0, 0, 0, 0, 0], [count * 4, 0, 0, 0, 0, 0], algos,
            {"kernel_launches": kernels, "staged_calls": 0 if arena else 1, "bulk_launches": 0, "generic_launches": kernels})
    for r, c in enumerate(comms):
        assert torch.equal(dsts[r], want_out)
        assert _delta(before[r], _counters(c)) == want
    _release(comms, arena, srcs, dsts)


@pytest.mark.parametrize("size", ["small", "large"])
@pytest.mark.parametrize("arena", [True, False], ids=["arena", "plain"])
@pytest.mark.parametrize("op", ["all_gather", "reduce_scatter"])
def test_forced_copy_all_gather_reduce_scatter_counts_twoshot(torch_cuda, coll_mod, group, op, arena, size):
    """A forced `copy` with several ranks runs the P2P (or copy-engine) kernels and is counted under their family, two-shot."""
    comms, streams = group
    count = SMALL if size == "small" else _large(torch_cuda, op, len(comms))
    _run(torch_cuda, coll_mod, comms, streams, op, "copy", arena, count)


@pytest.mark.parametrize("count", [0, SMALL, 1 << 21])
@pytest.mark.parametrize("op", OPS)
def test_unsupported_type_pair_is_refused_before_any_work(torch_cuda, coll_mod, group, op, count):
    """bf16 -> fp16 has no kernel: every op refuses it up front, whatever the size, with no counter moved and nothing enqueued."""
    torch = torch_cuda
    comms, _ = group
    c = comms[0]
    n = len(comms)
    src = torch.zeros(max(count, 1) * n, dtype=torch.bfloat16, device="cuda")      # the C API directly: real pointers also for count 0
    dst = torch.zeros(max(count, 1) * n, dtype=torch.float16, device="cuda")
    L, h, st = coll_mod.load(), c._h, c._stream(None)
    ep = C.byref(coll_mod.Epilogue(coll_mod.BF16, coll_mod.F16, 1.0))
    s, d = C.c_void_p(src.data_ptr()), C.c_void_p(dst.data_ptr())
    call = {"all_reduce": lambda: L.b200collAllReduce(s, d, count, ep, coll_mod.SUM, h, st),
            "all_gather": lambda: L.b200collAllGather(s, d, count, ep, h, st),
            "reduce_scatter": lambda: L.b200collReduceScatter(s, d, count, ep, coll_mod.SUM, h, st),
            "all_to_all": lambda: L.b200collAllToAll(s, d, count, ep, h, st),
            "broadcast": lambda: L.b200collBroadcast(s, d, count, ep, 0, h, st),
            "reduce": lambda: L.b200collReduce(s, d, count, ep, coll_mod.SUM, 0, h, st)}[op]
    c.set_algo("auto")
    before = _counters(c)
    assert call() == INVALID_ARGUMENT
    torch.cuda.synchronize()
    assert _delta(before, _counters(c)) == _delta(before, before)
