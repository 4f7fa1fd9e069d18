"""GPU tests for libb200coll (run with `pytest -m gpu` on a B200 box). Every numerics check compares the CUDA kernel with a
plain PyTorch fp32 reference of the same op. On a one-GPU box the P2P protocols are exercised with virtual ranks that
share cuda:0 (in-process group, one stream per rank); NVLS/multicast and true multi-process tests need >= 2 GPUs."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PERF = os.path.join(ROOT, "build", "b200coll_perf")


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


@pytest.fixture
def group(torch_cuda, coll_mod, request):
    n = getattr(request, "param", 2)
    comms = coll_mod.Comm.init_all([0] * n, arena_mb=96)
    streams = [torch_cuda.cuda.Stream() for _ in comms]
    yield comms, streams
    torch_cuda.cuda.synchronize()
    for c in comms:
        c.destroy()


def fill(torch, comms, count, dtype):
    srcs = []
    for r, c in enumerate(comms):
        t = c.empty(count, dtype)
        t.copy_((((torch.arange(count, device="cuda") * (2 * r + 3) + r) % 17) - 8).to(dtype) * 0.25)
        srcs.append(t)
    torch.cuda.synchronize()
    return srcs


def run_all(torch, comms, streams, fn):
    for r, c in enumerate(comms):
        fn(r, c, streams[r])
    torch.cuda.synchronize()
    for c in comms:
        c.check_async_error()


def test_self_check_and_arena_tensor_aliasing(torch_cuda, coll_mod):
    ok, report = coll_mod.self_check()
    assert ok, report
    (c,) = coll_mod.Comm.init_all([0], arena_mb=16)
    t = c.empty(1024, torch_cuda.bfloat16)
    assert c.is_symmetric(t) and t.data_ptr() == t._b200coll_buf.ptr       # zero-copy view of arena memory
    t.fill_(3.0)
    out = c.empty(1024, torch_cuda.float32)
    c.all_reduce(t, out, scale=0.5)                                        # nranks == 1: fused scale/cast copy kernel
    torch_cuda.cuda.synchronize()
    assert torch_cuda.equal(out, torch_cuda.full((1024,), 1.5, device="cuda"))
    assert c.stats()["kernel_launches"] == 1
    first = t.data_ptr()
    c.release(out); c.release(t)                                           # explicit, deterministic hand-back: the next allocation reuses the space
    assert c.empty(1024, torch_cuda.bfloat16).data_ptr() == first
    with pytest.raises(ValueError):
        c.release(torch_cuda.empty(4, device="cuda"))
    c.destroy()


@pytest.mark.parametrize("group", [2, 4], indirect=True)
@pytest.mark.parametrize("algo", ["ll", "ll2", "oneshot", "twoshot"])
@pytest.mark.parametrize("count", [8, 1000, 1 << 15])
def test_all_reduce_matches_fp32_reference(torch_cuda, group, algo, count):
    torch = torch_cuda
    comms, streams = group
    srcs = fill(torch, comms, count, torch.bfloat16)
    dsts = [c.empty(count, torch.bfloat16) for c in comms]
    want = sum(s.float() for s in srcs)
    for c in comms:
        c.set_algo(algo)
    run_all(torch, comms, streams, lambda r, c, st: c.all_reduce(srcs[r], dsts[r], stream=st))
    for d in dsts:
        assert torch.equal(d.float(), want)
    for a, b in zip(dsts, dsts[1:]):
        assert torch.equal(a, b)                # every rank holds bit-identical results


@pytest.mark.parametrize("group", [4], indirect=True)
def test_in_place_and_repeated_launches_rotate_lamport_buffers(torch_cuda, group):
    torch = torch_cuda
    comms, streams = group
    for it, (algo, count) in enumerate([("ll", 4096), ("ll2", 64), ("ll", 9000), ("ll2", 70001), ("ll2", 16), ("ll", 4096), ("ll2", 4096), ("ll", 128), ("ll", 128)]):
        # shrinking/growing sizes and alternating one-/two-shot Lamport kernels: stale-slot clearing (lo and hi halves) must follow
        for c in comms:
            c.set_algo(algo)
        srcs = fill(torch, comms, count, torch.bfloat16)
        want = sum(s.float() for s in srcs)
        run_all(torch, comms, streams, lambda r, c, st: c.all_reduce(srcs[r], stream=st))
        for s in srcs:
            assert torch.equal(s.float(), want), f"iteration {it} count {count}"


@pytest.mark.parametrize("group", [2], indirect=True)
@pytest.mark.parametrize("in_dt,out_dt,scale", [("bfloat16", "float32", 0.5), ("float32", "bfloat16", 0.25), ("float16", "float16", 2.0), ("bfloat16", "float8_e4m3fn", 0.125)])
def test_fused_scale_cast_epilogue(torch_cuda, group, in_dt, out_dt, scale):
    torch = torch_cuda
    comms, streams = group
    count = 4096
    srcs = fill(torch, comms, count, getattr(torch, in_dt))
    dsts = [c.empty(count, getattr(torch, out_dt)) for c in comms]
    want = (sum(s.float() for s in srcs) * scale)
    for algo in ("ll", "twoshot"):
        for c in comms:
            c.set_algo(algo)
        run_all(torch, comms, streams, lambda r, c, st: c.all_reduce(srcs[r], dsts[r], scale=scale, stream=st))
        for d in dsts:
            if out_dt == "float8_e4m3fn":
                assert torch.allclose(d.float(), want.to(torch.float8_e4m3fn).float())
            else:
                assert torch.equal(d.float(), want.to(getattr(torch, out_dt)).float()), algo


@pytest.mark.parametrize("group", [4], indirect=True)
@pytest.mark.parametrize("algo", ["ll", "twoshot"])
def test_all_gather_reduce_scatter_all_to_all(torch_cuda, group, algo):
    torch = torch_cuda
    comms, streams = group
    n, count = len(comms), 2048
    for c in comms:
        c.set_algo(algo)
    srcs = fill(torch, comms, count, torch.bfloat16)
    gat = [c.empty(count * n, torch.bfloat16) for c in comms]
    run_all(torch, comms, streams, lambda r, c, st: c.all_gather(srcs[r], gat[r], stream=st))
    for g in gat:
        assert torch.equal(g, torch.cat(srcs))
    big = fill(torch, comms, count * n, torch.bfloat16)
    rs = [c.empty(count, torch.bfloat16) for c in comms]
    run_all(torch, comms, streams, lambda r, c, st: c.reduce_scatter(big[r], rs[r], stream=st))
    total = sum(b.float() for b in big)
    for r in range(n):
        assert torch.equal(rs[r].float(), total[r * count:(r + 1) * count])
    a2a = [c.empty(count * n, torch.bfloat16) for c in comms]
    run_all(torch, comms, streams, lambda r, c, st: c.all_to_all(big[r], a2a[r], stream=st))
    for r in range(n):
        want = torch.cat([big[s][r * count:(r + 1) * count] for s in range(n)])
        assert torch.equal(a2a[r], want)


@pytest.mark.parametrize("group", [2, 4], indirect=True)
def test_copy_engine_path_all_gather_all_to_all_broadcast(torch_cuda, group):
    """Identity epilogue and >= 1 MiB: the payload moves through the cp.async.bulk ring (k_bulk) instead of LDG/STG — all-gather, all-to-all
    and the P2P broadcast, odd chunk counts so the last chunk of a segment is short; bit-exact against plain tensor ops."""
    torch = torch_cuda
    comms, streams = group
    n = len(comms)
    count = (1 << 20) + 40 * 8                                      # 2 MiB + 640 B per rank: 129 chunks of 16 KiB, the last one short
    srcs = []
    for r, c in enumerate(comms):
        t = c.empty(count * n, torch.bfloat16)
        t.copy_(((torch.arange(count * n, device="cuda") * (2 * r + 3) + 7 * r) % 251 - 125).to(torch.bfloat16))
        srcs.append(t)
    torch.cuda.synchronize()
    before = comms[0].stats()["bulk_launches"]
    gat = [c.empty(count * n, torch.bfloat16) for c in comms]
    run_all(torch, comms, streams, lambda r, c, st: c.all_gather(srcs[r][:count], gat[r], stream=st))
    for g in gat:
        assert torch.equal(g, torch.cat([s[:count] for s in srcs]))
    a2a = [c.empty(count * n, torch.bfloat16) for c in comms]
    for rep in range(2):                                            # twice: the ring's mbarrier phases and the barrier epochs carry over
        run_all(torch, comms, streams, lambda r, c, st: c.all_to_all(srcs[r], a2a[r], stream=st))
        for r in range(n):
            assert torch.equal(a2a[r], torch.cat([srcs[s][r * count:(r + 1) * count] for s in range(n)]))
    for root in range(n):
        outs = [c.empty(count, torch.bfloat16) for c in comms]
        run_all(torch, comms, streams, lambda r, c, st: c.broadcast(srcs[r][:count], outs[r], root=root, stream=st))
        for o in outs:
            assert torch.equal(o, srcs[root][:count])
        for c, o in zip(comms, outs):
            c.release(o)
    assert comms[0].stats()["bulk_launches"] - before == 1 + 2 + n   # every one of those calls took the copy-engine kernel


def test_copy_engine_path_one_rank_copy(torch_cuda, coll_mod):
    torch = torch_cuda
    (c,) = coll_mod.Comm.init_all([0], arena_mb=96)
    count = (12 << 20) + 8 * 37
    src = c.empty(count, torch.bfloat16)
    src.copy_((torch.arange(count, device="cuda") % 509 - 254).to(torch.bfloat16))
    dst = c.empty(count, torch.bfloat16)
    dst.zero_()
    c.all_reduce(src, dst)
    torch.cuda.synchronize()
    assert torch.equal(dst, src) and c.stats()["bulk_launches"] == 1
    plain = torch.empty(count, dtype=torch.bfloat16, device="cuda")      # destination outside the arena
    c.all_reduce(src, plain)
    torch.cuda.synchronize()
    assert torch.equal(plain, src) and c.stats()["bulk_launches"] == 2
    c.destroy()


@pytest.mark.parametrize("group", [2, 4], indirect=True)
@pytest.mark.parametrize("count", [8, 1003, 1 << 16])
def test_broadcast_and_reduce_rooted(torch_cuda, group, count):
    """ncclBroadcast / ncclReduce semantics incl. a count that is not a whole number of 16-byte vectors, every root,
    in-place, and the fused cast/scale epilogue (fp32 reference)."""
    torch = torch_cuda
    comms, streams = group
    n = len(comms)
    srcs = fill(torch, comms, count, torch.bfloat16)
    for root in range(n):
        outs = [c.empty(count, torch.bfloat16) for c in comms]
        for o in outs:
            o.fill_(55.0)
        torch.cuda.synchronize()
        run_all(torch, comms, streams, lambda r, c, st: c.broadcast(srcs[r], outs[r], root=root, stream=st))
        for o in outs:
            assert torch.equal(o, srcs[root]), root
        red = [c.empty(count, torch.float32) for c in comms]
        for o in red:
            o.fill_(55.0)
        torch.cuda.synchronize()
        run_all(torch, comms, streams, lambda r, c, st: c.reduce(srcs[r], red[r], root=root, scale=0.5, stream=st))   # bf16 in, fp32 out, x0.5 fused
        want = sum(t.float() for t in srcs) * 0.5
        for r in range(n):
            assert torch.equal(red[r], want if r == root else torch.full_like(want, 55.0)), (root, r)
    # in-place broadcast from rank 1 with a fused fp32 -> (scale 2) -> fp32 epilogue
    bufs = [c.empty(count, torch.float32) for c in comms]
    for r, b in enumerate(bufs):
        b.copy_(torch.arange(count, device="cuda").float() * 0.5 + r)
    torch.cuda.synchronize()
    want = bufs[1].clone() * 2.0
    run_all(torch, comms, streams, lambda r, c, st: c.broadcast(bufs[r], root=1, scale=2.0, stream=st))
    for b in bufs:
        assert torch.equal(b, want)
    for c in comms:
        st = c.stats()
        assert st["calls"][4] == n + 1 and st["calls"][5] == n          # broadcast, reduce counters (b200collOp_t order)


@pytest.mark.parametrize("group", [2], indirect=True)
def test_rooted_ops_outside_the_arena_are_staged(torch_cuda, group):
    torch = torch_cuda
    comms, streams = group
    count = (1 << 20) + 24
    srcs = [(((torch.arange(count, device="cuda") * (r + 2)) % 9) - 4).to(torch.bfloat16) for r in range(len(comms))]
    dsts = [torch.full((count,), 9.0, dtype=torch.bfloat16, device="cuda") for _ in comms]
    run_all(torch, comms, streams, lambda r, c, st: c.broadcast(srcs[r], dsts[r], root=1, stream=st))
    for d in dsts:
        assert torch.equal(d, srcs[1])
    red = [torch.full((count,), 9.0, dtype=torch.bfloat16, device="cuda") for _ in comms]
    run_all(torch, comms, streams, lambda r, c, st: c.reduce(srcs[r], red[r], root=0, stream=st))
    assert torch.equal(red[0].float(), sum(s.float() for s in srcs)) and torch.equal(red[1], torch.full_like(red[1], 9.0))
    assert all(c.stats()["staged_calls"] == 2 for c in comms)


@pytest.mark.parametrize("group", [4], indirect=True)
def test_all_to_all_v_expert_dispatch(torch_cuda, group):
    """Skewed per-peer row counts (MoE dispatch shape): rows land at the offsets the receiver advertised."""
    torch = torch_cuda
    comms, streams = group
    n, hidden = len(comms), 256
    rows = [[(3 * s + 5 * d) % 7 for d in range(n)] for s in range(n)]                 # rows[s][d]: s -> d
    send = []
    cap = max(max(sum(rows[s]) for s in range(n)), max(sum(rows[s][d] for s in range(n)) for d in range(n))) + 1
    for s, c in enumerate(comms):
        t = c.empty(cap * hidden, torch.bfloat16)            # symmetric allocation: same size, same order on every rank
        t.copy_(((torch.arange(t.numel(), device="cuda") + 100 * s) % 251).to(torch.bfloat16))
        send.append(t)
    recv = [c.empty(cap * hidden, torch.bfloat16) for c in comms]
    for t in recv:
        t.zero_()
    torch.cuda.synchronize()
    send_off = [[sum(rows[s][:d]) for d in range(n)] for s in range(n)]
    recv_off = [[sum(rows[x][d] for x in range(s)) for s in range(n)] for d in range(n)]  # recv_off[d][s]: where s's rows start at d
    run_all(torch, comms, streams, lambda r, c, st: c.all_to_all_v(send[r], recv[r], hidden, rows[r], send_off[r], [recv_off[d][r] for d in range(n)], stream=st))
    for d in range(n):
        for s in range(n):
            got = recv[d][recv_off[d][s] * hidden:(recv_off[d][s] + rows[s][d]) * hidden]
            want = send[s][send_off[s][d] * hidden:(send_off[s][d] + rows[s][d]) * hidden]
            assert torch.equal(got, want), (s, d)


@pytest.mark.parametrize("group", [2], indirect=True)
def test_buffers_outside_the_arena_are_staged(torch_cuda, group):
    torch = torch_cuda
    comms, streams = group
    count = 1 << 20                                             # 2 MiB > LL limit: must take the staging path
    srcs = [(((torch.arange(count, device="cuda") * (r + 2)) % 9) - 4).to(torch.bfloat16) for r in range(len(comms))]
    dsts = [torch.empty(count, dtype=torch.bfloat16, device="cuda") for _ in comms]
    run_all(torch, comms, streams, lambda r, c, st: c.all_reduce(srcs[r], dsts[r], stream=st))
    want = sum(s.float() for s in srcs)
    for d in dsts:
        assert torch.equal(d.float(), want)
    assert all(c.stats()["staged_calls"] == 1 for c in comms)


@pytest.mark.parametrize("group", [2], indirect=True)
def test_cuda_graph_replay(torch_cuda, group):
    """Epochs and Lamport phases live in device memory, so a captured collective replays correctly."""
    torch = torch_cuda
    comms, streams = group
    count = 2048
    srcs = fill(torch, comms, count, torch.bfloat16)
    dsts = [c.empty(count, torch.bfloat16) for c in comms]
    graphs = []
    for algo in ("ll", "ll2", "twoshot"):
        for c in comms:
            c.set_algo(algo)
        graphs = []
        for r, c in enumerate(comms):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=streams[r]):
                c.all_reduce(srcs[r], dsts[r], stream=streams[r])
            graphs.append(g)
        for it in range(5):
            for r in range(len(comms)):
                srcs[r].add_(1.0)
            torch.cuda.synchronize()
            want = sum(s.float() for s in srcs)
            for r, g in enumerate(graphs):
                with torch.cuda.stream(streams[r]):
                    g.replay()
            torch.cuda.synchronize()
            for d in dsts:
                assert torch.equal(d.float(), want), (algo, it)


def test_watchdog_reports_instead_of_hanging(torch_cuda, coll_mod):
    """Only one of two ranks launches: its spin must time out, record a fault and return (SURVEY §5.3)."""
    torch = torch_cuda
    comms = coll_mod.Comm.init_all([0, 0], arena_mb=32, timeout_ms=300)
    src = comms[0].empty(1024, torch.bfloat16); src.fill_(1.0)
    comms[0].set_algo("twoshot")
    comms[0].all_reduce(src)
    torch.cuda.synchronize()
    with pytest.raises(coll_mod.B200CollError, match="watchdog"):
        comms[0].check_async_error()
    with pytest.raises(coll_mod.B200CollError):
        comms[0].all_reduce(src)                  # poisoned communicator refuses further work
    for c in comms:
        c.destroy()


def test_perf_tool_virtual_ranks_zero_errors(torch_cuda, coll_lib):
    assert os.path.exists(PERF), "build/b200coll_perf missing (python -c 'import __graft_entry__ as g; g.build()')"
    for op in ("all_reduce", "all_gather", "reduce_scatter", "alltoall", "broadcast", "reduce"):
        r = subprocess.run([PERF, "--devs", "0,0,0,0", "--op", op, "-b", "1K", "-e", "1M", "-f", "4", "--iters", "3", "--warmup", "1"], capture_output=True, text=True, timeout=120,
                           env={**os.environ, "B200COLL_TIMEOUT_MS": "5000"})
        assert r.returncode == 0, r.stdout + r.stderr
        assert "errors=0" in r.stdout


def test_nccl_tests_names_and_launcher_rank_mode(torch_cuda, coll_lib):
    """`all_reduce_perf -b .. -e .. -g 1 -w .. -n .. -c 1` as the reference's pods invoke nccl-tests: the op comes from argv[0], and
    with a launcher's rank variables in the environment (torchrun's here; OpenMPI's / PMI's are read the same way) each process is
    one rank of the job. Two ranks share cuda:0 when the box has a single GPU."""
    exe = os.path.join(ROOT, "build", "all_reduce_perf")
    assert os.path.islink(exe), "build/all_reduce_perf symlink missing (make -C coll)"
    ngpu = torch_cuda.cuda.device_count()
    base = {**os.environ, "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(20000 + os.getpid() % 20000), "B200COLL_TIMEOUT_MS": "5000"}
    procs = [subprocess.Popen([exe, "-b", "1K", "-e", "1M", "-f", "4", "-g", "1", "-w", "1", "-n", "3", "-c", "1", "-d", "bfloat16", "-o", "sum"],
                              env={**base, "RANK": str(r), "LOCAL_RANK": str(r % ngpu)}, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "# Avg bus bandwidth" in outs[0][0] and "# Out of bounds values : 0 OK" in outs[0][0] and "op=all_reduce nranks=2" in outs[0][0]
    assert outs[1][0] == ""                                  # only rank 0 prints the table
    r = subprocess.run([os.path.join(ROOT, "build", "broadcast_perf"), "-g", "2", "-b", "4K", "-e", "64K", "-f", "4", "-n", "2", "-w", "1"], capture_output=True, text=True, timeout=120,
                       env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
    assert r.returncode == 0 and "op=broadcast nranks=2" in r.stdout and "FAILED" not in r.stdout, r.stdout + r.stderr


def test_multi_gpu_procs_nvls(torch_cuda, coll_lib):
    n = torch_cuda.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    devs = ",".join(str(i) for i in range(n))
    for algo in ("auto", "nvls", "twoshot"):
        r = subprocess.run([PERF, "--devs", devs, "--procs", "--op", "all_reduce", "--algo", algo, "-b", "1K", "-e", "64M", "-f", "16", "--iters", "3", "--warmup", "1"],
                           capture_output=True, text=True, timeout=180, env={**os.environ, "B200COLL_TIMEOUT_MS": "5000"})
        assert r.returncode == 0 and "errors=0" in r.stdout, r.stdout + r.stderr
    for op in ("all_gather", "alltoall", "broadcast"):     # one process driving every GPU (threads): the copy-engine kernel's shared-memory opt-in is per device
        r = subprocess.run([PERF, "--devs", devs, "--op", op, "-b", "4M", "-e", "64M", "-f", "16", "--iters", "2", "--warmup", "1"],
                           capture_output=True, text=True, timeout=180, env={**os.environ, "B200COLL_TIMEOUT_MS": "5000"})
        assert r.returncode == 0 and "errors=0" in r.stdout, r.stdout + r.stderr
    for op in ("broadcast", "reduce"):                     # multimem.st fan-out / multimem.ld_reduce by the root (N >= 3) or P2P (N == 2)
        r = subprocess.run([PERF, "--devs", devs, "--procs", "--op", op, "-b", "1K", "-e", "64M", "-f", "16", "--iters", "3", "--warmup", "1"],
                           capture_output=True, text=True, timeout=180, env={**os.environ, "B200COLL_TIMEOUT_MS": "5000"})
        assert r.returncode == 0 and "errors=0" in r.stdout, r.stdout + r.stderr


def test_bench_contract_one_gpu(torch_cuda, tmp_path):
    import json
    import numpy as np
    dump = tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--max", "16M", "--dump-outputs", str(dump)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(line) == 1
    d = json.loads(line[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches"):
        assert k in d
    assert d["n_gpus"] == 1 and d["gpu_launches"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0
    assert d["e2e"]["d2h_bytes_per_step"] == d["e2e"]["h2d_bytes_per_step"]          # the whole result comes back, not a sample of it
    assert d["verified_vs_torch_fp32"] is True and d["e2e"]["verified_vs_torch_fp32"] is True
    assert len(d["e2e"]["table"]) == len(d["table"]) and all(r["e2e_us"] > 0 for r in d["e2e"]["table"])      # per-size end-to-end rows are published
    assert d["impl"] == "ours" and d["backend"].startswith("libb200coll") and "backend" not in d["config"]   # config is identical on both arms
    assert d["steps"] == 3 and d["e2e"]["steps"] == 3                                  # --steps sets the timed steps of both sweeps
    arrays = {p.stem: np.load(p) for p in dump.glob("*.npy")}
    assert set(arrays) == {f"all_reduce_{k}_{1024 << i:010d}B" for k in ("oop", "e2e") for i in range(15)}    # 1K..16M, one rank: no in-place pass
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values()) and sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert all((a == 0.25).all() for k, a in arrays.items() if "_e2e_" in k)              # host input 0.25 everywhere, one rank: the sum is the input
    elems = {k: int(k.split("_")[-1][:-1]) // 2 for k in arrays}
    sample = max(a.size for a in arrays.values())
    assert sample < elems["all_reduce_oop_0016777216B"] and all(a.size == min(elems[k], sample) for k, a in arrays.items())   # small outputs whole, large ones sampled



@pytest.mark.parametrize("group", [2], indirect=True)
def test_all_reduce_from_host_pipelines_copy_and_collective(torch_cuda, group):
    torch = torch_cuda
    comms, streams = group
    count = (5 << 20) + 1024                                     # several 4 MiB chunks and a ragged tail
    hosts = [(((torch.arange(count) * (r + 2)) % 11) - 5).to(torch.bfloat16).pin_memory() for r in range(len(comms))]
    outs = [c.empty(count, torch.bfloat16) for c in comms]
    for rep in range(3):                                         # staging buffers are reused across calls
        for r, c in enumerate(comms):
            with torch.cuda.stream(streams[r]):
                c.all_reduce_from_host(hosts[r], outs[r], chunk_bytes=4 << 20)
        torch.cuda.synchronize()
        want = sum(h.float() for h in hosts).cuda()
        for o in outs:
            assert torch.equal(o.float(), want)
    for c in comms:
        c.check_async_error()


@pytest.mark.parametrize("group", [2], indirect=True)
def test_all_reduce_host_zero_copy_single_chunk_and_pipeline(torch_cuda, group, monkeypatch):
    """b200collAllReduceHost (coll/src/hostpath.cu): pinned host in, pinned host out, one call. Three regimes — a single kernel that
    reads and writes host memory over PCIe, copy/all-reduce/copy on the caller's stream, and the chunked three-leg pipeline (ragged last
    chunk, staging rings reused and regrown across calls) — against an fp32 reference on data whose sums are not exact in bf16."""
    torch = torch_cuda
    from container_engine_accelerators_b200.parallel import harness
    comms, streams = group
    n = len(comms)
    gen = harness._gen_expected(torch, "all_reduce", 0, n, 0, "cpu")
    for count in (1 << 12, (1 << 18) + 8, (1 << 19) + 24, (5 << 20) + 13, (9 << 20) + 5):      # one-shot / two-shot Lamport zero-copy, one chunk, 3 and 5 chunks with a ragged tail
        idx = torch.arange(count)
        ins = [gen(r, idx).to(torch.bfloat16) for r in range(n)]
        h_in = [comms[0].host_empty(count, torch.bfloat16), torch.empty(count, dtype=torch.bfloat16).pin_memory()]      # the library's NUMA-placed memory and plain torch pinned memory
        h_out = [torch.empty(count, dtype=torch.bfloat16).pin_memory(), comms[1].host_empty(count, torch.bfloat16)]
        for r in range(n):
            h_in[r].copy_(ins[r]); h_out[r].fill_(77.0)
        for rep in range(2):
            for r, c in enumerate(comms):
                c.all_reduce_host(h_in[r], h_out[r], stream=streams[r])
            torch.cuda.synchronize()
            want = sum(x.float() for x in ins)
            for r in range(n):
                assert harness.reduction_ok(torch, h_out[r].float(), want, torch.bfloat16, n), (count, rep, r)
        comms[0].host_release(h_in[0]); comms[1].host_release(h_out[1])
    st = comms[0].stats()
    assert st["host_calls"] == 10 and st["host_zero_copy"] == 4 and st["host_pipelined"] == 4, st
    for c in comms:
        c.check_async_error()
    node, cpus = comms[0].numa()
    assert node >= -1 and isinstance(cpus, str)


def test_all_reduce_host_one_rank_fused_epilogue(torch_cuda, coll_mod):
    """One rank: the host step is copy-in | fused scale/cast kernel | copy-back; bf16 in, fp32 out, scale 0.5, in the pipelined regime."""
    torch = torch_cuda
    (c,) = coll_mod.Comm.init_all([0], arena_mb=64)
    count = (6 << 20) + 5
    h_in = c.host_empty(count, torch.bfloat16)
    h_in.copy_(((torch.arange(count) % 251) - 125).to(torch.bfloat16))
    h_out = c.host_empty(count, torch.float32)
    c.all_reduce_host(h_in, h_out, scale=0.5)
    torch.cuda.synchronize()
    assert torch.equal(h_out, h_in.float() * 0.5)
    tiny_in, tiny_out = h_in[:1000], h_out[:1000]
    tiny_out.zero_()
    c.all_reduce_host(tiny_in, tiny_out, scale=2.0)                # zero-copy regime: the copy kernel reads and writes host memory
    torch.cuda.synchronize()
    assert torch.equal(tiny_out, tiny_in.float() * 2.0)
    assert c.stats()["host_zero_copy"] == 1 and c.stats()["host_pipelined"] == 1
    c.destroy()


# ------------------------------------------------------------------------------------------------- NCCL-API shim
class _NcclShim:
    """ctypes view of libb200coll_nccl.so with NCCL's own prototypes (what an nccl-tests binary would call)."""
    F32, F16, BF16, U8, I64 = 7, 6, 9, 1, 4
    SUM, AVG = 0, 4

    def __init__(self):
        import ctypes as C
        self.C = C
        self.L = L = C.CDLL(os.path.join(ROOT, "coll", "lib", "libb200coll_nccl.so"))
        vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
        L.ncclGetErrorString.restype = C.c_char_p
        L.ncclCommInitAll.argtypes = [C.POINTER(vp), ci, C.POINTER(ci)]
        L.ncclCommDestroy.argtypes = [vp]
        L.ncclAllReduce.argtypes = [vp, vp, sz, ci, ci, vp, vp]
        L.ncclAllGather.argtypes = [vp, vp, sz, ci, vp, vp]
        L.ncclReduceScatter.argtypes = [vp, vp, sz, ci, ci, vp, vp]
        L.ncclBroadcast.argtypes = [vp, vp, sz, ci, ci, vp, vp]
        L.ncclReduce.argtypes = [vp, vp, sz, ci, ci, ci, vp, vp]
        L.ncclSend.argtypes = [vp, sz, ci, ci, vp, vp]
        L.ncclRecv.argtypes = [vp, sz, ci, ci, vp, vp]
        L.ncclAlltoAll.argtypes = [vp, vp, sz, ci, vp, vp]
        L.ncclGather.argtypes = [vp, vp, sz, ci, ci, vp, vp]
        L.ncclScatter.argtypes = [vp, vp, sz, ci, ci, vp, vp]
        L.ncclRedOpCreatePreMulSum.argtypes = [C.POINTER(ci), vp, ci, ci, vp]
        L.ncclRedOpDestroy.argtypes = [ci, vp]
        L.ncclCommCount.argtypes = [vp, C.POINTER(ci)]
        L.ncclCommUserRank.argtypes = [vp, C.POINTER(ci)]
        L.ncclCommGetAsyncError.argtypes = [vp, C.POINTER(ci)]

    def ck(self, rc):
        assert rc == 0, self.L.ncclGetErrorString(rc).decode()


def test_nccl_api_shim_collectives(torch_cuda, coll_lib):
    """An NCCL-API program (plain cudaMalloc buffers, NCCL dtypes/ops/handles) running on libb200coll through the shim."""
    torch = torch_cuda
    s = _NcclShim()
    C, L, n = s.C, s.L, 2
    comms = (C.c_void_p * n)()
    s.ck(L.ncclCommInitAll(comms, n, (C.c_int * n)(0, 0)))
    try:
        cnt, rk, ver = C.c_int(), C.c_int(), C.c_int()
        s.ck(L.ncclCommCount(comms[1], C.byref(cnt))); s.ck(L.ncclCommUserRank(comms[1], C.byref(rk))); s.ck(L.ncclGetVersion(C.byref(ver)))
        assert (cnt.value, rk.value) == (2, 1) and ver.value >= 22000
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

        for count in (1000, 3 << 19):                                           # Lamport path, then staged (3 MiB of bf16 > 512 KiB)
            src = [(((torch.arange(count, device="cuda") * (r + 3)) % 13) - 6).to(torch.bfloat16) for r in range(n)]
            dst = [torch.empty(count, dtype=torch.bfloat16, device="cuda") for _ in range(n)]
            every(lambda r: L.ncclAllReduce(p(src[r]), p(dst[r]), count, s.BF16, s.SUM, comms[r], st[r]))
            want = sum(t.float() for t in src)
            assert all(torch.equal(d.float(), want) for d in dst)
        # ncclAvg and a pre-multiplied sum (host scalar 0.25, fp32)
        src = [torch.full((4096,), float(r + 1), device="cuda") for r in range(n)]
        dst = [torch.empty(4096, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclAllReduce(p(src[r]), p(dst[r]), 4096, s.F32, s.AVG, comms[r], st[r]))
        assert all(torch.equal(d, torch.full_like(d, 1.5)) for d in dst)
        op, scalar = C.c_int(), C.c_float(0.25)
        s.ck(L.ncclRedOpCreatePreMulSum(C.byref(op), C.byref(scalar), s.F32, 1, comms[0]))
        assert op.value >= 5
        every(lambda r: L.ncclAllReduce(p(src[r]), p(dst[r]), 4096, s.F32, op.value, comms[r], st[r]))
        assert all(torch.equal(d, torch.full_like(d, 0.75)) for d in dst)
        s.ck(L.ncclRedOpDestroy(op.value, comms[0]))
        assert L.ncclAllReduce(p(src[0]), p(dst[0]), 4096, s.F32, op.value, comms[0], st[0]) != 0          # stale handle is refused
        # the rest of ncclRedOp_t x ncclDataType_t (generic P2P kernel): what PyTorch's int64 all-reduces and `all_reduce_perf -o max -d int32` send
        I32, U8, F64, MAX, MIN, PROD = 2, 1, 8, 2, 3, 1
        for count in (1003, (3 << 18) + 5):                                     # staged through the arena (plain cudaMalloc buffers), scalar tail
            i32 = [((torch.arange(count, device="cuda") * (7 * r + 3)) % 2001 - 1000).to(torch.int32) for r in range(n)]
            o32 = [torch.empty(count, dtype=torch.int32, device="cuda") for _ in range(n)]
            every(lambda r: L.ncclAllReduce(p(i32[r]), p(o32[r]), count, I32, MAX, comms[r], st[r]))
            assert all(torch.equal(o, torch.maximum(i32[0], i32[1])) for o in o32)
            i64 = [(torch.arange(count, device="cuda", dtype=torch.int64) * (r + 1) << 33) - 5 for r in range(n)]
            every(lambda r: L.ncclAllReduce(p(i64[r]), p(i64[r]), count, s.I64, s.SUM, comms[r], st[r]))      # in place, values beyond 2^32
            assert all(torch.equal(t, (torch.arange(count, device="cuda", dtype=torch.int64) * 3 << 33) - 10) for t in i64)
        u8 = [((torch.arange(4096, device="cuda") * (r + 5)) % 251).to(torch.uint8) for r in range(n)]
        o8 = [torch.empty(4096, dtype=torch.uint8, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclAllReduce(p(u8[r]), p(o8[r]), 4096, U8, MIN, comms[r], st[r]))
        assert all(torch.equal(o, torch.minimum(u8[0], u8[1])) for o in o8)
        f64 = [torch.linspace(0.5, 2.0, 2048, device="cuda", dtype=torch.float64) * (r + 1) for r in range(n)]
        o64 = [torch.empty(2048, dtype=torch.float64, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclAllReduce(p(f64[r]), p(o64[r]), 2048, F64, PROD, comms[r], st[r]))
        assert all(torch.equal(o, f64[0] * f64[1]) for o in o64)
        bmax = [torch.empty(1000, dtype=torch.bfloat16, device="cuda") for _ in range(n)]
        bsrc = [(((torch.arange(1000, device="cuda") * (r + 3)) % 13) - 6).to(torch.bfloat16) for r in range(n)]
        every(lambda r: L.ncclAllReduce(p(bsrc[r]), p(bmax[r]), 1000, s.BF16, MAX, comms[r], st[r]))
        assert all(torch.equal(o, torch.maximum(bsrc[0], bsrc[1])) for o in bmax)
        rs32 = [torch.empty(512, dtype=torch.int32, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclReduceScatter(p(i32[r]), p(rs32[r]), 512, I32, s.SUM, comms[r], st[r]))
        assert all(torch.equal(rs32[r], (i32[0] + i32[1])[r * 512:(r + 1) * 512]) for r in range(n))
        rd32 = [torch.full((1003,), -9, dtype=torch.int32, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclReduce(p(i32[r]), p(rd32[r]), 1003, I32, MIN, 1, comms[r], st[r]))
        assert torch.equal(rd32[1], torch.minimum(i32[0], i32[1])[:1003]) and bool((rd32[0] == -9).all())
        assert L.ncclAllReduce(p(i32[0]), p(o32[0]), 8, I32, s.AVG, comms[0], st[0]) != 0                    # avg: floating point only
        # all-gather / reduce-scatter
        part = [torch.arange(2048, device="cuda", dtype=torch.float16) + 2048 * r for r in range(n)]
        full = [torch.empty(2048 * n, dtype=torch.float16, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclAllGather(p(part[r]), p(full[r]), 2048, s.F16, comms[r], st[r]))
        assert all(torch.equal(f, torch.cat(part)) for f in full)
        rs = [torch.empty(2048, dtype=torch.float16, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclReduceScatter(p(full[r]), p(rs[r]), 2048, s.F16, s.SUM, comms[r], st[r]))
        assert all(torch.equal(rs[r], (full[0].float() * n)[r * 2048:(r + 1) * 2048].half()) for r in range(n))
        # broadcast moves bits for any dtype (int64 here, odd byte count refused for uint8), reduce lands on the root only
        ints = [torch.arange(1001, device="cuda", dtype=torch.int64) * (r + 1) - 7 for r in range(n)]
        every(lambda r: L.ncclBroadcast(p(ints[r]), p(ints[r]), 1001, s.I64, 1, comms[r], st[r]))
        assert torch.equal(ints[0], ints[1]) and ints[0][1000].item() == 1000 * 2 - 7
        assert L.ncclBroadcast(p(ints[0]), p(ints[0]), 3, s.U8, 0, comms[0], st[0]) != 0
        red = [torch.full((4096,), -1.0, device="cuda") for _ in range(n)]
        every(lambda r: L.ncclReduce(p(src[r]), p(red[r]) if r == 0 else None, 4096, s.F32, s.SUM, 0, comms[r], st[r]))
        assert torch.equal(red[0], torch.full_like(red[0], 3.0)) and torch.equal(red[1], torch.full_like(red[1], -1.0))
        # nccl-tests' alltoall: grouped send/recv to every peer
        a2a_in = [torch.arange(n * 512, device="cuda", dtype=torch.float32) + 10000 * r for r in range(n)]
        a2a_out = [torch.empty(n * 512, device="cuda") for _ in range(n)]

        def grouped(r):
            s.ck(L.ncclGroupStart())
            for peer in range(n):
                s.ck(L.ncclSend(C.c_void_p(a2a_in[r].data_ptr() + peer * 512 * 4), 512, s.F32, peer, comms[r], st[r]))
                s.ck(L.ncclRecv(C.c_void_p(a2a_out[r].data_ptr() + peer * 512 * 4), 512, s.F32, peer, comms[r], st[r]))
            return L.ncclGroupEnd()
        every(grouped)
        for r in range(n):
            assert torch.equal(a2a_out[r], torch.cat([a2a_in[q][r * 512:(r + 1) * 512] for q in range(n)]))
    finally:
        torch.cuda.synchronize()
        for c in comms:
            L.ncclCommDestroy(c)


def test_unmodified_nccl_program_runs_on_the_shim(torch_cuda, coll_lib):
    """coll/tests/nccl_client.c includes the SYSTEM's <nccl.h> and speaks only the NCCL C API (ncclCommInitAll, grouped per-device
    calls like nccl-tests in one-process mode): int32 max / sum, int64 sum, uint8 min, float sum / prod, double max, broadcast,
    all-gather, a send/recv ring. Linked against libb200coll_nccl.so it must pass its own host-side checks (the drop-in claim of the
    transport installer, reference: gpudirect-tcpx/nccl-config.yaml:22,61 — the benchmark binary is whatever NCCL program the pod runs)."""
    client = os.path.join(ROOT, "build", "nccl_client")
    if not os.path.exists(client):
        pytest.skip("build/nccl_client not built (no system nccl.h)")
    n = torch_cuda.cuda.device_count()
    args = [client, "2"] if n >= 2 else [client, "2", "--same-device"]
    r = subprocess.run(args, capture_output=True, text=True, timeout=180, env={**os.environ, "B200COLL_TIMEOUT_MS": "8000", "B200COLL_ARENA_MB": "256"})
    assert r.returncode == 0 and "all checks passed" in r.stdout and "WRONG" not in r.stdout, r.stdout + r.stderr
    assert r.stdout.count(" ok") >= 10


# ------------------------------------------------------------------------------------------------- point to point


def _pattern(torch, nbytes, seed):
    return ((torch.arange(nbytes, device="cuda", dtype=torch.int64) * (2 * seed + 7) + seed * 31) % 251).to(torch.uint8)


@pytest.mark.parametrize("group", [2, 4], indirect=True)
@pytest.mark.parametrize("nbytes", [16, 1003, (1 << 20) + 48, (3 << 20) + 5])
@pytest.mark.parametrize("arena_recv", [True, False])
def test_send_recv_ring_step(torch_cuda, coll_mod, group, nbytes, arena_recv):
    """Grouped send to the right / recv from the left (nccl-tests sendrecv): bytes arrive untouched, for sizes that are not a multiple
    of a vector, in place in the arena or through staging windows smaller than the message; repeated so sequence numbers advance."""
    torch = torch_cuda
    comms, streams = group
    n = len(comms)
    for c in comms:
        c.set_p2p_window(1 << 20)                   # 3 MiB + 5 B through 1 MiB windows: four chunks, both windows reused
    srcs = [c.empty(nbytes, torch.uint8) for c in comms]
    dsts = [c.empty(nbytes, torch.uint8) if arena_recv else torch.empty(nbytes, dtype=torch.uint8, device="cuda") for c in comms]
    for rep in range(3):
        for r in range(n):
            srcs[r].copy_(_pattern(torch, nbytes, r + 10 * rep))
            dsts[r].fill_(0xEE)
        torch.cuda.synchronize()
        with coll_mod.group():
            for r, c in enumerate(comms):
                c.send(srcs[r], (r + 1) % n, stream=streams[r])
                c.recv(dsts[r], (r - 1) % n, stream=streams[r])
        torch.cuda.synchronize()
        for r, c in enumerate(comms):
            c.check_async_error()
            assert torch.equal(dsts[r], srcs[(r - 1) % n]), (rep, r)
    st = comms[0].stats()
    assert st["p2p_sends"] == 3 and st["p2p_recvs"] == 3 and st["p2p_bytes"] == 6 * nbytes
    assert (st["staged_calls"] > 0) == (not arena_recv)


@pytest.mark.parametrize("group", [2], indirect=True)
def test_send_recv_pipeline_handover_and_self(torch_cuda, coll_mod, group):
    """Ungrouped calls: rank 0 sends, rank 1 receives (each blocks its own stream until the other arrives); then the reverse direction
    with another size; send/recv to self inside a group is a local copy."""
    torch = torch_cuda
    comms, streams = group
    a = comms[0].empty(1 << 16, torch.float32); a.copy_(torch.arange(1 << 16, device="cuda", dtype=torch.float32))
    b = comms[1].empty(1 << 16, torch.float32); b.zero_()
    comms[0].send(a, 1, stream=streams[0])
    comms[1].recv(b, 0, stream=streams[1])
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    back = torch.empty(100, dtype=torch.bfloat16, device="cuda")            # 200 bytes, not in the arena
    comms[1].send(b[:50].view(torch.bfloat16), 0, stream=streams[1])
    comms[0].recv(back, 1, stream=streams[0])
    torch.cuda.synchronize()
    assert torch.equal(back.view(torch.float32), a[:50])
    mine = torch.empty(1 << 10, dtype=torch.float32, device="cuda")
    with coll_mod.group():
        comms[0].send(a[:1 << 10], 0, stream=streams[0])
        comms[0].recv(mine, 0, stream=streams[0])
    torch.cuda.synchronize()
    assert torch.equal(mine, a[:1 << 10])
    for c in comms:
        c.check_async_error()


@pytest.mark.parametrize("group", [4], indirect=True)
def test_send_recv_irregular_group_and_graph_replay(torch_cuda, coll_mod, group):
    """One group with different sizes per pair and two messages for one pair (second one runs in a follow-up kernel); then a captured
    ring step replayed five times."""
    torch = torch_cuda
    comms, streams = group
    n = len(comms)
    size = lambda s, d: 4096 * (1 + s) + 16 * d
    out = {(s, d): comms[s].empty(size(s, d), torch.uint8) for s in range(n) for d in range(n) if s != d}
    inn = {(s, d): comms[d].empty(size(s, d), torch.uint8) for s in range(n) for d in range(n) if s != d}
    for (s, d), t in out.items():
        t.copy_(_pattern(torch, t.numel(), 17 * s + d))
    extra_out = comms[0].empty(777, torch.uint8); extra_out.copy_(_pattern(torch, 777, 99))
    extra_in = torch.zeros(777, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    with coll_mod.group():
        for r, c in enumerate(comms):
            for p in range(n):
                if p != r:
                    c.send(out[(r, p)], p, stream=streams[r])
                    c.recv(inn[(p, r)], p, stream=streams[r])
        comms[0].send(extra_out, 1, stream=streams[0])                      # a second message 0 -> 1 in the same group
        comms[1].recv(extra_in, 0, stream=streams[1])
    torch.cuda.synchronize()
    for k in out:
        assert torch.equal(out[k], inn[k]), k
    assert torch.equal(extra_in, extra_out)
    # graph replay: sequence numbers live in device memory
    count = 1 << 14
    srcs = [c.empty(count, torch.float32) for c in comms]
    dsts = [c.empty(count, torch.float32) for c in comms]
    graphs = []
    for r, c in enumerate(comms):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=streams[r]):
            with coll_mod.group():
                c.send(srcs[r], (r + 1) % n, stream=streams[r])
                c.recv(dsts[r], (r - 1) % n, stream=streams[r])
        graphs.append(g)
    for it in range(5):
        for r in range(n):
            srcs[r].fill_(float(10 * it + r))
        torch.cuda.synchronize()
        for r, g in enumerate(graphs):
            with torch.cuda.stream(streams[r]):
                g.replay()
        torch.cuda.synchronize()
        for r in range(n):
            assert torch.equal(dsts[r], srcs[(r - 1) % n]), (it, r)
    for c in comms:
        c.check_async_error()


def test_send_without_a_receiver_times_out(torch_cuda, coll_mod):
    torch = torch_cuda
    comms = coll_mod.Comm.init_all([0, 0], arena_mb=32, timeout_ms=300)
    src = comms[0].empty(1024, torch.bfloat16); src.fill_(1.0)
    comms[0].send(src, 1)
    torch.cuda.synchronize()
    with pytest.raises(coll_mod.B200CollError, match="code=3"):
        comms[0].check_async_error()
    for c in comms:
        c.destroy()


def test_sendrecv_perf_virtual_ranks_zero_errors(torch_cuda, coll_lib):
    for op in ("sendrecv", "gather", "scatter", "hypercube"):                      # nccl-tests names; all of them are groups of send / recv
        exe = os.path.join(ROOT, "build", f"{op}_perf")
        assert os.path.islink(exe)
        r = subprocess.run([exe, "--devs", "0,0,0,0", "-b", "64", "-e", "4M", "-f", "4", "-w", "2", "-n", "5", "-c", "1"], capture_output=True, text=True, timeout=300,
                           env={**{k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}, "B200COLL_TIMEOUT_MS": "5000"})
        assert r.returncode == 0, r.stdout + r.stderr
        assert f"op={op}" in r.stdout and "# Out of bounds values : 0 OK" in r.stdout, r.stdout


def test_nccl_api_shim_send_recv(torch_cuda, coll_lib):
    """ncclSend / ncclRecv through the shim for shapes that are not the all-to-all pattern: a lone pair outside any group (uint8, odd
    count) and a grouped exchange of int64 with different counts per direction, issued for both communicators inside one group."""
    torch = torch_cuda
    s = _NcclShim()
    C, L, n = s.C, s.L, 2
    comms = (C.c_void_p * n)()
    s.ck(L.ncclCommInitAll(comms, n, (C.c_int * n)(0, 0)))
    try:
        streams = [torch.cuda.Stream() for _ in range(n)]
        st = [C.c_void_p(x.cuda_stream) for x in streams]
        p = lambda t: C.c_void_p(t.data_ptr())
        a = _pattern(torch, 1001, 3)
        b = torch.zeros(1001, dtype=torch.uint8, device="cuda")
        s.ck(L.ncclSend(p(a), 1001, s.U8, 1, comms[0], st[0]))
        s.ck(L.ncclRecv(p(b), 1001, s.U8, 0, comms[1], st[1]))
        torch.cuda.synchronize()
        assert torch.equal(a, b)
        x01 = torch.arange(300, device="cuda", dtype=torch.int64) * 3 - 1
        x10 = torch.arange(5000, device="cuda", dtype=torch.int64) * -7
        y01 = torch.zeros(300, dtype=torch.int64, device="cuda")
        y10 = torch.zeros(5000, dtype=torch.int64, device="cuda")
        s.ck(L.ncclGroupStart())
        s.ck(L.ncclSend(p(x01), 300, s.I64, 1, comms[0], st[0])); s.ck(L.ncclRecv(p(y10), 5000, s.I64, 1, comms[0], st[0]))
        s.ck(L.ncclSend(p(x10), 5000, s.I64, 0, comms[1], st[1])); s.ck(L.ncclRecv(p(y01), 300, s.I64, 0, comms[1], st[1]))
        s.ck(L.ncclGroupEnd())
        torch.cuda.synchronize()
        assert torch.equal(x01, y01) and torch.equal(x10, y10)
        # integer all-gather: words on the bit-exact kernels (an int64 -1 must survive; small enough that floats would take the Lamport path)
        part = [torch.full((1000,), -1, device="cuda", dtype=torch.int64) for _ in range(n)]
        for r in range(n):
            part[r][::3] = r + 5
        full = [torch.zeros(1000 * n, dtype=torch.int64, device="cuda") for _ in range(n)]
        for r in range(n):
            s.ck(L.ncclAllGather(p(part[r]), p(full[r]), 1000, s.I64, comms[r], st[r]))
        torch.cuda.synchronize()
        assert all(torch.equal(f, torch.cat(part)) for f in full)
        # NCCL 2.28 host APIs: gather to rank 1, scatter from rank 0 (both inside one group across the two communicators), int64 all-to-all
        gathered = [torch.zeros(1000 * n, dtype=torch.int64, device="cuda") for _ in range(n)]
        s.ck(L.ncclGroupStart())
        for r in range(n):
            s.ck(L.ncclGather(p(part[r]), p(gathered[r]), 1000, s.I64, 1, comms[r], st[r]))
        s.ck(L.ncclGroupEnd())
        torch.cuda.synchronize()
        assert torch.equal(gathered[1], torch.cat(part)) and gathered[0].eq(0).all()
        pieces = [torch.zeros(1000, dtype=torch.int64, device="cuda") for _ in range(n)]
        s.ck(L.ncclGroupStart())
        for r in range(n):
            s.ck(L.ncclScatter(p(gathered[1]) if r == 0 else None, p(pieces[r]), 1000, s.I64, 0, comms[r], st[r]))
        s.ck(L.ncclGroupEnd())
        torch.cuda.synchronize()
        assert all(torch.equal(pieces[r], part[r]) for r in range(n))                             # rank 0 scattered what rank 1 had gathered
        a2a_in = [torch.arange(2048 * n, device="cuda", dtype=torch.int64) * (1 if r == 0 else -1) for r in range(n)]
        a2a_out = [torch.zeros(2048 * n, dtype=torch.int64, device="cuda") for _ in range(n)]
        for r in range(n):
            s.ck(L.ncclAlltoAll(p(a2a_in[r]), p(a2a_out[r]), 2048, s.I64, comms[r], st[r]))
        torch.cuda.synchronize()
        for r in range(n):
            assert torch.equal(a2a_out[r], torch.cat([a2a_in[q][r * 2048:(r + 1) * 2048] for q in range(n)]))
        for r in range(n):
            err = C.c_int(-1)
            s.ck(L.ncclCommGetAsyncError(comms[r], C.byref(err)))
            assert err.value == 0
    finally:
        torch.cuda.synchronize()
        for c in comms:
            L.ncclCommDestroy(c)


# ------------------------------------------------------------------------------------------------- communicator split
def _split_rank(rank, world, key, q):
    try:
        import torch
        from container_engine_accelerators_b200.ops import coll
        torch.cuda.set_device(0)
        comm = coll.Comm.init_rank(rank, world, key, arena_mb=32, timeout_ms=10000)
        pair = comm.split(color=rank // 2, key=-rank, arena_mb=16)               # {0,1} and {2,3}; negative keys reverse the order inside
        assert pair is not None and pair.nranks == 2 and pair.rank == 1 - rank % 2
        x = pair.empty(4096, torch.float32); x.fill_(float(rank + 1))
        pair.all_reduce(x)
        torch.cuda.synchronize()
        want = float((rank // 2) * 4 + 3)                                         # 1+2 or 3+4
        assert torch.equal(x, torch.full_like(x, want)), (rank, x[0].item(), want)
        lone = comm.split(color=0 if rank == 3 else -1)                           # everybody takes part, only rank 3 gets a communicator
        assert (lone is None) == (rank != 3) and (lone is None or lone.nranks == 1)
        y = comm.empty(1024, torch.float32); y.fill_(1.0)
        comm.all_reduce(y)                                                        # the parent still works after two splits
        torch.cuda.synchronize()
        assert torch.equal(y, torch.full_like(y, float(world)))
        for c in (lone, pair, comm):
            if c is not None:
                c.check_async_error(); c.destroy()
        q.put((rank, "ok"))
    except Exception as e:                                                        # noqa: BLE001 - reported to the parent
        import traceback
        q.put((rank, traceback.format_exc() + repr(e)))



def test_comm_split_four_processes(torch_cuda, coll_mod):
    """ncclCommSplit semantics across four processes (sharing cuda:0 on a one-GPU box): colours, key ordering, a rank without a colour,
    and the parent staying usable."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    key = f"split-test-{os.getpid()}"
    procs = [ctx.Process(target=_split_rank, args=(r, 4, key, q)) for r in range(4)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=180) for _ in procs)
    for p in procs:
        p.join(30)
    assert results == {r: "ok" for r in range(4)}, results
