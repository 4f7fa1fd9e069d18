"""libb200coll host-side logic that needs no GPU: tuner table, config/env, unique ids, graceful no-driver paths, and the
Unix-socket rendezvous (SCM_RIGHTS) exercised across real processes with memfd descriptors."""
import ctypes as C
import multiprocessing as mp
import os
import time
import struct
import subprocess

import pytest

from container_engine_accelerators_b200.ops import coll


@pytest.fixture(scope="module")
def lib(coll_lib):
    return coll.load()


def test_version_and_names(lib):
    assert lib.b200collGetVersion() >= 1
    assert [lib.b200collAlgoName(i).decode() for i in range(7)] == coll.ALGO_NAMES
    assert [lib.b200collTypeSize(t) for t in (coll.F32, coll.F16, coll.BF16, coll.FP8_E4M3)] == [4, 2, 2, 1]


@pytest.mark.parametrize("op,nbytes,n,nvls,want", [
    (coll.OP_ALLREDUCE, 1024, 1, True, "copy"),
    (coll.OP_ALLREDUCE, 1024, 8, True, "ll"), (coll.OP_ALLREDUCE, 256 << 10, 8, True, "ll"), (coll.OP_ALLREDUCE, 512 << 10, 8, True, "nvls"), (coll.OP_ALLREDUCE, 512 << 10, 8, False, "ll2"), (coll.OP_ALLREDUCE, 4 << 20, 8, True, "nvls"),
    (coll.OP_ALLREDUCE, 1 << 30, 8, True, "nvls"), (coll.OP_ALLREDUCE, 1 << 30, 8, False, "twoshot"),
    (coll.OP_ALLREDUCE, 1 << 30, 2, True, "twoshot"),            # N=2: NVLS would bounce my own half through the switch
    (coll.OP_ALLGATHER, 4096, 4, True, "ll"), (coll.OP_ALLGATHER, 64 << 20, 8, True, "twoshot"),
    (coll.OP_REDUCESCATTER, 64 << 20, 8, True, "nvls"), (coll.OP_REDUCESCATTER, 64 << 20, 8, False, "twoshot"),
    (coll.OP_ALLTOALL, 1 << 10, 8, True, "ll"), (coll.OP_ALLTOALL, 32 << 20, 8, True, "twoshot"),
])
def test_tuner_table(lib, op, nbytes, n, nvls, want):
    assert coll.tuner_pick(op, nbytes, n, nvls) == want


def test_tuner_file_override(coll_lib, tmp_path):
    import subprocess, sys
    tbl = tmp_path / "t.tbl"
    tbl.write_text("# op nmin nmax nvls max_bytes algo\nall_reduce 2 8 * 1024 oneshot\nall_reduce 2 8 * inf twoshot\n")
    code = "from container_engine_accelerators_b200.ops import coll; print(coll.tuner_pick(0, 512, 8, True), coll.tuner_pick(0, 1<<20, 8, True), coll.tuner_pick(1, 64, 8, True))"
    r = subprocess.run([sys.executable, "-c", code], env={**os.environ, "B200COLL_TUNER_FILE": str(tbl)}, capture_output=True, text=True)
    assert r.stdout.split() == ["oneshot", "twoshot", "ll"], r.stderr


def test_config_defaults_follow_env(lib, monkeypatch):
    monkeypatch.setenv("B200COLL_ARENA_MB", "123"); monkeypatch.setenv("B200COLL_NVLS", "0"); monkeypatch.setenv("B200COLL_TIMEOUT_MS", "777")
    cfg = coll.Comm.make_config()
    assert (cfg.arena_bytes, cfg.enable_nvls, cfg.timeout_ms) == (123 << 20, 0, 777)


def test_unique_id_from_string_is_deterministic(lib):
    a, b, c = coll.UniqueId(), coll.UniqueId(), coll.UniqueId()
    lib.b200collUniqueIdFromString(b"127.0.0.1:29500/x", C.byref(a)); lib.b200collUniqueIdFromString(b"127.0.0.1:29500/x", C.byref(b)); lib.b200collUniqueIdFromString(b"127.0.0.1:29501/x", C.byref(c))
    assert a.internal == b.internal != c.internal
    lib.b200collGetUniqueId(C.byref(a)); lib.b200collGetUniqueId(C.byref(b))
    assert a.internal != b.internal


@pytest.mark.skipif(os.path.exists("/dev/nvidiactl"), reason="GPU box: the no-driver path is not reachable")
def test_no_driver_is_reported_not_crashed(lib):
    ok, report = coll.self_check()
    assert not ok and "driver" in report
    with pytest.raises(coll.B200CollError) as ei:
        coll.Comm.init_all([0], arena_mb=8)
    assert ei.value.code == coll.NO_DRIVER


def _boot_rank(lib_path, name, rank, n, q):
    L = C.CDLL(lib_path)
    fd = os.memfd_create(f"r{rank}")
    os.write(fd, f"payload-from-rank-{rank}".encode())
    out = (C.c_int * n)()
    bc = C.c_int(-1)
    rc = L.b200collBootstrapSelfTest(name.encode(), rank, n, fd, out, C.byref(bc), 20000)
    got = []
    if rc == 0:
        # pread, not lseek+read: descriptors passed with SCM_RIGHTS share one open file description (one offset) across ranks
        for r in range(n):
            got.append(os.pread(out[r], 64, 0).decode())
        got.append(os.pread(bc.value, 64, 0).decode())
    q.put((rank, rc, got))


@pytest.mark.parametrize("n", [2, 5])
def test_bootstrap_fd_exchange_across_processes(coll_lib, n):
    ctx = mp.get_context("fork")
    q = ctx.Queue()
    name = f"pytest-{os.getpid()}-{n}"
    procs = [ctx.Process(target=_boot_rank, args=(coll_lib, name, r, n, q)) for r in range(n)]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=60) for _ in range(n))
    for p in procs:
        p.join(10)
    want = [f"payload-from-rank-{r}" for r in range(n)] + ["payload-from-rank-0"]
    for rank, rc, got in results:
        assert rc == 0 and got == want, (rank, rc, got)


def _boot_rank_env(lib_path, name, rank, n, q, secret, timeout_ms):
    if secret is not None:
        os.environ["B200COLL_RENDEZVOUS_SECRET"] = secret
    L = C.CDLL(lib_path)
    fd = os.memfd_create(f"r{rank}")
    out = (C.c_int * n)()
    bc = C.c_int(-1)
    rc = L.b200collBootstrapSelfTest(name.encode(), rank, n, fd, out, C.byref(bc), timeout_ms)
    q.put((rank, rc, L.b200collBootstrapSelfTestRejected()))


def test_bootstrap_drops_strangers_and_keeps_waiting(coll_lib):
    """The rendezvous name can be guessed by other processes on the host (it is derived from MASTER_ADDR:PORT). A connection that does
    not carry the job's token is dropped — it neither joins (it would receive every rank's arena descriptor) nor aborts the job."""
    import socket
    ctx = mp.get_context("fork")
    q = ctx.Queue()
    name = f"pytest-intruder-{os.getpid()}"
    p0 = ctx.Process(target=_boot_rank_env, args=(coll_lib, name, 0, 2, q, "s3cret", 20000))
    p0.start()
    addr = b"\0b200coll-" + name.encode()
    deadline = time.time() + 10
    while True:                                   # the stranger: right socket, plausible rank numbers, no token
        s = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        try:
            s.connect(addr)
            break
        except OSError:
            s.close()
            assert time.time() < deadline
            time.sleep(0.01)
    s.sendall(struct.pack("iiQ", 1, 2, 0x1234))
    time.sleep(0.2)
    p1 = ctx.Process(target=_boot_rank_env, args=(coll_lib, name, 1, 2, q, "s3cret", 20000))
    p1.start()
    results = sorted(q.get(timeout=60) for _ in range(2))
    p0.join(10); p1.join(10)
    assert s.recv(16) == b""                      # closed by rank 0, nothing was sent to it
    s.close()
    assert results[0][:2] == (0, 0) and results[1][:2] == (1, 0), results
    assert results[0][2] == 1                     # rank 0 counted exactly one rejected connection


def test_bootstrap_rank_with_the_wrong_secret_cannot_join(coll_lib):
    ctx = mp.get_context("fork")
    q = ctx.Queue()
    name = f"pytest-secret-{os.getpid()}"
    procs = [ctx.Process(target=_boot_rank_env, args=(coll_lib, name, 0, 2, q, "right", 1500)),
             ctx.Process(target=_boot_rank_env, args=(coll_lib, name, 1, 2, q, "wrong", 1500))]
    for p in procs:
        p.start()
    results = sorted(q.get(timeout=60) for _ in range(2))
    for p in procs:
        p.join(10)
    assert results[0][1] != 0 and results[1][1] != 0, results      # rank 0 timed out waiting; rank 1 was dropped


def test_bootstrap_times_out_when_a_rank_is_missing(coll_lib):
    L = C.CDLL(coll_lib)
    L.b200collGetLastError.restype = C.c_char_p
    out = (C.c_int * 2)()
    bc = C.c_int(-1)
    fd = os.memfd_create("x")
    rc = L.b200collBootstrapSelfTest(f"pytest-timeout-{os.getpid()}".encode(), 0, 2, fd, out, C.byref(bc), 300)
    assert rc == 1 and b"timed out" in L.b200collGetLastError()


def test_nccl_shim_exports_the_api_nccl_tests_links_against(coll_lib):
    """Every NCCL entry point nccl-tests' *_perf binaries reference must resolve, or the dynamic loader refuses to start them."""
    import subprocess
    shim = os.path.join(os.path.dirname(coll_lib), "libb200coll_nccl.so")
    syms = {l.split()[-1] for l in subprocess.run(["nm", "-D", "--defined-only", shim], capture_output=True, text=True, check=True).stdout.splitlines() if " T " in l}
    need = {"ncclGetVersion", "ncclGetUniqueId", "ncclGetErrorString", "ncclGetLastError", "ncclCommInitRank", "ncclCommInitRankConfig", "ncclCommInitAll", "ncclCommDestroy",
            "ncclCommFinalize", "ncclCommAbort", "ncclCommCount", "ncclCommUserRank", "ncclCommCuDevice", "ncclCommGetAsyncError", "ncclCommSplit", "ncclCommRegister",
            "ncclCommDeregister", "ncclMemAlloc", "ncclMemFree", "ncclAllReduce", "ncclAllGather", "ncclReduceScatter", "ncclBroadcast", "ncclBcast", "ncclReduce", "ncclSend",
            "ncclRecv", "ncclGroupStart", "ncclGroupEnd", "ncclRedOpCreatePreMulSum", "ncclRedOpDestroy",
            # NCCL 2.28 (the version the shim advertises): an nccl-tests built against that header references these as well
            "ncclAlltoAll", "ncclGather", "ncclScatter", "ncclCommWindowRegister", "ncclCommWindowDeregister", "ncclCommInitRankScalable", "ncclCommShrink",
            "ncclCommRevoke", "ncclGroupSimulateEnd"}
    # and nothing the installed NCCL header declares is missing from the shim
    import re
    try:                                                           # the header of the NCCL wheel that torch runs on, else the system one
        import nvidia.nccl
        wheel = [os.path.join(d, "include", "nccl.h") for d in nvidia.nccl.__path__]
    except ImportError:
        wheel = []
    hdr = next((p for p in wheel + ["/usr/include/nccl.h"] if os.path.exists(p)), None)
    if hdr:
        declared = set(re.findall(r"^\s*(?:ncclResult_t|const char\*)\s+(nccl[A-Za-z]+)\s*\(", open(hdr).read(), re.M))
        assert declared <= syms, sorted(declared - syms)
    assert need <= syms, sorted(need - syms)
    L = C.CDLL(shim)
    L.ncclGetErrorString.restype = C.c_char_p
    v = C.c_int()
    assert L.ncclGetVersion(C.byref(v)) == 0 and v.value >= 22000
    assert L.ncclGroupEnd() != 0                                   # unbalanced group
    if not os.path.exists("/dev/nvidiactl"):
        comms = (C.c_void_p * 1)()
        rc = L.ncclCommInitAll(comms, 1, (C.c_int * 1)(0))
        assert rc != 0 and L.ncclGetErrorString(rc)               # no driver: an error code, not a crash


def test_bench_output_dump_samples_the_same_elements_within_budget(tmp_path):
    """bench.py --dump-outputs: small outputs whole; large ones reduced to a sample that depends on their length only (so two builds
    dump the same elements), sorted, without repeats, with the first and last 1024 elements; float32 .npy files within 64 MiB."""
    import importlib.util
    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("bench_main", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    runs = []
    for _ in range(2):
        d = bench.OutputDump(63)
        d("small", torch.arange(256, dtype=torch.bfloat16))
        for n in (d.per_array + 1, 10_000_019):
            d(f"n{n}", torch.arange(n, dtype=torch.float32))           # exact in float32 below 2**24: the values are the sampled indices
        d.write(str(tmp_path / f"run{len(runs)}"))
        runs.append({p.stem: np.load(p) for p in (tmp_path / f"run{len(runs)}").glob("*.npy")})
    assert runs[0].keys() == runs[1].keys() == {"small", f"n{d.per_array + 1}", "n10000019"}
    assert all(np.array_equal(runs[0][k], runs[1][k]) and runs[0][k].dtype == np.float32 for k in runs[0])
    assert np.array_equal(runs[0]["small"], np.arange(256, dtype=np.float32))
    for n in (d.per_array + 1, 10_000_019):
        idx = runs[0][f"n{n}"].astype(np.int64)
        assert len(idx) == d.per_array and (np.diff(idx) > 0).all() and idx.min() == 0 and idx.max() == n - 1
        assert np.array_equal(idx[:1024], np.arange(1024)) and np.array_equal(idx[-1024:], np.arange(n - 1024, n))
    assert d.per_array * 4 * 63 <= bench.DUMP_LIMIT


def test_harness_bandwidth_accounting_follows_nccl_tests():
    """bench.py's numbers are only comparable with nccl-tests if the bus-bandwidth factors are the same: 2(n-1)/n for all_reduce,
    (n-1)/n for all_gather / reduce_scatter / alltoall, 1 for the rooted ops, and the average is over every (size, placement) measured."""
    from container_engine_accelerators_b200.parallel import harness as h
    assert h.bus_factor("all_reduce", 8) == pytest.approx(1.75) and h.bus_factor("all_gather", 8) == pytest.approx(0.875)
    assert h.bus_factor("reduce_scatter", 2) == 0.5 and h.bus_factor("alltoall", 4) == 0.75
    assert h.bus_factor("broadcast", 8) == 1.0 and h.bus_factor("reduce", 8) == 1.0 and h.bus_factor("all_reduce", 1) == 1.0
    assert h.bus_factor("sendrecv", 8) == 1.0 and h.bus_factor("gather", 8) == pytest.approx(0.875) and h.bus_factor("scatter", 4) == 0.75      # nccl-tests' factors
    assert set(h.P2P_OPS) == {"sendrecv", "gather", "scatter"} and h.ALL_OPS[:6] == h.OPS
    rows = [h.Row(nbytes=1 << 20, count=1 << 19, algo="nvls", oop_us=10.0, ip_us=20.0), h.Row(nbytes=1 << 30, count=1 << 29, algo="nvls", oop_us=2000.0, ip_us=-1.0, e2e_us=40000.0)]
    b = rows[0].bw("all_reduce", 8)
    assert b["oop_algbw"] == pytest.approx((1 << 20) / 10.0 / 1e3) and b["oop_busbw"] == pytest.approx(b["oop_algbw"] * 1.75) and b["ip_busbw"] == pytest.approx(b["oop_busbw"] / 2)
    s = h.summarize(rows, "all_reduce", 8)
    per = [rows[0].bw("all_reduce", 8)["oop_busbw"], rows[0].bw("all_reduce", 8)["ip_busbw"], rows[1].bw("all_reduce", 8)["oop_busbw"]]
    assert s["measurements"] == 3 and s["avg_busbw"] == pytest.approx(sum(per) / 3) and s["peak_busbw"] == pytest.approx(max(per))
    assert s["sweep_ms"] == pytest.approx((10 + 20 + 2000) / 1e3) and s["avg_e2e_busbw"] == pytest.approx((1 << 30) / 40000.0 / 1e3 * 1.75)
    table = h.format_table(rows, "all_reduce", 8, "title")
    assert table.splitlines()[0] == "# title" and table.splitlines()[-1].startswith("# Avg bus bandwidth : ") and "nvls" in table
    js = h.rows_json(rows, "all_reduce", 8)
    assert js[0]["bytes"] == 1 << 20 and "e2e_us" not in js[0] and js[1]["e2e_us"] == 40000.0 and js[1]["ip_us"] == -1.0
    assert h.OPS.index("broadcast") == coll_op_ids()["broadcast"] and h.OPS.index("alltoall") == coll_op_ids()["alltoall"]


def coll_op_ids():
    """b200collOp_t values from the public header (the harness indexes the tuner with OPS.index(op))."""
    import re
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "coll", "include", "b200coll.h")).read()
    names = {"AllReduce": "all_reduce", "AllGather": "all_gather", "ReduceScatter": "reduce_scatter", "AllToAll": "alltoall", "Broadcast": "broadcast", "Reduce": "reduce"}
    return {names[m.group(1)]: int(m.group(2)) for m in re.finditer(r"b200collOp(\w+) = (\d+)", header) if m.group(1) in names}


def test_ctypes_structs_match_the_c_header(tmp_path):
    """The Python binding restates the public structs; compile a probe against coll/include/b200coll.h (plain C, no CUDA) and compare
    sizes, member offsets and enumerators, so a header change cannot silently shear the binding."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "probe.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "b200coll.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu\n", sizeof(b200collStats), sizeof(b200collCommInfo), sizeof(b200collConfig), sizeof(b200collFault), sizeof(b200collEpilogue), sizeof(b200collUniqueId));
  printf("%zu %zu %zu %zu\n", offsetof(b200collStats, bytes), offsetof(b200collStats, algo_calls), offsetof(b200collStats, kernel_launches), offsetof(b200collStats, staged_calls));
  printf("%d %d %d %d %d %d %d\n", b200collNumOps, b200collNumAlgos, b200collFloat32, b200collFloat16, b200collBfloat16, b200collFloat8e4m3, b200collAvg);
  printf("%d %d %d %d %d %d\n", b200collOpAllReduce, b200collOpAllGather, b200collOpReduceScatter, b200collOpAllToAll, b200collOpBroadcast, b200collOpReduce);
  return 0;
}''')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(root, "coll", "include"), str(src), "-o", str(exe)], check=True)      # the header is valid C99
    lines = [list(map(int, l.split())) for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()]
    assert lines[0] == [C.sizeof(coll.Stats), C.sizeof(coll.CommInfo), C.sizeof(coll.Config), C.sizeof(coll.Fault), C.sizeof(coll.Epilogue), C.sizeof(coll.UniqueId)]
    assert lines[1] == [coll.Stats.bytes.offset, coll.Stats.algo_calls.offset, coll.Stats.kernel_launches.offset, coll.Stats.staged_calls.offset]
    assert lines[2] == [len(coll.Stats().calls), len(coll.ALGO_NAMES), coll.F32, coll.F16, coll.BF16, coll.FP8_E4M3, coll.AVG]
    assert lines[3][:4] == [coll.OP_ALLREDUCE, coll.OP_ALLGATHER, coll.OP_REDUCESCATTER, coll.OP_ALLTOALL] and lines[3][4:] == [4, 5]


def test_nccl_shim_declarations_match_nccl_h(tmp_path, coll_lib):
    """The shim re-declares NCCL's enums and prototypes (it cannot include nccl.h and define the same symbols). When a real nccl.h is
    installed, check the enumerator values and that every prototype the shim exports is call-compatible with NCCL's declaration."""
    import re
    import subprocess
    if not os.path.exists("/usr/include/nccl.h"):
        pytest.skip("no system nccl.h to compare against")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    shim = open(os.path.join(root, "coll", "src", "nccl_shim.cc")).read()
    enums = dict(re.findall(r"\b(nccl[A-Z]\w+) = (\d+)", shim))
    assert len(enums) >= 20
    checks = "\n".join(f'_Static_assert({name} == {val}, "{name}");' for name, val in enums.items())
    # call every exported entry point through NCCL's own prototypes: a signature mismatch is a compile error
    src = tmp_path / "probe.c"
    src.write_text(f'''
#include <cuda_runtime.h>
#include <nccl.h>
{checks}
void use(void) {{
  ncclComm_t c = 0; ncclUniqueId id; int v; void* p = 0; ncclRedOp_t op; cudaStream_t s = 0; ncclResult_t r;
  ncclGetVersion(&v); ncclGetUniqueId(&id); ncclCommInitRank(&c, 2, id, 0); ncclCommInitAll(&c, 1, 0); ncclCommDestroy(c); ncclCommFinalize(c); ncclCommAbort(c);
  ncclCommCount(c, &v); ncclCommUserRank(c, &v); ncclCommCuDevice(c, &v); ncclCommGetAsyncError(c, &r); ncclMemAlloc(&p, 8); ncclMemFree(p);
  ncclAllReduce(p, p, 1, ncclFloat, ncclSum, c, s); ncclAllGather(p, p, 1, ncclFloat, c, s); ncclReduceScatter(p, p, 1, ncclFloat, ncclSum, c, s);
  ncclBroadcast(p, p, 1, ncclFloat, 0, c, s); ncclBcast(p, 1, ncclFloat, 0, c, s); ncclReduce(p, p, 1, ncclFloat, ncclSum, 0, c, s);
  ncclSend(p, 1, ncclFloat, 0, c, s); ncclRecv(p, 1, ncclFloat, 0, c, s); ncclGroupStart(); ncclGroupEnd();
  ncclRedOpCreatePreMulSum(&op, p, ncclFloat, ncclScalarHostImmediate, c); ncclRedOpDestroy(op, c); ncclCommRegister(c, p, 8, &p); ncclCommDeregister(c, p);
  (void)ncclGetErrorString(r); (void)ncclGetLastError(c);
}}
int main(void) {{ return 0; }}
''')
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I/usr/local/cuda/include", "-fsyntax-only", str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    # the shim's own signatures, re-declared next to NCCL's: C linkage forbids two different parameter lists for one name
    sigs = re.findall(r"^((?:ncclResult_t|const char\*) nccl\w+\([^)]*\))\s*\{", shim, re.M)
    assert len(sigs) >= 28
    decl = tmp_path / "decl.cc"
    decl.write_text("#include <cuda_runtime.h>\n#include <nccl.h>\nextern \"C\" {\n" + "\n".join(re.sub(r"/\*.*?\*/", "", x) + ";" for x in sigs) + "\n}\nint main() { return 0; }\n")
    r = subprocess.run(["g++", "-std=c++17", "-I/usr/local/cuda/include", "-fsyntax-only", str(decl)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    # and the shim defines each of those names
    syms = subprocess.run(["nm", "-D", "--defined-only", os.path.join(os.path.dirname(coll_lib), "libb200coll_nccl.so")], capture_output=True, text=True, check=True).stdout
    for name in re.findall(r"\b(nccl[A-Z]\w+)\(", src.read_text()):
        assert f" T {name}\n" in syms, name


def _plan_p2p(lib_path, rank, n, ops, loopback=0, window=0):
    """ops: (is_send, peer, nbytes, in_arena). Returns (rc, [launch dicts]) from the library's planner hook (no GPU involved)."""
    import ctypes as C
    import re
    L = C.CDLL(lib_path)
    k = len(ops)
    out = C.create_string_buffer(1 << 16)
    arr = lambda t, xs: (t * k)(*xs)
    rc = L.b200collDebugPlanP2p(rank, n, loopback, C.c_size_t(window), k, arr(C.c_int, [o[0] for o in ops]), arr(C.c_int, [o[1] for o in ops]),
                                arr(C.c_size_t, [o[2] for o in ops]), arr(C.c_int, [o[3] for o in ops]), out, len(out))
    launches = []
    for line in out.value.decode().splitlines():
        kv = {k_: int(v) for k_, v in re.findall(r"(\w+)=(\d+)", line)}
        cta = re.search(r"ctas=\[(\d+),(\d+)\)", line)
        if line.startswith("launch"):
            launches.append({**kv, "ops": []})
        elif line.startswith("self copy"):
            launches.append({"self_copy": kv["bytes"], "ops": []})
        else:
            launches[-1]["ops"].append({**kv, "kind": line.split()[0], "staged": " staged " in line, "ctas": (int(cta.group(1)), int(cta.group(2)))})
    return rc, launches


def test_point_to_point_planner_layout_and_rounds(coll_lib):
    """Host side of send / recv (coll/src/collectives.cu p2p_flush / p2p_launch), checked without a GPU: CTA counts depend only on the
    message size (so both ends of a pair agree), sends occupy the low CTAs, staged receives get disjoint window pairs inside the staging
    area, a second message for the same pair waits for a follow-up kernel, self pairs are local copies."""
    MiB = 1 << 20
    for nbytes, want in [(16, 1), (128 << 10, 1), ((128 << 10) + 1, 2), (MiB, 8), (2 * MiB, 16), (1 << 30, 16)]:
        rc, (send,) = _plan_p2p(coll_lib, 0, 8, [(1, 3, nbytes, 1)])
        rc2, (recv,) = _plan_p2p(coll_lib, 3, 8, [(0, 0, nbytes, 1)])
        assert rc == 0 and rc2 == 0 and send["ctas"] == want and send["ops"][0]["lanes"] == want == recv["ops"][0]["lanes"], nbytes      # lane j of the send meets lane j of the recv
        assert recv["ctas"] == 1                     # a receive into the arena only exchanges flags: one CTA looks after all its lanes
    assert _plan_p2p(coll_lib, 0, 4, [(1, 1, 1 << 30, 1)], loopback=1)[1][0]["ctas"] == 2                     # virtual ranks share one GPU's SMs
    # a ring step: one launch, send in the low CTAs, arena receive written in place
    rc, (ring,) = _plan_p2p(coll_lib, 0, 8, [(0, 7, MiB, 1), (1, 1, MiB, 1)])
    assert rc == 0 and [o["kind"] for o in ring["ops"]] == ["send", "recv"] and ring["ops"][0]["ctas"] == (0, 8) and ring["ops"][1]["ctas"] == (8, 9) and ring["ops"][1]["lanes"] == 8
    assert not ring["ops"][1]["staged"] and ring["staged"] == 0
    # three receives outside the arena: three window pairs, disjoint, inside the 64 MiB staging area that starts at 25 MiB
    rc, (l,) = _plan_p2p(coll_lib, 1, 4, [(0, p, 40 * MiB, 0) for p in (0, 2, 3)])
    assert rc == 0 and l["staged"] == 3
    spans = sorted((o["off"], o["off"] + 2 * o["window"]) for o in l["ops"])
    assert spans[0][0] == 25 * MiB and spans[-1][1] <= 89 * MiB and all(a[1] <= b[0] for a, b in zip(spans, spans[1:]))
    assert all(o["window"] % 512 == 0 and o["chunks"] == -(-40 * MiB // o["window"]) for o in l["ops"])
    # the receiver may cap its windows; a message that fits one window is a single chunk
    rc, (l,) = _plan_p2p(coll_lib, 1, 2, [(0, 0, 3 * MiB + 5, 0)], window=MiB)
    assert l["ops"][0]["window"] == MiB and l["ops"][0]["chunks"] == 4
    assert _plan_p2p(coll_lib, 1, 2, [(0, 0, 1000, 0)], window=MiB)[1][0]["ops"][0]["chunks"] == 1
    # two messages 0 -> 1 in one group share a mailbox: the second runs in a follow-up kernel; empty messages vanish; self pairs are copies
    rc, ls = _plan_p2p(coll_lib, 0, 2, [(1, 1, 4096, 1), (1, 1, 777, 1), (0, 1, 64, 1), (1, 1, 0, 1), (1, 0, 256, 1), (0, 0, 256, 0)])
    assert rc == 0 and ls[0] == {"self_copy": 256, "ops": []}
    assert [(len(l["ops"]), l["sends"], l["recvs"]) for l in ls[1:]] == [(2, 1, 1), (1, 1, 0)] and ls[2]["ops"][0]["bytes"] == 777
    # misuse is refused before anything is launched
    assert _plan_p2p(coll_lib, 0, 2, [(1, 0, 64, 1)])[0] == 5               # send to self without the matching recv: invalid usage
    assert _plan_p2p(coll_lib, 0, 2, [(1, 2, 64, 1)])[0] == 4               # peer out of range: invalid argument


def test_point_to_point_protocol_under_host_emulation(coll_lib):
    """coll/src/p2p.cuh — the text nvcc compiles into k_p2p — built by g++ with every CTA of every rank a thread (coll/tests/p2p_emu.cc):
    ring steps with growing and shrinking sizes, staged receives through windows far smaller than the message, all-pairs groups,
    lone send / recv, watchdog and size-mismatch faults. Then the same under ThreadSanitizer where the toolchain has it: every payload
    byte must be ordered by a release/acquire pair on a flag. (This harness found the first version's window-sharing bug before any GPU
    saw the kernel.)"""
    import shutil
    root = os.path.dirname(os.path.dirname(coll_lib))
    r = subprocess.run(["make", "-C", root, "../build/p2p_emu"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    exe = os.path.join(os.path.dirname(root), "build", "p2p_emu")
    for extra in ([], ["--quick", "--threads", "4"]):            # one host thread per CTA, then four (bar.sync placement, strided loops)
        r = subprocess.run([exe] + extra, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0 and "all scenarios passed" in r.stdout, r.stdout + r.stderr
    if shutil.which("/usr/bin/g++") is None:
        pytest.skip("no system g++ for the ThreadSanitizer flavour")
    b = subprocess.run(["make", "-C", root, "../build/p2p_emu_tsan"], capture_output=True, text=True)
    if b.returncode != 0 and "tsan" in (b.stdout + b.stderr).lower():
        pytest.skip("toolchain has no libtsan")
    assert b.returncode == 0, b.stdout + b.stderr
    for extra in (["--quick"], ["--quick", "--threads", "2"]):
        r = subprocess.run([exe + "_tsan"] + extra, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "data race" not in r.stderr and "all scenarios passed" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_comm_split_plan_orders_by_key_then_rank(coll_lib):
    """b200collCommSplit's membership rule (ncclCommSplit's): same color -> same communicator, ranks ordered by (key, old rank)."""
    import itertools
    L = C.CDLL(coll_lib)

    def plan(colors, keys, rank):
        n = len(colors)
        nr, ns = C.c_int(-1), C.c_int(-1)
        rc = L.b200collDebugSplitPlan(n, rank, (C.c_int * n)(*colors), (C.c_int * n)(*keys), C.byref(nr), C.byref(ns))
        assert rc == 0
        return nr.value, ns.value

    # tensor-parallel pairs out of 8 ranks, and the data-parallel groups across them
    assert [plan([r // 2 for r in range(8)], [0] * 8, r) for r in range(8)] == [(r % 2, 2) for r in range(8)]
    assert [plan([r % 2 for r in range(8)], [0] * 8, r) for r in range(8)] == [(r // 2, 4) for r in range(8)]
    # keys reverse the order inside a colour; equal keys fall back to the old rank
    assert [plan([0, 0, 0, 1], [5, 3, 3, 0], r) for r in range(4)] == [(2, 3), (0, 3), (1, 3), (0, 1)]
    # exhaustively for 4 ranks and small colour / key alphabets: new ranks of a colour are exactly 0..size-1, ordered by (key, rank)
    for colors in itertools.product(range(2), repeat=4):
        for keys in itertools.product(range(2), repeat=4):
            got = [plan(colors, keys, r) for r in range(4)]
            for col in set(colors):
                members = sorted((keys[r], r) for r in range(4) if colors[r] == col)
                assert [got[r] for _, r in members] == [(i, len(members)) for i in range(len(members))]
    assert L.b200collDebugSplitPlan(9, 0, None, None, None, None) != 0


def test_pytorch_pluggable_allocator_entry_points(coll_lib):
    """b200collTorchAlloc / b200collTorchFree have the signature torch.cuda.memory.CUDAPluggableAllocator wants; without an allocator
    communicator they fail softly (nullptr = PyTorch's out-of-memory path), never crash."""
    L = C.CDLL(coll_lib)
    L.b200collTorchAlloc.argtypes = [C.c_size_t, C.c_int, C.c_void_p]; L.b200collTorchAlloc.restype = C.c_void_p
    L.b200collTorchFree.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]; L.b200collTorchFree.restype = None
    assert L.b200collTorchAlloc(1 << 20, 0, None) is None
    L.b200collTorchFree(None, 0, 0, None); L.b200collTorchFree(C.c_void_p(0x1000), 16, 0, None)      # no communicator: ignored
    from torch.cuda.memory import CUDAPluggableAllocator
    alloc = CUDAPluggableAllocator(coll_lib, "b200collTorchAlloc", "b200collTorchFree")                # resolves both symbols
    assert alloc.allocator() is not None


def test_epoch_barrier_under_host_emulation_classic_and_multicast_counter(coll_lib):
    """coll/src/barrier.cuh (what every barrier-based kernel calls) compiled for the host, CTAs as thread groups, under ThreadSanitizer:
    the shipped flag exchange, and the multicast-counter variant (-DB200COLL_VARIANT_MCBAR, an A/B candidate that has never met a GPU)
    with multimem.red emulated as an add to the same word of every arena. Launches alternate grid sizes and ranks enter late; stamps
    written between the two barriers must be readable by every peer right after the second one."""
    import shutil
    if shutil.which("/usr/bin/g++") is None:
        pytest.skip("no system g++ for the ThreadSanitizer build")
    root = os.path.dirname(os.path.dirname(coll_lib))
    for target, what in (("barrier_emu_tsan", "(flags)"), ("barrier_emu_tsan_mc", "(flags + multicast counter)")):
        b = subprocess.run(["make", "-C", root, f"../build/{target}"], capture_output=True, text=True)
        if b.returncode != 0 and "tsan" in (b.stdout + b.stderr).lower():
            pytest.skip("toolchain has no libtsan")
        assert b.returncode == 0, b.stdout + b.stderr
        r = subprocess.run([os.path.join(os.path.dirname(root), "build", target), "5"], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "data race" not in r.stderr and f"barrier_emu {what}: all launches consistent" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_cpulist_parser_matches_sysfs_format(coll_lib):
    """coll/src/hostpath.cu binds a rank to its GPU's CPUs from sysfs' local_cpulist ("0-31,64-95"); the parser is pure."""
    L = C.CDLL(coll_lib)
    L.b200collDebugParseCpuList.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.c_int]
    out = (C.c_int * 512)()

    def parse(text):
        n = L.b200collDebugParseCpuList(text.encode(), out, 512)
        return list(out[:n])
    assert parse("0-31,64-95") == list(range(32)) + list(range(64, 96))
    assert parse("3") == [3] and parse("") == [] and parse("0,2,4-5\n") == [0, 2, 4, 5]
    assert parse("7-7,1") == [1, 7] and parse("garbage") == [] and parse("2-") == []


def test_benchmark_self_check_rejects_low_precision_accumulation():
    """bench.py verifies reductions with data whose sums are not exact in bf16, within one bf16 ulp of the fp32-accumulated result
    (harness.reduction_ok). A reduction that accumulates in bf16 — what multimem.ld_reduce does without .acc::f32 — must fail it,
    a correctly rounded fp32 accumulation in any order must pass."""
    import torch
    from container_engine_accelerators_b200.parallel import harness as h
    n = 8
    gen = h._gen_expected(torch, "all_reduce", 0, n, 0, "cpu")
    idx = torch.arange(1 << 16)
    ins = [gen(r, idx) for r in range(n)]
    assert all(torch.equal(x, x.to(torch.bfloat16).float()) for x in ins)                 # inputs are bf16 values
    want = sum(ins)
    assert (want.to(torch.bfloat16).float() != want).float().mean() > 0.5                 # most sums need rounding: the check has teeth
    assert h.reduction_ok(torch, want.to(torch.bfloat16).float(), want, torch.bfloat16, n)
    assert h.reduction_ok(torch, sum(reversed(ins)).to(torch.bfloat16).float(), want, torch.bfloat16, n)
    acc = torch.zeros_like(want).to(torch.bfloat16)
    for x in ins:
        acc = (acc.float() + x).to(torch.bfloat16)
    assert not h.reduction_ok(torch, acc.float(), want, torch.bfloat16, n)
    half = torch.zeros_like(want).to(torch.float16)
    for x in ins:
        half = (half.float() + x).to(torch.float16)
    off_by_two = want.to(torch.bfloat16).float() + 2 * h.bf16_ulp(torch, want)
    assert not h.reduction_ok(torch, off_by_two, want, torch.bfloat16, n)


_LOCALITY_SCRIPT = r"""
import ctypes as C, json, os, sys
lib_path, root = sys.argv[1], sys.argv[2]
L = C.CDLL(lib_path)
L.b200collDebugApplyLocality.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_int)]
start = sorted(os.sched_getaffinity(0))
changed = C.c_int(-1)
out = {}
def run(name, sub, mode):
    node = L.b200collDebugApplyLocality(os.path.join(root, sub).encode(), mode, C.byref(changed))
    out[name] = [node, changed.value, sorted(os.sched_getaffinity(0))]
run("missing", "nope", 1); run("observe_only", "gpu", 0); run("outside", "far", 1); run("bind", "gpu", 1); run("again", "gpu", 1)
print(json.dumps({"start": start, "out": out}))
"""


def test_rank_is_bound_to_the_cpus_of_its_gpu(coll_lib, tmp_path):
    """What CommInitRank does with the GPU's sysfs directory (coll/src/hostpath.cu apply_gpu_locality): read numa_node, narrow the
    calling thread to the GPU-local CPUs it is allowed to use, leave it alone when the list lies outside its cpuset, when told to only
    observe (B200COLL_AFFINITY=0) or when the directory does not exist. This placement is what keeps eight ranks' host buffers on the
    right socket (profiles/host_path.md: 45 ms instead of 134 ms per GiB at 8 GPUs)."""
    cpus = sorted(os.sched_getaffinity(0))
    if len(cpus) < 3:
        pytest.skip("needs at least three usable CPUs")
    local = cpus[:2]
    (tmp_path / "gpu").mkdir(); (tmp_path / "gpu" / "numa_node").write_text("1\n"); (tmp_path / "gpu" / "local_cpulist").write_text(f"{local[0]},{local[1]}\n")
    (tmp_path / "far").mkdir(); (tmp_path / "far" / "numa_node").write_text("0\n"); (tmp_path / "far" / "local_cpulist").write_text("4090-4095\n")
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-c", _LOCALITY_SCRIPT, coll_lib, str(tmp_path)], capture_output=True, text=True, timeout=60)      # its own process: the affinity change must not leak
    assert r.returncode == 0, r.stderr
    res = json.loads(r.stdout)
    start, out = res["start"], res["out"]
    assert start == cpus
    assert out["missing"] == [-1, 0, cpus]
    assert out["observe_only"] == [1, 0, cpus]
    assert out["outside"] == [0, 0, cpus]
    assert out["bind"] == [1, 1, local]
    assert out["again"] == [1, 0, local]                     # already there: nothing to change
    assert sorted(os.sched_getaffinity(0)) == cpus           # the test process itself was never touched
