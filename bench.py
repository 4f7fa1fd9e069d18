#!/usr/bin/env python
"""Headline benchmark: all_reduce_perf bus GB/s, 1 KB - 1 GB, bf16 sum (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29500 \
        bench.py --gpus 8 --steps 20 --warmup 5
    ... --impl reference      # stock NCCL through its C API, NCCL's own defaults (see nccl_ref.py); reference-sym adds ncclMemAlloc + symmetric windows

A "step" is one pass over the 21-size sweep (1 KB..1 GB, x2), out-of-place and in-place. Following the
reference's nccl-tests protocol each size's `--steps` iterations are launched back to back and timed with
CUDA events on the launching stream (after `--warmup` untimed launches), bracketed by a cross-rank barrier
and torch.cuda.synchronize(); every number is the max over ranks. `value` is nccl-tests' "Avg bus bandwidth".
The end-to-end sweep (host in, host out) runs `--steps` steps as well. Rank 0 prints ONE JSON line.

The send buffer is filled from a seeded hash before the sweep, so the same arguments give the same inputs on
every run (harness.fill_inputs says why the receive buffer is not). `--dump-outputs DIR` makes rank 0
write what the last timed step of every size returned, as DIR/<op>_<oop|ip|e2e>_<bytes>B.npy in float32:
whole outputs when small, otherwise a fixed sample of their elements (first and last ones included), at
most 64 MiB in all. Two builds run with the same arguments can then be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


DUMP_LIMIT = 64 << 20      # bytes of .npy payload --dump-outputs may write, all arrays together


def parse_size(s: str) -> int:
    s = s.strip().upper()
    mult = {"K": 1 << 10, "M": 1 << 20, "G": 1 << 30}
    return int(float(s[:-1]) * mult[s[-1]]) if s[-1] in mult else int(s)


def positive_int(s: str) -> int:
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


class OutputDump:
    """Collects the outputs handed to harness.sweep's on_output as float32 copies: whole when they hold at most `per_array` elements,
    otherwise the first and last 1024 elements plus one element from each of `per_array - 2048` equal stretches in between, at an
    offset given by a hash of the stretch's number. The sample depends on the output's length only, so two runs with the same
    arguments sample the same elements. Copies of device outputs stay on the device until write(): the capture between two timed
    windows is a few kernel launches on the sweep's stream, with no host synchronisation and no idle GPU."""

    def __init__(self, n_arrays: int):
        self.per_array = max(4096, DUMP_LIMIT // 4 // max(1, n_arrays))
        self.arrays = {}

    def __call__(self, name: str, t) -> None:
        import torch
        n = t.numel()
        if n > self.per_array:
            edge, k = 1024, self.per_array - 2048
            span = n - 2 * edge
            j = torch.arange(k, device=t.device)
            mid = edge + j * span // k + (((j * 2654435761) & 0xFFFFFFFF) >> 8) % (span // k)
            t = t[torch.cat([torch.arange(edge, device=t.device), mid, torch.arange(n - edge, n, device=t.device)])]
        self.arrays[name] = t.to(torch.float32, copy=True)

    def write(self, out_dir: str) -> None:
        import numpy as np
        total = sum(a.numel() * 4 for a in self.arrays.values())
        assert total <= DUMP_LIMIT, f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT}"
        os.makedirs(out_dir, exist_ok=True)
        for name, a in self.arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-sym"], help="reference = stock NCCL on plain buffers (what nccl-tests does); reference-sym = the same on ncclMemAlloc memory with symmetric windows registered (NCCL's own fast path)")
    ap.add_argument("--op", default="all_reduce", choices=["all_reduce", "all_gather", "reduce_scatter", "alltoall", "broadcast", "reduce", "sendrecv", "gather", "scatter"])
    ap.add_argument("--min", default="1K")
    ap.add_argument("--max", default="1G")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--table", action="store_true", help="also print the nccl-tests style table to stderr")
    ap.add_argument("--extra-ops", default="", help="comma list of further collectives to sweep in the same process group; results go to --extra-out, never to stdout")
    ap.add_argument("--extra-out", default="gpurun_out/extra_ops.json")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of every size returned to DIR/<name>.npy (float32, at most 64 MiB in all)")
    args = ap.parse_args()
    warmup = max(3, args.warmup)

    try:
        import torch
    except Exception as e:   # pragma: no cover
        print(json.dumps({"impl": args.impl, "unavailable": f"torch import failed: {e}"}))
        return 0
    from container_engine_accelerators_b200.parallel import harness
    from container_engine_accelerators_b200.utils.clocks import ClockSampler

    dist = harness.Dist()
    if dist.world != args.gpus:
        if dist.rank == 0:
            print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={dist.world}; launch with torchrun --nproc-per-node {args.gpus}", file=sys.stderr)
        return 2
    if not torch.cuda.is_available():
        if dist.rank == 0:
            print(json.dumps({"impl": args.impl, "unavailable": "no CUDA device visible"}))
        return 0
    torch.cuda.set_device(dist.local_rank)
    dtype = torch.bfloat16
    min_b, max_b = parse_size(args.min), parse_size(args.max)
    cap = max(max_b, harness.WINDOW) // 2 + 4096

    if args.impl == "reference-sym":
        os.environ["B200_REF_SYM"] = "1"
    if args.impl.startswith("reference"):
        try:
            backend = harness.NcclBackend(dist, cap, dtype)
        except Exception as e:
            if dist.rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": f"stock NCCL could not be initialised: {e}"[:300]}))
            return 0
    else:
        backend = harness.OursBackend(dist, cap, dtype)   # raises if libb200coll.so is missing: no silent fallback

    n = dist.world
    verified = harness.verify(backend, dist, args.op, dtype)
    harness.fill_inputs(backend, dist)
    dump = None
    if args.dump_outputs and dist.rank == 0:
        n_sizes = sum(1 for k in range(64) if min_b << k <= max_b)
        dump = OutputDump(3 * n_sizes)          # at most out-of-place, in-place and end-to-end per size
    launches0 = backend.launches()
    t_wall = time.time()
    with ClockSampler(dist.local_rank) as clk:
        rows = harness.sweep(backend, dist, args.op, dtype, args.steps, warmup, min_b, max_b, placements=(0, 1), on_output=dump)
    launches = backend.launches() - launches0
    clocks = clk.summary()
    e2e = None
    e2e_rows = []
    if not args.no_e2e:
        e2e_ok = harness.verify_e2e(backend, dist, dtype) if args.op == "all_reduce" else True
        hl0 = backend.launches()
        e2e_steps = args.steps
        e2e_rows = harness.sweep(backend, dist, args.op, dtype, e2e_steps, min(warmup, 3), min_b, max_b, placements=(), e2e=True, on_output=dump)
        s2 = harness.summarize(e2e_rows, args.op, n)
        e2e = {"value": round(s2["avg_e2e_busbw"] or 0.0, 3), "unit": "GB/s", "h2d_bytes_per_step": int(sum(r.in_bytes for r in e2e_rows)),
               "d2h_bytes_per_step": int(sum(r.out_bytes for r in e2e_rows)), "steps": e2e_steps, "verified_vs_torch_fp32": bool(e2e_ok),
               "peak_busbw": round(max((r.bw(args.op, n)["e2e_busbw"] for r in e2e_rows), default=0.0), 2),
               "gpu_launches_incl_warmup": int(backend.launches() - hl0),
               "note": ("per size, every step: this rank's input starts in pinned host memory and the WHOLE result ends in pinned host memory. "
                        + ("ours: one call of the public API per step, Comm.all_reduce_host (b200collAllReduceHost: a zero-copy kernel over PCIe for tiny messages; "
                           "host->device copy, all-reduce and device->host copy overlapped chunk by chunk for large ones)" if args.impl == "ours" and args.op == "all_reduce"
                           else "copy in, the collective, copy the result back, on one stream (what a user of a device-pointer collective API writes)")),
               "table": [{"bytes": r.nbytes, "e2e_us": round(r.e2e_us, 2), "e2e_busbw": round(r.bw(args.op, n)["e2e_busbw"], 2)} for r in e2e_rows]}
        verified = verified and e2e_ok
    wall = time.time() - t_wall
    summ = harness.summarize(rows, args.op, n)
    if dist.rank == 0:
        if args.table:
            print(harness.format_table(rows, args.op, n, f"{backend.version} {args.op} nranks={n}"), file=sys.stderr)
        metric = f"{args.op}_perf avg bus GB/s 1KB-1GB bf16 sum (nccl-tests protocol, device-timed, max over ranks)"
        if n == 1:
            metric += " [1 rank: busbw factor is 0 by definition, value is algbw of the fused scale/cast copy]"
        out = {
            "metric": metric, "value": round(summ["avg_busbw"], 3), "unit": "GB/s", "n_gpus": n, "steps": args.steps, "warmup": warmup,
            "ms_per_step": round(summ["sweep_ms"], 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic (deterministic random-like bf16 buffers; no network, no dataset)",
            "impl": "reference" if args.impl.startswith("reference") else "ours", "backend": backend.version,
            "config": {"model": "none (collective benchmark: the reference has no model code)", "benchmark": f"{args.op}_perf", "sizes": f"{args.min}..{args.max} x2",
                       "global_batch": None, "seq_len": None, "parallelism": f"1 rank per GPU x{n}", "placements": "out-of-place + in-place",
                       "l2": "buffers rotate through a 192 MiB window (> 126 MB L2); sizes >= 192 MiB exceed L2 by themselves",
                       "timed_region": "per size: host barrier + device synchronize, then a device-side rendezvous of all ranks' streams, then the first event; the same on both arms",
                       "aggregate": "nccl-tests bus bandwidth (per-link hardware rate), not multiplied by N",
                       "scaling_note": "bus bandwidth is normalised per GPU by construction: perfect scaling is a CONSTANT value from 2 to 8 GPUs (aggregate_bus_gbs = value x N is the whole-job rate); "
                                       "the 1-GPU value has no bus in it (an HBM copy with the fused epilogue) and is not a base for efficiency"},
            "peak_busbw": round(summ["peak_busbw"], 2), "aggregate_bus_gbs": round(summ["avg_busbw"] * n, 2), "verified_vs_torch_fp32": bool(verified),
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"], "power_w_max": clocks["power_w_max"]},
            "gpu_launches": int(summ["measurements"] * args.steps) if args.impl == "ours" else 0,
            "verify": "random bf16 data (sums not exact in bf16) vs an fp32 torch reference within 1 bf16 ulp, at sizes taking the Lamport, NVLS / two-shot and scalar-tail paths" if args.op == "all_reduce" else "vs fp32 torch reference", "gpu_launches_incl_warmup": int(launches), "e2e": e2e, "wall_s": round(wall, 2), "table": harness.rows_json(rows, args.op, n),
        }
        if args.impl.startswith("reference"):
            out["reference_note"] = ("the reference repo ships no collective code or Python package; its nccl-test manifests run NCCL's *_perf on the node "
                                     "(net plugins are off the intra-node path), so this arm is the image's stock libnccl called through its C API with the "
                                     "NCCL's own defaults (B200_REF_PROFILE=1 applies the reference's multi-node env profile, gpudirect-tcpxo/README.md:71-103); pip install of /root/reference: see DESIGN.md")
        print(json.dumps(out), flush=True)
    if dump is not None:
        dump.write(args.dump_outputs)
    if args.extra_ops:
        extra = {}
        for op in [o for o in args.extra_ops.split(",") if o and o != args.op]:
            ok = harness.verify(backend, dist, op, dtype) if n > 1 else True
            rws = harness.sweep(backend, dist, op, dtype, args.steps, warmup, min_b, max_b, placements=(0, 1))
            sm = harness.summarize(rws, op, n)
            extra[op] = {"avg_busbw": round(sm["avg_busbw"], 3), "peak_busbw": round(sm["peak_busbw"], 2), "verified": bool(ok), "table": harness.rows_json(rws, op, n)}
            if dist.rank == 0 and args.table:
                print(harness.format_table(rws, op, n, f"{backend.version} {op} nranks={n}"), file=sys.stderr)
        if dist.rank == 0:
            os.makedirs(os.path.dirname(args.extra_out) or ".", exist_ok=True)
            with open(args.extra_out, "w") as f:
                json.dump({"impl": args.impl, "n_gpus": n, "backend": backend.version, "ops": extra}, f)
    backend.close()
    dist.close()
    return 0 if (verified or args.impl.startswith("reference")) else 3      # the reference arm's numerics are reported (verified_vs_torch_fp32), not enforced


if __name__ == "__main__":
    sys.exit(main())
