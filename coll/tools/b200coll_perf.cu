// b200coll_perf — nccl-tests-style benchmark + correctness checker for libb200coll.
// The reference's benchmark protocol (reference: gpudirect-tcpx/nccl-config.yaml:61-62,
// gpudirect-rdma/nccl-test-a4x-max-jobset.yaml:141-153): `-b <min> -e <max> -f 2 -g 1 -w 5 --iters 100 -c 1`,
// one rank per GPU, out-of-place and in-place, time = avg over iters, algbw = bytes/time,
// busbw = algbw * {AR: 2(N-1)/N; AG/RS/A2A: (N-1)/N}.
//
// Modes:  default      one process, one host thread per rank, ranks from --devs (repeat a device id for
//                      virtual ranks on one GPU: protocol tests on a single-GPU box)
//         --procs      fork one process per rank and rendezvous over the Unix-socket bootstrap
// Timing: CUDA events on each rank's stream around `iters` back-to-back launches, max over ranks.
// Buffers rotate through a >L2 window so every timed launch sees cold lines.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <fcntl.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/wait.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include "../include/b200coll.h"

#define RT(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "CUDA %s:%d %s -> %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); exit(2); } } while (0)
#define CC(x) do { b200collResult_t r_ = (x); if (r_ != b200collSuccess) { fprintf(stderr, "b200coll %s:%d %s -> %s (%s)\n", __FILE__, __LINE__, #x, b200collGetErrorString(r_), b200collGetLastError()); exit(3); } } while (0)

struct Opts {
  std::string op = "all_reduce";
  std::vector<int> devs;
  int nranks = 0;
  bool procs = false;
  size_t min_bytes = 1024, max_bytes = 1ull << 30;
  int factor = 2;
  b200collDataType_t in_dt = b200collBfloat16, out_dt = b200collBfloat16;
  float scale = 1.0f;
  std::string algo = "auto";
  int iters = 20, warmup = 5, check = 1;
  int inplace = 2;   // 0 out-of-place only, 1 in-place only, 2 both
  int max_ctas = 0;
  size_t window = 192ull << 20;
  std::string json;
  int skew_us = 0;   // delay rank 0's launches (race hunting)
  struct Shape { int kind, ctas, threads; };
  std::vector<Shape> shapes;   // --sweep kind:ctas:threads,... (launch-shape tuning inside one process)
};

static size_t parse_size(const char* s) {
  char* end; double v = strtod(s, &end);
  if (*end == 'K' || *end == 'k') v *= 1024; else if (*end == 'M' || *end == 'm') v *= 1 << 20; else if (*end == 'G' || *end == 'g') v *= 1 << 30;
  return (size_t)v;
}
static b200collDataType_t parse_dt(const char* s) {
  if (!strcmp(s, "f32") || !strcmp(s, "float")) return b200collFloat32;
  if (!strcmp(s, "f16") || !strcmp(s, "half")) return b200collFloat16;
  if (!strcmp(s, "bf16") || !strcmp(s, "bfloat16")) return b200collBfloat16;
  if (!strcmp(s, "fp8") || !strcmp(s, "e4m3")) return b200collFloat8e4m3;
  if (!strcmp(s, "e5m2")) return b200collFloat8e5m2;
  fprintf(stderr, "bad dtype %s\n", s); exit(1);
}
static const char* dt_name(b200collDataType_t t) { return t == b200collFloat32 ? "f32" : t == b200collFloat16 ? "f16" : t == b200collBfloat16 ? "bf16" : t == b200collFloat8e5m2 ? "e5m2" : "e4m3"; }

// deterministic input: multiples of 0.25 in [-2, 2] so sums over <= 8 ranks are exact in bf16/f16/f32 (and in the fp32 accumulator
// of the fp8 paths: every such value is an e4m3 and an e5m2 value)
static inline float gen(int rank, size_t i) { return (float)((int)((i * 7 + (size_t)rank * 13 + (i >> 9)) % 17) - 8) * 0.25f; }

template <typename T> __global__ void k_fill(T* p, size_t n, int rank, size_t base) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    size_t g = base + i;
    float v = (float)((int)((g * 7 + (size_t)rank * 13 + (g >> 9)) % 17) - 8) * 0.25f;
    p[i] = T(v);
  }
}
static void fill(void* p, size_t n, b200collDataType_t dt, int rank, size_t base, cudaStream_t st) {
  if (dt == b200collFloat32) k_fill<float><<<256, 256, 0, st>>>((float*)p, n, rank, base);
  else if (dt == b200collFloat16) k_fill<__half><<<256, 256, 0, st>>>((__half*)p, n, rank, base);
  else if (dt == b200collFloat8e4m3) k_fill<__nv_fp8_e4m3><<<256, 256, 0, st>>>((__nv_fp8_e4m3*)p, n, rank, base);
  else if (dt == b200collFloat8e5m2) k_fill<__nv_fp8_e5m2><<<256, 256, 0, st>>>((__nv_fp8_e5m2*)p, n, rank, base);
  else k_fill<__nv_bfloat16><<<256, 256, 0, st>>>((__nv_bfloat16*)p, n, rank, base);
}

static float to_f(const void* p, size_t i, b200collDataType_t dt) {
  switch (dt) {
    case b200collFloat32: return ((const float*)p)[i];
    case b200collFloat16: return __half2float(((const __half*)p)[i]);
    case b200collBfloat16: return __bfloat162float(((const __nv_bfloat16*)p)[i]);
    case b200collFloat8e5m2: return (float)(((const __nv_fp8_e5m2*)p)[i]);
    default: return (float)(((const __nv_fp8_e4m3*)p)[i]);
  }
}
// An exact fp32 result after the collective's saturating, round-to-nearest cast to `dt`.
static float round_to(b200collDataType_t dt, float v) {
  if (dt == b200collFloat8e4m3) return (float)__nv_fp8_e4m3(v);
  if (dt == b200collFloat8e5m2) return (float)__nv_fp8_e5m2(v);
  return v;
}

struct Shared {   // cross-process (mmap MAP_SHARED) or cross-thread rendezvous for timing
  std::atomic<int> arrive[4];
  float ms[B200COLL_MAX_RANKS];
  long errors[B200COLL_MAX_RANKS];
};

static void spin_barrier(Shared* sh, int which, int n, int* gen) {
  (*gen)++;
  sh->arrive[which].fetch_add(1);
  const time_t t0 = time(nullptr);
  while (sh->arrive[which].load() < (*gen) * n) {
    sched_yield();
    if (time(nullptr) - t0 > 90) { fprintf(stderr, "host barrier %d timed out (a rank died?)\n", which); _exit(6); }
  }
}

constexpr int kRoot = 0;   // rooted ops (broadcast, reduce) are driven from rank 0, like nccl-tests' default

struct RankCtx { int rank, nranks; b200collComm_t comm; int dev; };

// expected value of output element e (element index in the op's output) for this rank
static float expected(const Opts& o, int rank, int n, size_t e, size_t count) {
  if (o.op == "all_reduce" || o.op == "reduce") { float s = 0; for (int r = 0; r < n; r++) s += gen(r, e); return s * o.scale; }
  if (o.op == "broadcast") return gen(kRoot, e) * o.scale;
  if (o.op == "sendrecv") return gen((rank + n - 1) % n, e);      // ring step: my output is my left neighbour's input, untouched
  if (o.op == "all_gather" || o.op == "gather" || o.op == "hypercube") { int src = (int)(e / count); return gen(src, e % count) * o.scale; }
  if (o.op == "scatter") return gen(kRoot, (size_t)rank * count + e);
  if (o.op == "reduce_scatter") { float s = 0; for (int r = 0; r < n; r++) s += gen(r, (size_t)rank * count + e); return s * o.scale; }
  /* alltoall */ { int src = (int)(e / count); return gen(src, (size_t)rank * count + e % count) * o.scale; }
}

static int run_rank(const Opts& o, RankCtx ctx, Shared* sh) {
  const int n = ctx.nranks, rank = ctx.rank;
  RT(cudaSetDevice(ctx.dev));
  cudaStream_t st; RT(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  cudaEvent_t e0, e1; RT(cudaEventCreate(&e0)); RT(cudaEventCreate(&e1));
  if (o.algo != "auto") {
    for (int a = 0; a < b200collNumAlgos; a++) if (o.algo == b200collAlgoName((b200collAlgo_t)a)) CC(b200collCommSetAlgo(ctx.comm, (b200collAlgo_t)a));
  }
  if (o.max_ctas > 0) CC(b200collCommSetMaxCtas(ctx.comm, o.max_ctas));
  const size_t is = b200collTypeSize(o.in_dt), os = b200collTypeSize(o.out_dt);
  const bool is_bc = o.op == "broadcast", is_rd = o.op == "reduce", is_sr = o.op == "sendrecv";
  if (is_sr && (o.in_dt != o.out_dt || o.scale != 1.0f)) { fprintf(stderr, "sendrecv moves opaque bytes: --in and --out must match and --scale must be 1\n"); return 2; }
  const bool is_ar = o.op == "all_reduce" || is_bc || is_rd || is_sr;      // "whole message" geometry: count elements in, count out
  const bool is_hc = o.op == "hypercube";          // nccl-tests hypercube_perf: an all-gather made of log2(n) pairwise exchanges of doubling size
  if (is_hc && (n & (n - 1))) { fprintf(stderr, "hypercube needs a power-of-two number of ranks\n"); return 2; }
  const bool is_ga = o.op == "gather" || is_hc, is_sc = o.op == "scatter";                 // nccl-tests gather_perf / scatter_perf: one send/recv group around the root
  if ((is_ga || is_sc) && (o.in_dt != o.out_dt || o.scale != 1.0f)) { fprintf(stderr, "%s moves opaque bytes: --in and --out must match and --scale must be 1\n", o.op.c_str()); return 2; }
  const bool is_ag = o.op == "all_gather" || is_ga, is_rs = o.op == "reduce_scatter" || is_sc;      // same buffer geometry
  if (!is_ar && !is_ag && !is_rs && o.op != "alltoall") { fprintf(stderr, "unknown --op %s\n", o.op.c_str()); return 2; }
  // nccl-tests convention: "size" is the larger of the two buffers in bytes of the input type
  const size_t max_in_bytes = o.max_bytes, max_out_bytes = o.max_bytes / is * os;
  const size_t send_cap = std::max(o.window, max_in_bytes), recv_cap = std::max(o.window / is * os, max_out_bytes);
  void *send = nullptr, *recv = nullptr;
  CC(b200collMemAlloc(ctx.comm, &send, send_cap + 4096));
  CC(b200collMemAlloc(ctx.comm, &recv, recv_cap + 4096));
  b200collEpilogue ep{o.in_dt, o.out_dt, o.scale};
  int gen_ctr[4] = {0, 0, 0, 0};
  std::vector<char> host;
  b200collCommInfo info; CC(b200collCommInfoGet(ctx.comm, &info));
  if (rank == 0) {
    printf("# b200coll_perf op=%s nranks=%d in=%s out=%s scale=%g algo=%s nvls=%d loopback=%d mode=%s\n", o.op.c_str(), n, dt_name(o.in_dt), dt_name(o.out_dt), o.scale, o.algo.c_str(),
           info.nvls, info.same_device_loopback, o.procs ? "procs" : "threads");
    printf("#%13s %12s %6s %8s | %10s %8s %8s %6s | %10s %8s %8s %6s\n", "size(B)", "count", "type", "algo", "oop us", "algbw", "busbw", "#wrong", "ip us", "algbw", "busbw", "#wrong");
    fflush(stdout);
  }
  FILE* jf = (rank == 0 && !o.json.empty()) ? fopen(o.json.c_str(), "a") : nullptr;
  long total_errors = 0;
  double busbw_sum = 0; int busbw_n = 0;   // nccl-tests' "Avg bus bandwidth": mean over every (size, placement) measured
  for (size_t bytes = o.min_bytes; bytes <= o.max_bytes; bytes *= o.factor) {
    // element counts per the op
    size_t count;          // the `count` argument of the API
    size_t in_elems, out_elems;
    if (is_ar) { count = bytes / is; in_elems = out_elems = count; }
    else if (is_ag) { count = bytes / is / n; in_elems = count; out_elems = count * n; }
    else if (is_rs) { count = bytes / is / n; in_elems = count * n; out_elems = count; }
    else { count = bytes / is / n; in_elems = out_elems = count * n; }
    const size_t E = 16 / is;
    if (!is_ar) count = count / E * E;
    if (count == 0) continue;
    if (!is_ar) { in_elems = is_ag ? count : count * n; out_elems = is_rs ? count : count * n; }
    const size_t in_b = in_elems * is, out_b = out_elems * os;
    const size_t slot_b = (std::max(in_b, out_b / os * is) + 4095) / 4096 * 4096;
    int slots = (int)std::min<size_t>(64, std::max<size_t>(1, o.window / slot_b));
    const size_t nshapes = o.shapes.empty() ? 1 : o.shapes.size();
    for (size_t si = 0; si < nshapes; si++) {
    if (!o.shapes.empty()) CC(b200collCommSetLaunchShape(ctx.comm, o.shapes[si].kind, o.shapes[si].ctas, o.shapes[si].threads));
    double res_us[2] = {-1, -1}; long res_err[2] = {0, 0};
    const char* algo_used = "?";
    for (int ip = 0; ip < 2; ip++) {
      if ((ip == 0 && o.inplace == 1) || (ip == 1 && o.inplace == 0)) continue;
      if (ip == 1 && (o.op == "alltoall" || is_sr || is_ga || is_sc || is != os)) continue;
      auto sbuf = [&](int slot) -> char* {
        char* base = ip ? (char*)recv : (char*)send;
        size_t off = (size_t)slot * slot_b;
        if (ip && is_ag) off += (size_t)rank * count * os;     // in-place all-gather: send = recv + rank*count
        return base + off;
      };
      auto rbuf = [&](int slot) -> char* {
        size_t off = (size_t)slot * (ip ? slot_b : slot_b / is * os);
        if (ip && is_rs) off += (size_t)rank * count * is;     // in-place reduce-scatter: recv = send + rank*count
        return (char*)recv + off;
      };
      auto launch = [&](int slot) {
        if (is_hc) {
          RT(cudaMemcpyAsync(rbuf(slot) + (size_t)rank * count * is, sbuf(slot), count * is, cudaMemcpyDeviceToDevice, st));
          for (int mask = 1; mask < n; mask <<= 1) {      // after the step with this mask every rank holds the 2*mask blocks of its sub-cube
            const int peer = rank ^ mask, mine0 = rank & ~(mask - 1), theirs0 = peer & ~(mask - 1);
            CC(b200collGroupStart());
            CC(b200collSend(rbuf(slot) + (size_t)mine0 * count * is, (size_t)mask * count * is, peer, ctx.comm, st));
            CC(b200collRecv(rbuf(slot) + (size_t)theirs0 * count * is, (size_t)mask * count * is, peer, ctx.comm, st));
            CC(b200collGroupEnd());
          }
        } else if (is_ga) {
          CC(b200collGroupStart());
          CC(b200collSend(sbuf(slot), count * is, kRoot, ctx.comm, st));
          if (rank == kRoot) for (int p = 0; p < n; p++) CC(b200collRecv(rbuf(slot) + (size_t)p * count * is, count * is, p, ctx.comm, st));
          CC(b200collGroupEnd());
        } else if (is_sc) {
          CC(b200collGroupStart());
          if (rank == kRoot) for (int p = 0; p < n; p++) CC(b200collSend(sbuf(slot) + (size_t)p * count * is, count * is, p, ctx.comm, st));
          CC(b200collRecv(rbuf(slot), count * is, kRoot, ctx.comm, st));
          CC(b200collGroupEnd());
        }
        else if (is_sr) {      // nccl-tests sendrecv_perf: one grouped send to the right neighbour and recv from the left one
          CC(b200collGroupStart());
          CC(b200collSend(sbuf(slot), count * is, (rank + 1) % n, ctx.comm, st));
          CC(b200collRecv(rbuf(slot), count * is, (rank + n - 1) % n, ctx.comm, st));
          CC(b200collGroupEnd());
        }
        else if (is_bc) CC(b200collBroadcast(sbuf(slot), rbuf(slot), count, &ep, kRoot, ctx.comm, st));
        else if (is_rd) CC(b200collReduce(sbuf(slot), rbuf(slot), count, &ep, b200collSum, kRoot, ctx.comm, st));
        else if (is_ar) CC(b200collAllReduce(sbuf(slot), rbuf(slot), count, &ep, b200collSum, ctx.comm, st));
        else if (is_ag) CC(b200collAllGather(sbuf(slot), rbuf(slot), count, &ep, ctx.comm, st));
        else if (is_rs) CC(b200collReduceScatter(sbuf(slot), rbuf(slot), count, &ep, b200collSum, ctx.comm, st));
        else CC(b200collAllToAll(sbuf(slot), rbuf(slot), count, &ep, ctx.comm, st));
      };
      // ---- correctness on slot 0 (fresh data, poisoned output)
      long errs = 0;
      if (o.check) {
        if (!ip) RT(cudaMemsetAsync(rbuf(0), 0x5A, out_b, st));
        if (ip && is_ag) fill(sbuf(0), in_elems, o.in_dt, rank, 0, st);
        else if (ip && is_rs) fill((char*)recv, in_elems, o.in_dt, rank, 0, st);
        else fill(sbuf(0), in_elems, o.in_dt, rank, 0, st);
        RT(cudaStreamSynchronize(st));
        spin_barrier(sh, 0, n, &gen_ctr[0]);
        if (o.skew_us && rank == 0) usleep(o.skew_us);
        launch(0);
        RT(cudaStreamSynchronize(st));
        spin_barrier(sh, 1, n, &gen_ctr[1]);
        b200collFault f;
        if (b200collCommGetAsyncError(ctx.comm, &f) != b200collSuccess) { fprintf(stderr, "rank %d WATCHDOG code=%u peer=%u block=%u expected=%u observed=%u op=%u\n", rank, f.code, f.peer, f.block, f.expected, f.observed, f.op); _exit(5); }
        const char* outp = (ip && is_rs) ? rbuf(0) : (ip ? (char*)recv : rbuf(0));
        const size_t check_elems = ((is_rd || (is_ga && !is_hc)) && rank != kRoot) ? 0 : out_elems;   // a rooted reduce defines the root's output only
        host.resize(check_elems * os);
        RT(cudaMemcpy(host.data(), outp, check_elems * os, cudaMemcpyDeviceToHost));
        const size_t stride = check_elems > (1u << 22) ? 61 : 1;   // sample large buffers
        for (size_t e = 0; e < check_elems; e += stride) {
          // fp8 inputs accumulate exactly in fp32 (the fill's sums are exact), so the result is the exact sum rounded once: no tolerance
          const bool fp8_in = o.in_dt == b200collFloat8e4m3 || o.in_dt == b200collFloat8e5m2;
          float want = expected(o, rank, n, e, count);
          if (fp8_in || o.out_dt == b200collFloat8e5m2) want = round_to(o.out_dt, want);
          const float got = to_f(host.data(), e, o.out_dt);
          const float tol = (!fp8_in && o.out_dt == b200collFloat8e4m3) ? fabsf(want) * 0.0725f + 0.002f : 0.0f;
          if (!(fabsf(got - want) <= tol)) { if (errs < 4) fprintf(stderr, "rank %d %s size %zu %s elem %zu: got %g want %g\n", rank, o.op.c_str(), bytes, ip ? "ip" : "oop", e, got, want); errs++; }
        }
      }
      // ---- timing
      for (int i = 0; i < o.warmup; i++) launch(i % slots);
      RT(cudaStreamSynchronize(st));
      spin_barrier(sh, 2, n, &gen_ctr[2]);
      RT(cudaEventRecord(e0, st));
      for (int i = 0; i < o.iters; i++) launch(i % slots);
      RT(cudaEventRecord(e1, st));
      RT(cudaEventSynchronize(e1));
      float ms = 0; RT(cudaEventElapsedTime(&ms, e0, e1));
      sh->ms[rank] = ms / o.iters; sh->errors[rank] = errs;
      spin_barrier(sh, 3, n, &gen_ctr[3]);
      float worst = 0; long es = 0;
      for (int r = 0; r < n; r++) { worst = std::max(worst, sh->ms[r]); es += sh->errors[r]; }
      res_us[ip] = worst * 1e3; res_err[ip] = es; total_errors += es;
      spin_barrier(sh, 0, n, &gen_ctr[0]);   // keep ms[] stable until everyone has read it
      b200collFault f;
      if (b200collCommGetAsyncError(ctx.comm, &f) != b200collSuccess) { fprintf(stderr, "rank %d WATCHDOG (timing) code=%u peer=%u block=%u expected=%u observed=%u\n", rank, f.code, f.peer, f.block, f.expected, f.observed); _exit(5); }
    }
    if (rank == 0) {
      size_t tb = is_ar ? count * is : count * is * n;   // nccl-tests "size"
      b200collOp_t opid = is_bc ? b200collOpBroadcast : is_rd ? b200collOpReduce : is_ar ? b200collOpAllReduce : is_ag ? b200collOpAllGather : is_rs ? b200collOpReduceScatter : b200collOpAllToAll;
      if (is_sr || is_ga || is_sc) algo_used = "p2p";
      else if (o.algo == "auto") algo_used = b200collAlgoName(b200collTunerPick(opid, is_ar ? count * is : count * is, n, info.nvls)); else algo_used = o.algo.c_str();
      const double factor = (is_bc || is_rd || is_sr) ? 1.0 : is_ar ? 2.0 * (n - 1) / n : (double)(n - 1) / n;
      double ab[2], bb[2];
      for (int ip = 0; ip < 2; ip++) { ab[ip] = res_us[ip] > 0 ? tb / res_us[ip] / 1e3 : 0; bb[ip] = n > 1 ? ab[ip] * factor : ab[ip]; if (res_us[ip] > 0) { busbw_sum += bb[ip]; busbw_n++; } }
      if (!o.shapes.empty()) printf("[k%d c%d t%d] ", o.shapes[si].kind, o.shapes[si].ctas, o.shapes[si].threads);
      printf("%14zu %12zu %6s %8s | %10.2f %8.2f %8.2f %6ld | %10.2f %8.2f %8.2f %6ld\n", tb, count, dt_name(o.in_dt), algo_used, res_us[0], ab[0], bb[0], res_err[0], res_us[1], ab[1], bb[1], res_err[1]);
      fflush(stdout);
      if (jf) {
        fprintf(jf, "{\"op\":\"%s\",\"nranks\":%d,\"bytes\":%zu,\"in\":\"%s\",\"out\":\"%s\",\"scale\":%g,\"algo\":\"%s\",\"oop_us\":%.3f,\"ip_us\":%.3f,\"oop_busbw\":%.3f,\"ip_busbw\":%.3f,\"errors\":%ld,\"mode\":\"%s\",\"shape\":\"%d:%d:%d\"}\n",
                o.op.c_str(), n, tb, dt_name(o.in_dt), dt_name(o.out_dt), o.scale, algo_used, res_us[0], res_us[1], bb[0], bb[1], res_err[0] + res_err[1], o.procs ? "procs" : "threads", o.shapes.empty() ? -1 : o.shapes[si].kind, o.shapes.empty() ? 0 : o.shapes[si].ctas, o.shapes.empty() ? 0 : o.shapes[si].threads);
        fflush(jf);
      }
    }
    }   // shapes
  }
  if (jf) fclose(jf);
  b200collStats s; CC(b200collCommStatsGet(ctx.comm, &s));
  if (rank == 0) {
    printf("# Out of bounds values : %ld %s\n", total_errors, total_errors ? "FAILED" : "OK");
    printf("# Avg bus bandwidth    : %g\n", busbw_n ? busbw_sum / busbw_n : 0.0);
    printf("# launches=%llu staged_calls=%llu errors=%ld\n", (unsigned long long)s.kernel_launches, (unsigned long long)s.staged_calls, total_errors);
    fflush(stdout);      // --procs children leave through _exit(): nothing buffered survives it
  }
  CC(b200collMemFree(ctx.comm, recv));
  CC(b200collMemFree(ctx.comm, send));
  RT(cudaStreamDestroy(st));
  return total_errors ? 4 : 0;
}

// nccl-tests compatibility (the reference's pods run `<op>_perf -b .. -e .. -f 2 -g 1 -w 5 --iters 100 -c 0` under mpirun,
// gpudirect-tcpx/nccl-config.yaml:61-62, gpudirect-rdma/nccl-test-a4x-max-jobset.yaml:153): the binary answers to those
// names through symlinks, takes the same flags, and when a launcher exported a rank (OpenMPI, PMI, torchrun) it is ONE rank
// of the job instead of forking its own.
static const char* op_from_argv0(const char* argv0) {
  const char* base = strrchr(argv0, '/'); base = base ? base + 1 : argv0;
  static const struct { const char* name; const char* op; } kNames[] = {{"all_reduce_perf", "all_reduce"}, {"all_gather_perf", "all_gather"}, {"reduce_scatter_perf", "reduce_scatter"},
                                                                        {"alltoall_perf", "alltoall"}, {"broadcast_perf", "broadcast"}, {"reduce_perf", "reduce"}, {"sendrecv_perf", "sendrecv"}, {"gather_perf", "gather"}, {"scatter_perf", "scatter"}, {"hypercube_perf", "hypercube"}};
  for (auto& k : kNames) if (!strcmp(base, k.name)) return k.op;
  return nullptr;
}
struct LauncherRank { int rank = -1, size = 0, local_rank = 0; std::string job; };
static LauncherRank launcher_rank() {
  LauncherRank l;
  static const char* kRank[] = {"OMPI_COMM_WORLD_RANK", "PMI_RANK", "PMIX_RANK", "RANK"};
  static const char* kSize[] = {"OMPI_COMM_WORLD_SIZE", "PMI_SIZE", "", "WORLD_SIZE"};
  static const char* kLocal[] = {"OMPI_COMM_WORLD_LOCAL_RANK", "MPI_LOCALRANKID", "", "LOCAL_RANK"};
  for (int i = 0; i < 4; i++) {
    const char* r = getenv(kRank[i]); const char* s = *kSize[i] ? getenv(kSize[i]) : nullptr;
    if (!r || !s) continue;
    l.rank = atoi(r); l.size = atoi(s);
    const char* lr = *kLocal[i] ? getenv(kLocal[i]) : nullptr;
    l.local_rank = lr ? atoi(lr) : l.rank;
    break;
  }
  // every rank must derive the same id: an explicit job id, else the launcher's, else the rendezvous address
  for (const char* k : {"B200COLL_JOB_ID", "OMPI_MCA_ess_base_jobid", "PMIX_NAMESPACE", "PMI_JOBID", "TORCHELASTIC_RUN_ID"}) if (const char* v = getenv(k)) { l.job = std::string(k) + "=" + v; break; }
  if (l.job.empty()) { const char* a = getenv("MASTER_ADDR"); const char* p = getenv("MASTER_PORT"); l.job = std::string(a ? a : "local") + ":" + (p ? p : "0"); }
  return l;
}

int main(int argc, char** argv) {
  Opts o;
  int gpus_per_proc = 0;
  if (const char* op = op_from_argv0(argv[0])) o.op = op;
  for (int i = 1; i < argc; i++) {
    std::string a = argv[i];
    auto next = [&]() -> const char* { if (i + 1 >= argc) { fprintf(stderr, "missing value for %s\n", a.c_str()); exit(1); } return argv[++i]; };
    if (a == "--op") o.op = next();
    else if (a == "--ranks") o.nranks = atoi(next());
    else if (a == "--devs") { std::string s = next(); size_t p = 0; while (p < s.size()) { o.devs.push_back(atoi(s.c_str() + p)); p = s.find(',', p); if (p == std::string::npos) break; p++; } }
    else if (a == "--procs") o.procs = true;
    else if (a == "-b" || a == "--min") o.min_bytes = parse_size(next());
    else if (a == "-e" || a == "--max") o.max_bytes = parse_size(next());
    else if (a == "-f" || a == "--factor") o.factor = atoi(next());
    else if (a == "--dtype" || a == "-d" || a == "--datatype") o.in_dt = o.out_dt = parse_dt(next());
    else if (a == "-g" || a == "--ngpus") gpus_per_proc = atoi(next());
    else if (a == "-o" || a == "--redop") { std::string v = next(); if (v != "sum") { fprintf(stderr, "only -o sum is benchmarked (avg is a fused scale: use --scale)\n"); return 1; } }
    else if (a == "-t" || a == "--nthreads" || a == "-m" || a == "--agg_iters" || a == "-p" || a == "--parallel_init" || a == "-z" || a == "--blocking" || a == "-a" || a == "--average" ||
             a == "-G" || a == "--cudagraph" || a == "-C" || a == "--report_cputime" || a == "-R" || a == "--local_register" || a == "-T" || a == "--timeout" || a == "-r" || a == "--root") (void)next();   // accepted, no effect here
    else if (a == "--out-dtype") o.out_dt = parse_dt(next());
    else if (a == "--scale") o.scale = (float)atof(next());
    else if (a == "--algo") o.algo = next();
    else if (a == "--iters" || a == "-n") o.iters = atoi(next());
    else if (a == "--warmup" || a == "-w") o.warmup = atoi(next());
    else if (a == "--check" || a == "-c") o.check = atoi(next());
    else if (a == "--inplace") o.inplace = atoi(next());
    else if (a == "--max-ctas") o.max_ctas = atoi(next());
    else if (a == "--window") o.window = parse_size(next());
    else if (a == "--json") o.json = next();
    else if (a == "--skew-us") o.skew_us = atoi(next());
    else if (a == "--sweep") {
      std::string v = next(); size_t p = 0;
      while (p < v.size()) {
        Opts::Shape sh{0, 0, 0};
        if (sscanf(v.c_str() + p, "%d:%d:%d", &sh.kind, &sh.ctas, &sh.threads) == 3) o.shapes.push_back(sh);
        p = v.find(',', p); if (p == std::string::npos) break; p++;
      }
    }
    else if (a == "--selfcheck") { char buf[4096]; b200collResult_t r = b200collSelfCheck(buf, sizeof(buf)); fputs(buf, stdout); return r == b200collSuccess ? 0 : 1; }
    else if (a == "-h" || a == "--help") {
      puts("b200coll_perf (also all_reduce_perf, all_gather_perf, reduce_scatter_perf, alltoall_perf, broadcast_perf, reduce_perf, sendrecv_perf, gather_perf, scatter_perf, hypercube_perf): nccl-tests style sweep on libb200coll\n"
           "  --op NAME                 collective (implied by the name the binary is called by)\n"
           "  -b/-e SIZE -f N           sweep from -b to -e bytes multiplying by -f (1K, 64M, 1G ...)\n"
           "  -g N | --ranks N | --devs a,b,..   ranks in this process (threads); --procs forks one process per rank instead\n"
           "  under mpirun / torchrun (OMPI_COMM_WORLD_*, PMI_*, RANK/WORLD_SIZE/LOCAL_RANK) each process is one rank; B200COLL_JOB_ID names the job\n"
           "  -w N -n/--iters N -c 0|1  warm-up, timed iterations, check results against the host reference\n"
           "  -d float|half|bfloat16|e4m3|e5m2   input type; --out-dtype T (same names) and --scale X fuse a cast / scale into the collective\n"
           "  --algo auto|ll|ll2|oneshot|twoshot|nvls   --inplace 0|1|2   --max-ctas N   --sweep kind:ctas:threads,...   --json FILE   --window SIZE\n"
           "  --selfcheck               report whether this node can run the NVLink fast paths (exit 1 if not)");
      return 0;
    }
    else { fprintf(stderr, "unknown flag %s\n", a.c_str()); return 1; }
  }
  if (o.factor < 2) o.factor = 2;
  const LauncherRank lr = launcher_rank();
  if (lr.size > 1 && o.devs.empty() && !o.procs) {
    // one rank of an mpirun / torchrun job (nccl-tests' -g 1 layout): rendezvous on the job id, timing page in /dev/shm
    if (gpus_per_proc > 1) { fprintf(stderr, "-g %d under a launcher is not supported: run one rank per GPU (-g 1)\n", gpus_per_proc); return 1; }
    if (lr.size > B200COLL_MAX_RANKS) { fprintf(stderr, "libb200coll is an intra-node transport: %d ranks > %d GPUs of one NVSwitch domain\n", lr.size, B200COLL_MAX_RANKS); return 1; }
    int nd = 0; RT(cudaGetDeviceCount(&nd));
    const int dev = nd > 0 ? lr.local_rank % nd : 0;
    unsigned h = 2166136261u; for (char ch : lr.job) h = (h ^ (unsigned char)ch) * 16777619u;
    char shm_name[64]; snprintf(shm_name, sizeof shm_name, "/b200coll_perf.%08x", h);
    int fd = shm_open(shm_name, O_CREAT | O_RDWR, 0600);
    if (fd < 0 || ftruncate(fd, sizeof(Shared)) != 0) { perror("shm_open"); return 1; }
    Shared* sh = (Shared*)mmap(nullptr, sizeof(Shared), PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (sh == MAP_FAILED) { perror("mmap"); return 1; }
    o.nranks = lr.size; o.procs = true;
    b200collConfig cfg; b200collConfigDefault(&cfg);
    const size_t is_ = b200collTypeSize(o.in_dt), os_ = b200collTypeSize(o.out_dt);
    if (!getenv("B200COLL_ARENA_MB")) cfg.arena_bytes = std::max(o.window, o.max_bytes) + std::max(o.window / is_ * os_, o.max_bytes / is_ * os_) + (64u << 20);
    b200collUniqueId id; CC(b200collUniqueIdFromString(("perf/" + lr.job).c_str(), &id));
    RT(cudaSetDevice(dev));
    b200collComm_t comm;
    CC(b200collCommInitRank(&comm, lr.size, &id, lr.rank, &cfg));
    // a crashed earlier job with the same id may have left counters behind: wipe the page between two host barriers,
    // i.e. after everybody mapped it and before anybody counts on it
    CC(b200collHostBarrier(comm));
    if (lr.rank == 0) memset((void*)sh, 0, sizeof(Shared));
    CC(b200collHostBarrier(comm));
    int rc = run_rank(o, RankCtx{lr.rank, lr.size, comm, dev}, sh);
    CC(b200collCommDestroy(comm));          // ends with a host barrier: every rank is past its last use of the page
    if (lr.rank == 0) shm_unlink(shm_name);
    return rc;
  }
  if (gpus_per_proc > 0 && o.devs.empty() && o.nranks == 0) o.nranks = gpus_per_proc;     // nccl-tests -g N without a launcher: N ranks in this process
  if (o.devs.empty()) {
    int nd = 0; cudaGetDeviceCount(&nd);
    if (o.nranks == 0) o.nranks = nd > 0 ? nd : 1;
    for (int i = 0; i < o.nranks; i++) o.devs.push_back(nd > 0 ? i % nd : 0);
  }
  o.nranks = (int)o.devs.size();
  const int n = o.nranks;
  Shared* sh = (Shared*)mmap(nullptr, sizeof(Shared), PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS, -1, 0);
  memset(sh, 0, sizeof(Shared));
  b200collConfig cfg; b200collConfigDefault(&cfg);
  // arena: two windows (+ max buffers) and slack
  const size_t is_ = b200collTypeSize(o.in_dt), os_ = b200collTypeSize(o.out_dt);
  size_t need = std::max(o.window, o.max_bytes) + std::max(o.window / is_ * os_, o.max_bytes / is_ * os_) + (64u << 20);
  if (!getenv("B200COLL_ARENA_MB")) cfg.arena_bytes = need;
  if (o.procs) {
    b200collUniqueId id; CC(b200collGetUniqueId(&id));
    std::vector<pid_t> kids;
    for (int r = 0; r < n; r++) {
      pid_t p = fork();
      if (p == 0) {
        RT(cudaSetDevice(o.devs[r]));
        b200collComm_t comm;
        CC(b200collCommInitRank(&comm, n, &id, r, &cfg));
        int rc = run_rank(o, RankCtx{r, n, comm, o.devs[r]}, sh);
        CC(b200collCommDestroy(comm));
        _exit(rc);
      }
      kids.push_back(p);
    }
    int worst = 0;
    for (pid_t p : kids) { int stt = 0; waitpid(p, &stt, 0); int rc = WIFEXITED(stt) ? WEXITSTATUS(stt) : 128; worst = std::max(worst, rc); }
    return worst;
  }
  std::vector<b200collComm_t> comms(n);
  CC(b200collCommInitAll(comms.data(), n, o.devs.data(), &cfg));
  std::vector<std::thread> th;
  std::vector<int> rcs(n, 0);
  for (int r = 0; r < n; r++) th.emplace_back([&, r] { rcs[r] = run_rank(o, RankCtx{r, n, comms[r], o.devs[r]}, sh); });
  for (auto& t : th) t.join();
  for (int r = 0; r < n; r++) CC(b200collCommDestroy(comms[r]));
  int worst = 0; for (int rc : rcs) worst = std::max(worst, rc);
  return worst;
}
