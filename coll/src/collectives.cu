// libb200coll collective entry points: argument validation, algorithm choice (tuner table +
// feasibility), staging for buffers outside the symmetric arena, type dispatch, kernel launch.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "comm.h"
#include "kernels.cuh"

namespace b200coll {

template <typename T> struct Tag { using type = T; };
using bf16 = __nv_bfloat16;
using f8 = __nv_fp8_e4m3;
using f8e5 = __nv_fp8_e5m2;

// Supported (in, out) pairs: same type, widen to f32, narrow f32 to 16-bit, quantise to e4m3 / e5m2, dequantise fp8 to a wider
// type (no cross-fp8 pair).
template <typename F>
static b200collResult_t dispatch_types(b200collDataType_t in, b200collDataType_t out, F&& f) {
  if (in == b200collFloat32) {
    switch (out) {
      case b200collFloat32: return f(Tag<float>{}, Tag<float>{});
      case b200collBfloat16: return f(Tag<float>{}, Tag<bf16>{});
      case b200collFloat16: return f(Tag<float>{}, Tag<__half>{});
      case b200collFloat8e4m3: return f(Tag<float>{}, Tag<f8>{});
      case b200collFloat8e5m2: return f(Tag<float>{}, Tag<f8e5>{});
      default: break;
    }
  } else if (in == b200collBfloat16) {
    switch (out) {
      case b200collBfloat16: return f(Tag<bf16>{}, Tag<bf16>{});
      case b200collFloat32: return f(Tag<bf16>{}, Tag<float>{});
      case b200collFloat8e4m3: return f(Tag<bf16>{}, Tag<f8>{});
      case b200collFloat8e5m2: return f(Tag<bf16>{}, Tag<f8e5>{});
      default: break;
    }
  } else if (in == b200collFloat16) {
    switch (out) {
      case b200collFloat16: return f(Tag<__half>{}, Tag<__half>{});
      case b200collFloat32: return f(Tag<__half>{}, Tag<float>{});
      case b200collFloat8e4m3: return f(Tag<__half>{}, Tag<f8>{});
      case b200collFloat8e5m2: return f(Tag<__half>{}, Tag<f8e5>{});
      default: break;
    }
  } else if (in == b200collFloat8e4m3) {
    switch (out) {
      case b200collFloat8e4m3: return f(Tag<f8>{}, Tag<f8>{});
      case b200collBfloat16: return f(Tag<f8>{}, Tag<bf16>{});
      case b200collFloat16: return f(Tag<f8>{}, Tag<__half>{});
      case b200collFloat32: return f(Tag<f8>{}, Tag<float>{});
      default: break;
    }
  } else if (in == b200collFloat8e5m2) {
    switch (out) {
      case b200collFloat8e5m2: return f(Tag<f8e5>{}, Tag<f8e5>{});
      case b200collBfloat16: return f(Tag<f8e5>{}, Tag<bf16>{});
      case b200collFloat16: return f(Tag<f8e5>{}, Tag<__half>{});
      case b200collFloat32: return f(Tag<f8e5>{}, Tag<float>{});
      default: break;
    }
  }
  set_last_error("unsupported (in_dtype, out_dtype) pair");
  return b200collInvalidArgument;
}

// No multicast (NVLS) kernel is built for an fp8 input: the switch reduces fp8 with an f16 accumulator only (ptxas refuses .acc::f32
// for e4m3x4 / e5m2x4), and those kernels have not yet run on a multi-GPU NVSwitch system. An fp8 call the tuner sends to NVLS takes
// two-shot, and the Lamport kernels write their slots with P2P stores instead of multimem.st. `if constexpr` keeps the fp8 multicast
// instantiations out of the library altogether.
template <typename T> constexpr bool kMcKernels = !IsFp8<T>::value;
static bool is_fp8(b200collDataType_t t) { return t == b200collFloat8e4m3 || t == b200collFloat8e5m2; }

// f(std::true_type{}) launches a kernel's multicast variant, f(std::false_type{}) its P2P one; only an input type with multicast
// kernels ever reaches the former.
template <typename InT, typename F>
static auto with_mc(bool mc, F&& f) {
  if constexpr (kMcKernels<InT>) { if (mc) return f(std::true_type{}); }
  return f(std::false_type{});
}

// What the algorithm of a fused collective depends on besides the communicator (ranks, multicast, forced algorithm, tuner table).
struct CallFacts {
  b200collOp_t op;
  size_t bytes;                  // as the tuner sees them
  b200collDataType_t in_dtype;
  bool sym_in, sym_out;          // inside the symmetric arena
  bool inplace, same_size;       // send == recv; input and output elements of equal size
};

// The algorithm a call runs: the forced algorithm or the tuner's pick, moved to one that can serve the call. b200collAlgoAuto means
// that no all-reduce algorithm can run on these buffers and the call is staged; `staging` then asks for the algorithm that runs
// between the two staging halves (symmetric, not in place), which follows no pick.
static b200collAlgo_t resolve_algo(const b200collComm* c, const CallFacts& f, bool staging = false) {
  const bool mc = c->nvls && !is_fp8(f.in_dtype);      // no multicast kernel for an fp8 input (above)
  b200collAlgo_t a = c->forced_algo != b200collAlgoAuto ? c->forced_algo : b200collTunerPick(f.op, f.bytes, c->nranks, c->nvls);
  switch (f.op) {
    case b200collOpAllReduce: {
      auto feasible = [&](b200collAlgo_t x) {
        switch (x) {
          case b200collAlgoLL: return f.bytes <= kLLOneShotMaxBytes;
          case b200collAlgoLL2: return f.same_size && f.bytes <= kLLOneShotMaxBytes * (size_t)c->nranks;
          case b200collAlgoOneShot: return f.sym_in && !f.inplace;
          case b200collAlgoTwoShot: return f.sym_in && f.sym_out;
          case b200collAlgoNvls: return mc && f.sym_in && f.sym_out;
          default: return false;
        }
      };
      if (!staging && feasible(a)) return a;
      for (b200collAlgo_t x : {b200collAlgoNvls, b200collAlgoTwoShot, b200collAlgoOneShot, b200collAlgoLL, b200collAlgoLL2})
        if (feasible(x) && !(x == b200collAlgoNvls && c->nranks == 2)) return x;
      return b200collAlgoAuto;
    }
    case b200collOpAllGather:
    case b200collOpReduceScatter:
      if (a == b200collAlgoLL2) a = b200collAlgoLL;
      if ((a == b200collAlgoLL && f.bytes > kLLOneShotMaxBytes) || (a == b200collAlgoNvls && !mc) || a == b200collAlgoOneShot || a == b200collAlgoCopy) a = b200collAlgoTwoShot;
      return a;
    case b200collOpAllToAll:
      if (a == b200collAlgoLL2) a = b200collAlgoLL;
      return (a == b200collAlgoLL && f.bytes <= kLLOneShotMaxBytes) ? b200collAlgoLL : b200collAlgoTwoShot;
    default:                     // broadcast, reduce: multimem or P2P
      return (a == b200collAlgoNvls && mc) ? b200collAlgoNvls : b200collAlgoTwoShot;
  }
}

#define LAUNCH_CHECK(c)                                                                                  \
  do {                                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                                \
    if (e__ != cudaSuccess) { set_last_error(std::string("kernel launch failed: ") + cudaGetErrorString(e__)); return b200collUnhandledCudaError; } \
    (c)->stats.kernel_launches++;                                                                        \
  } while (0)

struct Grid { int blocks, threads; };

// Every kernel goes through cudaLaunchKernelEx so that back-to-back collectives can use programmatic dependent launch
// (on by default, B200COLL_PDL=0 disables): the next kernel's launch latency overlaps the current kernel's execution; each kernel starts with
// griddepcontrol.launch_dependents + griddepcontrol.wait, so it still observes its predecessor's completed memory.
// Never with virtual ranks (several communicators on one GPU): a pre-launched dependent grid parks its CTAs on SMs
// that another rank's current kernel still needs, and ranks that spin on each other then deadlock (seen at 1 MiB with
// 4 ranks on one B200). With one rank per GPU every CTA of kernel i is resident before kernel i+1 may start.
// Measured on 2 x B200 (profiles/latency_ab.md): the overlap wins ~1 us per back-to-back call up to 4 KiB (4.4 vs 5.5 us at 1 KiB) and
// LOSES 0.5 - 1 us from 16 KiB up (the early-launched grid sits on the SMs while its predecessor still needs them, and its
// griddepcontrol.wait returns only after the predecessor's memory flush). So only launches whose message is at most
// B200COLL_PDL_MAX_KB (default 8) carry the attribute; launch_ll sets the flag for the launch it is about to make.
static thread_local bool t_pdl_small = false;
static size_t pdl_max_bytes() {
  static const size_t v = [] { const char* e = getenv("B200COLL_PDL_MAX_KB"); return (size_t)(e && *e ? atol(e) : 8) << 10; }();
  return v;
}
static bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("B200COLL_PDL"); return !(e && *e == '0'); }();      // on unless B200COLL_PDL=0
  return on && t_pdl_small && g_loopback_comms.load(std::memory_order_relaxed) == 0;
}
template <typename... KArgs, typename... Args>
static void launch_k_smem(void (*kernel)(KArgs...), int blocks, int threads, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)blocks); cfg.blockDim = dim3((unsigned)threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr;
  if (pdl_enabled()) {
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr; cfg.numAttrs = 1;
  }
  (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);   // the error is picked up by LAUNCH_CHECK's cudaGetLastError
}
template <typename... KArgs, typename... Args>
static void launch_k(void (*kernel)(KArgs...), int blocks, int threads, cudaStream_t st, Args&&... args) {
  launch_k_smem(kernel, blocks, threads, 0, st, std::forward<Args>(args)...);
}

// Pick the smallest block size that still covers `vecs` with <= max_ctas blocks (small work spreads over more SMs),
// unless the family's shape pins the thread count.
enum { kShapeNvls = 0, kShapeP2p = 1, kShapeLL = 2, kShapeNvlsRs = 3, kShapeRooted = 4 };
static Grid pick_grid(const b200collComm* c, int kind, size_t vecs, int unroll) {
  static const int forced = [] { const char* e = getenv("B200COLL_FORCE_THREADS"); return e ? atoi(e) : 0; }();
  const int max_ctas = std::max(1, std::min(c->shape[kind].max_ctas > 0 ? c->shape[kind].max_ctas : c->max_ctas, c->max_ctas));
  int pinned = c->shape[kind].threads;
  if (forced >= 32 && forced <= 512) pinned = forced;
  if (pinned) {
    size_t b = (vecs + (size_t)pinned * unroll - 1) / ((size_t)pinned * unroll);
    return Grid{(int)std::max<size_t>(1, std::min<size_t>(b, (size_t)max_ctas)), pinned};
  }
  for (int t : {128, 256, 512}) {
    size_t b = (vecs + (size_t)t * unroll - 1) / ((size_t)t * unroll);
    if (b <= (size_t)max_ctas || t == 512) return Grid{(int)std::max<size_t>(1, std::min<size_t>(b, (size_t)max_ctas)), t};
  }
  return Grid{1, 128};
}

static size_t arena_off(b200collComm* c, const void* p) { return reinterpret_cast<CUdeviceptr>(p) - c->peer_va[c->rank]; }

b200collResult_t copy_rows(char* dst, size_t dst_pitch, const char* src, size_t src_pitch, size_t bytes, int rows, cudaStream_t st) {
  for (int r = 0; r < rows; r++) {
    const cudaError_t e = cudaMemcpyAsync(dst + (size_t)r * dst_pitch, src + (size_t)r * src_pitch, bytes, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) { set_last_error(cudaGetErrorString(e)); return b200collUnhandledCudaError; }
  }
  return b200collSuccess;
}

static bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }
static size_t out_align(size_t in_sz, size_t out_sz) { return std::min<size_t>(16, 16 / in_sz * out_sz); }

static b200collResult_t check_common(b200collComm* c, const void* send, void* recv, const b200collEpilogue* ep) {
  if (!c || !send || !recv || !ep) { set_last_error("null argument"); return b200collInvalidArgument; }
  if (dispatch_types(ep->in_dtype, ep->out_dtype, [](auto, auto) { return b200collSuccess; }) != b200collSuccess) {
    set_last_error("unsupported (in_dtype, out_dtype) pair (fp32 / fp16 / bf16 / fp8 e4m3 / fp8 e5m2 in and out; integer and fp64 payloads: reductions take the generic path, data movement takes them as words)");
    return b200collInvalidArgument;
  }
  const size_t is = b200collTypeSize(ep->in_dtype), os = b200collTypeSize(ep->out_dtype);
  if (!aligned(send, 16) || !aligned(recv, out_align(is, os))) { set_last_error("send must be 16-byte aligned and recv aligned to one output vector"); return b200collInvalidArgument; }
  if (c->fault_host && *const_cast<volatile uint32_t*>(&c->fault_host->code) != 0) { set_last_error("communicator is poisoned by an earlier watchdog fault"); return b200collRemoteError; }
  return b200collSuccess;
}

// B200COLL_NVTX=1: one NVTX mark per collective ("b200coll all_reduce nvls 67108864 B") so timelines show which algorithm
// a call took (SURVEY §5.1: the reference only passes NCCL_DEBUG through to opaque payloads).
static void account(b200collComm* c, b200collOp_t op, size_t bytes, b200collAlgo_t algo) {
  c->stats.calls[op]++; c->stats.bytes[op] += bytes; c->stats.algo_calls[algo]++;
  if ((c->stats_tick++ & 0xFF) == 0) stats_page_publish(c);      // keep the exported counters fresh without the application polling
  static const bool nvtx = [] { const char* e = getenv("B200COLL_NVTX"); return e && *e && *e != '0'; }();
  if (nvtx || debug_level() >= 2) {
    static const char* kOps[] = {"all_reduce", "all_gather", "reduce_scatter", "alltoall", "broadcast", "reduce"};
    char msg[96];
    snprintf(msg, sizeof(msg), "b200coll %s %s %zu B", kOps[op], b200collAlgoName(algo), bytes);
    if (nvtx) nvtxMarkA(msg);
    dbg(2, "rank %d: %s", c->rank, msg);
  }
}

// ------------------------------------------------------------------------------------------------ symmetry cross-check (debug)
// The zero-copy paths address peers by MY arena offset and pick the algorithm from MY view of the buffers: ranks that pass different
// offsets (allocation order drifted), counts or placements would read and write wrong peer addresses or run different kernels with
// different barrier counts. B200COLL_CHECK=1 compares (op, algorithm, count, offsets) across ranks over the bootstrap channel before
// every such launch and fails the call with InvalidUsage instead (host-synchronous, multi-process communicators only: a debugging aid).
static b200collResult_t cross_check(b200collComm* c, b200collOp_t op, b200collAlgo_t algo, size_t count, size_t off_a, size_t off_b) {
  static const bool on = [] { const char* e = getenv("B200COLL_CHECK"); return e && *e && *e != '0'; }();
  if (!on || !c->boot || c->nranks == 1) return b200collSuccess;
  struct Sig { unsigned long long op, algo, count, a, b; } mine = {(unsigned long long)op, (unsigned long long)algo, count, off_a, off_b};
  std::vector<char> all;
  const std::string e = c->boot->allgather(&mine, sizeof(mine), &all);
  if (!e.empty()) { set_last_error("cross-check: bootstrap: " + e); return b200collSystemError; }
  for (int r = 0; r < c->nranks; r++) {
    Sig s; memcpy(&s, all.data() + (size_t)r * sizeof(Sig), sizeof(Sig));
    if (memcmp(&s, &mine, sizeof(Sig)) != 0) {
      char msg[256];
      snprintf(msg, sizeof msg, "ranks disagree on a symmetric collective: rank %d has (op %llu, algo %s, count %llu, offsets %llu / %llu), rank %d has (op %llu, algo %s, count %llu, offsets %llu / %llu)",
               c->rank, mine.op, b200collAlgoName((b200collAlgo_t)mine.algo), mine.count, mine.a, mine.b, r, s.op, b200collAlgoName((b200collAlgo_t)s.algo), s.count, s.a, s.b);
      set_last_error(msg);
      return b200collInvalidUsage;
    }
  }
  return b200collSuccess;
}

// ------------------------------------------------------------------------------------------------ copy-engine path (k_bulk)
// B200COLL_BULK=0 turns it off (A/B against the LDG/STG kernels); B200COLL_BULK_MIN_KB moves the threshold (default 1024: below it the
// ring's set-up costs more than it saves). Only for the identity epilogue and sizes that are multiples of 16 bytes.
static bool bulk_enabled() {
  static const bool on = [] { const char* e = getenv("B200COLL_BULK"); return !(e && *e == '0'); }();
  return on;
}
static size_t bulk_min_bytes() {
  static const size_t v = [] { const char* e = getenv("B200COLL_BULK_MIN_KB"); return (size_t)(e && *e ? atol(e) : 1024) << 10; }();
  return v;
}
static b200collResult_t launch_bulk(b200collComm* c, BulkArgs& a, bool sync, b200collOp_t op, cudaStream_t st) {
  // the opt-in to 64 KiB of dynamic shared memory is per device (one process may drive several GPUs: InitAll, nccl-tests -g N)
  static std::atomic<unsigned long long> attr_done{0};
  const unsigned long long bit = 1ull << (c->device & 63);
  if (!(attr_done.load(std::memory_order_acquire) & bit)) {
    cudaFuncSetAttribute(k_bulk<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBulkSmemBytes);
    cudaFuncSetAttribute(k_bulk<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBulkSmemBytes);
    attr_done.fetch_or(bit, std::memory_order_release);
  }
  a.chunk_prefix[0] = 0;
  for (int g = 0; g < a.nseg; g++) a.chunk_prefix[g + 1] = a.chunk_prefix[g] + (a.bytes[g] + kBulkChunk - 1) / kBulkChunk;
  for (int g = a.nseg + 1; g <= kMaxRanks; g++) a.chunk_prefix[g] = a.chunk_prefix[a.nseg];
  static const int env_ctas = [] { const char* e = getenv("B200COLL_BULK_CTAS"); return e ? atoi(e) : 0; }();
  // 3 CTAs of 64 KiB shared memory fit on an SM; peers: stay within the collective cap so that every rank's grid is co-resident
  int cap = sync ? std::min(c->max_ctas, 2 * std::max(1, c->sm_count)) : 3 * std::max(1, c->sm_count);
  if (env_ctas > 0) cap = std::min(env_ctas, sync ? c->max_ctas : env_ctas);
  // every rank must launch the same grid (block b meets block b in the barriers): size it from what all ranks know — for rooted and
  // personalised ops the caller passes the symmetric chunk count in chunk_prefix[kMaxRanks] ... the largest segment list is the same on
  // every rank for all-gather / all-to-all (equal counts); broadcast and all-to-all-v pass `grid_hint`.
  const unsigned long long chunks = std::max<unsigned long long>(a.chunk_prefix[a.nseg], c->bulk_grid_hint);
  c->bulk_grid_hint = 0;
  const int blocks = (int)std::max<unsigned long long>(1, std::min<unsigned long long>(chunks, (unsigned long long)cap));
  if (sync) launch_k_smem(k_bulk<true>, blocks, kBulkThreads, kBulkSmemBytes, st, c->dev, a, (uint32_t)op);
  else launch_k_smem(k_bulk<false>, blocks, kBulkThreads, kBulkSmemBytes, st, c->dev, a, (uint32_t)op);
  LAUNCH_CHECK(c);
  c->stats.bulk_launches++;
  return b200collSuccess;
}

// ------------------------------------------------------------------------------------------------ nranks == 1
static b200collResult_t copy_scale(b200collComm* c, const void* send, void* recv, size_t count, const b200collEpilogue* ep, float scale, cudaStream_t st) {
  if (send == recv && ep->in_dtype == ep->out_dtype && scale == 1.0f) return b200collSuccess;
  const size_t nbytes = count * b200collTypeSize(ep->in_dtype);
  if (bulk_enabled() && ep->in_dtype == ep->out_dtype && scale == 1.0f && nbytes >= bulk_min_bytes() && nbytes % 16 == 0 && aligned(recv, 16)) {
    BulkArgs a = {};
    a.nseg = 1; a.src[0] = static_cast<const char*>(send); a.bytes[0] = nbytes; a.dst_local = static_cast<char*>(recv);
    return launch_bulk(c, a, false, b200collOpAllReduce, st);
  }
  return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
    using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
    // streaming copy: no peers to wait for, so oversubscribe the chip (8 CTAs of 256 threads per SM) instead of the collective cap
    const size_t vecs = count / Epv<InT>::value + 1;
    Grid g{(int)std::max<size_t>(1, std::min<size_t>((vecs + 1023) / 1024, (size_t)std::max(1, c->sm_count) * 8)), 256};
    launch_k(k_copy_scale<InT, OutT>, g.blocks, g.threads, st, static_cast<const InT*>(send), static_cast<OutT*>(recv), count, scale);
    LAUNCH_CHECK(c);
    return b200collSuccess;
  });
}

// ------------------------------------------------------------------------------------------------ LL (all ops)
static b200collResult_t launch_ll(b200collComm* c, b200collOp_t op, const void* send, void* recv, size_t count, const b200collEpilogue* ep, float scale, cudaStream_t st) {
  return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
    using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
    constexpr int E = Epv<InT>::value;
    const size_t nv = (count + E - 1) / E;
    Grid g = pick_grid(c, kShapeLL, nv, 1);
    const InT* in = static_cast<const InT*>(send); OutT* out = static_cast<OutT*>(recv);
    struct PdlScope { PdlScope(bool v) { t_pdl_small = v; } ~PdlScope() { t_pdl_small = false; } } pdl_scope(count * sizeof(InT) <= pdl_max_bytes());
    if (op == b200collOpAllReduce)
      with_mc<InT>(c->nvls, [&](auto mc) { launch_k(k_ll<InT, OutT, false, true, decltype(mc)::value>, g.blocks, g.threads, st, c->dev, in, out, count, scale, op); });
    else if (op == b200collOpAllGather)
      with_mc<InT>(c->nvls, [&](auto mc) { launch_k(k_ll<InT, OutT, false, false, decltype(mc)::value>, g.blocks, g.threads, st, c->dev, in, out, count, scale, op); });
    else if (op == b200collOpReduceScatter)
      launch_k(k_ll<InT, OutT, true, true, false>, g.blocks, g.threads, st, c->dev, in, out, count, scale, op);
    else
      launch_k(k_ll<InT, OutT, true, false, false>, g.blocks, g.threads, st, c->dev, in, out, count, scale, op);
    LAUNCH_CHECK(c);
    return b200collSuccess;
  });
}

// Two-shot Lamport all-reduce (same in/out type only; any local pointers, in-place allowed).
static b200collResult_t launch_ll2(b200collComm* c, const void* send, void* recv, size_t count, const b200collEpilogue* ep, float scale, cudaStream_t st) {
  return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
    using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
    if constexpr (std::is_same_v<InT, OutT>) {
      constexpr int E = Epv<InT>::value;
      const size_t nslice = ((count + E - 1) / E + c->nranks - 1) / c->nranks;
      Grid g = pick_grid(c, kShapeLL, nslice, 1);
      with_mc<InT>(c->nvls, [&](auto mc) { launch_k(k_ll_twoshot<InT, OutT, decltype(mc)::value>, g.blocks, g.threads, st, c->dev, static_cast<const InT*>(send), static_cast<OutT*>(recv), count, scale, b200collOpAllReduce); });
      LAUNCH_CHECK(c);
      return b200collSuccess;
    } else {
      set_last_error("two-shot LL needs in_dtype == out_dtype");
      return b200collInvalidArgument;
    }
  });
}

// ------------------------------------------------------------------------------------------------ all-reduce on symmetric buffers
static b200collResult_t ar_symmetric(b200collComm* c, b200collAlgo_t algo, const void* send, void* recv, size_t count, const b200collEpilogue* ep, float scale, cudaStream_t st) {
  const int identity = (ep->in_dtype == ep->out_dtype && scale == 1.0f) ? 1 : 0;
  return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
    using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
    constexpr int E = Epv<InT>::value;
    const size_t nvec = count / E;
    const size_t in_off = arena_off(c, send);
    if (algo == b200collAlgoOneShot) {
      Grid g = pick_grid(c, kShapeP2p, nvec, 2);
      launch_k(k_pull_reduce<InT, OutT, true, false>, g.blocks, g.threads, st, c->dev, in_off, static_cast<OutT*>(recv), count, scale, b200collOpAllReduce);
    } else if (algo == b200collAlgoTwoShot) {
      Grid g = pick_grid(c, kShapeP2p, nvec / c->nranks + 1, 2);
      launch_k(k_ar_twoshot<InT, OutT>, g.blocks, g.threads, st, c->dev, in_off, arena_off(c, recv), count, scale, b200collOpAllReduce);
    } else {
      // U=4 vectors in flight per thread. U=1 (more, thinner passes so multimem.st overlaps the next ld_reduce) was measured on
      // 8xB200 and lost to U=4 at every mid size (512 KiB: 20.1 vs 16.0 us, 8 MiB: 38.7 vs 33.9 us): it needs 4x the CTAs, and every
      // extra CTA adds 8 flag stores + a membar.sys to both barriers.
      const bool launched = with_mc<InT>(true, [&](auto mc) {
        if constexpr (decltype(mc)::value) {
          Grid g = pick_grid(c, kShapeNvls, nvec / c->nranks + 1, 4);
          launch_k(k_ar_nvls<InT, OutT, 4>, g.blocks, g.threads, st, c->dev, in_off, arena_off(c, recv), count, scale, identity, b200collOpAllReduce);
        }
        return decltype(mc)::value;
      });
      if (!launched) { set_last_error("no NVLS all-reduce kernel for fp8 inputs"); return b200collInternalError; }
    }
    LAUNCH_CHECK(c);
    return b200collSuccess;
  });
}


// ------------------------------------------------------------------------------------------------ point to point
namespace {

struct PendingP2p { bool send; const void* sbuf; void* rbuf; size_t bytes; int peer; b200collComm* comm; cudaStream_t st; };
thread_local int g_group_depth = 0;
thread_local std::vector<PendingP2p> g_group;
thread_local std::string* g_p2p_dry = nullptr;     // b200collDebugPlanP2p: describe the launches instead of making them (no CUDA call at all)

// CTAs per operation: a pure function of the message size and of settings every rank shares, so CTA j of a send always
// meets CTA j of the matching recv. Virtual ranks share one GPU's SMs between all their kernels: keep them small.
int p2p_blocks(const b200collComm* c, size_t bytes) {
  static const int env_max = [] { const char* e = getenv("B200COLL_P2P_MAX_BLOCKS"); return e ? atoi(e) : 0; }();
  int cap = c->loopback ? 2 : 16;                 // 16 CTAs per operation: sendrecv at 8 GPUs reaches 647 GB/s with it (profiles/other_ops_n8_r2.md); B200COLL_P2P_MAX_BLOCKS overrides
  if (env_max >= 1 && env_max <= kP2pMaxBlocks) cap = env_max;
  const size_t want = (bytes + (128u << 10) - 1) / (128u << 10);
  return (int)std::max<size_t>(1, std::min<size_t>(want, (size_t)cap));
}

// One kernel for `ops` (at most one send and one recv per peer, no self operations, no empty messages).
b200collResult_t p2p_launch(b200collComm* c, const std::vector<PendingP2p>& ops, cudaStream_t st) {
  P2pArgs a = {};
  int nstaged = 0;
  for (const PendingP2p& o : ops) if (!o.send && !b200collIsSymmetric(c, o.rbuf, o.bytes)) nstaged++;
  // staged receives share the two staging halves: each gets an equal slice, cut into two windows
  const size_t share = nstaged ? (2 * kStageHalfBytes / (size_t)nstaged) / 1024 * 1024 : 0;
  const size_t window = c->p2p_window ? std::min(c->p2p_window, share / 2) : share / 2;
  int blocks = 0, staged_seen = 0;
  size_t moved = 0;
  for (int pass = 0; pass < 2; pass++) {          // sends first, then recvs
    for (const PendingP2p& o : ops) {
      if (o.send != (pass == 0)) continue;
      const int i = a.nops++;
      a.first_block[i] = blocks;
      a.lanes[i] = p2p_blocks(c, o.bytes);
      blocks += (!o.send && b200collIsSymmetric(c, o.rbuf, o.bytes)) ? 1 : a.lanes[i];      // a direct receive only exchanges flags: one CTA for all lanes
      a.peer[i] = o.peer;
      a.bytes[i] = o.bytes;
      moved += o.bytes;
      if (o.send) {
        a.nsend++;
        a.src[i] = static_cast<const char*>(o.sbuf);
        c->stats.p2p_sends++;
      } else {
        a.dst[i] = static_cast<char*>(o.rbuf);
        c->stats.p2p_recvs++;
        if (b200collIsSymmetric(c, o.rbuf, o.bytes)) {
          a.staged[i] = 0; a.win_off[i] = arena_off(c, o.rbuf); a.win_bytes[i] = o.bytes;
        } else {
          a.staged[i] = 1; a.win_off[i] = kOffStage + (size_t)staged_seen * share; a.win_bytes[i] = window;
          staged_seen++;
          c->stats.staged_calls++;
        }
      }
    }
  }
  a.first_block[a.nops] = blocks;
  c->stats.p2p_bytes += moved;
  if (g_p2p_dry) {
    char line[192];
    snprintf(line, sizeof line, "launch ctas=%d sends=%d recvs=%d staged=%d\n", blocks, a.nsend, a.nops - a.nsend, nstaged);
    *g_p2p_dry += line;
    for (int i = 0; i < a.nops; i++) {
      const unsigned long long chunks = (i < a.nsend || a.bytes[i] <= a.win_bytes[i]) ? 1 : (a.bytes[i] + a.win_bytes[i] - 1) / a.win_bytes[i];
      if (i < a.nsend) snprintf(line, sizeof line, "  send peer=%d bytes=%llu lanes=%d ctas=[%d,%d)\n", a.peer[i], a.bytes[i], a.lanes[i], a.first_block[i], a.first_block[i + 1]);
      else if (!a.staged[i]) snprintf(line, sizeof line, "  recv peer=%d bytes=%llu lanes=%d ctas=[%d,%d) direct off=%llu\n", a.peer[i], a.bytes[i], a.lanes[i], a.first_block[i], a.first_block[i + 1], a.win_off[i]);
      else snprintf(line, sizeof line, "  recv peer=%d bytes=%llu lanes=%d ctas=[%d,%d) staged off=%llu window=%llu chunks=%llu\n", a.peer[i], a.bytes[i], a.lanes[i], a.first_block[i], a.first_block[i + 1], a.win_off[i], a.win_bytes[i], chunks);
      *g_p2p_dry += line;
    }
    return b200collSuccess;
  }
  static const bool nvtx = [] { const char* e = getenv("B200COLL_NVTX"); return e && *e && *e != '0'; }();
  if (nvtx || debug_level() >= 2) {
    char msg[96];
    snprintf(msg, sizeof(msg), "b200coll p2p %d send %d recv %zu B", a.nsend, a.nops - a.nsend, moved);
    if (nvtx) nvtxMarkA(msg);
    dbg(2, "rank %d: %s (%d CTAs, %d staged)", c->rank, msg, blocks, nstaged);
  }
  if ((c->stats_tick++ & 0xFF) == 0) stats_page_publish(c);
  launch_k(k_p2p, blocks, kP2pThreads, st, c->dev, a, (uint32_t)b200collNumOps);
  LAUNCH_CHECK(c);
  return b200collSuccess;
}

b200collResult_t p2p_flush(std::vector<PendingP2p>& all) {
  // per communicator, in order of first appearance
  while (!all.empty()) {
    b200collComm* c = all.front().comm;
    const cudaStream_t st = all.front().st;
    std::vector<PendingP2p> mine, rest;
    for (const PendingP2p& o : all) (o.comm == c ? mine : rest).push_back(o);
    all.swap(rest);
    if (c->fault_host && *const_cast<volatile uint32_t*>(&c->fault_host->code) != 0) { set_last_error("communicator is poisoned by an earlier watchdog fault"); return b200collRemoteError; }
    // a group may span communicators on several GPUs of this process (nccl-tests -g N): launch each on its own device
    struct DeviceGuard {
      int prev = -1; bool switched = false;
      explicit DeviceGuard(int want) { if (!g_p2p_dry && cudaGetDevice(&prev) == cudaSuccess && prev != want) switched = cudaSetDevice(want) == cudaSuccess; }
      ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
    } guard(c->device);
    // self operations: the i-th send to myself pairs with the i-th recv from myself
    std::vector<PendingP2p> self_s, self_r, remote;
    for (const PendingP2p& o : mine) {
      if (o.bytes == 0) continue;
      if (o.peer == c->rank) (o.send ? self_s : self_r).push_back(o); else remote.push_back(o);
    }
    if (self_s.size() != self_r.size()) { set_last_error("send/recv to self must come in matching pairs inside one group"); return b200collInvalidUsage; }
    for (size_t i = 0; i < self_s.size(); i++) {
      if (self_s[i].bytes != self_r[i].bytes) { set_last_error("send/recv to self: sizes differ"); return b200collInvalidArgument; }
      if (self_s[i].sbuf == self_r[i].rbuf) continue;
      if (g_p2p_dry) { *g_p2p_dry += "self copy bytes=" + std::to_string(self_s[i].bytes) + "\n"; continue; }
      cudaError_t e = cudaMemcpyAsync(self_r[i].rbuf, self_s[i].sbuf, self_s[i].bytes, cudaMemcpyDeviceToDevice, st);
      if (e != cudaSuccess) { set_last_error(cudaGetErrorString(e)); return b200collUnhandledCudaError; }
    }
    // rounds: a kernel carries at most one send and one recv per peer (they share a mailbox); later ones wait for the next round
    while (!remote.empty()) {
      bool has_send[kMaxRanks] = {}, has_recv[kMaxRanks] = {};
      std::vector<PendingP2p> now, later;
      for (const PendingP2p& o : remote) {
        bool* seen = o.send ? has_send : has_recv;
        if (seen[o.peer]) later.push_back(o); else { seen[o.peer] = true; now.push_back(o); }
      }
      b200collResult_t rc = p2p_launch(c, now, st);
      if (rc != b200collSuccess) return rc;
      remote.swap(later);
    }
  }
  return b200collSuccess;
}

b200collResult_t p2p_enqueue(bool send, const void* sbuf, void* rbuf, size_t bytes, int peer, b200collComm* c, cudaStream_t st) {
  const void* buf = send ? sbuf : rbuf;
  if (!c || (!buf && bytes)) { set_last_error("null argument"); return b200collInvalidArgument; }
  if (peer < 0 || peer >= c->nranks) { set_last_error("send/recv peer out of range"); return b200collInvalidArgument; }
  if (!aligned(buf, 16)) { set_last_error("send/recv buffers must be 16-byte aligned"); return b200collInvalidArgument; }
  if (bytes >> kP2pValueBits) { set_last_error("send/recv message too large"); return b200collInvalidArgument; }
  g_group.push_back(PendingP2p{send, sbuf, rbuf, bytes, peer, c, st});
  if (g_group_depth > 0) return b200collSuccess;
  std::vector<PendingP2p> ops;
  ops.swap(g_group);
  return p2p_flush(ops);
}

}  // namespace

}  // namespace b200coll

using namespace b200coll;

extern "C" {

b200collResult_t b200collAllReduce(const void* send, void* recv, size_t count, const b200collEpilogue* ep, b200collRedOp_t rop, b200collComm_t c, b200collStream_t stream) {
  if (c && send && recv && ep && needs_generic(ep, rop)) return generic_reduce(c, b200collOpAllReduce, send, recv, count, ep, rop, 0, static_cast<cudaStream_t>(stream));
  if ((int)rop < 0 || (int)rop > (int)b200collMax) { set_last_error("unknown reduction operator"); return b200collInvalidArgument; }
  b200collResult_t rc = check_common(c, send, recv, ep);
  if (rc != b200collSuccess) return rc;
  if (count == 0) return b200collSuccess;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t is = b200collTypeSize(ep->in_dtype), os = b200collTypeSize(ep->out_dtype);
  const size_t bytes = count * is;
  const float scale = ep->scale * (rop == b200collAvg ? 1.0f / (float)c->nranks : 1.0f);
  const bool inplace = send == recv;
  if (inplace && is != os) { set_last_error("in-place all-reduce needs in_dtype and out_dtype of equal size"); return b200collInvalidArgument; }
  if (c->nranks == 1) { account(c, b200collOpAllReduce, bytes, b200collAlgoCopy); return copy_scale(c, send, recv, count, ep, scale, st); }
  const bool sym_in = b200collIsSymmetric(c, send, bytes), sym_out = b200collIsSymmetric(c, recv, count * os);
  CallFacts f = {b200collOpAllReduce, bytes, ep->in_dtype, sym_in, sym_out, inplace, is == os};
  const b200collAlgo_t algo = resolve_algo(c, f);
  if (algo == b200collAlgoLL) { account(c, b200collOpAllReduce, bytes, algo); return launch_ll(c, b200collOpAllReduce, send, recv, count, ep, scale, st); }
  if (algo == b200collAlgoLL2) { account(c, b200collOpAllReduce, bytes, algo); return launch_ll2(c, send, recv, count, ep, scale, st); }
  if (algo != b200collAlgoAuto) {
    rc = cross_check(c, b200collOpAllReduce, algo, count, arena_off(c, send), arena_off(c, recv));
    if (rc != b200collSuccess) return rc;
    account(c, b200collOpAllReduce, bytes, algo);
    return ar_symmetric(c, algo, send, recv, count, ep, scale, st);
  }
  // ---- staged: buffers outside the arena and too big for LL
  f.sym_in = f.sym_out = true; f.inplace = false;
  const b200collAlgo_t inner = resolve_algo(c, f, /*staging=*/true);
  return run_staged(c, count, stage_chunk(std::max(is, os), 1), {send, is, 1}, {recv, os, 1}, st, [&](size_t, size_t n) {
    account(c, b200collOpAllReduce, n * is, inner);
    return ar_symmetric(c, inner, stage_ptr(c, 0), stage_ptr(c, 1), n, ep, scale, st);
  });
}

b200collResult_t b200collAllGather(const void* send, void* recv, size_t sendcount, const b200collEpilogue* ep, b200collComm_t c, b200collStream_t stream) {
  b200collResult_t rc = check_common(c, send, recv, ep);
  if (rc != b200collSuccess) return rc;
  if (sendcount == 0) return b200collSuccess;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t is = b200collTypeSize(ep->in_dtype), os = b200collTypeSize(ep->out_dtype);
  const size_t bytes = sendcount * is;
  const float scale = ep->scale;
  if (c->nranks == 1) { account(c, b200collOpAllGather, bytes, b200collAlgoCopy); return copy_scale(c, send, recv, sendcount, ep, scale, st); }
  if (sendcount % (16 / is) != 0) { set_last_error("all-gather sendcount must be a multiple of 16 bytes / sizeof(in_dtype)"); return b200collInvalidArgument; }
  const bool sym_out = b200collIsSymmetric(c, recv, (size_t)c->nranks * sendcount * os);
  const b200collAlgo_t algo = resolve_algo(c, {b200collOpAllGather, bytes, ep->in_dtype});
  if (algo == b200collAlgoLL) { account(c, b200collOpAllGather, bytes, algo); return launch_ll(c, b200collOpAllGather, send, recv, sendcount, ep, scale, st); }
  const int identity = (ep->in_dtype == ep->out_dtype && scale == 1.0f) ? 1 : 0;
  auto push = [&](const void* s, void* r, size_t n) -> b200collResult_t {
    account(c, b200collOpAllGather, n * is, algo);
    return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
      using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
      Grid g = pick_grid(c, algo == b200collAlgoNvls ? kShapeNvls : kShapeP2p, n / Epv<InT>::value, 4);
      with_mc<InT>(algo == b200collAlgoNvls, [&](auto mc) { launch_k(k_ag_push<InT, OutT, decltype(mc)::value>, g.blocks, g.threads, st, c->dev, static_cast<const InT*>(s), arena_off(c, r), n, scale, identity, b200collOpAllGather); });
      LAUNCH_CHECK(c);
      return b200collSuccess;
    });
  };
  if (sym_out) {
    rc = cross_check(c, b200collOpAllGather, algo, sendcount, arena_off(c, recv), 0);
    if (rc != b200collSuccess) return rc;
  }
  if (bulk_enabled() && sym_out && identity && bytes >= bulk_min_bytes() && bytes % 16 == 0 && algo != b200collAlgoNvls) {     // copy-engine push (kernels.cuh k_bulk)
    account(c, b200collOpAllGather, bytes, algo);
    BulkArgs a = {};
    a.nseg = 1; a.src[0] = static_cast<const char*>(send); a.bytes[0] = bytes;
    a.dst_off[0] = arena_off(c, recv) + (size_t)c->rank * bytes; a.dst_mask[0] = (1u << c->nranks) - 1;
    return launch_bulk(c, a, true, b200collOpAllGather, st);
  }
  if (sym_out) return push(send, recv, sendcount);
  // staged: gather chunks into staging half 1 laid out [nranks][chunk], then scatter locally into recv
  return run_staged(c, sendcount, stage_chunk(os, c->nranks), {}, {recv, os, c->nranks}, st,
                    [&](size_t done, size_t n) { return push(static_cast<const char*>(send) + done * is, stage_ptr(c, 1), n); });
}

b200collResult_t b200collReduceScatter(const void* send, void* recv, size_t recvcount, const b200collEpilogue* ep, b200collRedOp_t rop, b200collComm_t c, b200collStream_t stream) {
  if (c && send && recv && ep && needs_generic(ep, rop)) return generic_reduce(c, b200collOpReduceScatter, send, recv, recvcount, ep, rop, 0, static_cast<cudaStream_t>(stream));
  if ((int)rop < 0 || (int)rop > (int)b200collMax) { set_last_error("unknown reduction operator"); return b200collInvalidArgument; }
  b200collResult_t rc = check_common(c, send, recv, ep);
  if (rc != b200collSuccess) return rc;
  if (recvcount == 0) return b200collSuccess;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t is = b200collTypeSize(ep->in_dtype), os = b200collTypeSize(ep->out_dtype);
  const size_t bytes = recvcount * is;
  const float scale = ep->scale * (rop == b200collAvg ? 1.0f / (float)c->nranks : 1.0f);
  if (c->nranks == 1) { account(c, b200collOpReduceScatter, bytes, b200collAlgoCopy); return copy_scale(c, send, recv, recvcount, ep, scale, st); }
  if (recvcount % (16 / is) != 0) { set_last_error("reduce-scatter recvcount must be a multiple of 16 bytes / sizeof(in_dtype)"); return b200collInvalidArgument; }
  const bool sym_in = b200collIsSymmetric(c, send, (size_t)c->nranks * bytes);
  const b200collAlgo_t algo = resolve_algo(c, {b200collOpReduceScatter, bytes, ep->in_dtype});
  if (algo == b200collAlgoLL) { account(c, b200collOpReduceScatter, bytes, algo); return launch_ll(c, b200collOpReduceScatter, send, recv, recvcount, ep, scale, st); }
  auto pull = [&](const void* s_slice_of_mine, void* r, size_t n) -> b200collResult_t {
    account(c, b200collOpReduceScatter, n * is, algo);
    return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
      using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
      Grid g = pick_grid(c, algo == b200collAlgoNvls ? kShapeNvlsRs : kShapeP2p, n / Epv<InT>::value, 2);
      with_mc<InT>(algo == b200collAlgoNvls, [&](auto mc) { launch_k(k_pull_reduce<InT, OutT, false, decltype(mc)::value>, g.blocks, g.threads, st, c->dev, arena_off(c, s_slice_of_mine), static_cast<OutT*>(r), n, scale, b200collOpReduceScatter); });
      LAUNCH_CHECK(c);
      return b200collSuccess;
    });
  };
  if (sym_in) {
    rc = cross_check(c, b200collOpReduceScatter, algo, recvcount, arena_off(c, send), 0);
    if (rc != b200collSuccess) return rc;
    return pull(static_cast<const char*>(send) + (size_t)c->rank * bytes, recv, recvcount);
  }
  // staged: copy chunk j of every slice into staging half 0 laid out [nranks][chunk]; each rank pulls its row
  return run_staged(c, recvcount, stage_chunk(is, c->nranks), {send, is, c->nranks}, {}, st,
                    [&](size_t done, size_t n) { return pull(stage_ptr(c, 0) + (size_t)c->rank * n * is, static_cast<char*>(recv) + done * os, n); });
}

// symmetric: every rank moves the same amount, so the grid may follow the work. Otherwise (all-to-all-v: each rank only knows its own
// rows) every rank launches the full P2P shape — block b of one rank meets block b of every other rank in the barriers, so the grids
// must agree, and CTAs without work only take the two barriers.
static b200collResult_t a2av_launch(b200collComm* c, const void* send, void* recv_sym, const A2AvArgs& a, const b200collEpilogue* ep, cudaStream_t st, bool symmetric) {
  const int identity = (ep->in_dtype == ep->out_dtype && ep->scale == 1.0f) ? 1 : 0;
  return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
    using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
    Grid g = pick_grid(c, kShapeP2p, symmetric ? (size_t)a.prefix[c->nranks] + 1 : ~(size_t)0 >> 8, 4);
    launch_k(k_a2av_push<InT, OutT>, g.blocks, g.threads, st, c->dev, static_cast<const InT*>(send), arena_off(c, recv_sym), a, ep->scale, identity, b200collOpAllToAll);
    LAUNCH_CHECK(c);
    return b200collSuccess;
  });
}

// Fill the flattened prefix in the kernel's staggered order (j -> peer rank+1+j).
static void a2av_prefix(const b200collComm* c, const unsigned long long* nvec_by_peer, A2AvArgs* a) {
  a->prefix[0] = 0;
  for (int j = 0; j < c->nranks; j++) {
    int p = c->rank + 1 + j; if (p >= c->nranks) p -= c->nranks;
    a->prefix[j + 1] = a->prefix[j] + nvec_by_peer[p];
  }
  for (int j = c->nranks + 1; j <= kMaxRanks; j++) a->prefix[j] = a->prefix[c->nranks];
}

b200collResult_t b200collAllToAll(const void* send, void* recv, size_t count, const b200collEpilogue* ep, b200collComm_t c, b200collStream_t stream) {
  b200collResult_t rc = check_common(c, send, recv, ep);
  if (rc != b200collSuccess) return rc;
  if (count == 0) return b200collSuccess;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t is = b200collTypeSize(ep->in_dtype), os = b200collTypeSize(ep->out_dtype);
  const size_t bytes = count * is;
  if (c->nranks == 1) { account(c, b200collOpAllToAll, bytes, b200collAlgoCopy); return copy_scale(c, send, recv, count, ep, ep->scale, st); }
  if (send == recv) { set_last_error("in-place all-to-all is not supported"); return b200collInvalidUsage; }
  const size_t E = 16 / is;
  if (count % E != 0) { set_last_error("all-to-all count must be a multiple of 16 bytes / sizeof(in_dtype)"); return b200collInvalidArgument; }
  const b200collAlgo_t algo = resolve_algo(c, {b200collOpAllToAll, bytes, ep->in_dtype});
  if (algo == b200collAlgoLL) { account(c, b200collOpAllToAll, bytes * c->nranks, algo); return launch_ll(c, b200collOpAllToAll, send, recv, count, ep, ep->scale, st); }
  const bool sym_out = b200collIsSymmetric(c, recv, (size_t)c->nranks * count * os);
  auto run = [&](const void* s, size_t s_stride_elems, void* r_sym, size_t n) -> b200collResult_t {
    // block p of this chunk starts at element p*s_stride_elems of s; lands at block `rank` (stride n) of r_sym on peer p
    A2AvArgs a = {};
    unsigned long long nv[kMaxRanks] = {};
    for (int p = 0; p < c->nranks; p++) { a.src_vec[p] = (unsigned long long)p * s_stride_elems / E; a.dst_vec[p] = (unsigned long long)c->rank * n / E; nv[p] = n / E; }
    a2av_prefix(c, nv, &a);
    account(c, b200collOpAllToAll, n * is * c->nranks, algo);
    return a2av_launch(c, s, r_sym, a, ep, st, true);
  };
  if (sym_out) {
    rc = cross_check(c, b200collOpAllToAll, algo, count, arena_off(c, recv), 0);
    if (rc != b200collSuccess) return rc;
  }
  if (bulk_enabled() && sym_out && is == os && ep->in_dtype == ep->out_dtype && ep->scale == 1.0f && bytes * c->nranks >= bulk_min_bytes() && bytes % 16 == 0) {
    account(c, b200collOpAllToAll, bytes * c->nranks, algo);
    BulkArgs a = {};
    a.nseg = c->nranks;
    for (int j = 0; j < c->nranks; j++) {             // staggered: segment j goes to rank+1+j, the last one is my own block
      int p = c->rank + 1 + j; if (p >= c->nranks) p -= c->nranks;
      a.src[j] = static_cast<const char*>(send) + (size_t)p * bytes; a.bytes[j] = bytes;
      a.dst_off[j] = arena_off(c, recv) + (size_t)c->rank * bytes; a.dst_mask[j] = 1u << p;
    }
    return launch_bulk(c, a, true, b200collOpAllToAll, st);
  }
  if (sym_out) return run(send, count, recv, count);
  return run_staged(c, count, stage_chunk(os, c->nranks), {}, {recv, os, c->nranks}, st,
                    [&](size_t done, size_t n) { return run(static_cast<const char*>(send) + done * is, count, stage_ptr(c, 1), n); });
}

b200collResult_t b200collAllToAllv(const void* send, void* recv, size_t row_elems, const int64_t* send_rows, const int64_t* send_row_off,
                                   const int64_t* recv_row_off_at_peer, const b200collEpilogue* ep, b200collComm_t c, b200collStream_t stream) {
  b200collResult_t rc = check_common(c, send, recv, ep);
  if (rc != b200collSuccess) return rc;
  if (!send_rows || !send_row_off || !recv_row_off_at_peer || row_elems == 0) { set_last_error("alltoallv: null/zero argument"); return b200collInvalidArgument; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t is = b200collTypeSize(ep->in_dtype), os = b200collTypeSize(ep->out_dtype);
  const size_t E = 16 / is;
  if (row_elems % E != 0) { set_last_error("alltoallv: row_elems must be a multiple of 16 bytes / sizeof(in_dtype)"); return b200collInvalidArgument; }
  if (send == recv) { set_last_error("in-place all-to-all is not supported"); return b200collInvalidUsage; }
  const size_t row_vecs = row_elems / E;
  if (c->nranks == 1) {
    account(c, b200collOpAllToAll, (size_t)send_rows[0] * row_elems * is, b200collAlgoCopy);
    if (send_rows[0] <= 0) return b200collSuccess;
    return copy_scale(c, static_cast<const char*>(send) + (size_t)send_row_off[0] * row_elems * is, static_cast<char*>(recv) + (size_t)recv_row_off_at_peer[0] * row_elems * os,
                      (size_t)send_rows[0] * row_elems, ep, ep->scale, st);
  }
  // The receive side is written by peers, so it must be symmetric; expert-dispatch buffers are long-lived, allocate them with MemAlloc.
  if (!b200collIsSymmetric(c, recv, 1)) { set_last_error("alltoallv: recv must come from b200collMemAlloc (peers write into it)"); return b200collInvalidUsage; }
  A2AvArgs a = {};
  unsigned long long nv[kMaxRanks] = {};
  size_t total_bytes = 0;
  for (int p = 0; p < c->nranks; p++) {
    if (send_rows[p] < 0 || send_row_off[p] < 0 || recv_row_off_at_peer[p] < 0) { set_last_error("alltoallv: negative count/offset"); return b200collInvalidArgument; }
    a.src_vec[p] = (unsigned long long)send_row_off[p] * row_vecs;
    a.dst_vec[p] = (unsigned long long)recv_row_off_at_peer[p] * row_vecs;
    nv[p] = (unsigned long long)send_rows[p] * row_vecs;
    total_bytes += (size_t)send_rows[p] * row_elems * is;
  }
  a2av_prefix(c, nv, &a);
  account(c, b200collOpAllToAll, total_bytes, b200collAlgoTwoShot);
  return a2av_launch(c, send, recv, a, ep, st, false);
}

b200collResult_t b200collBroadcast(const void* send, void* recv, size_t count, const b200collEpilogue* ep, int root, b200collComm_t c, b200collStream_t stream) {
  // send is only read on the root; other ranks may pass any aligned non-null pointer (their recv is the usual choice).
  b200collResult_t rc = check_common(c, send, recv, ep);
  if (rc != b200collSuccess) return rc;
  if (root < 0 || root >= c->nranks) { set_last_error("broadcast root out of range"); return b200collInvalidArgument; }
  if (count == 0) return b200collSuccess;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t is = b200collTypeSize(ep->in_dtype), os = b200collTypeSize(ep->out_dtype);
  const float scale = ep->scale;
  if (c->nranks == 1) { account(c, b200collOpBroadcast, count * is, b200collAlgoCopy); return copy_scale(c, send, recv, count, ep, scale, st); }
  if (send == recv && is != os) { set_last_error("in-place broadcast needs in_dtype and out_dtype of equal size"); return b200collInvalidArgument; }
  const b200collAlgo_t algo = resolve_algo(c, {b200collOpBroadcast, count * is, ep->in_dtype});
  const int identity = (ep->in_dtype == ep->out_dtype && scale == 1.0f) ? 1 : 0;
  auto push = [&](const void* s, void* r_sym, size_t n) -> b200collResult_t {
    account(c, b200collOpBroadcast, n * is, algo);
    return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
      using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
      Grid g = pick_grid(c, algo == b200collAlgoNvls ? kShapeRooted : kShapeP2p, std::max<size_t>(1, n / Epv<InT>::value), 4);
      with_mc<InT>(algo == b200collAlgoNvls, [&](auto mc) { launch_k(k_bcast<InT, OutT, decltype(mc)::value>, g.blocks, g.threads, st, c->dev, static_cast<const InT*>(s), arena_off(c, r_sym), n, scale, identity, root, b200collOpBroadcast); });
      LAUNCH_CHECK(c);
      return b200collSuccess;
    });
  };
  if (bulk_enabled() && algo == b200collAlgoTwoShot && identity && count * is >= bulk_min_bytes() && (count * is) % 16 == 0 && b200collIsSymmetric(c, recv, count * os)) {
    account(c, b200collOpBroadcast, count * is, algo);
    BulkArgs a = {};
    if (c->rank == root) { a.nseg = 1; a.src[0] = static_cast<const char*>(send); a.bytes[0] = count * is; a.dst_off[0] = arena_off(c, recv); a.dst_mask[0] = (1u << c->nranks) - 1; }
    c->bulk_grid_hint = (count * is + kBulkChunk - 1) / kBulkChunk;      // non-root ranks carry no segment but must launch the root's grid
    return launch_bulk(c, a, true, b200collOpBroadcast, st);
  }
  if (b200collIsSymmetric(c, recv, count * os)) return push(send, recv, count);
  // staged: the root pushes a chunk into everybody's staging half 1, each rank copies it out locally
  return run_staged(c, count, stage_chunk(std::max(is, os), 1), {}, {recv, os, 1}, st,
                    [&](size_t done, size_t n) { return push(static_cast<const char*>(send) + done * is, stage_ptr(c, 1), n); });
}

b200collResult_t b200collReduce(const void* send, void* recv, size_t count, const b200collEpilogue* ep, b200collRedOp_t rop, int root, b200collComm_t c, b200collStream_t stream) {
  // recv is only written on the root; other ranks may pass any aligned non-null pointer.
  if (c && send && recv && ep && needs_generic(ep, rop)) {
    if (root < 0 || root >= c->nranks) { set_last_error("reduce root out of range"); return b200collInvalidArgument; }
    return generic_reduce(c, b200collOpReduce, send, recv, count, ep, rop, root, static_cast<cudaStream_t>(stream));
  }
  if ((int)rop < 0 || (int)rop > (int)b200collMax) { set_last_error("unknown reduction operator"); return b200collInvalidArgument; }
  b200collResult_t rc = check_common(c, send, recv, ep);
  if (rc != b200collSuccess) return rc;
  if (root < 0 || root >= c->nranks) { set_last_error("reduce root out of range"); return b200collInvalidArgument; }
  if (count == 0) return b200collSuccess;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t is = b200collTypeSize(ep->in_dtype), os = b200collTypeSize(ep->out_dtype);
  const float scale = ep->scale * (rop == b200collAvg ? 1.0f / (float)c->nranks : 1.0f);
  if (c->nranks == 1) { account(c, b200collOpReduce, count * is, b200collAlgoCopy); return copy_scale(c, send, recv, count, ep, scale, st); }
  if (send == recv && is != os) { set_last_error("in-place reduce needs in_dtype and out_dtype of equal size"); return b200collInvalidArgument; }
  const b200collAlgo_t algo = resolve_algo(c, {b200collOpReduce, count * is, ep->in_dtype});
  auto pull = [&](const void* s_sym, void* r, size_t n) -> b200collResult_t {
    account(c, b200collOpReduce, n * is, algo);
    return dispatch_types(ep->in_dtype, ep->out_dtype, [&](auto ti, auto to) -> b200collResult_t {
      using InT = typename decltype(ti)::type; using OutT = typename decltype(to)::type;
      Grid g = pick_grid(c, algo == b200collAlgoNvls ? kShapeRooted : kShapeP2p, std::max<size_t>(1, n / Epv<InT>::value), algo == b200collAlgoNvls ? 4 : 2);
      with_mc<InT>(algo == b200collAlgoNvls, [&](auto mc) { launch_k(k_reduce_root<InT, OutT, decltype(mc)::value>, g.blocks, g.threads, st, c->dev, arena_off(c, s_sym), static_cast<OutT*>(r), n, scale, root, b200collOpReduce); });
      LAUNCH_CHECK(c);
      return b200collSuccess;
    });
  };
  if (b200collIsSymmetric(c, send, count * is)) return pull(send, recv, count);
  // staged: every rank copies a chunk of its send buffer into staging half 0, the root reduces the chunk into recv
  return run_staged(c, count, stage_chunk(std::max(is, os), 1), {send, is, 1}, {}, st,
                    [&](size_t done, size_t n) { return pull(stage_ptr(c, 0), static_cast<char*>(recv) + done * os, n); });
}

b200collResult_t b200collGroupStart(void) { g_group_depth++; return b200collSuccess; }
b200collResult_t b200collGroupEnd(void) {
  if (g_group_depth == 0) { set_last_error("group end without a matching group start"); return b200collInvalidUsage; }
  if (--g_group_depth > 0) return b200collSuccess;
  std::vector<PendingP2p> ops;
  ops.swap(g_group);
  return p2p_flush(ops);
}
b200collResult_t b200collSend(const void* buf, size_t bytes, int peer, b200collComm_t c, b200collStream_t stream) {
  return p2p_enqueue(true, buf, nullptr, bytes, peer, c, static_cast<cudaStream_t>(stream));
}
b200collResult_t b200collRecv(void* buf, size_t bytes, int peer, b200collComm_t c, b200collStream_t stream) {
  return p2p_enqueue(false, nullptr, buf, bytes, peer, c, static_cast<cudaStream_t>(stream));
}

b200collResult_t b200collDebugPlanP2p(int rank, int nranks, int loopback, size_t window, int nops, const int* is_send, const int* peer, const size_t* bytes,
                                      const int* in_arena, char* out, size_t outlen) {
  if (!out || outlen == 0 || nops < 0 || nranks < 1 || nranks > kMaxRanks || rank < 0 || rank >= nranks) return b200collInvalidArgument;
  b200collComm fake;                                   // never touches the GPU: no arena, no streams, only the fields the planner reads
  fake.rank = rank; fake.nranks = nranks; fake.loopback = loopback != 0; fake.p2p_window = window / 512 * 512;
  fake.peer_va[rank] = (CUdeviceptr)1 << 40; fake.arena.total = (size_t)64 << 30;
  std::string text;
  size_t heap = kOffHeap, outside = (size_t)1 << 44;
  b200collResult_t rc = b200collSuccess;
  g_p2p_dry = &text;
  g_group_depth++;
  for (int i = 0; i < nops && rc == b200collSuccess; i++) {
    size_t& cursor = in_arena[i] ? heap : outside;
    void* buf = reinterpret_cast<void*>((in_arena[i] ? (size_t)fake.peer_va[rank] : 0) + cursor);
    cursor += (bytes[i] + 4095) / 4096 * 4096 + 4096;
    rc = is_send[i] ? b200collSend(buf, bytes[i], peer[i], &fake, nullptr) : b200collRecv(buf, bytes[i], peer[i], &fake, nullptr);
  }
  g_group_depth--;
  std::vector<PendingP2p> ops;
  ops.swap(g_group);
  if (rc == b200collSuccess) rc = p2p_flush(ops);
  g_p2p_dry = nullptr;
  snprintf(out, outlen, "%s", text.c_str());
  return rc;
}

b200collResult_t b200collBarrier(b200collComm_t c, b200collStream_t stream) {
  if (!c) return b200collInvalidArgument;
  if (c->nranks == 1) return b200collSuccess;
  launch_k(k_barrier, 1, 32, static_cast<cudaStream_t>(stream), c->dev, 99u);
  LAUNCH_CHECK(c);
  return b200collSuccess;
}

}  // extern "C"
