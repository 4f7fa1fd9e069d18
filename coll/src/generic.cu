// libb200coll: reductions outside the fp-sum fast paths — min / max / prod on every type, and every operator on the integer types
// and fp64 — so that the library (and libb200coll_nccl.so on top of it) accepts what an unmodified NCCL consumer sends: PyTorch's
// int64 all-reduces, nccl-tests `-o max -d int32`, a MIN over step counters (reference role: the installed NCCL,
// gpudirect-tcpxo/README.md:66-70, takes all of ncclRedOp_t x ncclDataType_t).
// One barrier-based P2P kernel (no Lamport path: its empty-slot marker is a NaN pattern, which is a legal integer; no NVLS: the
// switch has no prod and no 64-bit integer min/max), accumulating in the element type (fp16 / bf16 / fp8 in fp32), in rank order, so every
// rank computes bit-identical results:
//   all-reduce      rank r pulls vector slice r from every peer, reduces, pushes the result into every peer's out   (two-shot)
//   reduce-scatter  rank r pulls its block from every peer, reduces into its local out
//   reduce          the root pulls everything; the other ranks only take the two barriers
// Buffers outside the symmetric arena go through the two staging halves, like the fp paths.
#include <algorithm>
#include <string>

#include "comm.h"
#include "device.cuh"

namespace b200coll {

enum { kModeAllReduce = 0, kModeToLocal = 1 };

template <typename T> struct GAcc { using type = T; };
template <> struct GAcc<__half> { using type = float; };
template <> struct GAcc<__nv_bfloat16> { using type = float; };
template <> struct GAcc<__nv_fp8_e4m3> { using type = float; };
template <> struct GAcc<__nv_fp8_e5m2> { using type = float; };
template <typename T> __device__ __forceinline__ typename GAcc<T>::type g_load(T v) { return (typename GAcc<T>::type)v; }
template <> __device__ __forceinline__ float g_load<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float g_load<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float g_load<__nv_fp8_e4m3>(__nv_fp8_e4m3 v) { return float(v); }
template <> __device__ __forceinline__ float g_load<__nv_fp8_e5m2>(__nv_fp8_e5m2 v) { return float(v); }
template <typename T> __device__ __forceinline__ T g_store(typename GAcc<T>::type v) { return (T)v; }
template <> __device__ __forceinline__ __half g_store<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 g_store<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __nv_fp8_e4m3 g_store<__nv_fp8_e4m3>(float v) { return __nv_fp8_e4m3(v); }   // saturating, like the fused paths
template <> __device__ __forceinline__ __nv_fp8_e5m2 g_store<__nv_fp8_e5m2>(float v) { return __nv_fp8_e5m2(v); }
// scalar tails read peers' elements with volatile loads; the fp8 classes cannot be copied from a volatile object
template <typename T> __device__ __forceinline__ typename GAcc<T>::type g_load_volatile(const char* base, size_t e) { return g_load<T>(reinterpret_cast<const volatile T*>(base)[e]); }
template <> __device__ __forceinline__ float g_load_volatile<__nv_fp8_e4m3>(const char* base, size_t e) { return ld_volatile_float<__nv_fp8_e4m3>(base, e); }
template <> __device__ __forceinline__ float g_load_volatile<__nv_fp8_e5m2>(const char* base, size_t e) { return ld_volatile_float<__nv_fp8_e5m2>(base, e); }

template <int OP, typename A> __device__ __forceinline__ A g_apply(A a, A b) {
  if (OP == b200collSum) return a + b;
  if (OP == b200collProd) return a * b;
  if (OP == b200collMin) return b < a ? b : a;
  return b > a ? b : a;
}

template <typename T, int OP>
__device__ __forceinline__ uint4 g_reduce_vec(const uint4* d, int n) {
  constexpr int E = 16 / (int)sizeof(T);
  using A = typename GAcc<T>::type;
  union V { uint4 u; T e[E]; };
  A acc[E];
  V first; first.u = d[0];
#pragma unroll
  for (int i = 0; i < E; i++) acc[i] = g_load<T>(first.e[i]);
#pragma unroll
  for (int j = 1; j < kMaxRanks; j++) if (j < n) {
    V v; v.u = d[j];
#pragma unroll
    for (int i = 0; i < E; i++) acc[i] = g_apply<OP, A>(acc[i], g_load<T>(v.e[i]));
  }
  V out;
#pragma unroll
  for (int i = 0; i < E; i++) out.e[i] = g_store<T>(acc[i]);
  return out.u;
}

// region = `count` elements at arena offset in_off of every rank. mode kModeAllReduce: my vector slice of the region is reduced and
// pushed to arena offset out_off of every rank. mode kModeToLocal: the whole region is reduced into out_local — by `worker` only when
// worker >= 0 (rooted reduce), by every rank otherwise (reduce-scatter: in_off already points at this rank's block).
template <typename T, int OP>
__global__ void __launch_bounds__(512) k_generic_reduce(COMM_PARAM, size_t in_off, size_t out_off, T* __restrict__ out_local, size_t count, int mode, int worker, uint32_t op) {
  pdl_prologue();
  constexpr int E = 16 / (int)sizeof(T);
  using A = typename GAcc<T>::type;
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;
  const size_t nvec = count / E;
  size_t v0 = 0, v1 = nvec;
  if (mode == kModeAllReduce) { v0 = nvec * c.rank / c.nranks; v1 = nvec * (c.rank + 1) / c.nranks; }
  const bool works = mode == kModeAllReduce || worker < 0 || worker == c.rank;
  if (works) {
    for (size_t v = v0 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < v1; v += (size_t)gridDim.x * blockDim.x) {
      uint4 d[kMaxRanks];
#pragma unroll
      for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) d[j] = ld_vec(c.peer[j] + in_off + v * 16);     // rank order: same result everywhere
      const uint4 r = g_reduce_vec<T, OP>(d, c.nranks);
      if (mode == kModeAllReduce) {
#pragma unroll
        for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
          int p = c.rank + j; if (p >= c.nranks) p -= c.nranks;
          st_vec(c.peer[p] + out_off + v * 16, r);
        }
      } else {
        st_vec(reinterpret_cast<char*>(out_local) + v * 16, r);
      }
    }
    // scalar tail (count not a multiple of one vector): all-reduce -> rank 0 for everybody, else whoever works
    if (blockIdx.x == 0 && (mode != kModeAllReduce || c.rank == 0)) {
      const size_t e = nvec * E + threadIdx.x;
      if (e < count) {
        A acc = g_load_volatile<T>(c.peer[0] + in_off, e);
        for (int r = 1; r < c.nranks; r++) acc = g_apply<OP, A>(acc, g_load_volatile<T>(c.peer[r] + in_off, e));
        const T o = g_store<T>(acc);
        if (mode == kModeAllReduce) { for (int r = 0; r < c.nranks; r++) reinterpret_cast<T*>(c.peer[r] + out_off)[e] = o; }
        else out_local[e] = o;
      }
    }
  }
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

template <typename T>
static b200collResult_t launch_generic(b200collComm* c, b200collRedOp_t rop, size_t in_off, size_t out_off, void* out_local, size_t count, int mode, int worker, uint32_t op, cudaStream_t st) {
  constexpr int E = 16 / (int)sizeof(T);
  const size_t vecs = (mode == kModeAllReduce ? count / E / c->nranks : count / E) + 1;
  const int cap = std::max(1, std::min(c->shape[1].max_ctas > 0 ? c->shape[1].max_ctas : c->max_ctas, c->max_ctas));
  int threads = 512;
  for (int t : {128, 256, 512}) if ((vecs + t - 1) / t <= (size_t)cap) { threads = t; break; }
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((vecs + threads - 1) / threads, (size_t)cap));
  T* ol = static_cast<T*>(out_local);
  switch (rop) {
    case b200collSum: k_generic_reduce<T, b200collSum><<<blocks, threads, 0, st>>>(c->dev, in_off, out_off, ol, count, mode, worker, op); break;
    case b200collProd: k_generic_reduce<T, b200collProd><<<blocks, threads, 0, st>>>(c->dev, in_off, out_off, ol, count, mode, worker, op); break;
    case b200collMin: k_generic_reduce<T, b200collMin><<<blocks, threads, 0, st>>>(c->dev, in_off, out_off, ol, count, mode, worker, op); break;
    case b200collMax: k_generic_reduce<T, b200collMax><<<blocks, threads, 0, st>>>(c->dev, in_off, out_off, ol, count, mode, worker, op); break;
    default: set_last_error("this reduction operator is not defined for this type (avg: floating point only, through the fused scale)"); return b200collInvalidArgument;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_last_error(std::string("kernel launch failed: ") + cudaGetErrorString(e)); return b200collUnhandledCudaError; }
  c->stats.kernel_launches++; c->stats.generic_launches++;
  return b200collSuccess;
}

static b200collResult_t dispatch_generic(b200collComm* c, b200collDataType_t dt, b200collRedOp_t rop, size_t in_off, size_t out_off, void* out_local, size_t count, int mode, int worker, uint32_t op, cudaStream_t st) {
  switch (dt) {
    case b200collInt8: return launch_generic<int8_t>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collUint8: return launch_generic<uint8_t>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collInt32: return launch_generic<int32_t>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collUint32: return launch_generic<uint32_t>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collInt64: return launch_generic<long long>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collUint64: return launch_generic<unsigned long long>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collFloat64: return launch_generic<double>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collFloat32: return launch_generic<float>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collFloat16: return launch_generic<__half>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collBfloat16: return launch_generic<__nv_bfloat16>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collFloat8e4m3: return launch_generic<__nv_fp8_e4m3>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    case b200collFloat8e5m2: return launch_generic<__nv_fp8_e5m2>(c, rop, in_off, out_off, out_local, count, mode, worker, op, st);
    default: set_last_error("unsupported dtype for a generic reduction"); return b200collInvalidArgument;
  }
}

bool needs_generic(const b200collEpilogue* ep, b200collRedOp_t rop) {
  const bool fp = ep->in_dtype == b200collFloat32 || ep->in_dtype == b200collFloat16 || ep->in_dtype == b200collBfloat16 ||
                  ep->in_dtype == b200collFloat8e4m3 || ep->in_dtype == b200collFloat8e5m2;
  return !fp || rop == b200collProd || rop == b200collMin || rop == b200collMax;
}

// which: b200collOpAllReduce (count = elements of the buffer), b200collOpReduceScatter (count = elements each rank receives),
// b200collOpReduce (count = elements, root). One rank: a copy. Non-symmetric buffers: chunked through the staging halves.
b200collResult_t generic_reduce(b200collComm* c, b200collOp_t which, const void* send, void* recv, size_t count, const b200collEpilogue* ep, b200collRedOp_t rop, int root, cudaStream_t st) {
  if (ep->in_dtype != ep->out_dtype || ep->scale != 1.0f) { set_last_error("min / max / prod and integer / fp64 reductions take no cast or scale (in_dtype == out_dtype, scale == 1)"); return b200collInvalidArgument; }
  if (rop == b200collAvg) { set_last_error("avg is defined for fp32 / fp16 / bf16 / fp8 only"); return b200collInvalidArgument; }
  const size_t es = b200collTypeSize(ep->in_dtype);
  if (es == 0) { set_last_error("bad dtype"); return b200collInvalidArgument; }
  if (reinterpret_cast<uintptr_t>(send) % 16 || reinterpret_cast<uintptr_t>(recv) % 16) { set_last_error("send and recv must be 16-byte aligned"); return b200collInvalidArgument; }
  if (c->fault_host && *const_cast<volatile uint32_t*>(&c->fault_host->code) != 0) { set_last_error("communicator is poisoned by an earlier watchdog fault"); return b200collRemoteError; }
  if (count == 0) return b200collSuccess;
  const int n = c->nranks;
  const size_t in_elems = which == b200collOpReduceScatter ? count * n : count;
  c->stats.calls[which]++; c->stats.bytes[which] += count * es; c->stats.algo_calls[b200collAlgoTwoShot]++;
  if (n == 1) {
    if (send != recv) { cudaError_t e = cudaMemcpyAsync(recv, send, count * es, cudaMemcpyDeviceToDevice, st); if (e != cudaSuccess) { set_last_error(cudaGetErrorString(e)); return b200collUnhandledCudaError; } }
    return b200collSuccess;
  }
  if (which == b200collOpReduceScatter && (count * es) % 16 != 0) { set_last_error("reduce-scatter recvcount must be a multiple of 16 bytes / sizeof(dtype)"); return b200collInvalidArgument; }
  char* const base = reinterpret_cast<char*>(c->peer_va[c->rank]);
  auto off = [&](const void* p) { return (size_t)(static_cast<const char*>(p) - base); };
  const bool sym_in = b200collIsSymmetric(c, send, in_elems * es);
  const bool sym_out = b200collIsSymmetric(c, recv, count * es);
  const uint32_t opid = (uint32_t)which;
  // m elements of every rank's input at arena offset in_off (all-reduce: result to arena offset out_off, else into out_local)
  auto launch = [&](size_t in_off, size_t out_off, char* out_local, size_t m) {
    if (which == b200collOpAllReduce) return dispatch_generic(c, ep->in_dtype, rop, in_off, out_off, nullptr, m, kModeAllReduce, -1, opid, st);
    if (which == b200collOpReduceScatter) return dispatch_generic(c, ep->in_dtype, rop, in_off + (size_t)c->rank * m * es, 0, out_local, m, kModeToLocal, -1, opid, st);
    return dispatch_generic(c, ep->in_dtype, rop, in_off, 0, out_local, m, kModeToLocal, root, opid, st);
  };
  char* const out = static_cast<char*>(recv);
  if (sym_in && (which != b200collOpAllReduce || sym_out)) return launch(off(send), off(recv), out, count);
  // staged: chunk through staging half 0 (inputs) and half 1 (all-reduce results)
  const int rows = which == b200collOpReduceScatter ? n : 1;
  return run_staged(c, count, stage_chunk(es, rows), {send, es, rows}, {which == b200collOpAllReduce ? recv : nullptr, es, 1}, st,
                    [&](size_t done, size_t m) { return launch(kOffStage, kOffStage + kStageHalfBytes, out + done * es, m); });
}

}  // namespace b200coll
