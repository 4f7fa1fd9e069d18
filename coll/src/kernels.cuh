// libb200coll kernels (sm_100a). One kernel per (algorithm); each is templated on <InT, OutT> so the
// cast/scale epilogue runs in registers between the reduction and the (peer / multicast) store —
// no separate elementwise kernel or extra HBM pass on any path (BASELINE.json north-star).
//
//   k_copy_scale      nranks==1                    out = cast(in*scale)
//   k_ll              Lamport flag-in-payload      all four ops, zero barriers, <= 512 KiB per source
//   k_pull_reduce     one-shot AR / P2P or NVLS RS barrier, pull (or multimem.ld_reduce), reduce, local store
//   k_ar_twoshot      P2P all-reduce               pull+reduce own slice, push result to every peer (single pass)
//   k_ar_nvls         NVLS all-reduce              multimem.ld_reduce own slice -> scale/cast -> multimem.st
//   k_ag_push         all-gather                   P2P push or one multimem.st per vector
//   k_a2av_push       all-to-all(v)                per-peer row ranges, flattened for load balance
//   k_bcast           broadcast                    root pushes (P2P or one multimem.st per vector); the others only synchronise
//   k_reduce_root     reduce                       the root pulls (or multimem.ld_reduce) the whole buffer; the others only synchronise
//   k_bulk            identity epilogue, >= 1 MiB   all-gather / broadcast / all-to-all(v) / one-rank copy through the copy engine (cp.async.bulk ring)
//   k_p2p             send / recv (grouped)        receiver posts where to write, sender pushes over NVLink and signals; no all-rank barrier
//   k_barrier
#pragma once
#include "device.cuh"

namespace b200coll {

constexpr int kThreads = 512;

template <typename InT, typename OutT, int E>
__device__ __forceinline__ void finish_store_local(OutT* dst, const float* acc, float scale) {
  float f[E];
#pragma unroll
  for (int i = 0; i < E; i++) f[i] = acc[i] * scale;
  uint32_t w[Pack<OutT, E>::W];
  Pack<OutT, E>::run(f, w);
  st_words<Pack<OutT, E>::W>(dst, w);
}

// ------------------------------------------------------------------------------------------------
template <typename InT, typename OutT>
__global__ void __launch_bounds__(kThreads) k_copy_scale(const InT* __restrict__ in, OutT* __restrict__ out, size_t count, float scale) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  constexpr int U = 4;                       // 4 x 16 B loads in flight per thread: HBM-latency hiding for a pure streaming kernel
  const size_t nvec = count / E;
  const size_t stride = (size_t)gridDim.x * blockDim.x * U;
  for (size_t base = (size_t)blockIdx.x * blockDim.x * U + threadIdx.x; base < nvec; base += stride) {
    uint4 d[U];
#pragma unroll
    for (int u = 0; u < U; u++) { const size_t v = base + (size_t)u * blockDim.x; if (v < nvec) d[u] = ld_vec(in + v * E); }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = base + (size_t)u * blockDim.x;
      if (v < nvec) { float acc[E] = {}; unpack_add<InT>(acc, d[u]); finish_store_local<InT, OutT, E>(out + v * E, acc, scale); }
    }
  }
  if (blockIdx.x == 0) {
    const size_t e = nvec * E + threadIdx.x;
    if (e < count) out[e] = from_float<OutT>(to_float<InT>(in[e]) * scale);
  }
}

// ------------------------------------------------------------------------------------------------
// Lamport path. Scratch slot (buf, src, i) of MY arena is written by rank `src` (or by the switch on
// its behalf) and read only by me. Three buffers rotate per launch: use k%3, clear (k-1)%3 (last
// touched one launch ago, next written two launches from now), (k+1)%3 was cleared by the previous
// launch. A slot is "empty" while any of its four words equals kLLSentinel.
__device__ __forceinline__ char* ll_slot(char* base, uint32_t buf, int src, size_t i) {
  return base + kOffLL + (((size_t)buf * kMaxRanks + src) * kLLMaxVecs + i) * 16;
}
__device__ __forceinline__ uint4 ll_sanitize(uint4 v) {
  if (v.x == kLLSentinel) v.x = kLLSanitized;
  if (v.y == kLLSentinel) v.y = kLLSanitized;
  if (v.z == kLLSentinel) v.z = kLLSanitized;
  if (v.w == kLLSentinel) v.w = kLLSanitized;
  return v;
}
__device__ __forceinline__ bool ll_ready(const uint4& v) {
  return v.x != kLLSentinel && v.y != kLLSentinel && v.z != kLLSentinel && v.w != kLLSentinel;
}
__device__ __forceinline__ uint4 ll_wait(const CommDev& c, const char* slot, int src, uint32_t op) {
  uint4 v = ld_vec_volatile(slot);
  if (!ll_ready(v)) {
    const unsigned long long t0 = globaltimer_ns();
    uint32_t spins = 0;
    while (true) {
      v = ld_vec_volatile(slot);
      if (ll_ready(v)) break;
      if (((++spins) & 0x3FF) == 0) {
        if (c.fault->code != 0 || globaltimer_ns() - t0 > c.timeout_ns) { record_fault(c, 2, src, 0, v.x, op); v = make_uint4(0, 0, 0, 0); break; }   // never hand a half-written slot to the reduction
      }
    }
  }
  return v;
}
template <typename InT, int E>
__device__ __forceinline__ uint4 load_in_guarded(const InT* in, size_t i, size_t count) {
  if ((i + 1) * E <= count) return ld_vec(in + i * E);
  union { InT e[E]; uint4 v; } u;
  u.v = make_uint4(0, 0, 0, 0);
#pragma unroll
  for (int k = 0; k < E; k++) if (i * E + k < count) u.e[k] = in[i * E + k];
  return u.v;
}
template <typename OutT, int E>
__device__ __forceinline__ void store_out_guarded(OutT* out, size_t i, size_t count, const float* acc, float scale) {
  if ((i + 1) * E <= count) {
    float f[E];
#pragma unroll
    for (int k = 0; k < E; k++) f[k] = acc[k] * scale;
    uint32_t w[Pack<OutT, E>::W];
    Pack<OutT, E>::run(f, w);
    st_words<Pack<OutT, E>::W>(out + i * E, w);
  } else {
#pragma unroll
    for (int k = 0; k < E; k++) if (i * E + k < count) out[i * E + k] = from_float<OutT>(acc[k] * scale);
  }
}

// SLICED=false: every peer gets my whole `count`-element input (AR, AG). SLICED=true: peer p gets block p (RS, A2A).
// SUM=true: out[i] = sum over sources (AR, RS). SUM=false: out[src*count + i] = source's data (AG, A2A).
template <typename InT, typename OutT, bool SLICED, bool SUM, bool MC>
__global__ void __launch_bounds__(kThreads) k_ll(COMM_PARAM, const InT* __restrict__ in, OutT* __restrict__ out, size_t count, float scale, uint32_t op) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  const uint32_t k = load_seq(c, kSeqLL);
  const uint32_t buf = k % 3, prev = (k + 2) % 3;
  const size_t nv = (count + E - 1) / E;
  const size_t used_prev = c.state[kLLUsedLo0 + prev], used_prev_hi = c.state[kLLUsedHi0 + prev];
  size_t span = nv > used_prev ? nv : used_prev;
  if (used_prev_hi > span) span = used_prev_hi;
  char* const me = c.peer[c.rank];
  const uint4 empty = make_uint4(kLLSentinel, kLLSentinel, kLLSentinel, kLLSentinel);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < span; i += (size_t)gridDim.x * blockDim.x) {
    uint4 own = make_uint4(0, 0, 0, 0);
    if (i < nv) {
      if (!SLICED) {
        own = ll_sanitize(load_in_guarded<InT, E>(in, i, count));
        if (MC) {
          const uint32_t w[4] = {own.x, own.y, own.z, own.w};
          mc_st_words(ll_slot(c.mc, buf, c.rank, i), w, 4);
        } else {
#pragma unroll
          for (int j = 1; j < kMaxRanks; j++) if (j < c.nranks) {
            int p = c.rank + j; if (p >= c.nranks) p -= c.nranks;
            st_vec_volatile(ll_slot(c.peer[p], buf, c.rank, i), own);
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
          int p = c.rank + j; if (p >= c.nranks) p -= c.nranks;
          uint4 v = ll_sanitize(ld_vec(in + (size_t)p * count + i * E));
          if (j == 0) own = v; else st_vec_volatile(ll_slot(c.peer[p], buf, c.rank, i), v);
        }
      }
    }
    if (i < used_prev) {
#pragma unroll
      for (int r = 0; r < kMaxRanks; r++) if (r < c.nranks) st_vec(ll_slot(me, prev, r, i), empty);
    }
    if (i < used_prev_hi) {
#pragma unroll
      for (int r = 0; r < kMaxRanks; r++) if (r < c.nranks) st_vec(ll_slot(me, prev, r, kLLHalfVecs + i), empty);
    }
    if (i < nv) {
      if (SUM) {
        float acc[E] = {};
#pragma unroll
        for (int r = 0; r < kMaxRanks; r++) if (r < c.nranks) {
          uint4 d = (r == c.rank) ? own : ll_wait(c, ll_slot(me, buf, r, i), r, op);
          unpack_add<InT>(acc, d);
        }
        store_out_guarded<OutT, E>(out, i, count, acc, scale);
      } else {
#pragma unroll
        for (int r = 0; r < kMaxRanks; r++) if (r < c.nranks) {
          uint4 d = (r == c.rank) ? own : ll_wait(c, ll_slot(me, buf, r, i), r, op);
          float acc[E] = {};
          unpack_add<InT>(acc, d);
          store_out_guarded<OutT, E>(out + (size_t)r * count, i, count, acc, scale);
        }
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && last_block_ticket(c)) {
    c.state[kLLUsedLo0 + buf] = (uint32_t)nv;
    c.state[kLLUsedHi0 + buf] = 0;
    c.state[kSeqLL] = k + 1;
  }
}

// ------------------------------------------------------------------------------------------------
// Two-shot Lamport all-reduce: zero barriers like k_ll, but each rank receives 2S instead of N*S bytes.
// Phase 1 (reduce-scatter): rank s pushes vector i of slice p into peer p's lo slot (buf, s, i); rank p sums the
// N copies of its slice in fp32, applies scale/cast. Phase 2 (all-gather): p publishes the finished vector into
// everybody's hi slot (buf, p, i) — one multimem.st when MC — and every rank copies the N slices into out.
// One thread owns vector i of *every* slice end to end, so there is no intra-kernel dependency between threads
// and in-place is safe (a thread reads all its inputs before its first write). Needs sizeof(OutT) == sizeof(InT).
template <typename OutT, int E>
__device__ __forceinline__ void store_raw_guarded(OutT* out, size_t vec, size_t count, const uint4& w) {
  if ((vec + 1) * E <= count) { st_vec(out + vec * E, w); return; }
  union { OutT e[E]; uint4 v; } u;
  u.v = w;
#pragma unroll
  for (int k = 0; k < E; k++) if (vec * E + k < count) out[vec * E + k] = u.e[k];
}

template <typename InT, typename OutT, bool MC>
__global__ void __launch_bounds__(kThreads) k_ll_twoshot(COMM_PARAM, const InT* __restrict__ in, OutT* __restrict__ out, size_t count, float scale, uint32_t op) {
  pdl_prologue();
  static_assert(sizeof(InT) == sizeof(OutT), "two-shot LL keeps one vector geometry for both phases");
  constexpr int E = Epv<InT>::value;
  const uint32_t k = load_seq(c, kSeqLL);
  const uint32_t buf = k % 3, prev = (k + 2) % 3;
  const size_t nvec = (count + E - 1) / E;
  const size_t nslice = (nvec + c.nranks - 1) / c.nranks;
  const size_t used_lo = c.state[kLLUsedLo0 + prev], used_hi = c.state[kLLUsedHi0 + prev];
  size_t span = nslice > used_lo ? nslice : used_lo;
  if (used_hi > span) span = used_hi;
  char* const me = c.peer[c.rank];
  const uint4 empty = make_uint4(kLLSentinel, kLLSentinel, kLLSentinel, kLLSentinel);
  const size_t my0 = (size_t)c.rank * nslice;
  const size_t my_len = my0 >= nvec ? 0 : (nvec - my0 < nslice ? nvec - my0 : nslice);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < span; i += (size_t)gridDim.x * blockDim.x) {
    uint4 own = make_uint4(0, 0, 0, 0);
    if (i < nslice) {
#pragma unroll
      for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
        int p = c.rank + j; if (p >= c.nranks) p -= c.nranks;
        const size_t v = (size_t)p * nslice + i;
        if (v < nvec) {
          uint4 d = ll_sanitize(load_in_guarded<InT, E>(in, v, count));
          if (j == 0) own = d; else st_vec_volatile(ll_slot(c.peer[p], buf, c.rank, i), d);
        }
      }
    }
    if (i < used_lo) {
#pragma unroll
      for (int r = 0; r < kMaxRanks; r++) if (r < c.nranks) st_vec(ll_slot(me, prev, r, i), empty);
    }
    if (i < used_hi) {
#pragma unroll
      for (int r = 0; r < kMaxRanks; r++) if (r < c.nranks) st_vec(ll_slot(me, prev, r, kLLHalfVecs + i), empty);
    }
    if (i < my_len) {
      float acc[E] = {};
#pragma unroll
      for (int r = 0; r < kMaxRanks; r++) if (r < c.nranks) {
        uint4 d = (r == c.rank) ? own : ll_wait(c, ll_slot(me, buf, r, i), r, op);
        unpack_add<InT>(acc, d);
      }
#pragma unroll
      for (int e = 0; e < E; e++) acc[e] *= scale;
      uint32_t w[4];
      Pack<OutT, E>::run(acc, w);
      const uint4 red = ll_sanitize(make_uint4(w[0], w[1], w[2], w[3]));
      if (MC) {
        const uint32_t rw[4] = {red.x, red.y, red.z, red.w};
        mc_st_words(ll_slot(c.mc, buf, c.rank, kLLHalfVecs + i), rw, 4);
      } else {
#pragma unroll
        for (int j = 1; j < kMaxRanks; j++) if (j < c.nranks) {
          int p = c.rank + j; if (p >= c.nranks) p -= c.nranks;
          st_vec_volatile(ll_slot(c.peer[p], buf, c.rank, kLLHalfVecs + i), red);
        }
      }
      store_raw_guarded<OutT, E>(out, my0 + i, count, red);
    }
    if (i < nslice) {
#pragma unroll
      for (int r = 0; r < kMaxRanks; r++) if (r < c.nranks && r != c.rank) {
        const size_t v = (size_t)r * nslice + i;
        if (v < nvec) store_raw_guarded<OutT, E>(out, v, count, ll_wait(c, ll_slot(me, buf, r, kLLHalfVecs + i), r, op));
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && last_block_ticket(c)) {
    c.state[kLLUsedLo0 + buf] = (uint32_t)nslice;
    c.state[kLLUsedHi0 + buf] = (uint32_t)nslice;
    c.state[kSeqLL] = k + 1;
  }
}

// ------------------------------------------------------------------------------------------------
// Scalar tail for the barrier-based all-reduce kernels: rank 0 reduces elements [e0, count) from every
// peer and writes the result into every peer's out (so in-place is safe).
template <typename InT, typename OutT>
__device__ __forceinline__ void ar_tail_rank0(const CommDev& c, size_t in_off, size_t out_off, size_t e0, size_t count, float scale) {
  if (c.rank != 0 || blockIdx.x != 0) return;
  const size_t e = e0 + threadIdx.x;
  if (e >= count) return;
  float acc = 0.f;
  for (int r = 0; r < c.nranks; r++) acc += ld_volatile_float<InT>(c.peer[r] + in_off, e);
  const OutT o = from_float<OutT>(acc * scale);
  for (int r = 0; r < c.nranks; r++) reinterpret_cast<OutT*>(c.peer[r] + out_off)[e] = o;
}

// out_local[i] = scale * sum_r peer_r[in_off + i]   (one-shot all-reduce; reduce-scatter with in_off pointing at my slice)
// FIXED_ORDER: sum in rank order so every rank computes bit-identical results (one-shot AR).
template <typename InT, typename OutT, bool FIXED_ORDER, bool MC>
__global__ void __launch_bounds__(kThreads) k_pull_reduce(COMM_PARAM, size_t in_off, OutT* __restrict__ out, size_t count, float scale, uint32_t op) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  constexpr int U = 2;
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;
  const size_t nvec = count / E;
  const size_t stride = (size_t)gridDim.x * blockDim.x * U;
  for (size_t base = (size_t)blockIdx.x * blockDim.x * U + threadIdx.x; base < nvec; base += stride) {
    if constexpr (MC) {   // constexpr: the non-MC instantiation must not reference mc_ld_reduce<InT> (none exists for fp8)
      uint4 d[U];
#pragma unroll
      for (int u = 0; u < U; u++) { const size_t v = base + (size_t)u * blockDim.x; if (v < nvec) d[u] = mc_ld_reduce<InT>(c.mc + in_off + v * 16); }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = base + (size_t)u * blockDim.x;
        if (v < nvec) { float acc[E] = {}; unpack_add<InT>(acc, d[u]); finish_store_local<InT, OutT, E>(out + v * E, acc, scale); }
      }
    } else {
      uint4 d[U][kMaxRanks];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = base + (size_t)u * blockDim.x;
        if (v < nvec) {
#pragma unroll
          for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
            int r = j;
            if (!FIXED_ORDER) { r = c.rank + j; if (r >= c.nranks) r -= c.nranks; }
            d[u][j] = ld_vec(c.peer[r] + in_off + v * 16);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = base + (size_t)u * blockDim.x;
        if (v < nvec) {
          float acc[E] = {};
#pragma unroll
          for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) unpack_add<InT>(acc, d[u][j]);
          finish_store_local<InT, OutT, E>(out + v * E, acc, scale);
        }
      }
    }
  }
  if (blockIdx.x == 0) {   // scalar tail, every rank for itself (out is local and distinct from in for these ops)
    const size_t e = nvec * E + threadIdx.x;
    if (e < count) {
      float acc = 0.f;
      for (int r = 0; r < c.nranks; r++) acc += ld_volatile_float<InT>(c.peer[r] + in_off, e);
      out[e] = from_float<OutT>(acc * scale);
    }
  }
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

// ------------------------------------------------------------------------------------------------
// Two-shot fused into one pass: rank r owns vector slice r; pulls it from every peer, reduces in fp32,
// applies scale/cast and pushes the finished vector into every peer's out. Bytes per GPU and direction:
// S(N-1)/N pulled + S(N-1)/N pushed -> bus bandwidth bound = link bandwidth.
template <typename InT, typename OutT>
__global__ void __launch_bounds__(kThreads) k_ar_twoshot(COMM_PARAM, size_t in_off, size_t out_off, size_t count, float scale, uint32_t op) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  constexpr int W = Pack<OutT, E>::W;
  constexpr int U = 2;
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;
  const size_t nvec = count / E;
  const size_t v0 = nvec * c.rank / c.nranks, v1 = nvec * (c.rank + 1) / c.nranks;
  const size_t stride = (size_t)gridDim.x * blockDim.x * U;
  for (size_t base = v0 + (size_t)blockIdx.x * blockDim.x * U + threadIdx.x; base < v1; base += stride) {
    uint4 d[U][kMaxRanks];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = base + (size_t)u * blockDim.x;
      if (v < v1) {
#pragma unroll
        for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
          int r = c.rank + j; if (r >= c.nranks) r -= c.nranks;
          d[u][j] = ld_vec(c.peer[r] + in_off + v * 16);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = base + (size_t)u * blockDim.x;
      if (v < v1) {
        float acc[E] = {};
#pragma unroll
        for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) unpack_add<InT>(acc, d[u][j]);
#pragma unroll
        for (int i = 0; i < E; i++) acc[i] *= scale;
        uint32_t w[W];
        Pack<OutT, E>::run(acc, w);
#pragma unroll
        for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
          int r = c.rank + j; if (r >= c.nranks) r -= c.nranks;
          st_words<W>(c.peer[r] + out_off + v * (E * sizeof(OutT)), w);
        }
      }
    }
  }
  ar_tail_rank0<InT, OutT>(c, in_off, out_off, nvec * E, count, scale);
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

// NVLS all-reduce: the switch does the reduction (fp32 accumulate) and the broadcast.
// Per GPU and direction: ~S(1+1/N) bytes -> algbw bound = link/(1+1/N).
// U = vectors in flight per thread. Large messages use U=4; mid sizes use U=1 so that a slice takes several passes and
// the multimem.st of pass k (ingress-heavy) overlaps the ld_reduce of pass k+1 (egress-heavy) instead of running back to back.
template <typename InT, typename OutT, int U>
__global__ void __launch_bounds__(kThreads) k_ar_nvls(COMM_PARAM, size_t in_off, size_t out_off, size_t count, float scale, int identity, uint32_t op) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  constexpr int W = Pack<OutT, E>::W;
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;
  const size_t nvec = count / E;
  const size_t v0 = nvec * c.rank / c.nranks, v1 = nvec * (c.rank + 1) / c.nranks;
  const size_t stride = (size_t)gridDim.x * blockDim.x * U;
  for (size_t base = v0 + (size_t)blockIdx.x * blockDim.x * U + threadIdx.x; base < v1; base += stride) {
    uint4 d[U];
#pragma unroll
    for (int u = 0; u < U; u++) { const size_t v = base + (size_t)u * blockDim.x; if (v < v1) d[u] = mc_ld_reduce<InT>(c.mc + in_off + v * 16); }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = base + (size_t)u * blockDim.x;
      if (v < v1) {
        uint32_t w[W];
        if (identity) {   // same dtype, scale == 1: forward the switch's result untouched
          const uint32_t raw[4] = {d[u].x, d[u].y, d[u].z, d[u].w};
#pragma unroll
          for (int i = 0; i < W && i < 4; i++) w[i] = raw[i];
        } else {
          float acc[E] = {};
          unpack_add<InT>(acc, d[u]);
#pragma unroll
          for (int i = 0; i < E; i++) acc[i] *= scale;
          Pack<OutT, E>::run(acc, w);
        }
        mc_st_wordsW<W>(c.mc + out_off + v * (E * sizeof(OutT)), w);
      }
    }
  }
  ar_tail_rank0<InT, OutT>(c, in_off, out_off, nvec * E, count, scale);
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

// ------------------------------------------------------------------------------------------------
// All-gather push: my `count` elements land at element offset rank*count of every peer's out.
// MC: one multimem.st per vector (egress S/N instead of S(N-1)/N).
template <typename InT, typename OutT, bool MC>
__global__ void __launch_bounds__(kThreads) k_ag_push(COMM_PARAM, const InT* __restrict__ in, size_t out_off, size_t count, float scale, int identity, uint32_t op) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  constexpr int W = Pack<OutT, E>::W;
  constexpr int U = 4;
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;
  const size_t nvec = count / E;
  const size_t dst0 = out_off + (size_t)c.rank * count * sizeof(OutT);
  const size_t stride = (size_t)gridDim.x * blockDim.x * U;
  for (size_t base = (size_t)blockIdx.x * blockDim.x * U + threadIdx.x; base < nvec; base += stride) {
    uint4 d[U];
#pragma unroll
    for (int u = 0; u < U; u++) { const size_t v = base + (size_t)u * blockDim.x; if (v < nvec) d[u] = ld_vec(in + v * E); }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = base + (size_t)u * blockDim.x;
      if (v < nvec) {
        uint32_t w[W];
        if (identity) {
          const uint32_t raw[4] = {d[u].x, d[u].y, d[u].z, d[u].w};
#pragma unroll
          for (int i = 0; i < W && i < 4; i++) w[i] = raw[i];
        } else {
          float acc[E] = {};
          unpack_add<InT>(acc, d[u]);
#pragma unroll
          for (int i = 0; i < E; i++) acc[i] *= scale;
          Pack<OutT, E>::run(acc, w);
        }
        const size_t off = dst0 + v * (E * sizeof(OutT));
        if (MC) {
          mc_st_wordsW<W>(c.mc + off, w);
        } else {
#pragma unroll
          for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
            int r = c.rank + j; if (r >= c.nranks) r -= c.nranks;
            st_words<W>(c.peer[r] + off, w);
          }
        }
      }
    }
  }
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

// ------------------------------------------------------------------------------------------------
// All-to-all(v) push. Per destination p: nvec[p] input vectors starting at vector src_vec[p] of my send
// buffer go to output-vector offset dst_vec[p] (units of E*sizeof(OutT) bytes) of peer p's recv buffer.
// The (peer, vector) space is flattened with a prefix table so skewed expert loads still spread over all CTAs.
struct A2AvArgs {
  unsigned long long src_vec[kMaxRanks];
  unsigned long long dst_vec[kMaxRanks];
  unsigned long long prefix[kMaxRanks + 1];   // prefix over the staggered order j = 0..nranks-1 (peer = rank+1+j)
};
template <typename InT, typename OutT>
__global__ void __launch_bounds__(kThreads) k_a2av_push(COMM_PARAM, const InT* __restrict__ in, size_t out_off, A2AvArgs a, float scale, int identity, uint32_t op) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  constexpr int W = Pack<OutT, E>::W;
  constexpr int U = 4;
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;
  const size_t total = a.prefix[c.nranks];
  const size_t stride = (size_t)gridDim.x * blockDim.x * U;
  for (size_t base = (size_t)blockIdx.x * blockDim.x * U + threadIdx.x; base < total; base += stride) {
    uint4 d[U];
    int pj[U];
    size_t lv[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t g = base + (size_t)u * blockDim.x;
      pj[u] = 0; lv[u] = 0;
      if (g < total) {
        int j = 0;
#pragma unroll
        for (int q = 1; q < kMaxRanks; q++) if (q < c.nranks && g >= a.prefix[q]) j = q;
        int p = c.rank + 1 + j; if (p >= c.nranks) p -= c.nranks;
        pj[u] = p; lv[u] = g - a.prefix[j];
        d[u] = ld_vec(in + (a.src_vec[p] + lv[u]) * E);
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t g = base + (size_t)u * blockDim.x;
      if (g < total) {
        uint32_t w[W];
        if (identity) {
          const uint32_t raw[4] = {d[u].x, d[u].y, d[u].z, d[u].w};
#pragma unroll
          for (int i = 0; i < W && i < 4; i++) w[i] = raw[i];
        } else {
          float acc[E] = {};
          unpack_add<InT>(acc, d[u]);
#pragma unroll
          for (int i = 0; i < E; i++) acc[i] *= scale;
          Pack<OutT, E>::run(acc, w);
        }
        st_words<W>(c.peer[pj[u]] + out_off + (a.dst_vec[pj[u]] + lv[u]) * (E * sizeof(OutT)), w);
      }
    }
  }
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

// ------------------------------------------------------------------------------------------------
// Broadcast: the root's `count` elements land at out_off of every rank (its own copy included, so in-place and
// out-of-place behave the same). MC: one multimem.st per vector -> root egress S instead of S(N-1).
// Every rank launches the same grid; non-root CTAs only take part in the two barriers.
template <typename InT, typename OutT, bool MC>
__global__ void __launch_bounds__(kThreads) k_bcast(COMM_PARAM, const InT* __restrict__ in, size_t out_off, size_t count, float scale, int identity, int root, uint32_t op) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  constexpr int W = Pack<OutT, E>::W;
  constexpr int U = 4;
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;          // every rank is done with the previous contents of its out
  if (c.rank == root) {
    const size_t nvec = count / E;
    const size_t stride = (size_t)gridDim.x * blockDim.x * U;
    for (size_t base = (size_t)blockIdx.x * blockDim.x * U + threadIdx.x; base < nvec; base += stride) {
      uint4 d[U];
#pragma unroll
      for (int u = 0; u < U; u++) { const size_t v = base + (size_t)u * blockDim.x; if (v < nvec) d[u] = ld_vec(in + v * E); }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = base + (size_t)u * blockDim.x;
        if (v < nvec) {
          uint32_t w[W];
          if (identity) {
            const uint32_t raw[4] = {d[u].x, d[u].y, d[u].z, d[u].w};
#pragma unroll
            for (int i = 0; i < W && i < 4; i++) w[i] = raw[i];
          } else {
            float acc[E] = {};
            unpack_add<InT>(acc, d[u]);
#pragma unroll
            for (int i = 0; i < E; i++) acc[i] *= scale;
            Pack<OutT, E>::run(acc, w);
          }
          const size_t off = out_off + v * (E * sizeof(OutT));
          if (MC) {
            mc_st_wordsW<W>(c.mc + off, w);
          } else {
#pragma unroll
            for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
              int r = c.rank + j; if (r >= c.nranks) r -= c.nranks;
              st_words<W>(c.peer[r] + off, w);
            }
          }
        }
      }
    }
    if (blockIdx.x == 0) {                          // scalar tail (count not a multiple of one vector)
      const size_t e = nvec * E + threadIdx.x;
      if (e < count) {
        OutT o = from_float<OutT>(to_float<InT>(in[e]) * scale);
        if constexpr (sizeof(InT) == sizeof(OutT)) {
          if (identity) { const InT x = in[e]; memcpy(&o, &x, sizeof(o)); }   // bit-exact, like the vector path (payload may not be a float at all)
        }
        for (int r = 0; r < c.nranks; r++) reinterpret_cast<OutT*>(c.peer[r] + out_off)[e] = o;
      }
    }
  }
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

// Rooted reduce: out@root[i] = scale * sum_r peer_r[in_off + i]. Every rank launches this same kernel with the same grid
// (a different kernel on the non-root ranks would need its own lazy module load, and with virtual ranks that load cannot
// complete while the root's kernel is already spinning on the GPU -> deadlock); non-root CTAs only take the two barriers:
// the first tells the root my send buffer is ready, the second tells me the root has finished reading it.
// MC: the root issues multimem.ld_reduce (the switch adds, the root receives S bytes instead of S(N-1)).
template <typename InT, typename OutT, bool MC>
__global__ void __launch_bounds__(kThreads) k_reduce_root(COMM_PARAM, size_t in_off, OutT* __restrict__ out, size_t count, float scale, int root, uint32_t op) {
  pdl_prologue();
  constexpr int E = Epv<InT>::value;
  constexpr int U = MC ? 4 : 2;      // the root alone must keep the link busy: four ld_reduce vectors in flight per thread on the NVLS path
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;
  if (c.rank == root) {
    const size_t nvec = count / E;
    const size_t stride = (size_t)gridDim.x * blockDim.x * U;
    for (size_t base = (size_t)blockIdx.x * blockDim.x * U + threadIdx.x; base < nvec; base += stride) {
      if constexpr (MC) {
        uint4 d[U];
#pragma unroll
        for (int u = 0; u < U; u++) { const size_t v = base + (size_t)u * blockDim.x; if (v < nvec) d[u] = mc_ld_reduce<InT>(c.mc + in_off + v * 16); }
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = base + (size_t)u * blockDim.x;
          if (v < nvec) { float acc[E] = {}; unpack_add<InT>(acc, d[u]); finish_store_local<InT, OutT, E>(out + v * E, acc, scale); }
        }
      } else {
        uint4 d[U][kMaxRanks];
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = base + (size_t)u * blockDim.x;
          if (v < nvec) {
#pragma unroll
            for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) d[u][j] = ld_vec(c.peer[j] + in_off + v * 16);   // rank order: deterministic sum
          }
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = base + (size_t)u * blockDim.x;
          if (v < nvec) {
            float acc[E] = {};
#pragma unroll
            for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) unpack_add<InT>(acc, d[u][j]);
            finish_store_local<InT, OutT, E>(out + v * E, acc, scale);
          }
        }
      }
    }
    if (blockIdx.x == 0) {   // scalar tail
      const size_t e = nvec * E + threadIdx.x;
      if (e < count) {
        float acc = 0.f;
        for (int r = 0; r < c.nranks; r++) acc += ld_volatile_float<InT>(c.peer[r] + in_off, e);
        out[e] = from_float<OutT>(acc * scale);
      }
    }
  }
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

// ------------------------------------------------------------------------------------------------
// Copy-engine data movement (TMA bulk copies): all-gather, broadcast, all-to-all(v) and the one-rank copy when the epilogue is the
// identity (same dtype, scale 1) — the bytes are never looked at, so no register ever holds them. One elected thread per CTA drives a
// shared-memory ring:   cp.async.bulk global -> shared (completion counted on an mbarrier)      [SASS: UBLKCP.S.G + SYNCS.ARRIVE.TRANS64]
//                       cp.async.bulk shared -> (peer) global, one per destination, one bulk group per chunk            [UBLKCP.G.S]
// Loads run kStages-1 chunks ahead of the stores; a slot is reloaded once the group that stored from it has finished READING it
// (cp.async.bulk.wait_group.read), so up to (kStages-1) loads and 2 store groups per CTA are in flight — enough outstanding bytes per SM
// for HBM (one rank) and for NVLink (peers) without spending registers or issue slots on the payload.
// The work is a list of segments (source range -> set of destinations), flattened into chunks and dealt round-robin to the CTAs:
//   one-rank copy   1 segment, local destination            all-gather   1 segment -> every rank's out[rank]
//   broadcast       root: 1 segment -> every rank; others: none (barriers only)
//   all-to-all(v)   one segment per peer (staggered start so that all ranks do not hit the same peer at once)
struct BulkArgs {
  int nseg;
  const char* src[kMaxRanks];
  unsigned long long bytes[kMaxRanks];            // multiple of 16
  unsigned long long chunk_prefix[kMaxRanks + 1]; // chunks before segment g
  unsigned long long dst_off[kMaxRanks];          // arena offset at the destination rank(s)
  unsigned dst_mask[kMaxRanks];                   // bit r: copy to rank r (peer[r] + dst_off)
  char* dst_local;                                // one-rank copy: plain local destination instead of arena destinations (nseg == 1)
};
constexpr int kBulkStages = 4;
constexpr uint32_t kBulkChunk = 16384;
constexpr int kBulkThreads = 32;
constexpr size_t kBulkSmemBytes = (size_t)kBulkStages * kBulkChunk;
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <bool SYNC>
__global__ void __launch_bounds__(kBulkThreads) k_bulk(COMM_PARAM, const __grid_constant__ BulkArgs a, uint32_t op) {
  pdl_prologue();
  extern __shared__ __align__(128) char ring[];                  // [kBulkStages][kBulkChunk]
  __shared__ __align__(8) unsigned long long full[kBulkStages];
  uint32_t s = 0;
  if (SYNC) {
    s = load_seq(c, kSeqBarrier);
    if (!barrier_blocks<false>(c, 2 * s + 1, op)) return;        // every rank is done with the previous contents of the destination
  }
  if (threadIdx.x == 0 && a.nseg > 0) {
    for (int i = 0; i < kBulkStages; i++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&full[i])));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned long long nchunks = a.chunk_prefix[a.nseg];
    const unsigned long long mine = nchunks > blockIdx.x ? (nchunks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;   // chunks blockIdx.x, +gridDim.x, ...
    auto locate = [&](unsigned long long k, int* seg, unsigned long long* off, uint32_t* n) {
      const unsigned long long g = blockIdx.x + k * gridDim.x;
      int sgi = 0;
#pragma unroll
      for (int q = 1; q < kMaxRanks; q++) if (q < a.nseg && g >= a.chunk_prefix[q]) sgi = q;
      const unsigned long long o = (g - a.chunk_prefix[sgi]) * kBulkChunk;
      *seg = sgi; *off = o;
      *n = (uint32_t)(a.bytes[sgi] - o < kBulkChunk ? a.bytes[sgi] - o : kBulkChunk);
    };
    auto load = [&](unsigned long long k) {
      int seg; unsigned long long off; uint32_t n;
      locate(k, &seg, &off, &n);
      const int slot = (int)(k % kBulkStages);
      const uint32_t bar = smem_u32(&full[slot]), dst_s = smem_u32(ring + (size_t)slot * kBulkChunk);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(n) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_s), "l"(a.src[seg] + off), "r"(n), "r"(bar) : "memory");
    };
    const unsigned long long ahead = kBulkStages - 1;
    for (unsigned long long k = 0; k < mine && k < ahead; k++) load(k);
    bool dead = false;
    for (unsigned long long k = 0; k < mine && !dead; k++) {
      const int slot = (int)(k % kBulkStages);
      const uint32_t parity = (uint32_t)((k / kBulkStages) & 1u);
      const uint32_t bar = smem_u32(&full[slot]), src_s = smem_u32(ring + (size_t)slot * kBulkChunk);
      uint32_t done = 0, spins = 0;
      const unsigned long long t0 = globaltimer_ns();
      while (!done) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (!done && ((++spins) & 0x3FF) == 0 && globaltimer_ns() - t0 > c.timeout_ns) { record_fault(c, 5, (uint32_t)c.rank, (uint32_t)k, slot, op); dead = true; break; }   // the copy engine never delivered: report, do not hang
      }
      if (dead) break;
      int seg; unsigned long long off; uint32_t n;
      locate(k, &seg, &off, &n);
      if (a.dst_local) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(a.dst_local + off), "r"(src_s), "r"(n) : "memory");
      } else {
        const unsigned mask = a.dst_mask[seg];
#pragma unroll
        for (int j = 0; j < kMaxRanks; j++) if (j < c.nranks) {
          int r = c.rank + j; if (r >= c.nranks) r -= c.nranks;
          if (mask & (1u << r)) asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(c.peer[r] + a.dst_off[seg] + off), "r"(src_s), "r"(n) : "memory");
        }
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      if (k + ahead < mine) {
        asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // every group but the one just committed has finished reading its slot: slot (k-1) % kStages is free
        load(k + ahead);
      }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");          // every store has been performed, not just read
    asm volatile("fence.proxy.async.global;" ::: "memory");             // order the copy engine's writes before the flag stores of the barrier
  }
  if (SYNC) {
    if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
    if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
  }
}

}  // namespace b200coll

#include "p2p.cuh"

namespace b200coll {

__global__ void k_barrier(COMM_PARAM, uint32_t op) {
  pdl_prologue();
  const uint32_t s = load_seq(c, kSeqBarrier);
  if (!barrier_blocks<true>(c, 2 * s + 2, op)) return;
  if (threadIdx.x == 0 && last_block_ticket(c)) c.state[kSeqBarrier] = s + 1;
}

__global__ void k_fill_u32(uint32_t* p, size_t n, uint32_t v) {
  pdl_prologue();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

}  // namespace b200coll
