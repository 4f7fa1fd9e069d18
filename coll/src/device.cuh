// Device-side primitives shared by every libb200coll kernel (sm_100a only).
//   * symmetric-arena addressing (peer[] table + multicast alias)
//   * epoch barrier over per-block flags in each rank's control page (monotonic, never reset)
//   * Lamport (flag-in-payload) slot protocol for the zero-barrier small-message path
//   * multimem.{ld_reduce,st} wrappers (NVLS: reduce / broadcast inside the NVSwitch)
//   * 16-byte vector load/convert/store for {f32,f16,bf16,e4m3,e5m2} in and out (fp8: 16 elements per vector)
// Every cross-GPU spin carries a globaltimer watchdog that records a b200collFault and bails
// out instead of hanging the GPU (SURVEY §5.3).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <stdint.h>
#include "../include/b200coll.h"
#include "layout.h"

namespace b200coll {

// How kernels receive the communicator: as a __grid_constant__ parameter, so that peer[t] with a run-time t is an indexed load from
// the constant bank (LDC c[0x0][R+0x380]). Passed by value the compiler copies the 104-byte struct to the stack of every thread
// (STACK:104 in cuobjdump --dump-resource-usage) and every lookup becomes a local-memory load; -DB200COLL_VARIANT_BYVALUE
// (make VARIANT=byvalue -> lib/libb200coll_byvalue.so) keeps that form for A/B runs.
#ifdef B200COLL_VARIANT_BYVALUE
#define COMM_PARAM CommDev c
#else
#define COMM_PARAM const __grid_constant__ CommDev c
#endif

// ---------------------------------------------------------------- misc
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// Takes scalars, not the CommDev: passing the kernel-parameter struct by reference to a noinline function forces a
// 104-byte stack copy of it in every kernel and turns each peer[] lookup into a local-memory load.
static __device__ __noinline__ void record_fault_impl(b200collFault* f, uint32_t rank, uint32_t code, uint32_t peer, uint32_t expected, uint32_t observed, uint32_t op) {
  if (atomicCAS(&f->code, 0u, code) == 0u) {
    f->rank = rank; f->peer = peer; f->block = blockIdx.x; f->expected = expected; f->observed = observed; f->op = op;
    __threadfence_system();
  }
}
__device__ __forceinline__ void record_fault(const CommDev& c, uint32_t code, uint32_t peer, uint32_t expected, uint32_t observed, uint32_t op) {
  record_fault_impl(c.fault, (uint32_t)c.rank, code, peer, expected, observed, op);
}

// Programmatic dependent launch: let the next kernel in the stream start launching now, then wait until the previous
// kernel's memory is visible. Both are no-ops unless the launch carried the programmatic-serialization attribute.
__device__ __forceinline__ void pdl_prologue() {
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ---------------------------------------------------------------- flags
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
// multimem.red: the switch applies the add to the word at this offset of EVERY rank's arena
__device__ __forceinline__ void mc_red_add_release_u32(void* mc_addr, uint32_t v) { asm volatile("multimem.red.release.sys.global.add.u32 [%0], %1;" ::"l"(mc_addr), "r"(v) : "memory"); }
__device__ __forceinline__ void mc_red_add_relaxed_u32(void* mc_addr, uint32_t v) { asm volatile("multimem.red.relaxed.sys.global.add.u32 [%0], %1;" ::"l"(mc_addr), "r"(v) : "memory"); }

}  // namespace b200coll

#include "barrier.cuh"

namespace b200coll {

// ---------------------------------------------------------------- vector memory ops
__device__ __forceinline__ uint4 ld_vec(const void* p) {   // streaming 16 B load (own or peer memory)
  uint4 v;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ uint4 ld_vec_volatile(const void* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_vec(void* p, const uint4& v) {
  asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_vec_volatile(void* p, const uint4& v) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---- NVLS
template <typename InT> __device__ __forceinline__ uint4 mc_ld_reduce(const void* mc_addr);
template <> __device__ __forceinline__ uint4 mc_ld_reduce<__nv_bfloat16>(const void* a) {
  uint4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(a) : "memory");
  return v;
}
template <> __device__ __forceinline__ uint4 mc_ld_reduce<__half>(const void* a) {
  uint4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.f16x2 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(a) : "memory");
  return v;
}
template <> __device__ __forceinline__ uint4 mc_ld_reduce<float>(const void* a) {
  uint4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(a) : "memory");
  return v;
}
__device__ __forceinline__ void mc_st_words(void* a, const uint32_t* w, int nwords) {
  // nwords in {1,2,4}
  if (nwords == 4)
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(a), "f"(__uint_as_float(w[0])), "f"(__uint_as_float(w[1])),
                 "f"(__uint_as_float(w[2])), "f"(__uint_as_float(w[3])) : "memory");
  else if (nwords == 2)
    asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1,%2};" ::"l"(a), "f"(__uint_as_float(w[0])), "f"(__uint_as_float(w[1])) : "memory");
  else
    asm volatile("multimem.st.relaxed.sys.global.u32 [%0], %1;" ::"l"(a), "r"(w[0]) : "memory");
}

// ---------------------------------------------------------------- type handling
template <typename T> struct Epv { static constexpr int value = 16 / (int)sizeof(T); };

template <typename InT> __device__ __forceinline__ void unpack_add(float* acc, const uint4& v);
template <> __device__ __forceinline__ void unpack_add<float>(float* acc, const uint4& v) {
  acc[0] += __uint_as_float(v.x); acc[1] += __uint_as_float(v.y); acc[2] += __uint_as_float(v.z); acc[3] += __uint_as_float(v.w);
}
template <> __device__ __forceinline__ void unpack_add<__nv_bfloat16>(float* acc, const uint4& v) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; i++) { acc[2 * i] += __uint_as_float(w[i] << 16); acc[2 * i + 1] += __uint_as_float(w[i] & 0xFFFF0000u); }
}
template <> __device__ __forceinline__ void unpack_add<__half>(float* acc, const uint4& v) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; i++) {
    __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
    float2 f = __half22float2(h);
    acc[2 * i] += f.x; acc[2 * i + 1] += f.y;
  }
}
// fp8: 16 elements per vector. fp8 -> f16 -> f32 is exact for both encodings (every e4m3 / e5m2 value is an f16 value); the low byte
// of each word is the lower-indexed element, as Pack<fp8> writes it.
template <__nv_fp8_interpretation_t K>
__device__ __forceinline__ void unpack_add_fp8(float* acc, const uint4& v) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; i++) {
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const __half2 p = __half2(__nv_cvt_fp8x2_to_halfraw2((__nv_fp8x2_storage_t)(w[i] >> (16 * h)), K));
      const float2 f = __half22float2(p);
      acc[4 * i + 2 * h] += f.x; acc[4 * i + 2 * h + 1] += f.y;
    }
  }
}
template <> __device__ __forceinline__ void unpack_add<__nv_fp8_e4m3>(float* acc, const uint4& v) { unpack_add_fp8<__NV_E4M3>(acc, v); }
template <> __device__ __forceinline__ void unpack_add<__nv_fp8_e5m2>(float* acc, const uint4& v) { unpack_add_fp8<__NV_E5M2>(acc, v); }

template <typename T> struct IsFp8 { static constexpr bool value = false; };
template <> struct IsFp8<__nv_fp8_e4m3> { static constexpr bool value = true; };
template <> struct IsFp8<__nv_fp8_e5m2> { static constexpr bool value = true; };

// pack E floats into E*sizeof(OutT)/4 words
template <typename OutT, int E> struct Pack;
template <int E> struct Pack<float, E> {
  static constexpr int W = E;
  static __device__ __forceinline__ void run(const float* f, uint32_t* w) {
#pragma unroll
    for (int i = 0; i < E; i++) w[i] = __float_as_uint(f[i]);
  }
};
template <int E> struct Pack<__nv_bfloat16, E> {
  static constexpr int W = E / 2;
  static __device__ __forceinline__ void run(const float* f, uint32_t* w) {
#pragma unroll
    for (int i = 0; i < E / 2; i++) { __nv_bfloat162 b = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]); w[i] = *reinterpret_cast<uint32_t*>(&b); }
  }
};
template <int E> struct Pack<__half, E> {
  static constexpr int W = E / 2;
  static __device__ __forceinline__ void run(const float* f, uint32_t* w) {
#pragma unroll
    for (int i = 0; i < E / 2; i++) { __half2 b = __floats2half2_rn(f[2 * i], f[2 * i + 1]); w[i] = *reinterpret_cast<uint32_t*>(&b); }
  }
};
template <int E> struct Pack<__nv_fp8_e4m3, E> {
  static constexpr int W = E / 4;
  static __device__ __forceinline__ void run(const float* f, uint32_t* w) {
#pragma unroll
    for (int i = 0; i < E / 4; i++) {
      uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(f[4 * i], f[4 * i + 1]), __NV_SATFINITE, __NV_E4M3);
      uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(f[4 * i + 2], f[4 * i + 3]), __NV_SATFINITE, __NV_E4M3);
      w[i] = lo | (hi << 16);
    }
  }
};
template <int E> struct Pack<__nv_fp8_e5m2, E> {
  static constexpr int W = E / 4;
  static __device__ __forceinline__ void run(const float* f, uint32_t* w) {
#pragma unroll
    for (int i = 0; i < E / 4; i++) {
      uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(f[4 * i], f[4 * i + 1]), __NV_SATFINITE, __NV_E5M2);
      uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(f[4 * i + 2], f[4 * i + 3]), __NV_SATFINITE, __NV_E5M2);
      w[i] = lo | (hi << 16);
    }
  }
};

template <int W> __device__ __forceinline__ void st_words(void* p, const uint32_t* w) {
  if constexpr (W == 16) {   // fp8 in, fp32 out: one input vector widens to 64 bytes
#pragma unroll
    for (int q = 0; q < 4; q++) st_vec(reinterpret_cast<char*>(p) + 16 * q, make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]));
    return;
  }
  if (W == 8) {
    st_vec(p, make_uint4(w[0], w[1], w[2], w[3]));
    st_vec(reinterpret_cast<char*>(p) + 16, make_uint4(w[4], w[5], w[6], w[7]));
  } else if (W == 4) {
    st_vec(p, make_uint4(w[0], w[1], w[2], w[3]));
  } else if (W == 2) {
    asm volatile("st.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(w[0]), "r"(w[1]) : "memory");
  } else {
    asm volatile("st.global.u32 [%0], %1;" ::"l"(p), "r"(w[0]) : "memory");
  }
}
template <int W> __device__ __forceinline__ void mc_st_wordsW(void* p, const uint32_t* w) {
  if (W == 8) { mc_st_words(p, w, 4); mc_st_words(reinterpret_cast<char*>(p) + 16, w + 4, 4); }
  else mc_st_words(p, w, W);
}

template <typename T> __device__ __forceinline__ float to_float(T v);
template <> __device__ __forceinline__ float to_float<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_float<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_float<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __nv_fp8_e4m3 from_float<__nv_fp8_e4m3>(float v) { return __nv_fp8_e4m3(v); }   // round to nearest, saturate to +-448
template <> __device__ __forceinline__ __nv_fp8_e5m2 from_float<__nv_fp8_e5m2>(float v) { return __nv_fp8_e5m2(v); }   // round to nearest, saturate to +-57344
template <> __device__ __forceinline__ float to_float<__nv_fp8_e4m3>(__nv_fp8_e4m3 v) { return float(v); }
template <> __device__ __forceinline__ float to_float<__nv_fp8_e5m2>(__nv_fp8_e5m2 v) { return float(v); }

// Element e of a peer's buffer, read with a volatile load (scalar tails). The fp8 classes cannot be copied from a volatile object,
// so their byte is loaded as a plain integer and reinterpreted.
template <typename T> __device__ __forceinline__ float ld_volatile_float(const char* base, size_t e) { return to_float<T>(reinterpret_cast<const volatile T*>(base)[e]); }
template <> __device__ __forceinline__ float ld_volatile_float<__nv_fp8_e4m3>(const char* base, size_t e) {
  __nv_fp8_e4m3 v; v.__x = reinterpret_cast<const volatile __nv_fp8_storage_t*>(base)[e]; return float(v);
}
template <> __device__ __forceinline__ float ld_volatile_float<__nv_fp8_e5m2>(const char* base, size_t e) {
  __nv_fp8_e5m2 v; v.__x = reinterpret_cast<const volatile __nv_fp8_storage_t*>(base)[e]; return float(v);
}

}  // namespace b200coll
