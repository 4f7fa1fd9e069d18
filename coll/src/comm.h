// Host-side communicator state for libb200coll.
#pragma once
#include <cuda.h>
#include <sched.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../include/b200coll.h"
#include "bootstrap.h"
#include "device.cuh"

namespace b200coll {

// Driver entry points resolved at run time (cudaGetDriverEntryPoint) so the library loads — and its
// CPU-side logic is testable — on a box without libcuda.
#define B200COLL_DRV_FUNCS(X)                                                                                          \
  X(cuMemCreate) X(cuMemRelease) X(cuMemMap) X(cuMemUnmap) X(cuMemAddressReserve) X(cuMemAddressFree)                   \
  X(cuMemSetAccess) X(cuMemExportToShareableHandle) X(cuMemImportFromShareableHandle)                                  \
  X(cuMemGetAllocationGranularity) X(cuMulticastCreate) X(cuMulticastAddDevice) X(cuMulticastBindMem)                  \
  X(cuMulticastUnbind) X(cuMulticastGetGranularity) X(cuDeviceGet) X(cuDeviceGetAttribute) X(cuGetErrorString)         \
  X(cuDriverGetVersion) X(cuDeviceGetUuid)

struct Drv {
#define X(n) decltype(&::n) n = nullptr;
  B200COLL_DRV_FUNCS(X)
#undef X
  bool ok = false;
  std::string why;
};
const Drv& drv();

void set_last_error(const std::string& s);
void dbg(int level, const char* fmt, ...);
int debug_level();

struct FreeBlock { size_t off, len; };

struct Arena {
  CUmemGenericAllocationHandle handle = 0;
  size_t total = 0;               // bytes, granularity-rounded (control + heap)
  int device = -1;
};

// Host path (hostpath.cu): copy streams, events and the two staging pairs of b200collAllReduceHost.
struct HostPath {
  cudaStream_t h2d = nullptr, d2h = nullptr;
  cudaEvent_t ev_start = nullptr, ev_in_ready[2] = {}, ev_in_free[2] = {}, ev_out_free[2] = {};
  void* in[2] = {};
  void* out[2] = {};
  size_t chunk_bytes = 0;
};

extern std::atomic<int> g_loopback_comms;   // live communicators whose ranks share a GPU (virtual ranks): PDL stays off

struct SharedGroup;   // in-process groups (InitAll) share ownership bookkeeping

}  // namespace b200coll

struct b200collComm {
  int rank = 0, nranks = 1, device = 0;
  b200collConfig cfg{};
  b200coll::Arena arena;
  CUdeviceptr peer_va[B200COLL_MAX_RANKS] = {};
  CUmemGenericAllocationHandle peer_handle[B200COLL_MAX_RANKS] = {};   // imported (multi-process) or borrowed (in-process)
  bool peer_handle_owned[B200COLL_MAX_RANKS] = {};
  CUdeviceptr mc_va = 0;
  CUmemGenericAllocationHandle mc_handle = 0;
  bool mc_owned = false, mc_bound = false;
  bool nvls = false, loopback = false, loopback_counted = false;
  int sm_count = 0, driver_version = 0;
  uint32_t* state_dev = nullptr;
  b200collFault* fault_host = nullptr;
  b200collFault* fault_dev = nullptr;
  b200coll::CommDev dev{};
  std::unique_ptr<b200coll::Bootstrap> boot;
  // symmetric heap allocator (offsets relative to arena base)
  std::vector<b200coll::FreeBlock> free_list;
  std::map<size_t, size_t> live;   // off -> len
  std::mutex mu;
  b200collAlgo_t forced_algo = b200collAlgoAuto;
  int max_ctas = 0;
  // NVLS all-reduce/all-gather, P2P, LL, NVLS reduce-scatter. Measured on 8xB200 (profiles/launch_shapes_n8.md): the
  // multimem all-reduce saturates with 16-64 CTAs x 256 threads and degrades above ~100 CTAs; the ld_reduce-only
  // reduce-scatter kernel (2 loads in flight per thread) needs 64 x 512.
  struct Shape { int max_ctas; int threads; } shape[5] = {{32, 256}, {0, 0}, {148, 0}, {64, 512}, {148, 512}};   // [4]: rooted NVLS ops — only the root moves data, so ONE rank must keep the link busy: 148 x 512 threads x 2-4 vectors = 2.4-4.8 MB in flight (at 32 x 256 the 8-GPU broadcast stopped at 372 GB/s, NCCL 655)
  b200collStats stats{};
  std::shared_ptr<b200coll::SharedGroup> group;
  void* stats_shm = nullptr;       // exported stats page (metrics exporter reads it)
  std::string stats_shm_name;
  std::string boot_name;                // rendezvous name this communicator was created under (multi-process only); splits derive theirs from it
  uint32_t split_seq = 0;               // CommSplit calls so far (a collective call, so the same on every rank)
  size_t p2p_window = 0;                // staged receives: bytes per staging window; 0 = an equal share of the staging area
  uint32_t stats_tick = 0;              // collective calls since init; the counters page is refreshed every 256
  unsigned long long bulk_grid_hint = 0; // chunks the largest rank of a rooted / personalised bulk launch has (set by the caller, consumed by launch_bulk)
  int numa_node = -1;                   // of this rank's GPU (sysfs), -1 unknown
  std::string local_cpulist;            // GPU-local CPUs as sysfs prints them
  cpu_set_t affinity_saved;             // the calling thread's mask before CommInitRank narrowed it
  bool affinity_changed = false;
  b200coll::HostPath host;
  std::map<void*, size_t> host_allocs;  // HostAlloc: base -> mapped length
};

namespace b200coll {

void stats_page_publish(b200collComm* c);   // comm.cu

// ---- staging (collectives.cu, generic.cu): buffers outside the symmetric arena go through the two staging halves, chunk by chunk.
// A chunk of n elements that starts at element `done` is copied into staging half 0 as `rows` rows (row r: elements
// [r * count + done, + n) of the user buffer -> [r * n, + n) of the half), the kernel runs, and the result is copied out of
// staging half 1 the same way. A null buffer skips that copy: the kernel reads or writes the user buffer itself.
struct StageIn { const void* buf; size_t elem; int rows; };
struct StageOut { void* buf; size_t elem; int rows; };

inline char* stage_ptr(b200collComm* c, int half) { return reinterpret_cast<char*>(c->peer_va[c->rank]) + kOffStage + (size_t)half * kStageHalfBytes; }
// elements per chunk when `rows` rows of `elem`-byte elements share one staging half
inline size_t stage_chunk(size_t elem, int rows) { return kStageHalfBytes / elem / rows / 64 * 64; }
// `rows` device-to-device copies of `bytes` each, row r from src + r * src_pitch to dst + r * dst_pitch
b200collResult_t copy_rows(char* dst, size_t dst_pitch, const char* src, size_t src_pitch, size_t bytes, int rows, cudaStream_t st);

template <typename F>
b200collResult_t run_staged(b200collComm* c, size_t count, size_t chunk, StageIn in, StageOut out, cudaStream_t st, F&& kernel) {
  c->stats.staged_calls++;
  for (size_t done = 0; done < count; done += chunk) {
    const size_t n = std::min(chunk, count - done);
    b200collResult_t rc = b200collSuccess;
    if (in.buf) rc = copy_rows(stage_ptr(c, 0), n * in.elem, static_cast<const char*>(in.buf) + done * in.elem, count * in.elem, n * in.elem, in.rows, st);
    if (rc == b200collSuccess) rc = kernel(done, n);
    if (rc == b200collSuccess && out.buf) rc = copy_rows(static_cast<char*>(out.buf) + done * out.elem, count * out.elem, stage_ptr(c, 1), n * out.elem, n * out.elem, out.rows, st);
    if (rc != b200collSuccess) return rc;
  }
  return b200collSuccess;
}

// generic.cu
bool needs_generic(const b200collEpilogue* ep, b200collRedOp_t rop);
b200collResult_t generic_reduce(b200collComm* c, b200collOp_t which, const void* send, void* recv, size_t count, const b200collEpilogue* ep, b200collRedOp_t rop, int root, cudaStream_t st);

// hostpath.cu
void bind_to_gpu_numa(b200collComm* c, bool allow_bind);   // allow_bind=false: only record the node (in-process groups spanning GPUs)
void restore_affinity_after_init(b200collComm* c);
void hostpath_destroy(b200collComm* c);

}  // namespace b200coll
