// libb200coll_nccl.so — the subset of the NCCL C API that nccl-tests' *_perf binaries (and most framework glue) call,
// implemented on libb200coll, so an unmodified `all_reduce_perf` can be pointed at this library (LD_PRELOAD or a
// libnccl.so.2 symlink in LD_LIBRARY_PATH=/usr/local/nvidia/lib64, which is how the reference's pods pick up the
// installer-dropped NCCL: gpudirect-rdma/nccl-test-a4.yaml:42-68). SURVEY §5.8-6.
// User buffers are ordinary cudaMalloc memory here, so calls take the Lamport path (<= 512 KiB) or the staged path;
// ncclMemAlloc hands out symmetric-arena memory once a communicator exists (zero-copy + NVLS).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../include/b200coll.h"

extern "C" {

typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef enum { ncclSuccess = 0, ncclUnhandledCudaError = 1, ncclSystemError = 2, ncclInternalError = 3, ncclInvalidArgument = 4, ncclInvalidUsage = 5, ncclRemoteError = 6, ncclInProgress = 7 } ncclResult_t;
typedef enum { ncclInt8 = 0, ncclUint8 = 1, ncclInt32 = 2, ncclUint32 = 3, ncclInt64 = 4, ncclUint64 = 5, ncclFloat16 = 6, ncclFloat32 = 7, ncclFloat64 = 8, ncclBfloat16 = 9,
               ncclFloat8e4m3 = 10, ncclFloat8e5m2 = 11, ncclNumTypes = 12 } ncclDataType_t;
typedef enum { ncclSum = 0, ncclProd = 1, ncclMax = 2, ncclMin = 3, ncclAvg = 4 } ncclRedOp_t;
typedef enum { ncclScalarDevice = 0, ncclScalarHostImmediate = 1 } ncclScalarResidence_t;
typedef struct ncclWindow_vidmem* ncclWindow_t;
typedef struct ncclSimInfo_opaque ncclSimInfo_t;
typedef struct ncclConfig_opaque ncclConfig_t;      /* blocking, cgaClusterSize, ...: nothing in it has an analogue here */

}  // extern "C"

namespace {

struct ShimComm { b200collComm_t comm; int nranks, rank, device; };
struct P2pOp { bool send; const void* sbuf; void* rbuf; size_t count; ncclDataType_t dt; int peer; ShimComm* comm; cudaStream_t stream; };
thread_local int g_group_depth = 0;
thread_local std::vector<P2pOp> g_group_ops;
std::mutex g_mu;
ShimComm* g_last_comm = nullptr;   // ncclMemAlloc has no communicator argument

ncclResult_t map_rc(b200collResult_t r) {
  switch (r) {
    case b200collSuccess: return ncclSuccess;
    case b200collUnhandledCudaError: return ncclUnhandledCudaError;
    case b200collSystemError: return ncclSystemError;
    case b200collInvalidArgument: return ncclInvalidArgument;
    case b200collInvalidUsage: return ncclInvalidUsage;
    case b200collRemoteError: return ncclRemoteError;
    default: return ncclInternalError;
  }
}

bool map_dt(ncclDataType_t dt, b200collDataType_t* out) {
  switch (dt) {
    case ncclFloat32: *out = b200collFloat32; return true;
    case ncclFloat16: *out = b200collFloat16; return true;
    case ncclBfloat16: *out = b200collBfloat16; return true;
    default: return false;   // integer / fp64 / fp8: reductions go through map_dt_reduce, data movement through map_dt_as_words
  }
}

// Every NCCL element type that libb200coll can reduce, fp8 included (NCCL reduces e4m3 / e5m2 since 2.24): fp8 sum / avg / PreMulSum
// run on the fused fp32-accumulating kernels, min / max / prod and the integer / fp64 types on the generic kernel.
bool map_dt_reduce(ncclDataType_t dt, b200collDataType_t* out) {
  switch (dt) {
    case ncclInt8: *out = b200collInt8; return true;
    case ncclUint8: *out = b200collUint8; return true;
    case ncclInt32: *out = b200collInt32; return true;
    case ncclUint32: *out = b200collUint32; return true;
    case ncclInt64: *out = b200collInt64; return true;
    case ncclUint64: *out = b200collUint64; return true;
    case ncclFloat64: *out = b200collFloat64; return true;
    case ncclFloat8e4m3: *out = b200collFloat8e4m3; return true;
    case ncclFloat8e5m2: *out = b200collFloat8e5m2; return true;
    default: return map_dt(dt, out);
  }
}

// ncclRedOpCreatePreMulSum: "multiply every input by a scalar, then sum". With one scalar per communicator call that is
// scale * sum, i.e. the library's fused epilogue scale. Handles are ncclNumOps + slot.
constexpr int kNcclNumOps = 5;
std::vector<float> g_premul;          // slot -> scalar (NaN = free)
bool map_op(ncclRedOp_t op, b200collRedOp_t* rop, float* scale) {
  *scale = 1.0f;
  if (op == ncclSum) { *rop = b200collSum; return true; }
  if (op == ncclAvg) { *rop = b200collAvg; return true; }
  if (op == ncclProd) { *rop = b200collProd; return true; }
  if (op == ncclMax) { *rop = b200collMax; return true; }
  if (op == ncclMin) { *rop = b200collMin; return true; }
  std::lock_guard<std::mutex> lk(g_mu);
  const int slot = (int)op - kNcclNumOps;
  if (slot < 0 || slot >= (int)g_premul.size() || g_premul[slot] != g_premul[slot]) return false;   // a stale or foreign handle
  *rop = b200collSum; *scale = g_premul[slot];
  return true;
}

size_t nccl_type_size(ncclDataType_t dt) {
  switch ((int)dt) {
    case ncclInt8: case ncclUint8: case ncclFloat8e4m3: case ncclFloat8e5m2: return 1;
    case ncclFloat16: case ncclBfloat16: return 2;
    case ncclInt32: case ncclUint32: case ncclFloat32: return 4;
    case ncclInt64: case ncclUint64: case ncclFloat64: return 8;
    default: return 0;
  }
}

// nccl-tests' alltoall (and most MoE glue) is a group of one send and one recv per peer, equal counts, contiguous blocks: that is
// the library's fused all-to-all kernel. Every rank of such a group sees the same shape, so the decision is the same everywhere.
// B200COLL_SHIM_FUSE_ALLTOALL=0 turns the shortcut off (needed only if ranks mix this shape with other group shapes in one step).
bool group_is_alltoall(const std::vector<P2pOp>& ops, const void** send0, void** recv0, size_t* count, b200collDataType_t* dt) {
  static const bool fuse = [] { const char* e = getenv("B200COLL_SHIM_FUSE_ALLTOALL"); return !(e && *e == '0'); }();
  if (!fuse || ops.empty()) return false;
  ShimComm* c = ops[0].comm;
  const int n = c->nranks;
  if ((int)ops.size() != 2 * n || !map_dt(ops[0].dt, dt)) return false;
  std::vector<const P2pOp*> sends(n, nullptr), recvs(n, nullptr);
  for (const P2pOp& o : ops) {
    if (o.comm != c || o.peer < 0 || o.peer >= n || o.dt != ops[0].dt || o.stream != ops[0].stream) return false;
    const P2pOp*& slot = (o.send ? sends : recvs)[o.peer];
    if (slot) return false;
    slot = &o;
  }
  const size_t cnt = ops[0].count, esz = b200collTypeSize(*dt);
  if (cnt == 0 || (cnt * esz) % 16 != 0) return false;
  for (int p = 0; p < n; p++) {
    if (!sends[p] || !recvs[p] || sends[p]->count != cnt || recvs[p]->count != cnt) return false;
    if ((const char*)sends[p]->sbuf != (const char*)sends[0]->sbuf + (size_t)p * cnt * esz) return false;
    if ((char*)recvs[p]->rbuf != (char*)recvs[0]->rbuf + (size_t)p * cnt * esz) return false;
  }
  *send0 = sends[0]->sbuf; *recv0 = recvs[0]->rbuf; *count = cnt;
  return true;
}

ncclResult_t flush_group() {
  std::vector<P2pOp> ops;
  ops.swap(g_group_ops);
  if (ops.empty()) return ncclSuccess;
  const void* s0; void* r0; size_t count; b200collDataType_t dt;
  if (group_is_alltoall(ops, &s0, &r0, &count, &dt)) {
    b200collEpilogue ep{dt, dt, 1.0f};
    return map_rc(b200collAllToAll(s0, r0, count, &ep, ops[0].comm->comm, ops[0].stream));
  }
  // anything else (ring steps, pipeline hand-overs, irregular exchanges): the library's point-to-point kernel, one launch per communicator
  b200collResult_t rc = b200collGroupStart();
  for (const P2pOp& o : ops) {
    if (rc != b200collSuccess) break;
    const size_t bytes = o.count * nccl_type_size(o.dt);
    rc = o.send ? b200collSend(o.sbuf, bytes, o.peer, o.comm->comm, o.stream) : b200collRecv(o.rbuf, bytes, o.peer, o.comm->comm, o.stream);
  }
  const b200collResult_t rc_end = b200collGroupEnd();
  return map_rc(rc != b200collSuccess ? rc : rc_end);
}

}  // namespace

extern "C" {

ncclResult_t ncclGetVersion(int* v) { if (!v) return ncclInvalidArgument; *v = 22809; return ncclSuccess; }   // advertises the 2.28 API level
const char* ncclGetErrorString(ncclResult_t r) { return b200collGetErrorString((b200collResult_t)r); }
const char* ncclGetLastError(ncclComm_t) { return b200collGetLastError(); }

ncclResult_t ncclGetUniqueId(ncclUniqueId* id) {
  if (!id) return ncclInvalidArgument;
  static_assert(sizeof(ncclUniqueId) == sizeof(b200collUniqueId), "id sizes must match");
  return map_rc(b200collGetUniqueId(reinterpret_cast<b200collUniqueId*>(id)));
}

ncclResult_t ncclCommInitRank(ncclComm_t* comm, int nranks, ncclUniqueId id, int rank) {
  if (!comm) return ncclInvalidArgument;
  ShimComm* s = new ShimComm{nullptr, nranks, rank, 0};
  cudaGetDevice(&s->device);
  b200collResult_t r = b200collCommInitRank(&s->comm, nranks, reinterpret_cast<const b200collUniqueId*>(&id), rank, nullptr);
  if (r != b200collSuccess) { delete s; return map_rc(r); }
  { std::lock_guard<std::mutex> lk(g_mu); g_last_comm = s; }
  *comm = reinterpret_cast<ncclComm_t>(s);
  return ncclSuccess;
}

ncclResult_t ncclCommInitAll(ncclComm_t* comms, int ndev, const int* devlist) {
  if (!comms || ndev < 1 || ndev > B200COLL_MAX_RANKS) return ncclInvalidArgument;
  b200collComm_t cs[B200COLL_MAX_RANKS];
  b200collResult_t r = b200collCommInitAll(cs, ndev, devlist, nullptr);
  if (r != b200collSuccess) return map_rc(r);
  for (int i = 0; i < ndev; i++) comms[i] = reinterpret_cast<ncclComm_t>(new ShimComm{cs[i], ndev, i, devlist ? devlist[i] : i});
  return ncclSuccess;
}

ncclResult_t ncclCommDestroy(ncclComm_t comm) {
  ShimComm* s = reinterpret_cast<ShimComm*>(comm);
  if (!s) return ncclInvalidArgument;
  { std::lock_guard<std::mutex> lk(g_mu); if (g_last_comm == s) g_last_comm = nullptr; }
  b200collResult_t r = b200collCommDestroy(s->comm);
  delete s;
  return map_rc(r);
}
// Config structs, registration handles and splits of newer NCCL APIs: accepted where a no-op is faithful, refused where it is not.
ncclResult_t ncclCommInitRankConfig(ncclComm_t* comm, int nranks, ncclUniqueId id, int rank, ncclConfig_t* /*config*/) {
  return ncclCommInitRank(comm, nranks, id, rank);
}
ncclResult_t ncclCommSplit(ncclComm_t comm, int color, int key, ncclComm_t* newcomm, ncclConfig_t* /*config*/) {
  if (!comm || !newcomm) return ncclInvalidArgument;
  ShimComm* parent = reinterpret_cast<ShimComm*>(comm);
  *newcomm = nullptr;
  b200collComm_t child = nullptr;
  const b200collResult_t r = b200collCommSplit(parent->comm, color, key, &child, nullptr);
  if (r != b200collSuccess || !child) return map_rc(r);        // NCCL_SPLIT_NOCOLOR: success with a NULL communicator
  b200collCommInfo info;
  if (b200collCommInfoGet(child, &info) != b200collSuccess) { b200collCommDestroy(child); return ncclInternalError; }
  ShimComm* s = new ShimComm{child, info.nranks, info.rank, info.device};
  { std::lock_guard<std::mutex> lk(g_mu); g_last_comm = s; }
  *newcomm = reinterpret_cast<ncclComm_t>(s);
  return ncclSuccess;
}
ncclResult_t ncclCommRegister(const ncclComm_t comm, void* buff, size_t, void** handle) {              // arena memory is registered by construction
  if (!comm || !handle) return ncclInvalidArgument;
  *handle = buff;
  return ncclSuccess;
}
ncclResult_t ncclCommDeregister(const ncclComm_t, void*) { return ncclSuccess; }
ncclResult_t ncclRedOpCreatePreMulSum(ncclRedOp_t* op, void* scalar, ncclDataType_t dt, ncclScalarResidence_t residence, ncclComm_t comm) {
  if (!op || !scalar || !comm) return ncclInvalidArgument;
  unsigned char raw[8] = {};
  const size_t sz = dt == ncclFloat64 ? 8 : dt == ncclFloat32 ? 4 : (dt == ncclFloat16 || dt == ncclBfloat16) ? 2 : 0;
  if (!sz) return ncclInvalidArgument;
  if (residence == ncclScalarHostImmediate) memcpy(raw, scalar, sz);
  else if (cudaMemcpy(raw, scalar, sz, cudaMemcpyDeviceToHost) != cudaSuccess) return ncclUnhandledCudaError;
  float v;
  if (dt == ncclFloat64) { double d; memcpy(&d, raw, 8); v = (float)d; }
  else if (dt == ncclFloat32) memcpy(&v, raw, 4);
  else { unsigned short h; memcpy(&h, raw, 2); if (dt == ncclBfloat16) { unsigned int w = (unsigned int)h << 16; memcpy(&v, &w, 4); } else { __half hh; memcpy(&hh, &h, 2); v = __half2float(hh); } }
  std::lock_guard<std::mutex> lk(g_mu);
  size_t slot = 0;
  while (slot < g_premul.size() && g_premul[slot] == g_premul[slot]) slot++;
  if (slot == g_premul.size()) g_premul.push_back(v); else g_premul[slot] = v;
  *op = (ncclRedOp_t)(kNcclNumOps + (int)slot);
  return ncclSuccess;
}
ncclResult_t ncclRedOpDestroy(ncclRedOp_t op, ncclComm_t) {
  std::lock_guard<std::mutex> lk(g_mu);
  const int slot = (int)op - kNcclNumOps;
  if (slot < 0 || slot >= (int)g_premul.size()) return ncclInvalidArgument;
  g_premul[slot] = __builtin_nanf("");
  return ncclSuccess;
}
ncclResult_t ncclCommFinalize(ncclComm_t) { return ncclSuccess; }
ncclResult_t ncclCommAbort(ncclComm_t comm) { return ncclCommDestroy(comm); }
ncclResult_t ncclCommCount(const ncclComm_t comm, int* n) { if (!comm || !n) return ncclInvalidArgument; *n = reinterpret_cast<ShimComm*>(comm)->nranks; return ncclSuccess; }
ncclResult_t ncclCommUserRank(const ncclComm_t comm, int* r) { if (!comm || !r) return ncclInvalidArgument; *r = reinterpret_cast<ShimComm*>(comm)->rank; return ncclSuccess; }
ncclResult_t ncclCommCuDevice(const ncclComm_t comm, int* d) { if (!comm || !d) return ncclInvalidArgument; *d = reinterpret_cast<ShimComm*>(comm)->device; return ncclSuccess; }
ncclResult_t ncclCommGetAsyncError(ncclComm_t comm, ncclResult_t* out) {
  if (!comm || !out) return ncclInvalidArgument;
  *out = map_rc(b200collCommGetAsyncError(reinterpret_cast<ShimComm*>(comm)->comm, nullptr));
  return ncclSuccess;
}

ncclResult_t ncclMemAlloc(void** ptr, size_t size) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_last_comm) return map_rc(b200collMemAlloc(g_last_comm->comm, ptr, size));
  return cudaMalloc(ptr, size) == cudaSuccess ? ncclSuccess : ncclUnhandledCudaError;
}
ncclResult_t ncclMemFree(void* ptr) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_last_comm && b200collIsSymmetric(g_last_comm->comm, ptr, 1)) return map_rc(b200collMemFree(g_last_comm->comm, ptr));
  return cudaFree(ptr) == cudaSuccess ? ncclSuccess : ncclUnhandledCudaError;
}

ncclResult_t ncclAllReduce(const void* send, void* recv, size_t count, ncclDataType_t dt, ncclRedOp_t op, ncclComm_t comm, cudaStream_t stream) {
  b200collDataType_t t;
  b200collRedOp_t rop; float scale;
  if (!comm || !map_dt_reduce(dt, &t) || !map_op(op, &rop, &scale)) return ncclInvalidArgument;
  b200collEpilogue ep{t, t, scale};
  return map_rc(b200collAllReduce(send, recv, count, &ep, rop, reinterpret_cast<ShimComm*>(comm)->comm, stream));
}
static bool map_dt_as_words(ncclDataType_t dt, size_t count, b200collDataType_t* t, size_t* n);
// All-gather moves bits, so integer types ride the fp kernels as words — on the barrier-based kernels only: the Lamport path marks empty
// slots with a NaN pattern and rewrites payload words equal to it (harmless for floats, wrong for an int32 -1).
struct BitExactScope {
  b200collComm_t c; b200collAlgo_t prev;
  explicit BitExactScope(b200collComm_t comm) : c(comm), prev(b200collCommGetAlgo(comm)) { b200collCommSetAlgo(c, b200collAlgoTwoShot); }
  ~BitExactScope() { b200collCommSetAlgo(c, prev); }
};
ncclResult_t ncclAllGather(const void* send, void* recv, size_t sendcount, ncclDataType_t dt, ncclComm_t comm, cudaStream_t stream) {
  if (!comm) return ncclInvalidArgument;
  b200collComm_t c = reinterpret_cast<ShimComm*>(comm)->comm;
  b200collDataType_t t;
  if (map_dt(dt, &t)) {
    b200collEpilogue ep{t, t, 1.0f};
    return map_rc(b200collAllGather(send, recv, sendcount, &ep, c, stream));
  }
  size_t n = 0;
  if (!map_dt_as_words(dt, sendcount, &t, &n)) return ncclInvalidArgument;
  b200collEpilogue ep{t, t, 1.0f};
  BitExactScope exact(c);
  return map_rc(b200collAllGather(send, recv, n, &ep, c, stream));
}
ncclResult_t ncclReduceScatter(const void* send, void* recv, size_t recvcount, ncclDataType_t dt, ncclRedOp_t op, ncclComm_t comm, cudaStream_t stream) {
  b200collDataType_t t;
  b200collRedOp_t rop; float scale;
  if (!comm || !map_dt_reduce(dt, &t) || !map_op(op, &rop, &scale)) return ncclInvalidArgument;
  b200collEpilogue ep{t, t, scale};
  return map_rc(b200collReduceScatter(send, recv, recvcount, &ep, rop, reinterpret_cast<ShimComm*>(comm)->comm, stream));
}

// Broadcast moves bits, so every NCCL dtype works: the payload is described to the library as f16/f32 words
// (scale 1, same type in and out = the bit-exact identity path). fp8 goes this way too, not through the typed fp8 kernels: NCCL's
// movement ops are bit-exact, and the Lamport path would rewrite a payload word that equals its empty-slot marker.
static bool map_dt_as_words(ncclDataType_t dt, size_t count, b200collDataType_t* t, size_t* n) {
  switch (dt) {
    case ncclInt8: case ncclUint8: case ncclFloat8e4m3: case ncclFloat8e5m2: if (count % 2) return false; *t = b200collFloat16; *n = count / 2; return true;
    case ncclFloat16: case ncclBfloat16: *t = b200collFloat16; *n = count; return true;
    case ncclInt32: case ncclUint32: case ncclFloat32: *t = b200collFloat32; *n = count; return true;
    case ncclInt64: case ncclUint64: case ncclFloat64: *t = b200collFloat32; *n = count * 2; return true;
    default: return false;
  }
}
ncclResult_t ncclBroadcast(const void* send, void* recv, size_t count, ncclDataType_t dt, int root, ncclComm_t comm, cudaStream_t stream) {
  b200collDataType_t t; size_t n = 0;
  if (!comm || !map_dt_as_words(dt, count, &t, &n)) return ncclInvalidArgument;
  b200collEpilogue ep{t, t, 1.0f};
  return map_rc(b200collBroadcast(send ? send : recv, recv, n, &ep, root, reinterpret_cast<ShimComm*>(comm)->comm, stream));
}
ncclResult_t ncclBcast(void* buf, size_t count, ncclDataType_t dt, int root, ncclComm_t comm, cudaStream_t stream) {   // legacy in-place form
  return ncclBroadcast(buf, buf, count, dt, root, comm, stream);
}
ncclResult_t ncclReduce(const void* send, void* recv, size_t count, ncclDataType_t dt, ncclRedOp_t op, int root, ncclComm_t comm, cudaStream_t stream) {
  b200collDataType_t t;
  b200collRedOp_t rop; float scale;
  if (!comm || !map_dt_reduce(dt, &t) || !map_op(op, &rop, &scale)) return ncclInvalidArgument;
  b200collEpilogue ep{t, t, scale};
  // NCCL lets non-root ranks pass recv == NULL; the library wants an aligned pointer it will not touch
  return map_rc(b200collReduce(send, recv ? recv : const_cast<void*>(send), count, &ep, rop, root, reinterpret_cast<ShimComm*>(comm)->comm, stream));
}

// ---- NCCL 2.28 additions that an nccl-tests built against that header references
ncclResult_t ncclAlltoAll(const void* send, void* recv, size_t count, ncclDataType_t dt, ncclComm_t comm, cudaStream_t stream) {
  if (!comm) return ncclInvalidArgument;
  b200collComm_t c = reinterpret_cast<ShimComm*>(comm)->comm;
  b200collDataType_t t;
  if (map_dt(dt, &t)) {
    b200collEpilogue ep{t, t, 1.0f};
    return map_rc(b200collAllToAll(send, recv, count, &ep, c, stream));
  }
  size_t n = 0;
  if (!map_dt_as_words(dt, count, &t, &n)) return ncclInvalidArgument;
  b200collEpilogue ep{t, t, 1.0f};
  BitExactScope exact(c);
  return map_rc(b200collAllToAll(send, recv, n, &ep, c, stream));
}
// Gather / scatter are one group of sends and receives around the root (the root's own block is a local copy inside the same group).
ncclResult_t ncclGather(const void* send, void* recv, size_t count, ncclDataType_t dt, int root, ncclComm_t comm, cudaStream_t stream) {
  const size_t esz = nccl_type_size(dt);
  if (!comm || !esz) return ncclInvalidArgument;
  ShimComm* s = reinterpret_cast<ShimComm*>(comm);
  if (root < 0 || root >= s->nranks) return ncclInvalidArgument;
  b200collResult_t rc = b200collGroupStart();
  if (rc == b200collSuccess) rc = b200collSend(send, count * esz, root, s->comm, stream);
  if (s->rank == root)
    for (int p = 0; p < s->nranks && rc == b200collSuccess; p++) rc = b200collRecv(static_cast<char*>(recv) + (size_t)p * count * esz, count * esz, p, s->comm, stream);
  const b200collResult_t rc_end = b200collGroupEnd();
  return map_rc(rc != b200collSuccess ? rc : rc_end);
}
ncclResult_t ncclScatter(const void* send, void* recv, size_t count, ncclDataType_t dt, int root, ncclComm_t comm, cudaStream_t stream) {
  const size_t esz = nccl_type_size(dt);
  if (!comm || !esz) return ncclInvalidArgument;
  ShimComm* s = reinterpret_cast<ShimComm*>(comm);
  if (root < 0 || root >= s->nranks) return ncclInvalidArgument;
  b200collResult_t rc = b200collGroupStart();
  if (s->rank == root)
    for (int p = 0; p < s->nranks && rc == b200collSuccess; p++) rc = b200collSend(static_cast<const char*>(send) + (size_t)p * count * esz, count * esz, p, s->comm, stream);
  if (rc == b200collSuccess) rc = b200collRecv(recv, count * esz, root, s->comm, stream);
  const b200collResult_t rc_end = b200collGroupEnd();
  return map_rc(rc != b200collSuccess ? rc : rc_end);
}
// Symmetric windows: memory from ncclMemAlloc is symmetric by construction, anything else is staged by the library — nothing to register.
ncclResult_t ncclCommWindowRegister(ncclComm_t comm, void* buff, size_t, ncclWindow_t* win, int) {
  if (!comm || !win) return ncclInvalidArgument;
  *win = reinterpret_cast<ncclWindow_t>(buff);
  return ncclSuccess;
}
ncclResult_t ncclCommWindowDeregister(ncclComm_t, ncclWindow_t) { return ncclSuccess; }
ncclResult_t ncclCommInitRankScalable(ncclComm_t* comm, int nranks, int rank, int nid, ncclUniqueId* ids, ncclConfig_t*) {      // several ids only speed up NCCL's own bootstrap
  if (!ids || nid < 1) return ncclInvalidArgument;
  return ncclCommInitRank(comm, nranks, ids[0], rank);
}
// Shrinking around ranks that no longer answer needs a rendezvous that does not involve them; this transport's bootstrap is a star through
// rank 0 of the parent, so it cannot promise that. Create the smaller communicator with ncclCommInitRank (or ncclCommSplit while all are alive).
ncclResult_t ncclCommShrink(ncclComm_t, int*, int, ncclComm_t* newcomm, ncclConfig_t*, int) { if (newcomm) *newcomm = nullptr; return ncclInvalidUsage; }
ncclResult_t ncclCommRevoke(ncclComm_t comm, int) { return ncclCommAbort(comm); }
ncclResult_t ncclGroupSimulateEnd(ncclSimInfo_t*) { return ncclInvalidUsage; }                                                   // no cost model to query

ncclResult_t ncclGroupStart(void) { g_group_depth++; return ncclSuccess; }
ncclResult_t ncclGroupEnd(void) {
  if (g_group_depth <= 0) return ncclInvalidUsage;
  if (--g_group_depth > 0) return ncclSuccess;
  return flush_group();
}
ncclResult_t ncclSend(const void* buf, size_t count, ncclDataType_t dt, int peer, ncclComm_t comm, cudaStream_t stream) {
  if (!comm || nccl_type_size(dt) == 0) return ncclInvalidArgument;
  g_group_ops.push_back(P2pOp{true, buf, nullptr, count, dt, peer, reinterpret_cast<ShimComm*>(comm), stream});
  return g_group_depth > 0 ? ncclSuccess : flush_group();      // outside a group: a group of one (blocks the stream until the peer's recv)
}
ncclResult_t ncclRecv(void* buf, size_t count, ncclDataType_t dt, int peer, ncclComm_t comm, cudaStream_t stream) {
  if (!comm || nccl_type_size(dt) == 0) return ncclInvalidArgument;
  g_group_ops.push_back(P2pOp{false, nullptr, buf, count, dt, peer, reinterpret_cast<ShimComm*>(comm), stream});
  return g_group_depth > 0 ? ncclSuccess : flush_group();
}

}  // extern "C"
