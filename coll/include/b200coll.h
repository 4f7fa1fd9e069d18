/*
 * libb200coll — intra-node collective library for 8×B200 (sm_100a) over NVLink 5 / NVSwitch.
 *
 * Role parity: this is the payload the transport-installer DaemonSet drops into
 * /home/kubernetes/bin/nvidia/lib64 and the device plugin's Allocate mounts into the pod —
 * the slot the reference fills with pre-built NCCL net plugins
 * (reference: fast-socket-installer/fast-socket-installer.yaml:41-45,
 *  gpudirect-rdma/nccl-rdma-installer.yaml:70-77, gpudirect-tcpxo/nccl-tcpxo-installer.yaml:83-91).
 * On a single NVSwitch box a *net* plugin is never on the data path, so the product here is the
 * collective itself: one-shot (Lamport/LL), two-shot P2P and NVLS-multimem kernels with the
 * cast/scale epilogue fused, chosen per (op, bytes, nranks) by a measured table (the
 * libnccl-tuner.so analogue, reference: gpudirect-tcpxo/README.md:80-81).
 *
 * C ABI, no C++ types cross the boundary. All collectives are asynchronous on `stream`
 * and never block the host on a peer.
 */
#ifndef B200COLL_H_
#define B200COLL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200COLL_VERSION_MAJOR 0
#define B200COLL_VERSION_MINOR 1
#define B200COLL_MAX_RANKS 8
#define B200COLL_UNIQUE_ID_BYTES 128

typedef struct b200collComm* b200collComm_t;
typedef struct { char internal[B200COLL_UNIQUE_ID_BYTES]; } b200collUniqueId;
typedef void* b200collStream_t; /* cudaStream_t */

typedef enum {
  b200collSuccess = 0,
  b200collUnhandledCudaError = 1,
  b200collSystemError = 2,
  b200collInternalError = 3,
  b200collInvalidArgument = 4,
  b200collInvalidUsage = 5,
  b200collRemoteError = 6,   /* a peer timed out or aborted (watchdog) */
  b200collInProgress = 7,
  b200collOutOfMemory = 8,
  b200collNoDriver = 9       /* libcuda / GPU not present (CPU-only box) */
} b200collResult_t;

typedef enum {
  b200collFloat32 = 0,
  b200collFloat16 = 1,
  b200collBfloat16 = 2,
  b200collFloat8e4m3 = 3,   /* fp8 e4m3 (OCP "fn": max 448): input and output type */
  /* the types below take the generic reduction path (src/generic.cu): same type in and out, no scale, any operator but avg */
  b200collInt8 = 4,
  b200collUint8 = 5,
  b200collInt32 = 6,
  b200collUint32 = 7,
  b200collInt64 = 8,
  b200collUint64 = 9,
  b200collFloat64 = 10,
  /* fp8 e5m2 (max 57344): input and output type, like e4m3 */
  b200collFloat8e5m2 = 11,
  b200collNumTypes = 12
} b200collDataType_t;

/* sum and avg of fp32 / fp16 / bf16 / fp8 e4m3 / fp8 e5m2 run on the fused fast paths (Lamport, two-shot, NVLS) and accumulate in fp32;
 * fp8 results are rounded to nearest and saturate to the largest finite value. prod, min, max — and every operator on the integer types
 * and fp64 — run on one barrier-based P2P kernel that accumulates in the element type (fp16 / bf16 / fp8 in fp32).
 * Supported (in_dtype, out_dtype) pairs: equal types; fp32 <-> bf16 / fp16 widen or narrow; fp32 / bf16 / fp16 -> e4m3 or e5m2
 * (quantise); e4m3 or e5m2 -> bf16 / fp16 / fp32 (dequantise, with the fused scale). There is no e4m3 <-> e5m2 pair. */
typedef enum { b200collSum = 0, b200collAvg = 1, b200collProd = 2, b200collMin = 3, b200collMax = 4 } b200collRedOp_t;

typedef enum {
  b200collOpAllReduce = 0,
  b200collOpAllGather = 1,
  b200collOpReduceScatter = 2,
  b200collOpAllToAll = 3,
  b200collOpBroadcast = 4,
  b200collOpReduce = 5,
  b200collNumOps = 6
} b200collOp_t;

/* Algorithm ids (tuner output; B200COLL_ALGO overrides). */
typedef enum {
  b200collAlgoAuto = 0,
  b200collAlgoLL = 1,        /* Lamport flag-in-payload push, zero barriers  (tiny)  */
  b200collAlgoOneShot = 2,   /* barrier + pull all peers + reduce in regs    (small) */
  b200collAlgoTwoShot = 3,   /* P2P pull-reduce own slice + push to peers    (mid/large, no multicast needed) */
  b200collAlgoNvls = 4,      /* multimem.ld_reduce / multimem.st through the switch (large) */
  b200collAlgoCopy = 5,      /* nranks == 1: fused scale/cast copy */
  b200collAlgoLL2 = 6,       /* two-shot Lamport all-reduce: zero barriers, 2S bytes received instead of N*S (mid) */
  b200collNumAlgos = 7
} b200collAlgo_t;

/* Fused epilogue: out = cast<out_dtype>(reduce(in) * scale). scale==1.0f and equal dtypes is the plain collective. */
typedef struct {
  b200collDataType_t in_dtype;
  b200collDataType_t out_dtype;
  float scale;
} b200collEpilogue;

typedef struct {
  size_t arena_bytes;        /* symmetric user heap per rank (default: env B200COLL_ARENA_MB or 2560 MiB) */
  int enable_nvls;           /* -1 auto (probe), 0 off, 1 require */
  int max_ctas;              /* 0 = auto */
  int timeout_ms;            /* device-side watchdog for every cross-GPU spin and the rendezvous: default 600000 (env B200COLL_TIMEOUT_MS), 0 = none, < 0 = default */
  int debug;                 /* 0 quiet, 1 info, 2 trace (env B200COLL_DEBUG) */
} b200collConfig;

typedef struct {
  int rank, nranks, device;
  int nvls;                  /* multicast window mapped */
  int p2p_ok;                /* full P2P matrix */
  int same_device_loopback;  /* virtual ranks share one GPU (test mode) */
  size_t arena_bytes;
  size_t arena_used;
  int sm_count;
  int driver_version;
} b200collCommInfo;

typedef struct {
  uint64_t calls[b200collNumOps];
  uint64_t bytes[b200collNumOps];
  uint64_t algo_calls[b200collNumAlgos];
  uint64_t kernel_launches;
  uint64_t staged_calls;     /* calls that went through the staging copy (unregistered buffers) */
  uint64_t p2p_sends, p2p_recvs, p2p_bytes;   /* point-to-point operations and the bytes they moved (sent + received) */
  uint64_t host_calls, host_bytes;            /* b200collAllReduceHost calls and the input bytes they carried */
  uint64_t host_zero_copy, host_pipelined;    /* ... of which: one-kernel zero-copy calls / chunked three-leg pipelines */
  uint64_t bulk_launches;                     /* kernels that moved their payload with the copy engine (cp.async.bulk ring) */
  uint64_t generic_launches;                  /* min / max / prod / integer / fp64 reduction kernels */
} b200collStats;

/* Device-written watchdog record (host-pinned). code != 0 means the comm is poisoned. */
typedef struct {
  uint32_t code;             /* 0 ok, 1 barrier timeout, 2 LL data timeout, 3 send/recv peer never showed up, 4 send/recv sizes differ, 5 bulk copy never completed (bulk variant) */
  uint32_t rank, peer, block;
  uint32_t expected, observed;
  uint32_t op, reserved;
} b200collFault;

const char* b200collGetErrorString(b200collResult_t r);
const char* b200collGetLastError(void);
int b200collGetVersion(void);

void b200collConfigDefault(b200collConfig* cfg);

/* --- multi-process: one rank per process, rendezvous over an abstract Unix socket (SCM_RIGHTS fd passing). */
b200collResult_t b200collGetUniqueId(b200collUniqueId* id);
/* Deterministic id from a string (e.g. "$MASTER_ADDR:$MASTER_PORT/0") so torchrun ranks need no side channel. */
b200collResult_t b200collUniqueIdFromString(const char* s, b200collUniqueId* id);
b200collResult_t b200collCommInitRank(b200collComm_t* comm, int nranks, const b200collUniqueId* id, int rank,
                                      const b200collConfig* cfg);
/* --- single process: n ranks, one per entry of devs (entries may repeat: virtual ranks on one GPU for tests). */
b200collResult_t b200collCommInitAll(b200collComm_t* comms, int n, const int* devs, const b200collConfig* cfg);
/* ncclCommSplit: a collective call on a multi-process communicator. Ranks that pass the same color >= 0 form a new communicator
 * (its own arena: cfg, or the parent's settings when NULL), ordered by (key, rank in the parent); color < 0 takes part and gets none. */
b200collResult_t b200collCommSplit(b200collComm_t comm, int color, int key, b200collComm_t* newcomm, const b200collConfig* cfg);
/* Test hook: the (rank, size) a split would give `rank`, from everybody's colors and keys. */
b200collResult_t b200collDebugSplitPlan(int nranks, int rank, const int* colors, const int* keys, int* new_rank, int* new_size);
b200collResult_t b200collCommDestroy(b200collComm_t comm);
b200collResult_t b200collCommInfoGet(b200collComm_t comm, b200collCommInfo* info);
b200collResult_t b200collCommStatsGet(b200collComm_t comm, b200collStats* stats);
b200collResult_t b200collCommGetAsyncError(b200collComm_t comm, b200collFault* fault);
/* Host-level barrier over the bootstrap channel (multi-process comms only; no-op for InitAll comms). */
b200collResult_t b200collHostBarrier(b200collComm_t comm);

/* --- symmetric memory: collective calls, same order and size on every rank (ncclMemAlloc analogue). */
b200collResult_t b200collMemAlloc(b200collComm_t comm, void** ptr, size_t bytes);
b200collResult_t b200collMemFree(b200collComm_t comm, void* ptr);
/* PyTorch glue: `torch.cuda.memory.CUDAPluggableAllocator(lib, "b200collTorchAlloc", "b200collTorchFree")` + `torch.cuda.MemPool` put
 * tensors into the arena of the communicator named by SetAllocatorComm (same allocation sequence on every rank, as for MemAlloc). */
b200collResult_t b200collSetAllocatorComm(b200collComm_t comm);
void* b200collTorchAlloc(size_t size, int device, void* stream);
void b200collTorchFree(void* ptr, size_t size, int device, void* stream);
/* 1 if [ptr, ptr+bytes) lies in this rank's symmetric arena. */
int b200collIsSymmetric(b200collComm_t comm, const void* ptr, size_t bytes);

/* --- collectives. count is in elements of ep->in_dtype.
 * Buffers inside the symmetric arena take the zero-copy paths; any other device pointer is staged. */
b200collResult_t b200collAllReduce(const void* send, void* recv, size_t count, const b200collEpilogue* ep,
                                   b200collRedOp_t op, b200collComm_t comm, b200collStream_t stream);
/* recv holds nranks*sendcount elements; rank r's contribution lands at r*sendcount. */
b200collResult_t b200collAllGather(const void* send, void* recv, size_t sendcount, const b200collEpilogue* ep,
                                   b200collComm_t comm, b200collStream_t stream);
/* send holds nranks*recvcount elements; rank r receives the reduction of slice r. */
b200collResult_t b200collReduceScatter(const void* send, void* recv, size_t recvcount, const b200collEpilogue* ep,
                                       b200collRedOp_t op, b200collComm_t comm, b200collStream_t stream);
/* send/recv hold nranks*count elements; block p of send goes to block `rank` of peer p's recv. */
b200collResult_t b200collAllToAll(const void* send, void* recv, size_t count, const b200collEpilogue* ep,
                                  b200collComm_t comm, b200collStream_t stream);
/* Expert-dispatch shape: rows of `row_elems` elements; send_rows[p] rows go to peer p starting at row
 * send_row_off[p] of send; they land at row recv_row_off[src] of the destination (all four arrays are
 * host arrays of length nranks; recv_row_off[src] = where rank `src`'s rows start in MY recv). */
b200collResult_t b200collAllToAllv(const void* send, void* recv, size_t row_elems, const int64_t* send_rows,
                                   const int64_t* send_row_off, const int64_t* recv_row_off_at_peer,
                                   const b200collEpilogue* ep, b200collComm_t comm, b200collStream_t stream);
/* Rooted collectives (ncclBroadcast / ncclReduce). Broadcast: root's send -> every rank's recv (cast/scale fused);
 * send is read on the root only. Reduce: root's recv = scale * sum over ranks of send; recv is written on the root only.
 * Ranks that do not use a buffer may pass any 16-byte aligned device pointer for it. */
b200collResult_t b200collBroadcast(const void* send, void* recv, size_t count, const b200collEpilogue* ep, int root,
                                   b200collComm_t comm, b200collStream_t stream);
b200collResult_t b200collReduce(const void* send, void* recv, size_t count, const b200collEpilogue* ep,
                                b200collRedOp_t op, int root, b200collComm_t comm, b200collStream_t stream);
b200collResult_t b200collBarrier(b200collComm_t comm, b200collStream_t stream);

/* --- host path (src/hostpath.cu). CommInitRank binds the calling thread to the CPUs of the GPU's NUMA node (B200COLL_AFFINITY=0:
 * leave it alone, 2: restore the previous mask after init). HostAlloc returns pinned, device-mapped host memory on that node.
 * AllReduceHost is the end-to-end step "pinned host -> GPU -> all-reduce -> pinned host" as one asynchronous call on `stream`:
 * tiny messages run as ONE kernel that reads and writes host memory over PCIe, large ones are chunked so that the host-to-device
 * copy of chunk i+1, the all-reduce of chunk i and the copy-back of chunk i-1 overlap. Same call on every rank; staging comes from
 * the symmetric heap on first use (a collective contract, like MemAlloc). */
b200collResult_t b200collHostAlloc(b200collComm_t comm, void** ptr, size_t bytes);
b200collResult_t b200collHostFree(b200collComm_t comm, void* ptr);
b200collResult_t b200collAllReduceHost(const void* host_send, void* host_recv, size_t count, const b200collEpilogue* ep,
                                       b200collRedOp_t op, b200collComm_t comm, b200collStream_t stream);
/* NUMA node of this rank's GPU (-1 unknown) and its local CPU list as sysfs prints it. */
b200collResult_t b200collCommNumaGet(b200collComm_t comm, int* numa_node, char* cpulist, size_t len);
/* Test hook (no GPU needed): what CommInitRank does with the GPU's sysfs directory (files numa_node, local_cpulist): returns the NUMA node
 * read (-1 if absent); with mode != 0 the calling thread's affinity is narrowed to the listed CPUs it is allowed to use (*changed = 1 if so). */
int b200collDebugApplyLocality(const char* sysfs_dir, int mode, int* changed);
/* Test hook: parse a sysfs cpulist ("0-31,64-95") into at most `max` CPU numbers; returns how many. */
int b200collDebugParseCpuList(const char* s, int* cpus, int max);

/* --- point to point (ncclSend / ncclRecv / ncclGroupStart / ncclGroupEnd). `bytes` of opaque data; buffers 16-byte aligned.
 * A send pairs with the peer's recv of the same size, in call order per pair. Everything between GroupStart and GroupEnd
 * (a ring step, a pipeline hand-over, any mix of peers) becomes ONE kernel per communicator, launched at GroupEnd on the
 * stream of the group's first operation; outside a group each call is a group of its own and blocks the stream until the
 * peer arrives (so "send then recv" on both sides of a pair deadlocks exactly as it does with NCCL: group them).
 * The receiver's buffer is written directly over NVLink when it lies in the symmetric arena; otherwise through staging. */
b200collResult_t b200collGroupStart(void);
b200collResult_t b200collGroupEnd(void);
b200collResult_t b200collSend(const void* buf, size_t bytes, int peer, b200collComm_t comm, b200collStream_t stream);
b200collResult_t b200collRecv(void* buf, size_t bytes, int peer, b200collComm_t comm, b200collStream_t stream);
/* Test hook (no GPU needed): plans one group of point-to-point operations for `rank` on a stand-in communicator and writes the
 * launches it would make as text: CTA ranges per operation, direct or staged receive, window layout, follow-up kernels. */
b200collResult_t b200collDebugPlanP2p(int rank, int nranks, int loopback, size_t window, int nops, const int* is_send, const int* peer,
                                      const size_t* bytes, const int* in_arena, char* out, size_t outlen);

/* --- tuner (libnccl-tuner.so analogue). */
b200collAlgo_t b200collTunerPick(b200collOp_t op, size_t bytes, int nranks, int nvls_available);
/* Force an algorithm for subsequent calls on this comm (b200collAlgoAuto restores the table). */
b200collResult_t b200collCommSetAlgo(b200collComm_t comm, b200collAlgo_t algo);
b200collAlgo_t b200collCommGetAlgo(b200collComm_t comm);   /* what SetAlgo (or B200COLL_ALGO) last forced; Auto = the tuner decides */
b200collResult_t b200collCommSetMaxCtas(b200collComm_t comm, int max_ctas);
/* Receives into buffers outside the arena go through two staging windows per operation; this caps the window size (a multiple of
 * 512 bytes; 0 = an equal share of the 64 MiB staging area). A private choice of the receiver: the sender follows what is posted. */
b200collResult_t b200collCommSetP2pWindow(b200collComm_t comm, size_t bytes);
/* Launch shape per kernel family: kind 0 = NVLS all-reduce/all-gather, 1 = P2P pull/push kernels, 2 = LL, 3 = NVLS reduce-scatter, 4 = NVLS broadcast / reduce (root only).
 * max_ctas <= 0 keeps the current cap; threads == 0 lets the library pick {128,256,512} by work size.
 * Defaults come from the 8xB200 sweep in profiles/ (NVLS wants few CTAs: 32 x 256 threads). */
b200collResult_t b200collCommSetLaunchShape(b200collComm_t comm, int kind, int max_ctas, int threads);
const char* b200collAlgoName(b200collAlgo_t a);
size_t b200collTypeSize(b200collDataType_t t);

/* --- start-up self check (guest-config-checker analogue, reference: gpudirect-tcpxo/README.md:84,239).
 * Writes a human-readable report into buf; returns b200collSuccess iff the box can run the fast paths. */
b200collResult_t b200collSelfCheck(char* buf, size_t buflen);

#ifdef __cplusplus
}
#endif
#endif /* B200COLL_H_ */
