// Size-based algorithm table — the libnccl-tuner.so + a3plus_tuner_config.textproto analogue
// (reference: gpudirect-tcpxo/README.md:80-81,831). The built-in rows are the crossovers measured on
// 8xB200 / NVSwitch (bench/tune.py regenerates them; see coll/tuner/b200_nvswitch.tbl). A file named by
// B200COLL_TUNER_FILE overrides the built-in rows; format, one row per line:
//     <op> <nranks_min> <nranks_max> <nvls 0|1|*> <max_bytes> <algo>
// First matching row wins; "bytes" is the per-rank message size (AR: whole buffer; AG: send bytes;
// RS: recv bytes; A2A: bytes per peer).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <strings.h>

#include <mutex>
#include <string>
#include <vector>

#include "../include/b200coll.h"

namespace b200coll {

struct Row { int op, nmin, nmax, nvls; unsigned long long max_bytes; int algo; };

static const unsigned long long INF = ~0ull;

// clang-format off
static const Row kBuiltin[] = {
  // ---- all-reduce (crossovers measured at 2, 4 and 8 x B200: profiles/allreduce_sweep.md, gpurun_out/s{2,4}_ar_*.txt)
  {b200collOpAllReduce,     2, 2, -1,  512ull << 10, b200collAlgoLL},      // 2 GPUs: LL 10.3 us vs two-shot LL 11.8 us at 512 KiB
  {b200collOpAllReduce,     2, 2, -1,  1ull << 20,   b200collAlgoLL2},     //          two-shot LL 13.0 us vs barrier two-shot 16.1 us at 1 MiB
  {b200collOpAllReduce,     2, 2, -1,  INF,          b200collAlgoTwoShot}, //          NVLS would bounce my own half through the switch
  {b200collOpAllReduce,     3, 4, -1,  512ull << 10, b200collAlgoLL},      // 4 GPUs: LL 12.3 us at 512 KiB
  {b200collOpAllReduce,     3, 4, -1,  2ull << 20,   b200collAlgoLL2},     //          two-shot LL 14.9 / 17.3 us vs NVLS 18.6 / 19.6 us at 1 / 2 MiB
  {b200collOpAllReduce,     5, 8, -1,  256ull << 10, b200collAlgoLL},      // 8 GPUs: LL 13.1 us vs NVLS 15.8 us at 256 KiB; NVLS 16.0 us vs LL 17.2 us at 512 KiB
  {b200collOpAllReduce,     5, 8,  0,  2ull << 20,   b200collAlgoLL2},     //          without multicast: two-shot LL before the barrier two-shot
  {b200collOpAllReduce,     3, 8,  1,  INF,          b200collAlgoNvls},
  {b200collOpAllReduce,     3, 8,  0,  INF,          b200collAlgoTwoShot},
  // ---- all-gather (bytes = per-rank contribution)
  {b200collOpAllGather,     2, 8, -1,  256ull << 10, b200collAlgoLL},     // 8xB200: 2 MiB total in 13 us (push+barrier: 17 us at 1 MiB)
  {b200collOpAllGather,     2, 8, -1,  INF,          b200collAlgoTwoShot},
  // ---- reduce-scatter (bytes = per-rank result)
  {b200collOpReduceScatter, 2, 8, -1,  256ull << 10, b200collAlgoLL},
  {b200collOpReduceScatter, 3, 8,  1,  INF,          b200collAlgoNvls},
  {b200collOpReduceScatter, 2, 8, -1,  INF,          b200collAlgoTwoShot},
  // ---- all-to-all (bytes = per-peer block)
  {b200collOpAllToAll,      2, 8, -1,  256ull << 10, b200collAlgoLL},
  {b200collOpAllToAll,      2, 8, -1,  INF,          b200collAlgoTwoShot},
  // ---- rooted ops (bytes = message): the switch does the fan-out / the reduction when it can
  {b200collOpBroadcast,     3, 8,  1,  INF,          b200collAlgoNvls},
  {b200collOpBroadcast,     2, 8, -1,  INF,          b200collAlgoTwoShot},
  {b200collOpReduce,        3, 8,  1,  INF,          b200collAlgoNvls},
  {b200collOpReduce,        2, 8, -1,  INF,          b200collAlgoTwoShot},
};
// clang-format on

static std::vector<Row> g_rows;
static std::once_flag g_once;

static int parse_op(const char* s) {
  if (!strcasecmp(s, "allreduce") || !strcasecmp(s, "all_reduce")) return b200collOpAllReduce;
  if (!strcasecmp(s, "allgather") || !strcasecmp(s, "all_gather")) return b200collOpAllGather;
  if (!strcasecmp(s, "reducescatter") || !strcasecmp(s, "reduce_scatter")) return b200collOpReduceScatter;
  if (!strcasecmp(s, "alltoall") || !strcasecmp(s, "all_to_all")) return b200collOpAllToAll;
  if (!strcasecmp(s, "broadcast") || !strcasecmp(s, "bcast")) return b200collOpBroadcast;
  if (!strcasecmp(s, "reduce")) return b200collOpReduce;
  return -1;
}

static void load_rows() {
  const char* path = getenv("B200COLL_TUNER_FILE");
  if (path && *path && strcasecmp(path, "UNUSED")) {
    FILE* f = fopen(path, "r");
    if (f) {
      char line[256];
      while (fgets(line, sizeof(line), f)) {
        char op[32], nv[8], algo[32], mb[32];
        int nmin, nmax;
        if (line[0] == '#' || sscanf(line, "%31s %d %d %7s %31s %31s", op, &nmin, &nmax, nv, mb, algo) != 6) continue;
        Row r;
        r.op = parse_op(op); r.nmin = nmin; r.nmax = nmax;
        r.nvls = nv[0] == '*' ? -1 : atoi(nv);
        r.max_bytes = (!strcasecmp(mb, "inf")) ? INF : strtoull(mb, nullptr, 0);
        r.algo = -1;
        for (int a = 0; a < b200collNumAlgos; a++) if (!strcasecmp(algo, b200collAlgoName((b200collAlgo_t)a))) r.algo = a;
        if (r.op >= 0 && r.algo >= 0) g_rows.push_back(r);
      }
      fclose(f);
    } else {
      fprintf(stderr, "[b200coll] warning: cannot open B200COLL_TUNER_FILE=%s; using built-in table\n", path);
    }
  }
  for (const Row& r : kBuiltin) g_rows.push_back(r);
}

}  // namespace b200coll

extern "C" {

const char* b200collAlgoName(b200collAlgo_t a) {
  switch (a) {
    case b200collAlgoAuto: return "auto";
    case b200collAlgoLL: return "ll";
    case b200collAlgoOneShot: return "oneshot";
    case b200collAlgoTwoShot: return "twoshot";
    case b200collAlgoNvls: return "nvls";
    case b200collAlgoCopy: return "copy";
    case b200collAlgoLL2: return "ll2";
    default: return "?";
  }
}

size_t b200collTypeSize(b200collDataType_t t) {
  switch (t) {
    case b200collFloat32: return 4;
    case b200collFloat16: return 2;
    case b200collBfloat16: return 2;
    case b200collFloat8e4m3: case b200collFloat8e5m2: return 1;
    case b200collInt8: case b200collUint8: return 1;
    case b200collInt32: case b200collUint32: return 4;
    case b200collInt64: case b200collUint64: case b200collFloat64: return 8;
    default: return 0;
  }
}

b200collAlgo_t b200collTunerPick(b200collOp_t op, size_t bytes, int nranks, int nvls) {
  if (nranks <= 1) return b200collAlgoCopy;
  std::call_once(b200coll::g_once, b200coll::load_rows);
  for (const b200coll::Row& r : b200coll::g_rows) {
    if (r.op != (int)op || nranks < r.nmin || nranks > r.nmax) continue;
    if (r.nvls >= 0 && r.nvls != (nvls ? 1 : 0)) continue;
    if ((unsigned long long)bytes > r.max_bytes) continue;
    return (b200collAlgo_t)r.algo;
  }
  return b200collAlgoTwoShot;
}

}  // extern "C"
