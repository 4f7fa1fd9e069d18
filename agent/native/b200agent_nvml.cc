// libb200agent_nvml.so — the node agent's one NVML binding (C ABI, consumed through ctypes).
//
// Covers the reference's native pieces with a single dlopen'd libnvidia-ml.so.1:
//   * the cgo helper nvmlDeviceGetAverageUsage (reference: pkg/gpu/nvidia/metrics/util.go:37-87) — integer
//     mean of NVML_GPU_UTILIZATION_SAMPLES newer than a timestamp; guarded against sampleCount == 0,
//     which the reference divides by (util.go:82);
//   * the Xid event loop nvmlEventSetCreate / RegisterEvents / EventSetWait / Free that the reference
//     reaches through a second binding (vendor/github.com/NVIDIA/gpu-monitoring-tools/bindings/go/nvml/bindings.go:108-186);
//   * device enumeration used by discovery (minor number, UUID, name, PCI bus id, memory, MIG mode).
// NVML is resolved at run time so the library loads (and its error paths are testable) on a GPU-less box;
// B200AGENT_NVML_LIB overrides the library path (tests point it at a fake NVML).
#include <dlfcn.h>
#include "nvml_abi.h"
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <mutex>
#include <vector>

extern "C" {

typedef struct {
  int index;
  int minor_number;
  char uuid[96];
  char name[96];
  char bus_id[32];
  unsigned long long mem_total;
  unsigned long long mem_used;
  int mig_mode_current;   // -1 unknown/unsupported
  int mig_mode_pending;
} b200nvml_device_info;

typedef struct {
  char uuid[96];           // empty when the event carried no device
  unsigned long long event_type;
  unsigned long long event_data;   // the Xid for nvmlEventTypeXidCriticalError
  unsigned int gpu_instance_id;    // 0xFFFFFFFF when not MIG
  unsigned int compute_instance_id;
} b200nvml_event;

enum { B200NVML_OK = 0, B200NVML_NO_LIB = -1, B200NVML_TIMEOUT = -2, B200NVML_NOT_SUPPORTED = -3, B200NVML_BAD_ARG = -4, B200NVML_NO_SAMPLES = -5 };

}  // extern "C"

namespace {

#define NVML_FUNCS(X)                                                                                        \
  X(nvmlInit_v2) X(nvmlShutdown) X(nvmlErrorString) X(nvmlDeviceGetCount_v2) X(nvmlDeviceGetHandleByIndex_v2) \
  X(nvmlDeviceGetHandleByUUID) X(nvmlDeviceGetMinorNumber) X(nvmlDeviceGetUUID) X(nvmlDeviceGetName)          \
  X(nvmlDeviceGetPciInfo_v3) X(nvmlDeviceGetMemoryInfo) X(nvmlDeviceGetMigMode) X(nvmlDeviceGetSamples)       \
  X(nvmlSystemGetDriverVersion) X(nvmlEventSetCreate) X(nvmlDeviceRegisterEvents) X(nvmlEventSetWait_v2)      \
  X(nvmlEventSetFree) X(nvmlDeviceGetSupportedEventTypes)

struct Api {
#define X(n) decltype(&::n) n = nullptr;
  NVML_FUNCS(X)
#undef X
  decltype(&::nvmlDeviceGetUtilizationRates) nvmlDeviceGetUtilizationRates = nullptr;   // optional: the sampler's fallback
  void* handle = nullptr;
  bool ok = false;
  char why[256] = {0};
};

Api g_api;
std::once_flag g_once;
char g_last_error[512];

void set_err(const char* what, nvmlReturn_t r) {
  const char* s = g_api.nvmlErrorString ? g_api.nvmlErrorString(r) : "?";
  snprintf(g_last_error, sizeof(g_last_error), "%s: %s (%d)", what, s, (int)r);
}

void load_api() {
  const char* path = getenv("B200AGENT_NVML_LIB");
  const char* cands[] = {path, "libnvidia-ml.so.1", "/usr/local/nvidia/lib64/libnvidia-ml.so.1", "/home/kubernetes/bin/nvidia/lib64/libnvidia-ml.so.1"};
  for (const char* c : cands) {
    if (!c || !*c) continue;
    g_api.handle = dlopen(c, RTLD_LAZY | RTLD_GLOBAL);
    if (g_api.handle) break;
  }
  if (!g_api.handle) { snprintf(g_api.why, sizeof(g_api.why), "cannot dlopen libnvidia-ml.so.1: %s", dlerror()); return; }
  bool all = true;
#define X(n)                                                              \
  g_api.n = reinterpret_cast<decltype(g_api.n)>(dlsym(g_api.handle, #n)); \
  if (!g_api.n) { all = false; snprintf(g_api.why, sizeof(g_api.why), "libnvidia-ml lacks %s", #n); }
  NVML_FUNCS(X)
#undef X
  g_api.nvmlDeviceGetUtilizationRates = reinterpret_cast<decltype(g_api.nvmlDeviceGetUtilizationRates)>(dlsym(g_api.handle, "nvmlDeviceGetUtilizationRates"));
  g_api.ok = all;
}

int need_api() {
  std::call_once(g_once, load_api);
  if (!g_api.ok) { snprintf(g_last_error, sizeof(g_last_error), "%s", g_api.why); return B200NVML_NO_LIB; }
  return B200NVML_OK;
}

struct EventSet { nvmlEventSet_t set; };

// Some drivers refuse the utilisation sample buffer with NOT_SUPPORTED (580.178 on a B200 sizes it, then will not fill it). The
// driver's utilisation rate is then the one sample there is: the share of its last sample period (1/6 s to 1 s) in which a kernel
// ran, read now. It is newer than any cut-off in the past and there is none newer than a cut-off in the future.
int utilization_rate(nvmlDevice_t d, unsigned long long since_us, unsigned int* util, nvmlReturn_t refused, const char* what) {
  if (!g_api.nvmlDeviceGetUtilizationRates) { set_err(what, refused); return (int)refused; }
  timespec now;
  clock_gettime(CLOCK_REALTIME, &now);
  if (since_us > (unsigned long long)now.tv_sec * 1000000ull + (unsigned long long)now.tv_nsec / 1000) {
    snprintf(g_last_error, sizeof(g_last_error), "no utilisation samples newer than the cut-off");
    return B200NVML_NO_SAMPLES;
  }
  nvmlUtilization_t u;
  nvmlReturn_t r = g_api.nvmlDeviceGetUtilizationRates(d, &u);
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceGetUtilizationRates", r); return (int)r; }
  *util = u.gpu;
  return B200NVML_OK;
}

}  // namespace

extern "C" {

const char* b200nvml_last_error(void) { return g_last_error; }

int b200nvml_init(void) {
  int rc = need_api();
  if (rc) return rc;
  nvmlReturn_t r = g_api.nvmlInit_v2();
  if (r != NVML_SUCCESS) { set_err("nvmlInit", r); return (int)r; }
  return B200NVML_OK;
}

int b200nvml_shutdown(void) {
  if (need_api()) return B200NVML_NO_LIB;
  return (int)g_api.nvmlShutdown();
}

int b200nvml_driver_version(char* buf, unsigned int len) {
  int rc = need_api();
  if (rc) return rc;
  nvmlReturn_t r = g_api.nvmlSystemGetDriverVersion(buf, len);
  if (r != NVML_SUCCESS) { set_err("nvmlSystemGetDriverVersion", r); return (int)r; }
  return B200NVML_OK;
}

int b200nvml_device_count(int* count) {
  int rc = need_api();
  if (rc) return rc;
  unsigned int n = 0;
  nvmlReturn_t r = g_api.nvmlDeviceGetCount_v2(&n);
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceGetCount", r); return (int)r; }
  *count = (int)n;
  return B200NVML_OK;
}

int b200nvml_device_info_get(int index, b200nvml_device_info* out) {
  int rc = need_api();
  if (rc) return rc;
  if (!out) return B200NVML_BAD_ARG;
  memset(out, 0, sizeof(*out));
  out->index = index; out->mig_mode_current = out->mig_mode_pending = -1;
  nvmlDevice_t d;
  nvmlReturn_t r = g_api.nvmlDeviceGetHandleByIndex_v2((unsigned)index, &d);
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceGetHandleByIndex", r); return (int)r; }
  unsigned int minor = 0;
  r = g_api.nvmlDeviceGetMinorNumber(d, &minor);
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceGetMinorNumber", r); return (int)r; }
  out->minor_number = (int)minor;
  if ((r = g_api.nvmlDeviceGetUUID(d, out->uuid, sizeof(out->uuid))) != NVML_SUCCESS) { set_err("nvmlDeviceGetUUID", r); return (int)r; }
  if ((r = g_api.nvmlDeviceGetName(d, out->name, sizeof(out->name))) != NVML_SUCCESS) { set_err("nvmlDeviceGetName", r); return (int)r; }
  nvmlPciInfo_t pci;
  if ((r = g_api.nvmlDeviceGetPciInfo_v3(d, &pci)) == NVML_SUCCESS) snprintf(out->bus_id, sizeof(out->bus_id), "%s", pci.busId);
  nvmlMemory_t mem;
  if (g_api.nvmlDeviceGetMemoryInfo(d, &mem) == NVML_SUCCESS) { out->mem_total = mem.total; out->mem_used = mem.used; }
  unsigned int cur = 0, pend = 0;
  if (g_api.nvmlDeviceGetMigMode(d, &cur, &pend) == NVML_SUCCESS) { out->mig_mode_current = (int)cur; out->mig_mode_pending = (int)pend; }
  return B200NVML_OK;
}

// Integer mean of the GPU-utilisation samples newer than since_us (NVML keeps ~100 samples, ~6/s).
int b200nvml_average_usage(const char* uuid, unsigned long long since_us, unsigned int* util) {
  int rc = need_api();
  if (rc) return rc;
  if (!uuid || !util) return B200NVML_BAD_ARG;
  nvmlDevice_t d;
  nvmlReturn_t r = g_api.nvmlDeviceGetHandleByUUID(uuid, &d);
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceGetHandleByUUID", r); return (int)r; }
  nvmlValueType_t vt;
  unsigned int count = 0;
  r = g_api.nvmlDeviceGetSamples(d, NVML_GPU_UTILIZATION_SAMPLES, since_us, &vt, &count, nullptr);   // size query
  if (r == NVML_ERROR_NOT_SUPPORTED) return utilization_rate(d, since_us, util, r, "nvmlDeviceGetSamples(size)");
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceGetSamples(size)", r); return (int)r; }
  if (count == 0) { snprintf(g_last_error, sizeof(g_last_error), "no utilisation samples newer than the cut-off"); return B200NVML_NO_SAMPLES; }
  std::vector<nvmlSample_t> samples(count);
  r = g_api.nvmlDeviceGetSamples(d, NVML_GPU_UTILIZATION_SAMPLES, since_us, &vt, &count, samples.data());
  if (r == NVML_ERROR_NOT_SUPPORTED) return utilization_rate(d, since_us, util, r, "nvmlDeviceGetSamples");
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceGetSamples", r); return (int)r; }
  if (count == 0) return B200NVML_NO_SAMPLES;
  unsigned long long sum = 0;
  for (unsigned int i = 0; i < count; i++) sum += samples[i].sampleValue.uiVal;
  *util = (unsigned int)(sum / count);
  return B200NVML_OK;
}

// ---- Xid events
int b200nvml_events_open(void** set_out) {
  int rc = need_api();
  if (rc) return rc;
  EventSet* es = new EventSet();
  nvmlReturn_t r = g_api.nvmlEventSetCreate(&es->set);
  if (r != NVML_SUCCESS) { delete es; set_err("nvmlEventSetCreate", r); return (int)r; }
  *set_out = es;
  return B200NVML_OK;
}

int b200nvml_events_register_xid(void* set, int index) {
  int rc = need_api();
  if (rc) return rc;
  if (!set) return B200NVML_BAD_ARG;
  nvmlDevice_t d;
  nvmlReturn_t r = g_api.nvmlDeviceGetHandleByIndex_v2((unsigned)index, &d);
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceGetHandleByIndex", r); return (int)r; }
  r = g_api.nvmlDeviceRegisterEvents(d, nvmlEventTypeXidCriticalError, static_cast<EventSet*>(set)->set);
  if (r == NVML_ERROR_NOT_SUPPORTED) { set_err("nvmlDeviceRegisterEvents", r); return B200NVML_NOT_SUPPORTED; }
  if (r != NVML_SUCCESS) { set_err("nvmlDeviceRegisterEvents", r); return (int)r; }
  return B200NVML_OK;
}

int b200nvml_events_wait(void* set, unsigned int timeout_ms, b200nvml_event* ev) {
  int rc = need_api();
  if (rc) return rc;
  if (!set || !ev) return B200NVML_BAD_ARG;
  memset(ev, 0, sizeof(*ev));
  nvmlEventData_t data;
  memset(&data, 0, sizeof(data));
  nvmlReturn_t r = g_api.nvmlEventSetWait_v2(static_cast<EventSet*>(set)->set, &data, timeout_ms);
  if (r == NVML_ERROR_TIMEOUT) return B200NVML_TIMEOUT;
  if (r != NVML_SUCCESS) { set_err("nvmlEventSetWait", r); return (int)r; }
  ev->event_type = data.eventType; ev->event_data = data.eventData;
  ev->gpu_instance_id = data.gpuInstanceId; ev->compute_instance_id = data.computeInstanceId;
  if (data.device) {
    if (g_api.nvmlDeviceGetUUID(data.device, ev->uuid, sizeof(ev->uuid)) != NVML_SUCCESS) ev->uuid[0] = 0;
  }
  return B200NVML_OK;
}

int b200nvml_events_close(void* set) {
  if (!set) return B200NVML_BAD_ARG;
  EventSet* es = static_cast<EventSet*>(set);
  if (g_api.ok) g_api.nvmlEventSetFree(es->set);
  delete es;
  return B200NVML_OK;
}

unsigned long long b200nvml_event_type_xid(void) { return nvmlEventTypeXidCriticalError; }

}  // extern "C"
