// libfake_nvml.so — a scripted stand-in for libnvidia-ml.so.1 so the native NVML binding and everything
// above it (discovery, duty-cycle sampler, Xid health loop) run end to end on a GPU-less CI box.
// Scripted by environment: FAKE_NVML_GPUS (count, default 2), FAKE_NVML_UTIL ("50,60,70" sample values,
// empty = no samples), FAKE_NVML_EVENTS (file with "gpu_index xid [gi ci]" lines; each Wait pops one line,
// "-1 xid" = event without a device), FAKE_NVML_NO_EVENTS=1 (RegisterEvents returns NOT_SUPPORTED),
// FAKE_NVML_SAMPLES_UNSUPPORTED=1 (GetSamples sizes the buffer but refuses to fill it, as some drivers do; GetUtilizationRates
// then reports the last FAKE_NVML_UTIL value).
#include "nvml_abi.h"
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>
#include <cstdint>

#include <dirent.h>
#include <ctype.h>
// FAKE_NVML_DEV_DIR: count nvidia<N> files there (lets a test hot-add a GPU by touching a file), else FAKE_NVML_GPUS.
static int gpus() {
  if (const char* d = getenv("FAKE_NVML_DEV_DIR")) {
    int n = 0;
    if (DIR* dir = opendir(d)) {
      while (dirent* e = readdir(dir)) {
        const char* s = e->d_name;
        if (strncmp(s, "nvidia", 6) != 0 || !s[6]) continue;
        bool digits = true;
        for (const char* p = s + 6; *p; p++) digits = digits && isdigit((unsigned char)*p);
        if (digits) n++;
      }
      closedir(dir);
    }
    return n;
  }
  const char* e = getenv("FAKE_NVML_GPUS");
  return e ? atoi(e) : 2;
}
static long g_event_pos = 0;

extern "C" {
nvmlReturn_t nvmlInit_v2(void) { return getenv("FAKE_NVML_INIT_FAIL") ? NVML_ERROR_DRIVER_NOT_LOADED : NVML_SUCCESS; }
nvmlReturn_t nvmlShutdown(void) { return NVML_SUCCESS; }
const char* nvmlErrorString(nvmlReturn_t r) { return r == NVML_SUCCESS ? "Success" : r == NVML_ERROR_NOT_SUPPORTED ? "Not Supported" : "fake error"; }
nvmlReturn_t nvmlDeviceGetCount_v2(unsigned int* n) { *n = (unsigned)gpus(); return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceGetHandleByIndex_v2(unsigned int i, nvmlDevice_t* d) { if ((int)i >= gpus()) return NVML_ERROR_INVALID_ARGUMENT; *d = (nvmlDevice_t)(uintptr_t)(i + 1); return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceGetHandleByUUID(const char* uuid, nvmlDevice_t* d) {
  int idx = -1;
  if (sscanf(uuid, "GPU-fake-%d", &idx) != 1 || idx < 0 || idx >= gpus()) return NVML_ERROR_NOT_FOUND;
  *d = (nvmlDevice_t)(uintptr_t)(idx + 1); return NVML_SUCCESS;
}
static int idx_of(nvmlDevice_t d) { return (int)(uintptr_t)d - 1; }
nvmlReturn_t nvmlDeviceGetMinorNumber(nvmlDevice_t d, unsigned int* m) { *m = (unsigned)idx_of(d); return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceGetUUID(nvmlDevice_t d, char* buf, unsigned int len) { snprintf(buf, len, "GPU-fake-%d", idx_of(d)); return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceGetName(nvmlDevice_t, char* buf, unsigned int len) { snprintf(buf, len, "NVIDIA B200"); return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceGetPciInfo_v3(nvmlDevice_t d, nvmlPciInfo_t* p) { memset(p, 0, sizeof(*p)); snprintf(p->busId, sizeof(p->busId), "00000000:%02X:00.0", 0x1B + idx_of(d)); return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceGetMemoryInfo(nvmlDevice_t, nvmlMemory_t* m) { m->total = 183359ull << 20; m->used = 1024ull << 20; m->free = m->total - m->used; return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceGetMigMode(nvmlDevice_t, unsigned int* c, unsigned int* p) { *c = *p = getenv("FAKE_NVML_MIG") ? 1 : 0; return NVML_SUCCESS; }
nvmlReturn_t nvmlSystemGetDriverVersion(char* buf, unsigned int len) { const char* v = getenv("FAKE_NVML_DRIVER"); snprintf(buf, len, "%s", v ? v : "580.159.03"); return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceGetSupportedEventTypes(nvmlDevice_t, unsigned long long* t) { *t = nvmlEventTypeXidCriticalError; return NVML_SUCCESS; }
static unsigned util_values(unsigned* vals) {
  const char* e = getenv("FAKE_NVML_UTIL");
  unsigned n = 0;
  if (e) { const char* p = e; while (*p && n < 128) { vals[n++] = (unsigned)strtoul(p, (char**)&p, 10); if (*p == ',') p++; else break; } }
  else { vals[0] = 40; vals[1] = 60; n = 2; }
  return e && !*e ? 0 : n;
}
nvmlReturn_t nvmlDeviceGetUtilizationRates(nvmlDevice_t, nvmlUtilization_t* u) {
  unsigned vals[128]; unsigned n = util_values(vals);
  u->gpu = n ? vals[n - 1] : 0; u->memory = 0;
  return NVML_SUCCESS;
}
nvmlReturn_t nvmlDeviceGetSamples(nvmlDevice_t, nvmlSamplingType_t, unsigned long long, nvmlValueType_t* vt, unsigned int* count, nvmlSample_t* samples) {
  unsigned vals[128]; unsigned n = util_values(vals);
  *vt = NVML_VALUE_TYPE_UNSIGNED_INT;
  if (!samples) { *count = n; return NVML_SUCCESS; }
  if (getenv("FAKE_NVML_SAMPLES_UNSUPPORTED")) return NVML_ERROR_NOT_SUPPORTED;
  if (*count > n) *count = n;
  for (unsigned i = 0; i < *count; i++) { samples[i].timeStamp = 1; samples[i].sampleValue.uiVal = vals[i]; }
  return NVML_SUCCESS;
}
nvmlReturn_t nvmlEventSetCreate(nvmlEventSet_t* s) { *s = (nvmlEventSet_t)malloc(8); return NVML_SUCCESS; }
nvmlReturn_t nvmlEventSetFree(nvmlEventSet_t s) { free(s); return NVML_SUCCESS; }
nvmlReturn_t nvmlDeviceRegisterEvents(nvmlDevice_t, unsigned long long, nvmlEventSet_t) { return getenv("FAKE_NVML_NO_EVENTS") ? NVML_ERROR_NOT_SUPPORTED : NVML_SUCCESS; }
nvmlReturn_t nvmlEventSetWait_v2(nvmlEventSet_t, nvmlEventData_t* data, unsigned int timeoutms) {
  const char* path = getenv("FAKE_NVML_EVENTS");
  if (path) {
    FILE* f = fopen(path, "r");
    if (f) {
      fseek(f, g_event_pos, SEEK_SET);
      char line[128];
      while (fgets(line, sizeof(line), f)) {
        g_event_pos = ftell(f);
        int idx = 0; unsigned long long xid = 0; unsigned gi = 0xFFFFFFFFu, ci = 0xFFFFFFFFu;
        int got = sscanf(line, "%d %llu %u %u", &idx, &xid, &gi, &ci);
        if (got < 2) continue;
        fclose(f);
        memset(data, 0, sizeof(*data));
        data->device = idx >= 0 ? (nvmlDevice_t)(uintptr_t)(idx + 1) : nullptr;
        data->eventType = nvmlEventTypeXidCriticalError; data->eventData = xid; data->gpuInstanceId = gi; data->computeInstanceId = ci;
        return NVML_SUCCESS;
      }
      fclose(f);
    }
  }
  usleep((timeoutms > 50 ? 50 : timeoutms) * 1000);
  return NVML_ERROR_TIMEOUT;
}
}
