// libb200probe.so — lifecycle, NVML enumeration and the passive health loop (C ABI, see
// include/b200probe.h).  No GPU work here; this file is the part of the library that replaces the
// reference plugin's NVML usage:
//   enumeration   <- what backs ListAndWatch for values.yaml:16-18 (/root/reference/values.yaml)
//   health loop   <- the plugin's XID/ECC event wait [RECALLED upstream checkHealth]; NVML contracts
//                    from nvml.h:9125 (nvmlEventSetCreate), :9161 (nvmlDeviceRegisterEvents),
//                    :9222 (nvmlEventSetWait_v2), event constants :2818,:2824,:2835.
// NVML is dlopen()ed from an overridable path so a mock libnvidia-ml drives the tests on a GPU-less box.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvml.h>
#include <pthread.h>
#include <time.h>
#include <unistd.h>

#include <cctype>
#include <cstdlib>
#include <string>
#include <vector>

#include "common.h"

namespace {

struct Nvml {
    void* lib = nullptr;
    nvmlReturn_t (*Init_v2)(void);
    nvmlReturn_t (*Shutdown)(void);
    const char* (*ErrorString)(nvmlReturn_t);
    nvmlReturn_t (*DeviceGetCount_v2)(unsigned int*);
    nvmlReturn_t (*DeviceGetHandleByIndex_v2)(unsigned int, nvmlDevice_t*);
    nvmlReturn_t (*DeviceGetUUID)(nvmlDevice_t, char*, unsigned int);
    nvmlReturn_t (*DeviceGetName)(nvmlDevice_t, char*, unsigned int);
    nvmlReturn_t (*DeviceGetMemoryInfo)(nvmlDevice_t, nvmlMemory_t*);
    nvmlReturn_t (*DeviceGetCudaComputeCapability)(nvmlDevice_t, int*, int*);
    nvmlReturn_t (*DeviceGetPciInfo_v3)(nvmlDevice_t, nvmlPciInfo_t*);
    nvmlReturn_t (*DeviceGetNumaNodeId)(nvmlDevice_t, unsigned int*);                 // optional
    nvmlReturn_t (*DeviceGetMigMode)(nvmlDevice_t, unsigned int*, unsigned int*);     // optional
    nvmlReturn_t (*DeviceGetSupportedEventTypes)(nvmlDevice_t, unsigned long long*);
    nvmlReturn_t (*DeviceRegisterEvents)(nvmlDevice_t, unsigned long long, nvmlEventSet_t);
    nvmlReturn_t (*EventSetCreate)(nvmlEventSet_t*);
    nvmlReturn_t (*EventSetWait_v2)(nvmlEventSet_t, nvmlEventData_t*, unsigned int);
    nvmlReturn_t (*EventSetFree)(nvmlEventSet_t);
    nvmlReturn_t (*DeviceGetNvLinkState)(nvmlDevice_t, unsigned int, nvmlEnableState_t*);    // optional
    nvmlReturn_t (*DeviceGetFieldValues)(nvmlDevice_t, int, nvmlFieldValue_t*);              // optional
    nvmlReturn_t (*DeviceGetGpuFabricInfoV)(nvmlDevice_t, nvmlGpuFabricInfoV_t*);            // optional
    nvmlReturn_t (*DeviceGetComputeRunningProcesses_v3)(nvmlDevice_t, unsigned int*, nvmlProcessInfo_t*);   // optional
    nvmlReturn_t (*DeviceGetUtilizationRates)(nvmlDevice_t, nvmlUtilization_t*);                          // optional
    nvmlReturn_t (*DeviceGetEccMode)(nvmlDevice_t, nvmlEnableState_t*, nvmlEnableState_t*);                // optional
    nvmlReturn_t (*DeviceGetTotalEccErrors)(nvmlDevice_t, nvmlMemoryErrorType_t, nvmlEccCounterType_t, unsigned long long*);   // optional
    nvmlReturn_t (*DeviceGetRemappedRows)(nvmlDevice_t, unsigned int*, unsigned int*, unsigned int*, unsigned int*);         // optional
};

struct Device {
    nvmlDevice_t h;
    b200probe_device_t info;
};

struct State {
    pthread_mutex_t mu = PTHREAD_MUTEX_INITIALIZER;
    bool inited = false;
    Nvml nvml;
    std::vector<Device> devs;
    // health
    bool health_open = false, health_disabled = false;
    nvmlEventSet_t evset = nullptr;
    std::vector<uint64_t> skip_xids;
    uint64_t unhealthy = 0;
    int waiters = 0;                      // threads inside nvmlEventSetWait_v2 with g.mu dropped
    pthread_cond_t no_waiters = PTHREAD_COND_INITIALIZER;
    // cuda
    bool cuda_ready = false;
    int cuda_count = 0;
    std::vector<std::string> cuda_uuid;
    std::vector<b200::DevProps> cuda_props;
    std::vector<char> cuda_touched;       // a probe of this process has run on the ordinal: the process owns a context there
};
State g;

struct Lock {
    Lock() { pthread_mutex_lock(&g.mu); }
    ~Lock() { pthread_mutex_unlock(&g.mu); }
};

thread_local char tl_err[512] = "";

int nvml_rc(nvmlReturn_t r) { return r == NVML_SUCCESS ? 0 : B200PROBE_NVML_BASE + (int)r; }

template <typename F>
bool sym(void* lib, const char* name, F& fn, bool required) {
    fn = reinterpret_cast<F>(dlsym(lib, name));
    if (!fn && required) b200::set_error("NVML symbol %s missing", name);
    return fn != nullptr || !required;
}

double now_us() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}

// Fill one device record.  Field order and failure policy follow the reference plugin's
// enumeration: a device whose UUID cannot be read is a hard error; optional attributes
// (NUMA node, MIG mode) degrade to -1.
int read_device(unsigned idx, Device* d) {
    Nvml& n = g.nvml;
    memset(&d->info, 0, sizeof(d->info));
    d->info.index = (int)idx;
    d->info.cuda_ordinal = -1;
    nvmlReturn_t r = n.DeviceGetHandleByIndex_v2(idx, &d->h);
    if (r != NVML_SUCCESS) { b200::set_error("nvmlDeviceGetHandleByIndex_v2(%u): %s", idx, n.ErrorString(r)); return nvml_rc(r); }
    r = n.DeviceGetUUID(d->h, d->info.uuid, sizeof(d->info.uuid));
    if (r != NVML_SUCCESS) { b200::set_error("nvmlDeviceGetUUID(%u): %s", idx, n.ErrorString(r)); return nvml_rc(r); }
    r = n.DeviceGetName(d->h, d->info.name, sizeof(d->info.name));
    if (r != NVML_SUCCESS) { b200::set_error("nvmlDeviceGetName(%u): %s", idx, n.ErrorString(r)); return nvml_rc(r); }
    nvmlMemory_t mem;
    r = n.DeviceGetMemoryInfo(d->h, &mem);
    if (r != NVML_SUCCESS) { b200::set_error("nvmlDeviceGetMemoryInfo(%u): %s", idx, n.ErrorString(r)); return nvml_rc(r); }
    d->info.mem_total = mem.total;
    r = n.DeviceGetCudaComputeCapability(d->h, &d->info.cc_major, &d->info.cc_minor);
    if (r != NVML_SUCCESS) { b200::set_error("nvmlDeviceGetCudaComputeCapability(%u): %s", idx, n.ErrorString(r)); return nvml_rc(r); }
    nvmlPciInfo_t pci;
    if (n.DeviceGetPciInfo_v3 && n.DeviceGetPciInfo_v3(d->h, &pci) == NVML_SUCCESS) {
        snprintf(d->info.pci_bus_id, sizeof(d->info.pci_bus_id), "%s", pci.busId);
    }
    unsigned numa = 0;
    d->info.numa_node = (n.DeviceGetNumaNodeId && n.DeviceGetNumaNodeId(d->h, &numa) == NVML_SUCCESS) ? (int)numa : -1;
    unsigned cur = 0, pend = 0;
    d->info.mig_enabled = (n.DeviceGetMigMode && n.DeviceGetMigMode(d->h, &cur, &pend) == NVML_SUCCESS) ? (int)cur : -1;
    unsigned long long ev = 0;
    if (n.DeviceGetSupportedEventTypes(d->h, &ev) == NVML_SUCCESS) d->info.supported_events = ev;
    return 0;
}

int enumerate_locked() {
    unsigned count = 0;
    nvmlReturn_t r = g.nvml.DeviceGetCount_v2(&count);
    if (r != NVML_SUCCESS) { b200::set_error("nvmlDeviceGetCount_v2: %s", g.nvml.ErrorString(r)); return nvml_rc(r); }
    if (count > B200PROBE_MAX_DEVICES) count = B200PROBE_MAX_DEVICES;
    std::vector<Device> devs(count);
    for (unsigned i = 0; i < count; ++i) {
        int rc = read_device(i, &devs[i]);
        if (rc) return rc;
    }
    // keep CUDA ordinals already resolved
    for (auto& d : devs)
        for (size_t c = 0; c < g.cuda_uuid.size(); ++c)
            if (g.cuda_uuid[c] == d.info.uuid) d.info.cuda_ordinal = (int)c;
    g.devs.swap(devs);
    return 0;
}

std::string format_cuda_uuid(const cudaUUID_t& u) {
    const unsigned char* b = reinterpret_cast<const unsigned char*>(u.bytes);
    char s[64];
    snprintf(s, sizeof(s), "GPU-%02x%02x%02x%02x-%02x%02x-%02x%02x-%02x%02x-%02x%02x%02x%02x%02x%02x", b[0], b[1], b[2],
             b[3], b[4], b[5], b[6], b[7], b[8], b[9], b[10], b[11], b[12], b[13], b[14], b[15]);
    return s;
}

int cuda_init_locked() {
    if (g.cuda_ready) return 0;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        b200::set_error("CUDA unavailable (%s); the probes have no CPU fallback", e == cudaSuccess ? "no devices" : cudaGetErrorString(e));
        cudaGetLastError();
        return B200PROBE_ENOCUDA;
    }
    g.cuda_count = n;
    g.cuda_uuid.resize(n);
    g.cuda_props.resize(n);
    g.cuda_touched.assign(n, 0);
    for (int i = 0; i < n; ++i) {
        cudaDeviceProp p;
        e = cudaGetDeviceProperties(&p, i);
        if (e != cudaSuccess) { b200::set_error("cudaGetDeviceProperties(%d): %s", i, cudaGetErrorString(e)); return b200::cuda_rc(e); }
        g.cuda_uuid[i] = format_cuda_uuid(p.uuid);
        g.cuda_props[i] = {p.multiProcessorCount, p.l2CacheSize, (int)p.sharedMemPerBlockOptin, p.major, p.minor};
    }
    for (auto& d : g.devs)
        for (int c = 0; c < n; ++c)
            if (g.cuda_uuid[c] == d.info.uuid) d.info.cuda_ordinal = c;
    g.cuda_ready = true;
    return 0;
}

// DP_DISABLE_HEALTHCHECKS grammar [RECALLED upstream getAdditionalXids]: comma list, blanks
// trimmed, malformed entries ignored.
void parse_skip_list(const char* s, std::vector<uint64_t>* out) {
    // application-level XIDs the reference treats as "GPU still healthy"
    static const uint64_t kAppXids[] = {13, 31, 43, 45, 68, 109};
    out->assign(kAppXids, kAppXids + sizeof(kAppXids) / sizeof(kAppXids[0]));
    if (!s) return;
    std::string tok;
    auto flush = [&]() {
        size_t a = 0, b = tok.size();
        while (a < b && isspace((unsigned char)tok[a])) ++a;
        while (b > a && isspace((unsigned char)tok[b - 1])) --b;
        if (b > a) {
            bool digits = true;
            for (size_t i = a; i < b; ++i) digits = digits && isdigit((unsigned char)tok[i]);
            if (digits && b - a <= 19) out->push_back(strtoull(tok.substr(a, b - a).c_str(), nullptr, 10));
        }
        tok.clear();
    };
    for (const char* p = s; *p; ++p) {
        if (*p == ',') flush(); else tok.push_back(*p);
    }
    flush();
}

uint64_t all_mask() {
    uint64_t m = 0;
    for (size_t i = 0; i < g.devs.size() && i < 64; ++i) m |= 1ull << i;
    return m;
}

int health_open_locked(const char* disable, uint64_t* at_open) {
    if (g.health_open) { if (at_open) *at_open = g.unhealthy; return 0; }
    std::string low = disable ? disable : "";
    for (auto& c : low) c = (char)tolower((unsigned char)c);
    if (low == "all") low = "xids";
    g.unhealthy = 0;
    if (low.find("xids") != std::string::npos) {   // loop disabled: every device stays Healthy
        g.health_disabled = true;
        g.health_open = true;
        if (at_open) *at_open = 0;
        return 0;
    }
    g.health_disabled = false;
    parse_skip_list(low.c_str(), &g.skip_xids);
    nvmlReturn_t r = g.nvml.EventSetCreate(&g.evset);
    if (r != NVML_SUCCESS) { b200::set_error("nvmlEventSetCreate: %s", g.nvml.ErrorString(r)); return nvml_rc(r); }
    const unsigned long long want = nvmlEventTypeXidCriticalError | nvmlEventTypeDoubleBitEccError | nvmlEventTypeSingleBitEccError;
    for (size_t i = 0; i < g.devs.size(); ++i) {
        unsigned long long supported = 0;
        r = g.nvml.DeviceGetSupportedEventTypes(g.devs[i].h, &supported);
        if (r != NVML_SUCCESS) { g.unhealthy |= 1ull << i; continue; }     // "unable to determine the supported events"
        r = g.nvml.DeviceRegisterEvents(g.devs[i].h, want & supported, g.evset);
        if (r != NVML_SUCCESS) g.unhealthy |= 1ull << i;                     // includes NOT_SUPPORTED ("too old")
    }
    g.health_open = true;
    if (at_open) *at_open = g.unhealthy;
    return 0;
}

int health_wait_locked(int timeout_ms, b200probe_health_event_t* ev) {
    b200probe_health_event_t local;
    if (!ev) ev = &local;
    memset(ev, 0, sizeof(*ev));
    ev->device_index = -1;
    if (!g.health_open) { b200::set_error("health_wait before health_open"); return B200PROBE_ESTATE; }
    if (g.health_disabled) { ev->rc_wait = NVML_ERROR_TIMEOUT; ev->skipped = 1; return 0; }
    nvmlEventData_t data;
    memset(&data, 0, sizeof(data));
    nvmlEventSet_t set = g.evset;
    auto wait = g.nvml.EventSetWait_v2;
    // The wait blocks up to timeout_ms: drop the lock so enumeration / other devices' probes proceed.  health_close and
    // shutdown wait for `waiters` to reach zero before they free the event set or unload NVML under a blocked waiter.
    ++g.waiters;
    pthread_mutex_unlock(&g.mu);
    nvmlReturn_t r = wait(set, &data, timeout_ms < 0 ? 0 : (unsigned)timeout_ms);
    pthread_mutex_lock(&g.mu);
    if (--g.waiters == 0) pthread_cond_broadcast(&g.no_waiters);
    if (!g.health_open || g.evset != set) {          // closed (or closed and reopened) while we were waiting: the event belongs to nobody
        ev->rc_wait = NVML_ERROR_TIMEOUT;
        ev->skipped = 1;
        return 0;
    }
    ev->rc_wait = (int)r;
    if (r == NVML_ERROR_TIMEOUT) return 0;
    if (r != NVML_SUCCESS) {               // "Error waiting for event: marking all devices as unhealthy"
        ev->newly_unhealthy = all_mask() & ~g.unhealthy;
        g.unhealthy |= all_mask();
        return 0;
    }
    ev->event_type = data.eventType;
    ev->event_data = data.eventData;
    ev->gpu_instance_id = data.gpuInstanceId;
    ev->compute_instance_id = data.computeInstanceId;
    if (data.eventType != nvmlEventTypeXidCriticalError) { ev->skipped = 1; return 0; }
    for (uint64_t x : g.skip_xids)
        if (x == data.eventData) { ev->skipped = 1; return 0; }
    char uuid[96];
    r = g.nvml.DeviceGetUUID(data.device, uuid, sizeof(uuid));
    if (r != NVML_SUCCESS) {               // cannot attribute the event: all devices unhealthy
        ev->newly_unhealthy = all_mask() & ~g.unhealthy;
        g.unhealthy |= all_mask();
        return 0;
    }
    for (size_t i = 0; i < g.devs.size(); ++i) {
        if (strcmp(g.devs[i].info.uuid, uuid) == 0) {
            ev->device_index = (int)i;
            ev->newly_unhealthy = (1ull << i) & ~g.unhealthy;
            g.unhealthy |= 1ull << i;
            return 0;
        }
    }
    ev->skipped = 1;                       // "Ignoring event for unexpected device"
    return 0;
}

}  // namespace

namespace b200 {
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(tl_err, sizeof(tl_err), fmt, ap);
    va_end(ap);
}
const char* get_error() { return tl_err; }

int cuda_ordinal_of(int nvml_idx, int* ordinal) {
    Lock l;
    if (!g.inited) { set_error("b200probe_init not called"); return B200PROBE_ENOTINIT; }
    if (nvml_idx < 0 || nvml_idx >= (int)g.devs.size()) { set_error("device index %d out of range", nvml_idx); return B200PROBE_ERANGE; }
    int rc = cuda_init_locked();
    if (rc) return rc;
    int o = g.devs[nvml_idx].info.cuda_ordinal;
    if (o < 0) { set_error("NVML device %d (%s) is not visible to CUDA", nvml_idx, g.devs[nvml_idx].info.uuid); return B200PROBE_ENOCUDA; }
    *ordinal = o;
    return 0;
}

int device_props(int ordinal, DevProps* out) {
    Lock l;
    int rc = cuda_init_locked();
    if (rc) return rc;
    if (ordinal < 0 || ordinal >= g.cuda_count) { set_error("CUDA ordinal %d out of range", ordinal); return B200PROBE_ERANGE; }
    *out = g.cuda_props[ordinal];
    g.cuda_touched[ordinal] = 1;          // every probe entry point passes here before it sets the device
    if (out->cc_major != 10) {
        set_error("CUDA device %d is sm_%d%d; the probe kernels are sm_100a-only", ordinal, out->cc_major, out->cc_minor);
        return B200PROBE_EARCH;
    }
    return 0;
}
}  // namespace b200

extern "C" {

int b200probe_abi_version(void) { return B200PROBE_ABI_VERSION; }

int b200probe_init(const char* path) {
    Lock l;
    if (g.inited) return 0;
    if (!path || !*path) path = getenv("B200PROBE_NVML_PATH");
    if (!path || !*path) path = "libnvidia-ml.so.1";
    void* lib = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    if (!lib) { b200::set_error("dlopen(%s): %s", path, dlerror()); return B200PROBE_ENVML; }
    Nvml n;
    n.lib = lib;
    bool ok = sym(lib, "nvmlInit_v2", n.Init_v2, true) && sym(lib, "nvmlShutdown", n.Shutdown, true) &&
              sym(lib, "nvmlErrorString", n.ErrorString, true) && sym(lib, "nvmlDeviceGetCount_v2", n.DeviceGetCount_v2, true) &&
              sym(lib, "nvmlDeviceGetHandleByIndex_v2", n.DeviceGetHandleByIndex_v2, true) &&
              sym(lib, "nvmlDeviceGetUUID", n.DeviceGetUUID, true) && sym(lib, "nvmlDeviceGetName", n.DeviceGetName, true) &&
              sym(lib, "nvmlDeviceGetMemoryInfo", n.DeviceGetMemoryInfo, true) &&
              sym(lib, "nvmlDeviceGetCudaComputeCapability", n.DeviceGetCudaComputeCapability, true) &&
              sym(lib, "nvmlDeviceGetSupportedEventTypes", n.DeviceGetSupportedEventTypes, true) &&
              sym(lib, "nvmlDeviceRegisterEvents", n.DeviceRegisterEvents, true) &&
              sym(lib, "nvmlEventSetCreate", n.EventSetCreate, true) && sym(lib, "nvmlEventSetWait_v2", n.EventSetWait_v2, true) &&
              sym(lib, "nvmlEventSetFree", n.EventSetFree, true);
    sym(lib, "nvmlDeviceGetPciInfo_v3", n.DeviceGetPciInfo_v3, false);
    sym(lib, "nvmlDeviceGetNumaNodeId", n.DeviceGetNumaNodeId, false);
    sym(lib, "nvmlDeviceGetMigMode", n.DeviceGetMigMode, false);
    sym(lib, "nvmlDeviceGetNvLinkState", n.DeviceGetNvLinkState, false);
    sym(lib, "nvmlDeviceGetFieldValues", n.DeviceGetFieldValues, false);
    sym(lib, "nvmlDeviceGetGpuFabricInfoV", n.DeviceGetGpuFabricInfoV, false);
    sym(lib, "nvmlDeviceGetComputeRunningProcesses_v3", n.DeviceGetComputeRunningProcesses_v3, false);
    sym(lib, "nvmlDeviceGetUtilizationRates", n.DeviceGetUtilizationRates, false);
    sym(lib, "nvmlDeviceGetEccMode", n.DeviceGetEccMode, false);
    sym(lib, "nvmlDeviceGetTotalEccErrors", n.DeviceGetTotalEccErrors, false);
    sym(lib, "nvmlDeviceGetRemappedRows", n.DeviceGetRemappedRows, false);
    if (!ok) { dlclose(lib); return B200PROBE_ENVML; }
    nvmlReturn_t r = n.Init_v2();
    if (r != NVML_SUCCESS) { b200::set_error("nvmlInit_v2: %s", n.ErrorString(r)); dlclose(lib); return nvml_rc(r); }
    g.nvml = n;
    int rc = enumerate_locked();
    if (rc) { n.Shutdown(); dlclose(lib); g.nvml = Nvml(); return rc; }
    g.inited = true;
    return 0;
}

// caller holds g.mu: a thread blocked in the event wait returns within its timeout; nothing it uses is freed before that
static void drain_waiters_locked() {
    g.health_open = false;                            // a waiter that wakes up sees the set is gone and reports a timeout
    while (g.waiters > 0) pthread_cond_wait(&g.no_waiters, &g.mu);
}

void b200probe_shutdown(void) {
    Lock l;
    if (!g.inited) return;
    drain_waiters_locked();
    if (g.evset) g.nvml.EventSetFree(g.evset);
    g.evset = nullptr;
    g.health_open = g.health_disabled = false;
    g.unhealthy = 0;
    g.nvml.Shutdown();
    dlclose(g.nvml.lib);
    g.nvml = Nvml();
    g.devs.clear();
    g.inited = false;
}

const char* b200probe_strerror(int rc) {
    switch (rc) {
        case B200PROBE_OK: return "ok";
        case B200PROBE_EINVAL: return "invalid argument";
        case B200PROBE_ENOTINIT: return "b200probe_init not called";
        case B200PROBE_ENVML: return "NVML library unavailable";
        case B200PROBE_ENOCUDA: return "CUDA device unavailable (no CPU fallback)";
        case B200PROBE_ERANGE: return "index or buffer out of range";
        case B200PROBE_EMISMATCH: return "data verification failed";
        case B200PROBE_ENOPEER: return "peer access unavailable";
        case B200PROBE_ENONCCL: return "NCCL library unavailable";
        case B200PROBE_EARCH: return "device is not sm_100";
        case B200PROBE_ENOMEM: return "out of memory";
        case B200PROBE_ESTATE: return "call sequence error";
        default: break;
    }
    if (rc >= B200PROBE_NCCL_BASE) return "NCCL error (rc - 3000 = ncclResult_t)";
    if (rc >= B200PROBE_NVML_BASE) return "NVML error (rc - 2000 = nvmlReturn_t)";
    if (rc >= B200PROBE_CUDA_BASE) return cudaGetErrorString((cudaError_t)(rc - B200PROBE_CUDA_BASE));
    return "unknown error";
}

int b200probe_last_error(char* buf, int cap) {
    if (!buf || cap <= 0) return B200PROBE_EINVAL;
    snprintf(buf, (size_t)cap, "%s", b200::get_error());
    return 0;
}

int b200probe_device_count(int* n) {
    if (!n) return B200PROBE_EINVAL;
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    *n = (int)g.devs.size();
    return 0;
}

int b200probe_device_info(int idx, b200probe_device_t* out) {
    if (!out) return B200PROBE_EINVAL;
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    if (idx < 0 || idx >= (int)g.devs.size()) return B200PROBE_ERANGE;
    *out = g.devs[idx].info;
    return 0;
}

int b200probe_enumerate(b200probe_device_t* out, int cap, int* n, double* usec) {
    if (!n) return B200PROBE_EINVAL;
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    if (g.health_open && !g.health_disabled) {
        // Handles registered with the event set must stay valid: report the cached list.
        if (usec) *usec = 0;
    } else {
        double t0 = now_us();
        int rc = enumerate_locked();
        if (rc) return rc;
        if (usec) *usec = now_us() - t0;
    }
    *n = (int)g.devs.size();
    if (out) {
        if (cap < *n) return B200PROBE_ERANGE;
        for (int i = 0; i < *n; ++i) out[i] = g.devs[i].info;
    }
    return 0;
}

int b200probe_health_open(const char* disable, uint64_t* at_open) {
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    return health_open_locked(disable, at_open);
}

int b200probe_health_wait(int timeout_ms, b200probe_health_event_t* ev) {
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    return health_wait_locked(timeout_ms, ev);
}

int b200probe_passive_health(int timeout_ms, uint64_t* mask) {
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    if (!g.health_open) {
        int rc = health_open_locked(getenv("DP_DISABLE_HEALTHCHECKS"), nullptr);
        if (rc) return rc;
    }
    int rc = health_wait_locked(timeout_ms, nullptr);
    if (mask) *mask = g.unhealthy;
    return rc;
}

int b200probe_health_mask(uint64_t* mask) {
    if (!mask) return B200PROBE_EINVAL;
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    *mask = g.unhealthy;
    return 0;
}

void b200probe_health_close(void) {
    Lock l;
    if (!g.inited || !g.health_open) return;
    drain_waiters_locked();
    if (g.evset) g.nvml.EventSetFree(g.evset);
    g.evset = nullptr;
    g.health_open = g.health_disabled = false;
    g.unhealthy = 0;
}

// Passive NVLink cross-check (SURVEY.md §8f.3): per-link state (nvml.h:8766), fabric registration
// + health mask (nvml.h:7220, :3453-3488) and the DATA/RAW throughput counters (nvml.h:2383-2386).
// Correlated with the active all-to-all by the host: a cold row in the pair matrix + an inactive
// link localises the fault; RAW-DATA counter deltas around an exchange give the protocol overhead.
int b200probe_nvlink_passive(int idx, b200probe_nvlink_status_t* out) {
    if (!out) return B200PROBE_EINVAL;
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    if (idx < 0 || idx >= (int)g.devs.size()) return B200PROBE_ERANGE;
    memset(out, 0, sizeof(*out));
    out->fabric_state = -1;
    nvmlDevice_t h = g.devs[idx].h;
    if (g.nvml.DeviceGetNvLinkState) {
        for (unsigned link = 0; link < NVML_NVLINK_MAX_LINKS; ++link) {
            nvmlEnableState_t st;
            nvmlReturn_t r = g.nvml.DeviceGetNvLinkState(h, link, &st);
            if (r != NVML_SUCCESS) continue;          // NOT_SUPPORTED / INVALID_ARGUMENT: link does not exist
            out->links_total++;
            if (st == NVML_FEATURE_ENABLED) { out->links_active++; out->active_mask |= 1u << link; }
        }
    }
    if (g.nvml.DeviceGetGpuFabricInfoV) {
        nvmlGpuFabricInfoV_t fi;
        memset(&fi, 0, sizeof(fi));
        fi.version = nvmlGpuFabricInfo_v2;
        if (g.nvml.DeviceGetGpuFabricInfoV(h, &fi) == NVML_SUCCESS) {
            out->fabric_state = (int)fi.state;
            out->fabric_status = (int)fi.status;
            out->fabric_health_mask = fi.healthMask;
        }
    }
    if (g.nvml.DeviceGetFieldValues) {
        nvmlFieldValue_t fv[4];
        memset(fv, 0, sizeof(fv));
        const unsigned ids[4] = {NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX, NVML_FI_DEV_NVLINK_THROUGHPUT_RAW_TX,
                                 NVML_FI_DEV_NVLINK_THROUGHPUT_RAW_RX};
        for (int i = 0; i < 4; ++i) { fv[i].fieldId = ids[i]; fv[i].scopeId = 0xFFFFFFFFu; }   // UINT_MAX: sum over all links
        if (g.nvml.DeviceGetFieldValues(h, 4, fv) == NVML_SUCCESS) {
            uint64_t v[4];
            int ok = 1;
            for (int i = 0; i < 4; ++i) {
                if (fv[i].nvmlReturn != NVML_SUCCESS) { ok = 0; v[i] = 0; continue; }
                v[i] = fv[i].valueType == NVML_VALUE_TYPE_UNSIGNED_LONG_LONG ? fv[i].value.ullVal
                     : fv[i].valueType == NVML_VALUE_TYPE_UNSIGNED_LONG ? fv[i].value.ulVal
                     : fv[i].valueType == NVML_VALUE_TYPE_UNSIGNED_INT ? fv[i].value.uiVal : 0;
            }
            out->data_tx_kib = v[0]; out->data_rx_kib = v[1]; out->raw_tx_kib = v[2]; out->raw_rx_kib = v[3];
            out->counters_ok = ok;
        }
    }
    return 0;
}

// Is somebody else using this GPU?  The active probes measure against idle-box figures and take SMs, HBM bandwidth and
// memory from whatever runs beside them, so the host asks before every round and skips (does not fail) a busy device.
int b200probe_device_busy(int idx, b200probe_busy_t* out) {
    if (!out) return B200PROBE_EINVAL;
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    if (idx < 0 || idx >= (int)g.devs.size()) return B200PROBE_ERANGE;
    memset(out, 0, sizeof(*out));
    out->compute_procs = out->util_gpu_pct = out->util_mem_pct = -1;
    nvmlDevice_t h = g.devs[idx].h;
    if (g.nvml.DeviceGetComputeRunningProcesses_v3) {
        std::vector<nvmlProcessInfo_t> procs(64);
        unsigned count = (unsigned)procs.size();
        nvmlReturn_t r = g.nvml.DeviceGetComputeRunningProcesses_v3(h, &count, procs.data());
        if (r == NVML_ERROR_INSUFFICIENT_SIZE) { procs.resize(count + 16); count = (unsigned)procs.size(); r = g.nvml.DeviceGetComputeRunningProcesses_v3(h, &count, procs.data()); }
        if (r == NVML_SUCCESS) {
            const unsigned self = (unsigned)getpid();
            int others = 0;
            bool saw_self = false;
            for (unsigned i = 0; i < count; ++i) { if (procs[i].pid == self) saw_self = true; else ++others; }
            // NVML reports pids of the HOST namespace: inside a container our own context shows up under a pid we cannot
            // recognise.  If this process has run a probe on the device and did not find itself, one of the entries is us.
            const int ord = g.devs[idx].info.cuda_ordinal;
            if (!saw_self && others > 0 && ord >= 0 && ord < (int)g.cuda_touched.size() && g.cuda_touched[ord]) --others;
            out->compute_procs = others;
        }
    }
    nvmlUtilization_t u;
    if (g.nvml.DeviceGetUtilizationRates && g.nvml.DeviceGetUtilizationRates(h, &u) == NVML_SUCCESS) { out->util_gpu_pct = (int)u.gpu; out->util_mem_pct = (int)u.memory; }
    nvmlMemory_t mem;
    if (g.nvml.DeviceGetMemoryInfo(h, &mem) == NVML_SUCCESS) out->mem_used = mem.used;
    out->busy = (out->compute_procs > 0 || out->util_gpu_pct >= B200PROBE_BUSY_UTIL_PCT) ? 1 : 0;
    return 0;
}

// Passive half of the HBM integrity probe: ECC mode (nvml.h:6249), the volatile corrected / uncorrected totals (:6349)
// and the row remapper's state (:7730).  b200probe_hbm_memtest takes this snapshot before and after its march.
int b200probe_hbm_ecc(int idx, b200probe_ecc_status_t* out) {
    if (!out) return B200PROBE_EINVAL;
    Lock l;
    if (!g.inited) return B200PROBE_ENOTINIT;
    if (idx < 0 || idx >= (int)g.devs.size()) return B200PROBE_ERANGE;
    out->ecc_mode = out->remap_corrected_rows = out->remap_uncorrected_rows = out->remap_pending = out->remap_failure = -1;
    out->corrected_volatile = out->uncorrected_volatile = -1;
    nvmlDevice_t h = g.devs[idx].h;
    nvmlEnableState_t cur, pend;
    if (g.nvml.DeviceGetEccMode && g.nvml.DeviceGetEccMode(h, &cur, &pend) == NVML_SUCCESS) out->ecc_mode = cur == NVML_FEATURE_ENABLED ? 1 : 0;
    unsigned long long v;
    if (g.nvml.DeviceGetTotalEccErrors) {
        if (g.nvml.DeviceGetTotalEccErrors(h, NVML_MEMORY_ERROR_TYPE_CORRECTED, NVML_VOLATILE_ECC, &v) == NVML_SUCCESS) out->corrected_volatile = (int64_t)v;
        if (g.nvml.DeviceGetTotalEccErrors(h, NVML_MEMORY_ERROR_TYPE_UNCORRECTED, NVML_VOLATILE_ECC, &v) == NVML_SUCCESS) out->uncorrected_volatile = (int64_t)v;
    }
    unsigned corr, unc, pending, failure;
    if (g.nvml.DeviceGetRemappedRows && g.nvml.DeviceGetRemappedRows(h, &corr, &unc, &pending, &failure) == NVML_SUCCESS) {
        out->remap_corrected_rows = (int)corr;
        out->remap_uncorrected_rows = (int)unc;
        out->remap_pending = pending ? 1 : 0;
        out->remap_failure = failure ? 1 : 0;
    }
    return 0;
}

uint32_t b200probe_pattern_word(uint64_t i, uint32_t seed) { return b200_pattern_word(i, seed); }

}  // extern "C"
