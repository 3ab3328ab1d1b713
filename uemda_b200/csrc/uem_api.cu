// Error channel, version and device binding of libuem_b200.
#include "uem_common.cuh"
#include <atomic>

static thread_local char g_err[512] = "";
int g_uem_refine_ctas_per_sm = 0;
int g_uem_region_ctas_per_sm = 0;
int g_uem_proto_ctas_per_sm = 0;
int g_uem_l2_stream = 1;
int g_uem_l2_keep = 0;
int g_uem_l2_region = 1;
int g_uem_l2_last_use = 1;

int uem_fail(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}

extern "C" const char* uem_last_error(void) { return g_err; }

extern "C" int uem_version(void) { return UEM_ABI_VERSION; }

static std::atomic<long long> g_launches{0};
void uem_note_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
extern "C" int64_t uem_kernel_launches(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

// optional cudaEvent_t pair recorded around the next fused-refine kernel launch on this thread
static thread_local void* g_ev_start = nullptr;
static thread_local void* g_ev_stop = nullptr;
extern "C" int uem_profile_refine_events(void* start, void* stop) {
    g_ev_start = start;
    g_ev_stop = stop;
    return 0;
}
void uem_take_profile_events(void** start, void** stop) {
    *start = g_ev_start;
    *stop = g_ev_stop;
    g_ev_start = g_ev_stop = nullptr;
}

extern "C" int uem_set_device(int device) {
    UEM_CUDA(cudaSetDevice(device));
    return 0;
}
