// runtime.cu -- error reporting, device check, launch accounting.
#include <stdarg.h>

#include <vector>

#include "common.cuh"

namespace gm {
static thread_local char g_err[1024] = "";
std::atomic<long long> g_launches{0};

bool g_profile = false;
struct ProfEvent { int cat; cudaEvent_t e0, e1; };
static std::vector<ProfEvent> g_prof_events;

void profile_begin(int category, cudaStream_t s) {
    ProfEvent ev{category, nullptr, nullptr};
    if (cudaEventCreate(&ev.e0) != cudaSuccess || cudaEventCreate(&ev.e1) != cudaSuccess) return;
    cudaEventRecord(ev.e0, s);
    g_prof_events.push_back(ev);
}
void profile_end(cudaStream_t s) {
    if (!g_prof_events.empty()) cudaEventRecord(g_prof_events.back().e1, s);
}

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace gm

extern "C" {
const char* gm_last_error(void) { return gm::g_err; }
int gm_abi_version(void) { return 6; }
int64_t gm_kernel_launch_count(void) { return gm::g_launches.load(); }

void gm_profile_enable(int on) { gm::g_profile = on != 0; }

int gm_profile_collect(double* ms, int32_t* launches) {
    for (int c = 0; c < gm::PROF_CATEGORIES; c++) {
        if (ms) ms[c] = 0.0;
        if (launches) launches[c] = 0;
    }
    for (auto& ev : gm::g_prof_events) {
        float t = 0.f;
        if (cudaEventSynchronize(ev.e1) == cudaSuccess && cudaEventElapsedTime(&t, ev.e0, ev.e1) == cudaSuccess) {
            if (ms) ms[ev.cat] += t;
            if (launches) launches[ev.cat] += 1;
        }
        cudaEventDestroy(ev.e0);
        cudaEventDestroy(ev.e1);
    }
    gm::g_prof_events.clear();
    cudaGetLastError();
    return GM_OK;
}

int gm_device_check(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        gm::set_error("no CUDA device (%s); libgraphmarl_b200 has no CPU fallback",
                      e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
        cudaGetLastError();
        return GM_ERR_NO_DEVICE;
    }
    int dev = 0, major = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (major != 10) {
        gm::set_error("device compute capability %d.x, built for sm_100a only", major);
        return GM_ERR_NO_DEVICE;
    }
    return GM_OK;
}
}
