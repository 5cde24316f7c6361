// common.cuh -- shared helpers of libgraphmarl_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>

#include "../../include/graphmarl_b200.h"

namespace gm {

void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define GM_CHECK_ARG(cond, ...)                 \
    do {                                        \
        if (!(cond)) {                          \
            gm::set_error(__VA_ARGS__);         \
            return GM_ERR_INVALID;              \
        }                                       \
    } while (0)

#define GM_CUDA(call)                                                                  \
    do {                                                                               \
        cudaError_t e__ = (call);                                                      \
        if (e__ != cudaSuccess) {                                                      \
            gm::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call,                 \
                          cudaGetErrorString(e__));                                    \
            return GM_ERR_CUDA;                                                        \
        }                                                                              \
    } while (0)

#define GM_LAUNCH_CHECK()                                                              \
    do {                                                                               \
        cudaError_t e__ = cudaGetLastError();                                          \
        if (e__ != cudaSuccess) {                                                      \
            gm::set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__,             \
                          cudaGetErrorString(e__));                                    \
            return GM_ERR_CUDA;                                                        \
        }                                                                              \
        gm::count_launch();                                                            \
    } while (0)

// optional per-launch timing with CUDA events on the launching stream (gm_profile_enable / gm_profile_collect)
enum { PROF_TC = 0, PROF_ENV = 1, PROF_AGG = 2, PROF_READOUT = 3, PROF_REPLAY = 4, PROF_CATEGORIES = 8 };
extern bool g_profile;
void profile_begin(int category, cudaStream_t s);
void profile_end(cudaStream_t s);
struct ProfileScope {
    cudaStream_t s;
    bool on;
    ProfileScope(int category, cudaStream_t stream) : s(stream), on(g_profile) {
        if (on) profile_begin(category, s);
    }
    ~ProfileScope() {
        if (on) profile_end(s);
    }
};

constexpr unsigned FULL = 0xffffffffu;
constexpr int kNumSMs = 148;

__host__ __device__ inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), counter-based draws for the device-side
// random source when the host supplies none.
// ---------------------------------------------------------------------------
struct Philox {
    uint32_t r[4];
    __device__ Philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed) {
        uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
        uint32_t c[4] = {c0, c1, c2, c3};
#pragma unroll
        for (int i = 0; i < 10; i++) {
            uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
            uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
            uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
            c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
        r[0] = c[0]; r[1] = c[1]; r[2] = c[2]; r[3] = c[3];
    }
};

// uniform double in [0,1) with 53 random bits, same construction as genrand_res53
__device__ inline double u53(uint32_t a, uint32_t b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) / 9007199254740992.0;
}

__device__ inline float apply_act(float x, int act) {
    switch (act) {
        case GM_ACT_LEAKY_RELU: return x >= 0.f ? x : x * 0.01f;
        case GM_ACT_RELU: return fmaxf(x, 0.f);
        case GM_ACT_TANH: return tanhf(x);
        case GM_ACT_SIGMOID: return 1.f / (1.f + expf(-x));
        case GM_ACT_ELU: return x > 0.f ? x : expm1f(x);
        default: return x;
    }
}

__device__ inline float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

}  // namespace gm
