// replay_sampler.cu -- the replay ring's index streams, bit-exact with numpy's Generator, on host and device.
//
// Reference: src/replaybuffer.py:101 (`np.random.default_rng(seed)`), :111-130 (get_batch):
//     single transitions : indices = rng.choice(count, batch, replace=True)
//     sequences          : start = (index % count + rng.choice(count - seq_len, batch)) % count,
//                          step o reads (start + o) % count
// numpy (un-vendored dependency of the reference, `numpy` unpinned in pyproject.toml:18, 2.3.5 here) implements
// default_rng(seed) as PCG64 (XSL-RR 128/64, 128-bit LCG) seeded from SeedSequence(seed).generate_state(4, uint64), and
// Generator.choice(n, size) without p as integers(0, n, size): Lemire's multiply-shift rejection on 32-bit halves of
// the 64-bit outputs (low half first, the high half is buffered).  Restated here from the published algorithms and
// pinned against numpy itself in tests/test_host_helpers.py and against the reference's recorded index streams in
// tests/golden/replay.npz.  The device form keeps the generator state in HBM so that sampling needs no host round trip.
#include "common.cuh"

namespace gm {

struct Pcg64 {
    uint64_t state_hi, state_lo, inc_hi, inc_lo, has_u32, buf;
};
static_assert(sizeof(Pcg64) == GM_PCG64_STATE_WORDS * 8, "state layout");

__host__ __device__ inline void mul128(uint64_t ah, uint64_t al, uint64_t bh, uint64_t bl, uint64_t& rh, uint64_t& rl) {
#ifdef __CUDA_ARCH__
    rl = al * bl;
    rh = __umul64hi(al, bl) + ah * bl + al * bh;
#else
    unsigned __int128 p = (unsigned __int128)al * bl;
    rl = (uint64_t)p;
    rh = (uint64_t)(p >> 64) + ah * bl + al * bh;
#endif
}

__host__ __device__ inline void pcg_step(Pcg64& g) {
    const uint64_t MH = 2549297995355413924ull, ML = 4865540595714422341ull;  // PCG_DEFAULT_MULTIPLIER_128
    uint64_t h, l;
    mul128(g.state_hi, g.state_lo, MH, ML, h, l);
    l += g.inc_lo;
    h += g.inc_hi + (l < g.inc_lo ? 1 : 0);
    g.state_hi = h;
    g.state_lo = l;
}

__host__ __device__ inline uint64_t pcg_u64(Pcg64& g) {
    pcg_step(g);
    const uint64_t x = g.state_hi ^ g.state_lo;
    const unsigned r = (unsigned)(g.state_hi >> 58);  // state >> 122
    return (x >> r) | (x << ((64 - r) & 63));
}

__host__ __device__ inline uint32_t pcg_u32(Pcg64& g) {
    if (g.has_u32) {
        g.has_u32 = 0;
        return (uint32_t)g.buf;
    }
    const uint64_t n = pcg_u64(g);
    g.has_u32 = 1;
    g.buf = n >> 32;
    return (uint32_t)n;
}

// Generator.integers(0, n): n <= 2^32 - 1 (ring capacities are far below)
__host__ __device__ inline int64_t pcg_bounded(Pcg64& g, int64_t n) {
    const uint64_t rng = (uint64_t)n - 1;
    if (rng == 0) return 0;
    if (rng == 0xFFFFFFFFull) return (int64_t)pcg_u32(g);
    const uint32_t excl = (uint32_t)rng + 1;
    uint64_t m = (uint64_t)pcg_u32(g) * excl;
    uint32_t leftover = (uint32_t)m;
    if (leftover < excl) {
        const uint32_t threshold = (0xFFFFFFFFu - (uint32_t)rng) % excl;
        while (leftover < threshold) {
            m = (uint64_t)pcg_u32(g) * excl;
            leftover = (uint32_t)m;
        }
    }
    return (int64_t)(m >> 32);
}

static void seed_sequence_pool(uint64_t seed, uint32_t pool[4]) {
    // numpy SeedSequence(seed): the integer as little-endian 32-bit words (at least one), pool of 4 words
    uint32_t ent[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    const int n_ent = ent[1] ? 2 : 1;
    uint32_t hc = 0x43b0d7e5u;
    auto hashmix = [&](uint32_t v) {
        v ^= hc;
        hc *= 0x931e8875u;
        v *= hc;
        v ^= v >> 16;
        return v;
    };
    auto mix = [](uint32_t x, uint32_t y) {
        uint32_t r = 0xca01f9ddu * x - 0x4973f715u * y;
        r ^= r >> 16;
        return r;
    };
    for (int i = 0; i < 4; i++) pool[i] = hashmix(i < n_ent ? ent[i] : 0u);
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++)
            if (i != j) pool[j] = mix(pool[j], hashmix(pool[i]));
}

__global__ void replay_indices_kernel(Pcg64* __restrict__ state, int64_t count, int64_t index, int batch, int seq_len,
                                      int64_t* __restrict__ out) {
    if (blockIdx.x || threadIdx.x) return;
    Pcg64 g = *state;
    if (seq_len <= 1) {
        for (int i = 0; i < batch; i++) out[i] = pcg_bounded(g, count);
    } else {
        const int64_t buffer_start = index % count;
        for (int i = 0; i < batch; i++) out[i] = (buffer_start + pcg_bounded(g, count - seq_len)) % count;
        for (int o = 1; o < seq_len; o++)
            for (int i = 0; i < batch; i++) out[(int64_t)o * batch + i] = (out[i] + o) % count;
    }
    *state = g;
}

// Per-env sequences on a ring that a batched step fills with B consecutive slots (one per env): the start step is drawn
// with the rule above counted in steps, then the env; row o is the slot of that env o steps later.
__global__ void env_sequences_kernel(Pcg64* __restrict__ state, int64_t steps_stored, int64_t head_step, int num_envs,
                                     int batch, int seq_len, int64_t* __restrict__ out) {
    if (blockIdx.x || threadIdx.x) return;
    Pcg64 g = *state;
    const int64_t first = head_step % steps_stored;
    for (int i = 0; i < batch; i++) out[i] = (first + pcg_bounded(g, steps_stored - seq_len)) % steps_stored;
    for (int i = 0; i < batch; i++) {
        const int64_t env = pcg_bounded(g, num_envs);
        const int64_t s0 = out[i];
        for (int o = 0; o < seq_len; o++) out[(int64_t)o * batch + i] = ((s0 + o) % steps_stored) * num_envs + env;
    }
    *state = g;
}

}  // namespace gm

using namespace gm;

extern "C" {

void gm_pcg64_seed(uint64_t* state, uint64_t seed) {
    uint32_t pool[4];
    seed_sequence_pool(seed, pool);
    uint32_t w[8];
    uint32_t hc = 0x8b51f9ddu;  // generate_state(4, uint64) = 8 uint32 words
    for (int i = 0; i < 8; i++) {
        uint32_t v = pool[i & 3];
        v ^= hc;
        hc *= 0x58f38dedu;
        v *= hc;
        v ^= v >> 16;
        w[i] = v;
    }
    uint64_t u[4];
    for (int i = 0; i < 4; i++) u[i] = (uint64_t)w[2 * i] | ((uint64_t)w[2 * i + 1] << 32);
    Pcg64 g{};
    // pcg_setseq_128_srandom_r(initstate = u0:u1, initseq = u2:u3)
    g.inc_hi = (u[2] << 1) | (u[3] >> 63);
    g.inc_lo = (u[3] << 1) | 1;
    pcg_step(g);
    g.state_lo += u[1];
    g.state_hi += u[0] + (g.state_lo < u[1] ? 1 : 0);
    pcg_step(g);
    *(Pcg64*)state = g;
}

void gm_pcg64_choice(uint64_t* state, int64_t n, int64_t size, int64_t* out) {
    Pcg64& g = *(Pcg64*)state;
    for (int64_t i = 0; i < size; i++) out[i] = pcg_bounded(g, n);
}

int gm_replay_sample_indices(uint64_t* state_dev, int64_t count, int64_t index, int32_t batch, int32_t seq_len, int64_t* out,
                             void* stream) {
    GM_CHECK_ARG(state_dev && out && batch > 0, "bad sampler arguments");
    GM_CHECK_ARG(count > 0 && count <= 0xFFFFFFFFll && (seq_len <= 1 || count - seq_len > 0), "count %lld / sequence length %d",
                 (long long)count, seq_len);
    replay_indices_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((Pcg64*)state_dev, count, index, batch, seq_len, out);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int gm_replay_sample_env_sequences(uint64_t* state_dev, int64_t steps_stored, int64_t head_step, int32_t num_envs,
                                   int32_t batch, int32_t seq_len, int64_t* out, void* stream) {
    GM_CHECK_ARG(state_dev && out && batch > 0 && num_envs > 0 && seq_len >= 1, "bad sampler arguments");
    GM_CHECK_ARG(steps_stored - seq_len > 0 && steps_stored <= 0xFFFFFFFFll && head_step >= 0,
                 "%lld stored steps / sequence length %d", (long long)steps_stored, seq_len);
    env_sequences_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((Pcg64*)state_dev, steps_stored, head_step, num_envs, batch,
                                                             seq_len, out);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

}  // extern "C"
