// gemm_sm100.cu -- tcgen05 / TMEM fused linear layer for sm_100a (GM_MATH_BF16X3, GM_MATH_BF16).
//
//   C[M,N] = epilogue( [seg0 | seg1][M,K] * W[N,K]^T )        (torch.nn.Linear layout)
//
// Arithmetic.  fp32 operands are split into bf16 hi + bf16 lo (x = hi + lo up to 2^-17 relative)
// and the product is formed from three tensor-core passes hi*hi + hi*lo + lo*hi accumulated in
// fp32 in TMEM ("bf16x3", relative error per product ~2^-16, inside the fp32 tolerance the parity
// tests state).  GM_MATH_BF16 runs the hi*hi pass only.
//
// Data flow.  Activations travel between layers "tile-packed" (gemm_sm100.cuh): already split to
// bf16 hi/lo and already in the shared-memory core-matrix layout of the tensor core, written by
// the producing layer's epilogue and pulled by the consuming layer with ONE bulk copy (TMA) per
// 32-wide k-block.  Only raw fp32 inputs (node observations, carried state, agent observations)
// go through the producer warps, which split them on the fly.
//
// Structure (one persistent CTA per SM, 18 warps, warp specialised):
//   warps 0-7   epilogue : tcgen05.ld accumulator rows TMEM -> registers (warp e: TMEM quadrant e%4,
//                          column half e/4), bias + activation or the whole LSTM cell pointwise (gates
//                          never leave the SM); stores fp32 rows and/or tile-packed bf16 hi/lo
//   warps 8-15  producer : fp32 segments only: 32-byte loads (8 rows x 128-byte lines per warp
//                          instruction), split to bf16 hi/lo, conflict-free 16-byte smem stores in the
//                          UMMA canonical K-major (no swizzle) layout; loads of k-block i+1 are in
//                          flight while k-block i is converted
//   warp  16    MMA      : one thread issues tcgen05.mma (M=128, N=BN, K=16) into TMEM,
//                          tcgen05.commit releases smem stages / publishes accumulators
//   warp  17    copies   : one thread streams weight tiles and tile-packed activation blocks with
//                          cp.async.bulk (TMA bulk copy) signalling the stage mbarrier
// smem ring of 4 stages x (A hi/lo 16 KiB + W hi/lo BN*128 B); 2 accumulator stages in TMEM.
// (Measured on B200: separate, deeper activation / weight rings with their own copy threads were slower.)
#include <cuda_bf16.h>

#include <stdlib.h>

#include <algorithm>
#include <utility>
#include <vector>

#include "common.cuh"
#include "gemm_sm100.cuh"
#include "linear_simt.cuh"

#ifndef GM_LSTM_SHARED_RCP
#define GM_LSTM_SHARED_RCP 1
#endif
// Timing probes (build with -DGM_TC_PROBES=1): GM_TC_DEBUG / GM_LN_DEBUG then switch off parts of the kernels to
// measure what bounds them.  Results are WRONG while a probe is active; the default build has none of this code.
#ifndef GM_TC_PROBES
#define GM_TC_PROBES 0
#endif


namespace gm {

namespace tc {

// GM_TC_PROBES: per-tile timeline of CTA 0 (SM clock) into the buffer GM_TC_TRACE_PTR points at: 8 slots per tile
// [0] MMA: accumulator free  [1] MMA: first stage full  [2] MMA: last k-block issued  [3] epilogue: accumulator full
// [4] epilogue: done  [5] copies: last stage of the tile requested  [6] LSTM epilogue: first 8-unit step loaded  [7] ... done
#if GM_TC_PROBES
#define GM_TRACE(ptr, tile, slot) do { if ((ptr) && blockIdx.x == 0 && (tile) < 64) ((long long*)(ptr))[(tile) * 8 + (slot)] = clock64(); } while (0)
#define GM_TRACE_VAL(ptr, tile, slot, val) do { if ((ptr) && blockIdx.x == 0 && (tile) < 64) ((long long*)(ptr))[(tile) * 8 + (slot)] = (val); } while (0)
#define GM_CLOCK() clock64()
#else
#define GM_TRACE(ptr, tile, slot) do { } while (0)
#define GM_TRACE_VAL(ptr, tile, slot, val) do { } while (0)
#define GM_CLOCK() 0ll
#endif

constexpr int BM = TC_BM, BK = TC_BK, STAGES = 4, ACC_STAGES = 2;
constexpr int EPI_WARPS = 8, PROD_WARPS = 8;
constexpr int MMA_WARP = 16, W_WARP = 17;
constexpr int THREADS = 32 * 18;
constexpr int A_PART_BYTES = BM * BK * 2;  // one bf16 part (hi or lo) of an A stage: 8 KiB
constexpr int SBO_BYTES = BK * 16;         // distance between 8-row groups: 512 B

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (sticky launch error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 22)) __trap();
    }
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// UMMA shared-memory descriptor, K-major, SWIZZLE_NONE: core matrix = 8 rows x 16 bytes stored
// as 128 contiguous bytes; LBO = distance between the two K core matrices of one MMA (128 B),
// SBO = distance between consecutive 8-row groups (BK/8 core matrices = 512 B).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    constexpr uint64_t LBO = 128 >> 4, SBO = SBO_BYTES >> 4;
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | (LBO << 16) | (SBO << 32) | (1ull << 46);
}
// instruction descriptor: D=f32, A=B=bf16, both K-major, M=128, N=BN
__host__ __device__ constexpr uint32_t umma_idesc(int BN) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

#define TMEM_LD16(addr, v)                                                                                        \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];" \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),  \
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),         \
                   "=r"(v[15])                                                                                      \
                 : "r"(addr)                                                                                        \
                 : "memory")
#define TMEM_LD8(addr, v)                                                                              \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"                \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) \
                 : "r"(addr)                                                                              \
                 : "memory")
#define TMEM_LD4(addr, v)                                                                      \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"                    \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])                                 \
                 : "r"(addr)                                                                      \
                 : "memory")
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
// x = hi + lo: hi = bf16(x), lo = bf16(x - hi), two values per packed conversion (6 instructions per pair)
__device__ __forceinline__ void split8(const float (&x)[8], uint4& hi, uint4& lo) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        h[i] = pack_bf16x2(x[2 * i], x[2 * i + 1]);  // low half = x[2i], high half = x[2i+1], round to nearest even
        const float f0 = __uint_as_float(h[i] << 16), f1 = __uint_as_float(h[i] & 0xffff0000u);
        l[i] = pack_bf16x2(x[2 * i] - f0, x[2 * i + 1] - f1);
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}

__device__ __forceinline__ void ld_global_v8(const float* ptr, float* v) {
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(ptr));
}
// coherent (not .nc) form: for data this thread wrote earlier in the same kernel
__device__ __forceinline__ void ld_global_v8_coherent(const float* ptr, float* v) {
    asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(ptr)
                 : "memory");
}
__device__ __forceinline__ void st_global_v8(float* ptr, const float* v) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(ptr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}

// one 8-float chunk of a row; widest vector the alignment allows, zero beyond kvalid
__device__ __forceinline__ void load_chunk(const float* __restrict__ row, int k, int kvalid, int align, float (&x)[8]) {
    if (k + 8 <= kvalid && align >= 8) {
        ld_global_v8(row + k, x);
    } else if (k + 8 <= kvalid && align >= 4) {
        float4 a = __ldg((const float4*)(row + k)), b = __ldg((const float4*)(row + k + 4));
        x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
    } else if (k + 8 <= kvalid && align >= 2) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            float2 a = __ldg((const float2*)(row + k + 2 * i));
            x[2 * i] = a.x; x[2 * i + 1] = a.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++) x[i] = (k + i < kvalid) ? __ldg(row + k + i) : 0.f;
    }
}

// Bare MUFU forms (no range fix-up code around them: the callers clamp the arguments).  The LSTM-cell epilogues work in
// base 2: the packed biases / LayerNorm parameters of the gates are pre-scaled by -log2(e) (i, f, o) and +2 log2(e) (g),
// so a gate costs one FFMA, one FMNMX, one EX2 and one FADD before the shared reciprocal.
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kGateI = -kLog2e, kGateG = 2.f * kLog2e;  // exponent scale of the sigmoid gates / of the tanh gate
constexpr float kExpClamp = 29.f;                         // 1 + 2^29 per factor keeps the four-factor product finite
// (h, c') of one hidden unit from the four gate EXPONENT arguments ei = -log2e*(i), ef, eo (sigmoid gates), eg = 2 log2e*(g)
// and the previous cell value: sig(i), sig(f), sig(o), tanh(g) from four exponentials and ONE reciprocal -- with
// A = 1+2^ei, F = 1+2^ef, O = 1+2^eo, G = 1+2^eg and R = 1/(A F O G): sig(i) = R F O G, sig(f) = R A O G,
// sig(o) = R A F G, tanh(g) = 1 - 2 R A F O.  Saturation error of the clamp < 4e-9.
__device__ __forceinline__ void lstm_unit(float ei, float ef, float eg, float eo, float c_prev, float& c_new, float& sig_o) {
    const float A = 1.f + ex2_approx(fminf(ei, kExpClamp)), F = 1.f + ex2_approx(fminf(ef, kExpClamp));
    const float O = 1.f + ex2_approx(fminf(eo, kExpClamp)), G = 1.f + ex2_approx(fminf(eg, kExpClamp));
    const float AF = A * F, OG = O * G;
    const float R = rcp_approx(AF * OG);
    const float t1 = R * OG, t2 = R * AF;
    const float i_ = t1 * F, f_ = t1 * A;
    sig_o = t2 * G;
    const float g_ = fmaf(t2 * O, -2.f, 1.f);
    c_new = fmaf(f_, c_prev, i_ * g_);
}
__device__ __forceinline__ float tanh_base2(float x) {  // tanh(x) = 1 - 2 / (1 + 2^(2 log2e x))
    return fmaf(rcp_approx(1.f + ex2_approx(fminf(x * kGateG, kExpClamp))), -2.f, 1.f);
}
// fast transcendental forms for the fused LSTM epilogue (abs. error ~1e-7, inside the stated tolerance)
__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float fast_tanh(float x) { return 1.f - __fdividef(2.f, __expf(2.f * x) + 1.f); }

__device__ __forceinline__ int ptr_align_floats(const float* p, int64_t ld) {
    if (p == nullptr) return 1;
    if (((uintptr_t)p & 31) == 0 && (ld & 7) == 0) return 8;
    if (((uintptr_t)p & 15) == 0 && (ld & 3) == 0) return 4;
    if (((uintptr_t)p & 7) == 0 && (ld & 1) == 0) return 2;
    return 1;
}

// byte offset of the 16-byte chunk (row r, k-chunk kc) inside one bf16 part of a [128 x 32] block
__device__ __forceinline__ uint32_t core_off(int r, int kc) { return (uint32_t)((r >> 3) * SBO_BYTES + kc * 128 + (r & 7) * 16); }

template <int BN, int PASSES, int EPI, int NCG>
// 18 warps: 5 on one SM sub-partition (16K registers each) -> 96 registers per thread at most
__global__ void __launch_bounds__(THREADS, 1) linear_tc_kernel(const TcArgs p) {
    constexpr int W_PART_BYTES = BN * BK * 2;  // one bf16 part of a weight stage
    constexpr int STAGE_BYTES = 2 * A_PART_BYTES + 2 * W_PART_BYTES;
    constexpr uint32_t IDESC = umma_idesc(BN);
    constexpr bool LN = EPI == EPI_LNLSTM;
    constexpr int ACC_COLS = LN ? 2 * BN : BN;  // LayerNormLSTM: separate accumulators for x W_ih^T and h W_hh^T
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES + 2 * ACC_STAGES];
    __shared__ uint32_t tmem_base_smem;
    __shared__ float qpart[EPI == EPI_QHEAD ? 2 : 1][EPI == EPI_QHEAD ? NCG - 1 : 1][EPI == EPI_QHEAD ? BM : 1][TC_MAX_ACT];
    // Q-head weights [n_act, N <= 256]: every epilogue thread needs all of them for every tile; from global memory (the L1
    // of this kernel is ~7 KiB) they made the Q-head epilogue the bound of the layer (17 K clocks per tile against 14.5 K
    // of MMAs, tools/tc_trace.py)
    __shared__ __align__(16) float qw_s[EPI == EPI_QHEAD ? TC_MAX_ACT : 1][EPI == EPI_QHEAD ? 256 : 4];
    // NCG == 4 ("wide" epilogue): warps 8-15 are epilogue warps too (no fp32 operands, hence no producers), four
    // column groups per TMEM quadrant
    static_assert(NCG == 2 || NCG == 4, "2 or 4 column groups");
    static_assert(!LN || NCG == 4, "the LayerNormLSTM epilogue is written for four column quarters");
    constexpr int EPI_W = NCG == 4 ? EPI_WARPS + PROD_WARPS : EPI_WARPS;  // NCG == 4: no producers (all operands tile-packed)
    __shared__ float ln_part[1][LN ? BM : 1][4][2];  // per row and column quarter: partial sum / centred sum of squares
    __shared__ float ln_cpart[1][LN ? BM : 1][8];    // per row: the quarters' partial sums of the LN_H pass
    // LayerNormLSTM: the cell's LayerNorm parameters (TcArgs::ln_params: column sums, per-tile affine + biases, ln_cell),
    // 8 KiB at H = 128; every epilogue thread reads them for every tile, as broadcast LDS.128 instead of 32-byte global loads
    __shared__ __align__(16) float ln_prm_s[LN ? 16 * BN : 4];
    __shared__ __align__(16) float ln_cin_s[LN ? 16 * 32 : 1][8];  // per epilogue thread: previous cell state of the tile's 8 units (cp.async)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_u32(&bars[0]), bar_empty = smem_u32(&bars[STAGES]);
    const uint32_t bar_tfull = smem_u32(&bars[2 * STAGES]), bar_tempty = smem_u32(&bars[2 * STAGES + ACC_STAGES]);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) {
            // the copy thread's expect_tx arrive, plus the 256 producer threads when a segment is fp32
            mbar_init(bar_full + 8 * s, 1 + (p.has_prod ? PROD_WARPS * 32 : 0));
            mbar_init(bar_empty + 8 * s, 1);  // tcgen05.commit
        }
        for (int a = 0; a < ACC_STAGES; a++) {
            mbar_init(bar_tfull + 8 * a, 1);           // tcgen05.commit
            mbar_init(bar_tempty + 8 * a, EPI_W * 32);  // every epilogue thread
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == MMA_WARP) {  // TMEM: ACC_STAGES x BN fp32 columns x 128 lanes
        uint32_t dst = smem_u32(&tmem_base_smem);
        uint32_t cols = ACC_STAGES * ACC_COLS;
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (EPI == EPI_QHEAD) {
        for (int i = threadIdx.x; i < p.n_act * p.N; i += THREADS) qw_s[i / p.N][i % p.N] = __ldg(p.q_w + i);
    }
    if (LN) {
        for (int i = threadIdx.x; i < 16 * BN; i += THREADS) ln_prm_s[i] = __ldg(p.ln_params + i);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_smem;

    // Work units: (M tile, N tile), unit u of the grid at mt = u / n_tiles, nt = u % n_tiles; CTA b takes units b, b + grid, ...
    const int n_tiles = p.n_tiles;
    const int n_ctas = (int)gridDim.x, cta = (int)blockIdx.x;
    // LayerNormLSTM: a CTA owns whole M tiles (row statistics couple the N tiles of a row)
    const int my_units = LN ? ((p.m_tiles - cta + n_ctas - 1) / n_ctas) * n_tiles
                            : (p.m_tiles * n_tiles - cta + n_ctas - 1) / n_ctas;
    const int kblocks = p.Kp / BK;
    const int kb_seg1 = p.K0p / BK;  // first k-block of segment 1
    auto unit_mt = [&](int i) { return LN ? cta + (i / n_tiles) * n_ctas : (cta + i * n_ctas) / n_tiles; };
    auto unit_nt = [&](int i) { return LN ? i % n_tiles : (cta + i * n_ctas) % n_tiles; };

    if (NCG == 2 && warp >= EPI_WARPS && warp < EPI_WARPS + PROD_WARPS) {
        // ================= producer: fp32 activations -> bf16 hi/lo core matrices ================
        // Warp pw owns tile rows [16pw, 16pw+16) as two 8-row groups.  Lane = (part = lane/8, r8 = lane%8):
        // one 32-byte load per lane = 8 rows x one 128-byte line per warp instruction, and the 8 lanes of a
        // quarter warp fill the 8 consecutive 16-byte rows of core matrix `part` of their group: conflict-free
        // stores (with r8 = lane/4 a quarter warp hit two bank groups four times).
        if (p.has_prod) {
            const int pw = warp - EPI_WARPS;
            const int r8 = lane & 7, part = lane >> 3;
            const int al0 = ptr_align_floats(p.A0, p.lda0), al1 = ptr_align_floats(p.A1, p.lda1);
            const bool prod0 = p.A0pk == nullptr, prod1 = p.K1 > 0 && p.A1pk == nullptr;
            const uint32_t total_it = (uint32_t)my_units * (uint32_t)kblocks;
            uint8_t* const st_base = smem + (2 * pw) * SBO_BYTES + r8 * 16 + part * 128;

            // fetch the two chunks (row groups g = 0,1) of iteration `it` into registers
            auto fetch = [&](uint32_t it, float (&x)[2][8]) {
#pragma unroll
                for (int g = 0; g < 2; g++)
#pragma unroll
                    for (int i = 0; i < 8; i++) x[g][i] = 0.f;
                if (it >= total_it) return;
                const int kb = (int)(it % kblocks);
                const bool seg1 = kb >= kb_seg1;
                if (seg1 ? !prod1 : !prod0) return;  // this k-block arrives by bulk copy
                const int k = (seg1 ? kb - kb_seg1 : kb) * BK + part * 8;
                const int64_t m0 = (int64_t)unit_mt((int)(it / kblocks)) * BM + pw * 16 + r8;
#pragma unroll
                for (int g = 0; g < 2; g++) {
                    const int64_t m = m0 + 8 * g;
                    if (m < p.M) {
                        if (seg1) load_chunk(p.A1 + m * p.lda1, k, p.K1, al1, x[g]);
                        else load_chunk(p.A0 + m * p.lda0, k, p.K0, al0, x[g]);
                    }
                }
            };
            // register ring of 3 k-blocks: the loads of k-blocks it+1 and it+2 are in flight while k-block
            // `it` is converted (2 x 32-byte loads per thread and k-block -> ~32 KB in flight per SM)
            float buf[3][2][8];
            fetch(0, buf[0]);
            fetch(1, buf[1]);
            for (uint32_t base = 0; base < total_it; base += 3) {
#pragma unroll
                for (int u = 0; u < 3; u++) {
                    const uint32_t it = base + u;
                    if (it >= total_it) break;
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    fetch(it + 2, buf[(u + 2) % 3]);
                    const int kb = (int)(it % kblocks);
                    const bool mine = (kb >= kb_seg1) ? prod1 : prod0;
                    mbar_wait(bar_empty + 8 * s, ph ^ 1);
                    if (mine) {
#pragma unroll
                        for (int g = 0; g < 2; g++) {
                            uint4 hi, lo;
                            split8(buf[u][g], hi, lo);
                            uint8_t* dst = st_base + s * STAGE_BYTES + g * SBO_BYTES;
                            *(uint4*)dst = hi;
                            if (PASSES == 3) *(uint4*)(dst + A_PART_BYTES) = lo;
                        }
                        fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
                    }
                    mbar_arrive(bar_full + 8 * s);
                }
            }
        }
    } else if (warp == W_WARP) {
        // ================= bulk copies: weight tile (+ tile-packed activations) per stage ==============
        if (lane == 0) {
            constexpr uint32_t w_bytes = (PASSES == 3 ? 2 : 1) * W_PART_BYTES;
            constexpr uint32_t a_bytes = (PASSES == 3 ? 2 : 1) * A_PART_BYTES;
            const int kb0_blocks = kb_seg1, kb1_blocks = kblocks - kb_seg1;
            uint32_t it = 0;
            for (int u = 0; u < my_units; u++) {
                const int mt = unit_mt(u), nt = unit_nt(u);
                for (int kb = 0; kb < kblocks; kb++, it++) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    const bool seg1 = kb >= kb_seg1;
                    const uint8_t* apk = seg1 ? p.A1pk : p.A0pk;
                    mbar_wait(bar_empty + 8 * s, ph ^ 1);  // the MMAs on this stage have retired
#if GM_TC_PROBES
                    if (p.a_stages & 8) {  // GM_TC_DEBUG & 8, timing probe: no copies at all (the MMAs run on stale shared memory)
                        mbar_arrive(bar_full + 8 * s);
                        continue;
                    }
#endif
                    mbar_arrive_expect_tx(bar_full + 8 * s, w_bytes + (apk ? a_bytes : 0u));
                    const uint8_t* src = p.Wp + ((size_t)nt * kblocks + kb) * (2 * W_PART_BYTES);
                    bulk_g2s(smem_base + s * STAGE_BYTES + 2 * A_PART_BYTES, src, w_bytes, bar_full + 8 * s);
                    if (apk) {
                        const size_t blk = seg1 ? ((size_t)mt * kb1_blocks + (kb - kb_seg1)) : ((size_t)mt * kb0_blocks + kb);
                        bulk_g2s(smem_base + s * STAGE_BYTES, apk + blk * TC_PK_BLOCK, a_bytes, bar_full + 8 * s);
                    }
                }
                GM_TRACE(p.trace, u, 5);
            }
        }
    } else if (warp == MMA_WARP) {
        // ================= MMA issuer ==================================================================
        if (lane == 0) {
            uint32_t it = 0;
            for (uint32_t tcount = 0; tcount < (uint32_t)my_units; tcount++) {
                const int as = tcount % ACC_STAGES;
                const uint32_t aph = (tcount / ACC_STAGES) & 1;
                mbar_wait(bar_tempty + 8 * as, aph ^ 1);  // epilogue drained this accumulator
                tc_fence_after();
                GM_TRACE(p.trace, tcount, 0);
                const uint32_t d0 = tmem_base + as * ACC_COLS;
                for (int kb = 0; kb < kblocks; kb++, it++) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(bar_full + 8 * s, ph);
                    tc_fence_after();
                    if (kb == 0) GM_TRACE(p.trace, tcount, 1);
                    const uint32_t a_hi = smem_base + s * STAGE_BYTES, a_lo = a_hi + A_PART_BYTES;
                    const uint32_t w_hi = a_hi + 2 * A_PART_BYTES, w_lo = w_hi + W_PART_BYTES;
                    // LayerNormLSTM: segment 1 accumulates into its own BN columns
                    const uint32_t d = d0 + ((LN && kb >= kb_seg1) ? BN : 0);
                    const int kfirst = LN ? (kb != 0 && kb != kb_seg1) : kb;  // 0 on the first k-block of an accumulator
#pragma unroll
                    for (int ks = 0; ks < BK / 16; ks++) {
#if GM_TC_PROBES
                        if ((LN && (p.accumulate & 2)) || (p.a_stages & 2)) break;  // timing probes: no MMAs
#endif
                        const uint32_t o = ks * 256;  // two 128-byte core matrices per K=16 step
                        if (PASSES == 3) {  // small terms first, then hi*hi
                            umma(d, umma_desc(a_lo + o), umma_desc(w_hi + o), IDESC, (kfirst | ks) != 0);
                            umma(d, umma_desc(a_hi + o), umma_desc(w_lo + o), IDESC, 1);
                            umma(d, umma_desc(a_hi + o), umma_desc(w_hi + o), IDESC, 1);
                        } else {
                            umma(d, umma_desc(a_hi + o), umma_desc(w_hi + o), IDESC, (kfirst | ks) != 0);
                        }
                    }
                    umma_commit(bar_empty + 8 * s);  // smem stage reusable once these MMAs retire
                }
                GM_TRACE(p.trace, tcount, 2);
                umma_commit(bar_tfull + 8 * as);  // accumulator complete
            }
        }
    } else {
        // ================= epilogue: TMEM -> registers -> global ==========================================
        // warp e reads TMEM lanes 32*(e%4).. (its hardware quadrant) and the column group e/4 (of NCG).
        const int quad = warp & 3, chalf = warp >> 2;
        const int r = quad * 32 + lane;  // accumulator lane == tile row
        float ln_csum = 0.f;             // LayerNormLSTM: running sum of this thread's pre-LN cell values of the row
        float ln_ma = 0.f, ln_ra = 0.f, ln_mb = 0.f, ln_rb = 0.f;  // ... and the row's LayerNorm statistics of the current M tile
        float* const ln_craw = (float*)(smem + STAGES * STAGE_BYTES);  // LayerNormLSTM only: [BN][BM] behind the ring
        for (uint32_t tcount = 0; tcount < (uint32_t)my_units; tcount++) {
            const int as = tcount % ACC_STAGES;
            const uint32_t aph = (tcount / ACC_STAGES) & 1;
            const int mt = unit_mt((int)tcount), nt = unit_nt((int)tcount);
            const int64_t m = (int64_t)mt * BM + r;
            const bool live = m < p.M;
            if constexpr (LN) {
#if GM_TC_PROBES
                if (p.accumulate & 1) {  // GM_LN_DEBUG timing probe: no epilogue work
                    mbar_wait(bar_tfull + 8 * as, aph);
                    tc_fence_after();
                    tc_fence_before();
                    mbar_arrive(bar_tempty + 8 * as);
                    continue;
                }
#endif
#include "gemm_sm100_lnlstm.inc"
            } else {
#if GM_TC_PROBES
                if ((p.a_stages & 1) && EPI != EPI_QHEAD) {  // GM_TC_DEBUG timing probe: no epilogue work
                    mbar_wait(bar_tfull + 8 * as, aph);
                    tc_fence_after();
                    tc_fence_before();
                    mbar_arrive(bar_tempty + 8 * as);
                    continue;
                }
#endif
#include "gemm_sm100_epilogue.inc"
                if (threadIdx.x == 0) GM_TRACE(p.trace, tcount, 4);
                tc_fence_before();
                mbar_arrive(bar_tempty + 8 * as);
            }
        }
        (void)ln_csum; (void)ln_craw; (void)ln_ma; (void)ln_ra; (void)ln_mb; (void)ln_rb; (void)ln_prm_s; (void)ln_cin_s;
    }

    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        uint32_t cols = ACC_STAGES * ACC_COLS;
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(cols) : "memory");
    }
}

#include "gemm_sm100_encfused.inc"

// -------------------------------------------------------------------------------------------------
// weight packing: fp32 W[N,K] (nn.Linear layout) -> bf16 hi/lo tiles in the UMMA canonical layout
//   out[nt][kb][part][g][kc][r][e]  (g = 8-row group, kc = 8-element K chunk, r = row in group)
// Packed K space: segment 0 = [0,K0p) (K0 real columns, zero padded), segment 1 from K0p.
// lstm != 0: packed row n of tile nt, n = gate*U + jj, comes from source row gate*H + nt*U + jj.
// -------------------------------------------------------------------------------------------------
__global__ void pack_w_kernel(const float* __restrict__ W, int64_t ldw, const float* __restrict__ W1, int64_t ldw1, int N,
                              int K0, int K1, int K0p, int Kp, int BN, int n_tiles, int lstm, int H,
                              uint8_t* __restrict__ out) {
    const int kblocks = Kp / BK;
    const int64_t total = (int64_t)n_tiles * kblocks * BN * (BK / 8);  // one thread per (row, 8-element chunk)
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        int kc = (int)(t % (BK / 8));
        int64_t u = t / (BK / 8);
        int row = (int)(u % BN);
        u /= BN;
        int kb = (int)(u % kblocks);
        int nt = (int)(u / kblocks);
        int n_src;
        if (lstm) {
            int U = BN / 4, gate = row / U, jj = row % U;
            n_src = gate * H + nt * U + jj;
            if (nt * U + jj >= H) n_src = -1;
        } else {
            n_src = nt * BN + row;
        }
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; e++) {
            int k = kb * BK + kc * 8 + e;
            float v = 0.f;
            if (n_src >= 0 && n_src < N) {
                if (k < K0p) {
                    if (k < K0) v = W[(int64_t)n_src * ldw + k];
                } else if (k - K0p < K1) {
                    // segment 1: the tail columns of W, or a second matrix (e.g. weight_hh next to weight_ih)
                    v = W1 ? W1[(int64_t)n_src * ldw1 + (k - K0p)] : W[(int64_t)n_src * ldw + K0 + (k - K0p)];
                }
            }
            x[e] = v;
        }
        uint4 hi, lo;
        split8(x, hi, lo);
        size_t base = ((size_t)nt * kblocks + kb) * (size_t)(2 * BN * BK * 2);
        size_t off = (size_t)(row >> 3) * SBO_BYTES + (size_t)kc * 128 + (size_t)(row & 7) * 16;
        *(uint4*)(out + base + off) = hi;
        *(uint4*)(out + base + (size_t)BN * BK * 2 + off) = lo;
    }
}

// tile-ordered bias (b + b2, zero padded to n_tiles*BN) stored behind the weight tiles
__global__ void pack_bias_kernel(const float* __restrict__ b, const float* __restrict__ b2, int N, int BN, int n_tiles,
                                 int lstm, int H, float* __restrict__ out) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_tiles * BN) return;
    int nt = idx / BN, row = idx % BN, n_src;
    if (lstm) {
        int U = BN / 4, gate = row / U, jj = row % U;
        n_src = (nt * U + jj < H) ? gate * H + nt * U + jj : -1;
    } else {
        n_src = nt * BN + row;
    }
    float v = 0.f;
    if (n_src >= 0 && n_src < N) v = (b ? b[n_src] : 0.f) + (b2 ? b2[n_src] : 0.f);
    // the LSTM epilogue works on base-2 exponent arguments: bias of gate g (tanh) scaled by 2 log2e, the others by -log2e
    if (lstm) v *= (row / (BN / 4) == 2) ? kGateG : kGateI;
    out[idx] = v;
}

// -------------------------------------------------------------------------------------------------
// LayerNormLSTM packing (EPI_LNLSTM, H = 128).  Stage 1 builds, per segment (0: weight_ih, 1: weight_hh), the fp32
// matrix Wx [H + 4H, H] that pack_w_kernel then splits like any linear layer with BN = 128:
//   rows [0, H)       : centred Gram matrix G[n][k] = sum_j (W[j][n] - mean_n)(W[j][k] - mean_k), fp64 accumulation
//   rows H + t*128 + c: weight row gate*H + unit, (half, gate, u) = (c/64, (c%64)/16, c%16), unit = t*32 + half*16 + u
// -------------------------------------------------------------------------------------------------
__global__ void lnlstm_stage_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, int H, float* __restrict__ wx) {
    const int rows = 5 * H;
    const int64_t total = 2ll * rows * H;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(idx % H);
        const int n = (int)((idx / H) % rows);
        const int seg = (int)(idx / ((int64_t)H * rows));
        const float* W = seg ? w_hh : w_ih;
        float v;
        if (n < H) {
            double sn = 0.0, sk = 0.0, snk = 0.0;
            for (int j = 0; j < 4 * H; j++) {
                const double a = W[(int64_t)j * H + n], b = W[(int64_t)j * H + k];
                sn += a; sk += b; snk += a * b;
            }
            v = (float)(snk - sn * sk / (4.0 * H));
        } else {
            const int tt = (n - H) / 128, c = (n - H) % 128;
            const int half = c / 64, gate = (c % 64) / 16, u = c % 16;
            v = W[(int64_t)(gate * H + tt * 32 + half * 16 + u) * H + k];
        }
        wx[idx] = v;
    }
}

// params: [colsum(W_ih) H | colsum(W_hh) H | per chunk tile: ln_input.weight, ln_hidden.weight, ln_input.bias +
// ln_hidden.bias + bias_ih (tile column order) | ln_cell.weight H | ln_cell.bias H]
__global__ void lnlstm_params_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, const float* __restrict__ b_ih,
                                     const float* __restrict__ ln_in_w, const float* __restrict__ ln_in_b,
                                     const float* __restrict__ ln_hid_w, const float* __restrict__ ln_hid_b,
                                     const float* __restrict__ ln_cell_w, const float* __restrict__ ln_cell_b, int H,
                                     float* __restrict__ out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_chunks = H / 32, total = 2 * H + n_chunks * 3 * 128 + 2 * H;
    if (idx >= total) return;
    if (idx < 2 * H) {
        const float* W = idx < H ? w_ih : w_hh;
        const int k = idx % H;
        double s = 0.0;
        for (int j = 0; j < 4 * H; j++) s += W[(int64_t)j * H + k];
        out[idx] = (float)s;
    } else if (idx < 2 * H + n_chunks * 3 * 128) {
        const int e = idx - 2 * H, tt = e / 384, which = (e % 384) / 128, c = e % 128;
        const int half = c / 64, gate = (c % 64) / 16, u = c % 16;
        const int src = gate * H + tt * 32 + half * 16 + u;
        // pre-scaled to base-2 exponent arguments like the LSTM biases (gate 2 = tanh gate)
        const float sc = gate == 2 ? kGateG : kGateI;
        out[idx] = sc * (which == 0 ? ln_in_w[src] : which == 1 ? ln_hid_w[src] : ln_in_b[src] + ln_hid_b[src] + b_ih[src]);
    } else {
        const int e = idx - (2 * H + n_chunks * 3 * 128);
        out[idx] = e < H ? ln_cell_w[e] : ln_cell_b[e - H];
    }
}

}  // namespace tc

// -------------------------------------------------------------------------------------------------
int tc_pick_bn(int N, int epi) {
    if (epi == EPI_LSTM || epi == EPI_QHEAD) return 256;
    if (epi == EPI_LNLSTM) return 128;
    return N <= 128 ? 128 : 256;
}

static int64_t lnlstm_param_floats(int H) { return 2 * H + (H / 32) * 3 * 128 + 2 * H; }

TcShape tc_shape(int N, int K0, int K1, int epi, int H) {
    TcShape s;
    s.BN = tc_pick_bn(N, epi);
    s.K0p = (int)round_up(K0, tc::BK);  // segment 1 starts on a k-block boundary
    s.Kp = s.K0p + (int)round_up(K1, tc::BK);
    s.n_tiles = (epi == EPI_LSTM) ? ceil_div(H, s.BN / 4) : (epi == EPI_LNLSTM) ? 1 + H / 32 : ceil_div(N, s.BN);
    s.w_bytes = (int64_t)s.n_tiles * (s.Kp / tc::BK) * 2 * s.BN * tc::BK * 2;
    s.packed_bytes = round_up(s.w_bytes + (int64_t)s.n_tiles * s.BN * 4, 256);
    if (epi == EPI_LNLSTM)  // weights | LN parameters | fp32 staging of the two [5H, H] source matrices
        s.packed_bytes = round_up(s.w_bytes + round_up(lnlstm_param_floats(H) * 4, 256) + 2ll * 5 * H * H * 4, 256);
    return s;
}

int tc_pack_lnlstm(const float* w_ih, const float* w_hh, const float* b_ih, const float* ln_in_w, const float* ln_in_b,
                   const float* ln_hid_w, const float* ln_hid_b, const float* ln_cell_w, const float* ln_cell_b, int H, void* out,
                   cudaStream_t s) {
    GM_CHECK_ARG(H == 128, "fused LayerNormLSTM cell is built for hidden == 128, got %d", H);
    GM_CHECK_ARG(w_ih && w_hh && b_ih && ln_in_w && ln_in_b && ln_hid_w && ln_hid_b && ln_cell_w && ln_cell_b,
                 "LayerNormLSTM cell parameters missing");
    TcShape sh = tc_shape(4 * H, H, H, EPI_LNLSTM, H);
    float* params = (float*)((char*)out + sh.w_bytes);
    float* wx = (float*)((char*)params + round_up(lnlstm_param_floats(H) * 4, 256));
    tc::lnlstm_stage_kernel<<<148 * 4, 256, 0, s>>>(w_ih, w_hh, H, wx);
    GM_LAUNCH_CHECK();
    tc::lnlstm_params_kernel<<<ceil_div((int)lnlstm_param_floats(H), 256), 256, 0, s>>>(w_ih, w_hh, b_ih, ln_in_w, ln_in_b, ln_hid_w,
                                                                                         ln_hid_b, ln_cell_w, ln_cell_b, H, params);
    GM_LAUNCH_CHECK();
    int64_t total = (int64_t)sh.n_tiles * (sh.Kp / tc::BK) * sh.BN * (tc::BK / 8);
    int blocks = (int)std::min<int64_t>((total + 255) / 256, 148 * 8);
    tc::pack_w_kernel<<<blocks, 256, 0, s>>>(wx, H, wx + (int64_t)5 * H * H, H, 5 * H, H, H, sh.K0p, sh.Kp, sh.BN, sh.n_tiles, 0, H,
                                             (uint8_t*)out);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int tc_pack_weights(const float* W, int64_t ldw, const float* W1, int64_t ldw1, const float* bias, const float* bias2, int N,
                    int K0, int K1, int epi, int H, void* out, cudaStream_t s) {
    TcShape sh = tc_shape(N, K0, K1, epi, H);
    int64_t total = (int64_t)sh.n_tiles * (sh.Kp / tc::BK) * sh.BN * (tc::BK / 8);
    int blocks = (int)std::min<int64_t>((total + 255) / 256, 148 * 8);
    tc::pack_w_kernel<<<blocks, 256, 0, s>>>(W, ldw, W1, ldw1, N, K0, K1, sh.K0p, sh.Kp, sh.BN, sh.n_tiles, epi == EPI_LSTM,
                                             H, (uint8_t*)out);
    GM_LAUNCH_CHECK();
    tc::pack_bias_kernel<<<ceil_div(sh.n_tiles * sh.BN, 256), 256, 0, s>>>(bias, bias2, N, sh.BN, sh.n_tiles, epi == EPI_LSTM, H,
                                                                          (float*)((char*)out + sh.w_bytes));
    GM_LAUNCH_CHECK();
    return GM_OK;
}

template <int BN, int PASSES, int EPI, int NCG = 2>
static int launch_tc(TcArgs a, cudaStream_t s) {
    constexpr int smem = tc::STAGES * (2 * tc::A_PART_BYTES + 2 * BN * tc::BK * 2) +
                         (EPI == EPI_LNLSTM ? BN * tc::BM * 4 : 0);  // + pre-LN cell values of one M tile
    static bool configured = false;
    auto kern = tc::linear_tc_kernel<BN, PASSES, EPI, NCG>;
    if (!configured) {
        GM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        configured = true;
    }
#if GM_TC_PROBES
    {
        static int dbg = -1;
        if (dbg < 0) { const char* e = getenv("GM_TC_DEBUG"); dbg = e ? atoi(e) : 0; }
        a.a_stages = dbg;  // the field is unused by this kernel otherwise
        static long long trace_ptr = -1;
        if (trace_ptr < 0) { const char* e = getenv("GM_TC_TRACE_PTR"); trace_ptr = e ? strtoll(e, nullptr, 0) : 0; }
        static int trace_epi = -2;
        if (trace_epi == -2) { const char* e = getenv("GM_TC_TRACE_EPI"); trace_epi = e ? atoi(e) : -1; }
        static int trace_kp = -2;  // optional filter: only the layer whose packed K equals this (e.g. 96 = encoder L1 at N = 20)
        if (trace_kp == -2) { const char* e = getenv("GM_TC_TRACE_KP"); trace_kp = e ? atoi(e) : -1; }
        a.trace = (EPI == trace_epi && (trace_kp <= 0 || a.Kp == trace_kp)) ? (void*)trace_ptr : nullptr;
    }
#endif
    // LayerNormLSTM: a CTA owns whole M tiles
    const int units = EPI == EPI_LNLSTM ? a.m_tiles : a.m_tiles * a.n_tiles;
    ProfileScope prof(PROF_TC, s);
    kern<<<std::min(units, kNumSMs), tc::THREADS, smem, s>>>(a);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

// ---- fused encoder layers 1 + 2 for sparse input rows (gemm_sm100_encfused.inc) -----------------------------------
bool enc_fused_ok(int D, int U1, int U2, int math) {
    return math == GM_MATH_BF16X3 && D >= 1 && (U1 % tc::BK) == 0 && U1 >= tc::BK && U2 >= 32 && U2 <= tc::EF_BN && (U2 % tc::BK) == 0 &&
           tc::ef_plan(D).nw >= 3;
}
int64_t enc_fused_w1t_bytes(int U1, int D) { return (int64_t)(U1 / tc::BK) * tc::ef_chunk_bytes(D); }

// D = input width, S static rows (dense [S, D], may be 0 / NULL): the chunks hold D + S rows, or (static_only) the S rows alone
int enc_fused_pack_w1t(const float* W1, const float* b1, int U1, int D, const float* static_rows, int S, int static_only, void* out,
                       cudaStream_t s) {
    tc::ef_pack_w1t_kernel<<<U1 / tc::BK, 256, 0, s>>>(W1, b1, U1, D, static_only ? 0 : D, static_rows, static_rows ? S : 0, (float*)out);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

// the caller's sparse rows [ceil(R/128)*128][24] (12 column indices then 12 values, of which the first 6 are read)
// -> Cpk = act(W2 act(W1 x + b1) + b2) tile-packed [R, U2].  D: rows of the W1^T chunks (input width + static rows)
int enc_fused_launch(const int32_t* sp_rows, int64_t R, int D, const void* w1t, const void* W2p, int U1, int U2, int act, uint8_t* Cpk,
                     cudaStream_t s) {
    GM_CHECK_ARG(sp_rows && w1t && W2p && Cpk && R > 0, "bad fused-encoder arguments");
    GM_CHECK_ARG(act == GM_ACT_LEAKY_RELU, "the fused encoder kernel is built for leaky_relu only");
    GM_CHECK_ARG((((uintptr_t)w1t | (uintptr_t)W2p | (uintptr_t)sp_rows) & 15) == 0 && ((uintptr_t)Cpk & 127) == 0,
                 "fused-encoder buffers must be 16 / 128-byte aligned");
    const int m_tiles = (int)((R + tc::BM - 1) / tc::BM);
    const tc::EfPlan plan = tc::ef_plan(D);
    GM_CHECK_ARG(plan.nw >= 3, "fused-encoder chunk of %d rows does not fit in shared memory", D);
    const int smem = plan.smem;
    static int configured = 0;
    if (configured < smem) {
        GM_CUDA(cudaFuncSetAttribute(tc::enc_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        configured = smem;
    }
    const TcShape sh = tc_shape(U2, U1, 0, EPI_LINEAR, 0);
    GM_CHECK_ARG(sh.BN == tc::EF_BN || U2 <= 128, "unexpected layer-2 tile");
    tc::EncFusedArgs a{};
    a.sp = sp_rows; a.w1t = (const uint8_t*)w1t; a.Wp = (const uint8_t*)W2p;
    a.bias_tile = (const float*)((const uint8_t*)W2p + sh.w_bytes);
    a.Cpk = Cpk; a.M = R; a.D = D; a.U1 = U1; a.U2 = U2; a.act = act; a.m_tiles = m_tiles;
    a.nw = plan.nw; a.na = plan.na;
#if GM_TC_PROBES
    {
        static long long trace_ptr = -1;
        if (trace_ptr < 0) { const char* e = getenv("GM_TC_TRACE_PTR"); trace_ptr = e ? strtoll(e, nullptr, 0) : 0; }
        static int trace_epi = -2;
        if (trace_epi == -2) { const char* e = getenv("GM_TC_TRACE_EPI"); trace_epi = e ? atoi(e) : -1; }
        a.trace = trace_epi == 9 ? (void*)trace_ptr : nullptr;
    }
#endif
    const int grid = std::min(m_tiles, kNumSMs);
    ProfileScope prof(PROF_TC, s);
    tc::enc_fused_kernel<<<grid, tc::THREADS, smem, s>>>(a);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int tc_launch(TcArgs a, int math, int epi, cudaStream_t s) {
    if (a.M <= 0) return GM_OK;
    TcShape sh = tc_shape(a.N, a.K0, a.K1, epi, a.H);
    a.K0p = sh.K0p;
    a.Kp = sh.Kp;
    a.n_tiles = sh.n_tiles;
    a.m_tiles = (int)((a.M + tc::BM - 1) / tc::BM);
    GM_CHECK_ARG(((uintptr_t)a.Wp & 255) == 0, "packed weights must be 256-byte aligned");
    a.bias_tile = (const float*)(a.Wp + sh.w_bytes);
    GM_CHECK_ARG((a.A0 != nullptr) != (a.A0pk != nullptr), "segment 0 needs exactly one of fp32 / tile-packed source");
    GM_CHECK_ARG(a.K1 == 0 || ((a.A1 != nullptr) != (a.A1pk != nullptr)), "segment 1 needs exactly one of fp32 / tile-packed source");
    GM_CHECK_ARG(a.A0pk == nullptr || ((a.K0 % tc::BK) == 0 && ((uintptr_t)a.A0pk & 127) == 0),
                 "tile-packed segment 0: K %% 32 and 128-byte alignment");
    GM_CHECK_ARG(a.K1 == 0 || a.A1pk == nullptr || ((a.K1 % tc::BK) == 0 && ((uintptr_t)a.A1pk & 127) == 0),
                 "tile-packed segment 1: K %% 32 and 128-byte alignment");
    a.has_prod = (a.A0 != nullptr) || (a.K1 > 0 && a.A1 != nullptr);
    if (epi == EPI_LNLSTM) {
        GM_CHECK_ARG(a.H == 128 && a.K0 == 128 && a.K1 == 128, "fused LayerNormLSTM cell needs hidden == 128 and two 128-wide segments");
        GM_CHECK_ARG(a.A0pk && a.A1pk, "fused LayerNormLSTM cell takes tile-packed operands only (its producer warps run the epilogue)");
        GM_CHECK_ARG(a.c_in && a.h_out && a.c_out && (a.ldc_in & 7) == 0 && (a.ldh & 7) == 0 && (a.ldco & 7) == 0 &&
                         (((uintptr_t)a.c_in | (uintptr_t)a.h_out | (uintptr_t)a.c_out) & 31) == 0 && ((uintptr_t)a.Hpk & 127) == 0,
                     "fused LayerNormLSTM epilogue needs 32-byte aligned state rows");
        a.ln_params = (const float*)(a.Wp + sh.w_bytes);
#if GM_TC_PROBES
        {
            static int dbg = -1;
            if (dbg < 0) { const char* e = getenv("GM_LN_DEBUG"); dbg = e ? atoi(e) : 0; }
            a.accumulate = dbg;
        }
#endif
        return launch_tc<128, 3, EPI_LNLSTM, 4>(a, s);  // always the three-pass product (SURVEY 7.4: LN amplifies rounding)
    }
    if (epi == EPI_LSTM) {
        GM_CHECK_ARG(a.H % 64 == 0, "fused LSTM epilogue needs hidden %% 64 == 0, got %d", a.H);
        GM_CHECK_ARG((a.ldc_in & 7) == 0 && (a.ldh & 7) == 0 && (a.ldco & 7) == 0 &&
                         (((uintptr_t)a.c_in | (uintptr_t)a.h_out | (uintptr_t)a.c_out) & 31) == 0 && ((uintptr_t)a.Hpk & 127) == 0,
                     "fused LSTM epilogue needs 32-byte aligned state rows");
    } else if (epi == EPI_QHEAD) {
        GM_CHECK_ARG(a.N <= 256 && (a.N & 3) == 0 && a.q_w && a.q_b && a.act_out && a.n_act >= 1 && a.n_act <= TC_MAX_ACT &&
                         ((uintptr_t)a.q_w & 15) == 0 && !a.accumulate,
                     "fused Q head needs a last hidden layer of <= 256 units (multiple of 4) and <= %d actions", TC_MAX_ACT);
    } else {
        GM_CHECK_ARG(a.C != nullptr || a.Cpk != nullptr, "no output");
        GM_CHECK_ARG(a.Cpk == nullptr || ((a.N % tc::BK) == 0 && ((uintptr_t)a.Cpk & 127) == 0 && !a.accumulate),
                     "tile-packed output needs N %% 32 == 0 and 128-byte alignment");
        GM_CHECK_ARG(!a.accumulate || a.C != nullptr, "accumulate needs an fp32 output");
    }
    const int passes = math == GM_MATH_BF16 ? 1 : 3;
    // all operands tile-packed: the producer warps have nothing to do and run the epilogue too (4 epilogue warps per
    // scheduler overlap MUFU and FP32 work better: GEMM time per step 0.69 -> 0.67 ms)
    if (!a.has_prod && passes == 3) {
        if (epi == EPI_LSTM) return launch_tc<256, 3, EPI_LSTM, 4>(a, s);
        if (epi == EPI_QHEAD) return launch_tc<256, 3, EPI_QHEAD, 4>(a, s);  // Q head: 4 column groups of 64, partials summed through smem
        if (epi == EPI_LINEAR) return sh.BN == 128 ? launch_tc<128, 3, EPI_LINEAR, 4>(a, s) : launch_tc<256, 3, EPI_LINEAR, 4>(a, s);
    }
    if (epi == EPI_LSTM) return passes == 3 ? launch_tc<256, 3, EPI_LSTM>(a, s) : launch_tc<256, 1, EPI_LSTM>(a, s);
    if (epi == EPI_QHEAD) return passes == 3 ? launch_tc<256, 3, EPI_QHEAD>(a, s) : launch_tc<256, 1, EPI_QHEAD>(a, s);
    if (sh.BN == 128) return passes == 3 ? launch_tc<128, 3, EPI_LINEAR>(a, s) : launch_tc<128, 1, EPI_LINEAR>(a, s);
    return passes == 3 ? launch_tc<256, 3, EPI_LINEAR>(a, s) : launch_tc<256, 1, EPI_LINEAR>(a, s);
}

// ---- generic entry used by gm_linear and the unfused layers: packs W into `ws`, then runs -------------
int64_t linear_tc_workspace_bytes(int64_t, int N, int K, int) { return tc_shape(N, K, 0, EPI_LINEAR, 0).packed_bytes + 256; }

int linear_tc(const LinearArgs& l, int math, void* ws, int64_t ws_bytes, cudaStream_t s) {
    TcShape sh = tc_shape(l.N, l.K, 0, EPI_LINEAR, 0);
    char* wsa = (char*)round_up((int64_t)ws, 256);
    GM_CHECK_ARG(ws != nullptr && ws_bytes - (wsa - (char*)ws) >= sh.packed_bytes,
                 "tensor-core linear needs %lld workspace bytes, got %lld", (long long)sh.packed_bytes + 256, (long long)ws_bytes);
    int rc = tc_pack_weights(l.W, l.ldw, nullptr, 0, l.bias, l.bias2, l.N, l.K, 0, EPI_LINEAR, 0, wsa, s);
    if (rc) return rc;
    TcArgs a{};
    a.A0 = l.A; a.lda0 = l.lda; a.K0 = l.K;
    a.Wp = (const uint8_t*)wsa;
    a.C = l.C; a.ldc = l.ldc; a.act = l.act; a.accumulate = l.accumulate;
    a.M = l.M; a.N = l.N;
    return tc_launch(a, math, EPI_LINEAR, s);
}

}  // namespace gm
