// netmon.cu -- NetMon forward (graph-observation module) for B graphs of N nodes.
//
// Reference: src/model.py:451-631 (NetMon.forward, _update_node_states, _get_neighbor_h,
// _get_global_h, output_to_network_obs), :213-229 (SimpleAggregation), :32-42 (MLP),
// src/layernormlstm.py:24-42.  SURVEY.md Appendix B is the distilled math.
//
// Data layout (HBM, fp32): rows r = b*N + v; state [R, ns*H] with h in the first H floats
// of a node's row and c in the next H (model.py:417-449); adjacency as padded ascending
// neighbour lists (self included when the mask has it) instead of the reference's dense
// [B,N,N] float mask, so aggregation is a sum over short lists and the readout is a pure gather.
//
// Aggregation on the tensor-core path (tile-packed output, see the launch site):
//   aggregate_pk_pipe_kernel  default: persistent CTAs, TMA bulk copies of whole graphs' hidden rows / lists into a
//                             3-stage shared-memory ring (producer warp + mbarriers), sums from shared memory
//   aggregate_pk_kernel       L2 gather, 8 rows x 32 columns per warp; the fallback for graphs that do not fit the ring.
//                             Two more forms measured in round 1 (a 4-row-per-line gather and a single-stage bulk-staged
//                             kernel, both slower, DESIGN.md section 5) were removed in round 2.
#include <cuda_bf16.h>

#include "common.cuh"
#include "gemm_sm100.cuh"
#include "linear_simt.cuh"
#include "netmon_rows.cuh"

namespace gm {

int linear_dispatch(const LinearArgs& a, int math, void* ws, int64_t ws_bytes, cudaStream_t s);  // gemm_dispatch.cu

// ---------------------------------------------------------------------------------------
// adjacency mask -> ascending neighbour lists (one warp per (graph, node) row)
// ---------------------------------------------------------------------------------------
__global__ void adj_to_lists_kernel(const float* __restrict__ mask, int B, int N, int DM, int* __restrict__ nbr,
                                    int* __restrict__ deg, int* __restrict__ overflow) {
    int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= B * N) return;
    const float* m = mask + (size_t)row * N;
    int cnt = 0;
    for (int c0 = 0; c0 < N; c0 += 32) {
        int c = c0 + lane;
        bool on = (c < N) && (m[c] != 0.f);
        unsigned bal = __ballot_sync(FULL, on);
        int pos = cnt + __popc(bal & ((1u << lane) - 1u));
        if (on && pos < DM) nbr[(size_t)row * DM + pos] = c;
        cnt += __popc(bal);
    }
    for (int q = cnt + lane; q < DM; q += 32) nbr[(size_t)row * DM + q] = -1;
    if (lane == 0) {
        deg[row] = min(cnt, DM);
        if (cnt > DM) atomicExch(overflow, 1);
    }
}

// ---------------------------------------------------------------------------------------
// aggregation: M[r] = sum (or mean) of h over the node's list (model.py:213-229)
// one warp per row, lanes stride the H floats as float4
// ---------------------------------------------------------------------------------------
__global__ void aggregate_kernel(const float* __restrict__ h, int64_t ldh, float* __restrict__ M, int B, int N, int H,
                                 const int* __restrict__ nbr, const int* __restrict__ deg, int DM,
                                 const int* __restrict__ list_index, int mean) {
    int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= (int64_t)B * N) return;
    int b = (int)(row / N), v = (int)(row - (int64_t)b * N);
    int li = list_index ? list_index[b] : b;
    const int* lst = nbr + ((size_t)li * N + v) * DM;
    int dg = deg[(size_t)li * N + v];
    const float* hb = h + (size_t)b * N * ldh;
    if ((H & 3) != 0 || (ldh & 3) != 0 || (((uintptr_t)h | (uintptr_t)M) & 15) != 0) {  // small / odd hidden sizes: scalar
        for (int c = lane; c < H; c += 32) {
            float acc = 0.f;
            for (int q = 0; q < dg; q++) acc += hb[(size_t)lst[q] * ldh + c];
            if (mean) acc /= (float)max(dg, 1);
            M[row * H + c] = acc;
        }
        return;
    }
    for (int c = lane * 4; c < H; c += 128) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int q = 0; q < dg; q++) {
            int u = lst[q];
            float4 x = *(const float4*)(hb + (size_t)u * ldh + c);
            acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
        }
        if (mean) { acc.x /= (float)max(dg, 1); acc.y /= (float)max(dg, 1); acc.z /= (float)max(dg, 1); acc.w /= (float)max(dg, 1); }
        *(float4*)(M + row * H + c) = acc;
    }
}

// ---------------------------------------------------------------------------------------
// aggregation for the tensor-core cell: same sum (ascending list order) but written tile-packed
// (bf16 hi/lo core matrices, gemm_sm100.cuh) so the update cell pulls M with bulk copies.
// warp = 8 rows x one 32-column k-block; lane = (r8 = lane/4, part = lane%4) owns 8 floats: every
// warp load touches 8 rows x one 128-byte line, every warp store fills 4 complete 128-byte lines.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t agg_pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}

// A block owns `rows_per_block` consecutive rows (whole graphs when the host can arrange it, a multiple of 8) and its
// warps walk the (8-row group, k-block) tasks of those rows: every 128-byte line of h that the block gathers is
// fetched from L2 once and re-read by the other list members (a row is in ~4 lists) from L1.
// The block first copies the neighbour lists and degrees of its rows into shared memory (one coalesced pass), so a
// task's dependent chain is "hidden rows -> store" instead of "list_index -> list/degree -> hidden rows -> store";
// with ~2.5 task rounds per warp the kernel is bound by that chain, not by bytes (ncu: DRAM 20 %, L2 18 %).
constexpr int AGG_THREADS = 256;
__global__ void __launch_bounds__(AGG_THREADS) aggregate_pk_kernel(const float* __restrict__ h, int64_t ldh, uint8_t* __restrict__ Mpk,
                                                                   int B, int N, int H, const int* __restrict__ nbr,
                                                                   const int* __restrict__ deg, int DM,
                                                                   const int* __restrict__ list_index, int mean, int write_lo,
                                                                   int rows_per_block) {
    extern __shared__ int agg_lists[];  // lists i32[rows_per_block][DM] | degrees i32[rows_per_block]
    const int lane = threadIdx.x & 31;
    const int kbs = H / TC_BK;
    const int64_t R = (int64_t)B * N;
    const int64_t row0 = (int64_t)blockIdx.x * rows_per_block;
    const int tasks = (rows_per_block >> 3) * kbs;
    int* s_deg = agg_lists + rows_per_block * DM;
    for (int t = threadIdx.x; t < rows_per_block * DM; t += (int)blockDim.x) {
        const int r = t / DM, q = t - r * DM;
        const int64_t row = row0 + r;
        int val = 0;
        if (row < R) {
            const unsigned row32 = (unsigned)row;
            const int b = (int)(row32 / (unsigned)N), v = (int)(row32 - (unsigned)b * (unsigned)N);
            const size_t node = (size_t)(list_index ? list_index[b] : b) * N + v;
            val = nbr[node * DM + q];
            if (q == 0) s_deg[r] = deg[node];
        }
        agg_lists[t] = val;
    }
    __syncthreads();
    for (int t = threadIdx.x >> 5; t < tasks; t += (int)(blockDim.x >> 5)) {
    const int rl = (t / kbs) * 8 + (lane >> 2);
    const int64_t row = row0 + rl;
    const int kb = t % kbs, part = lane & 3;
    if (row >= R) continue;
    const unsigned row32 = (unsigned)row;  // the host checks B*N < 2^31
    const int b = (int)(row32 / (unsigned)N);
    const int* lst = agg_lists + rl * DM;
    const int dg = s_deg[rl];
    const float* hb = h + (size_t)b * N * ldh + kb * TC_BK + part * 8;
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = 0.f;
    // first four list entries with all eight 16-byte loads in flight, then the (rare) rest; ascending list order
    {
        float4 a[4], c[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const float4* src = (const float4*)(hb + (size_t)lst[q < dg ? q : 0] * ldh);
            a[q] = q < dg ? __ldg(src) : make_float4(0.f, 0.f, 0.f, 0.f);
            c[q] = q < dg ? __ldg(src + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
            if (q < dg) {
                x[0] += a[q].x; x[1] += a[q].y; x[2] += a[q].z; x[3] += a[q].w;
                x[4] += c[q].x; x[5] += c[q].y; x[6] += c[q].z; x[7] += c[q].w;
            }
        }
    }
    for (int q = 4; q < dg; q++) {
        const float4* src = (const float4*)(hb + (size_t)lst[q] * ldh);
        float4 a = __ldg(src), c = __ldg(src + 1);
        x[0] += a.x; x[1] += a.y; x[2] += a.z; x[3] += a.w; x[4] += c.x; x[5] += c.y; x[6] += c.z; x[7] += c.w;
    }
    if (mean) {
        const float d = (float)max(dg, 1);
#pragma unroll
        for (int i = 0; i < 8; i++) x[i] = x[i] / d;
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        hi[i] = agg_pack2(x[2 * i], x[2 * i + 1]);
        lo[i] = agg_pack2(x[2 * i] - __uint_as_float(hi[i] << 16), x[2 * i + 1] - __uint_as_float(hi[i] & 0xffff0000u));
    }
    const int64_t mt = row / TC_BM;
    const int r = (int)(row - mt * TC_BM);
    uint8_t* dst = Mpk + ((size_t)mt * kbs + kb) * TC_PK_BLOCK + (size_t)(r >> 3) * (TC_BK * 16) + part * 128 + (r & 7) * 16;
    *(uint4*)dst = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if (write_lo) *(uint4*)(dst + TC_BM * TC_BK * 2) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

__device__ __forceinline__ uint32_t agg_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Persistent, pipelined form of the bulk-staged aggregation: one CTA per SM slot walks its row blocks through a 3-stage
// shared-memory ring.  Warp 0 is the producer: lane 0 posts the stage's transaction count and issues the bulk copy of the
// block's hidden rows, all 32 lanes stage the neighbour lists / degrees with ordinary loads (their two dependent latencies
// are the producer's, not the consumers'), then arrive on the stage's "full" mbarrier.  The other warps consume: wait for
// "full", form the sums from shared memory, store the packed tile rows, release the stage on its "empty" mbarrier.  No
// consumer warp ever waits on global memory, so loads of block i+1, i+2 overlap the arithmetic and stores of block i.
constexpr int AGG_STAGES = 3;
constexpr int AGG_PIPE_THREADS = 32 * 11, AGG_PIPE_CTAS = 3;  // 1 producer + 10 consumer warps, 3 CTAs per SM

__device__ __forceinline__ void agg_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (!done) {  // bounded: a protocol bug traps instead of hanging the GPU
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(bar), "r"(parity)
                     : "memory");
        if (!done && ++spins > (1u << 26)) __trap();
    }
}

// HC / DMC: compile-time hidden size / list width (0 = use the runtime arguments); the <128, 4> instance turns the row, tile and
// task index arithmetic of the consumer loop into shifts.
template <int HC, int DMC>
__global__ void __launch_bounds__(AGG_PIPE_THREADS, AGG_PIPE_CTAS) aggregate_pk_pipe_kernel(const float* __restrict__ h, int64_t ldh, uint8_t* __restrict__ Mpk,
                                                                   int B, int N, int H_rt, const int* __restrict__ nbr,
                                                                   const int* __restrict__ deg, int DM_rt,
                                                                   const int* __restrict__ list_index, int mean, int write_lo,
                                                                   int rows_per_block, int n_blocks, int stage_bytes) {
    const int H = HC ? HC : H_rt, DM = DMC ? DMC : DM_rt;
    extern __shared__ __align__(128) uint8_t agg_sm[];  // full[3], empty[3] mbarriers | 3 x (rows f32[rpb][H] | lists | degrees)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_cons = (int)(blockDim.x >> 5) - 1;
    const int kbs = H / TC_BK;
    const int64_t R = (int64_t)B * N;
    const uint32_t full0 = agg_smem_u32(agg_sm), empty0 = full0 + 8 * AGG_STAGES;
    if (threadIdx.x == 0) {
        for (int st = 0; st < AGG_STAGES; st++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(full0 + 8 * st), "r"(32) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(empty0 + 8 * st), "r"(n_cons) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    int it = 0;
    if (warp == 0) {  // ---- producer ----
        // a block holds whole graphs and a graph's lists / degrees are contiguous: when they are 16-byte granular they move
        // as bulk copies too, and the producer touches global memory only for the (prefetched) list index of each graph
        const int gpb = rows_per_block / N;  // graphs per block (<= 32)
        const bool bulk_lists = ((N * DM) & 3) == 0 && (N & 3) == 0 && (((uintptr_t)nbr | (uintptr_t)deg) & 15) == 0;
        auto graph_list = [&](int blk) -> int {  // lane g: list index of the block's g-th graph (or -1)
            const int b = blk * gpb + lane;
            if (blk >= n_blocks || lane >= gpb || b >= B) return -1;
            return list_index ? list_index[b] : b;
        };
        int li_next = graph_list(blockIdx.x);
        for (int blk = blockIdx.x; blk < n_blocks; blk += (int)gridDim.x, it++) {
            const int st = it % AGG_STAGES;
            const uint32_t ph = (uint32_t)(it / AGG_STAGES) & 1u;
            const int li_mine = li_next;
            li_next = graph_list(blk + (int)gridDim.x);
            if (it >= AGG_STAGES) agg_mbar_wait(empty0 + 8 * st, ph ^ 1u);
            uint8_t* base = agg_sm + 128 + (size_t)st * stage_bytes;
            float* s_h = (float*)base;
            int* s_lst = (int*)(base + (size_t)rows_per_block * H * 4);
            int* s_deg = s_lst + rows_per_block * DM;
            const int64_t row0 = (int64_t)blk * rows_per_block;
            const int nrows = (int)min((int64_t)rows_per_block, R - row0);
            const int ngraphs = nrows / N;
            const uint32_t bar = full0 + 8 * st;
            const uint32_t row_bytes = (uint32_t)H * 4u;
            if (lane == 0) {
                const uint32_t tx = row_bytes * (uint32_t)nrows + (bulk_lists ? (uint32_t)ngraphs * (uint32_t)(N * (DM + 1)) * 4u : 0u);
                asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(tx) : "memory");
                if (ldh == H) {
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                     agg_smem_u32(s_h)),
                                 "l"(h + row0 * ldh), "r"(row_bytes * (uint32_t)nrows), "r"(bar)
                                 : "memory");
                } else {
                    for (int r = 0; r < nrows; r++)
                        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                         agg_smem_u32(s_h + (size_t)r * H)),
                                     "l"(h + (row0 + r) * ldh), "r"(row_bytes), "r"(bar)
                                     : "memory");
                }
            }
            __syncwarp();  // the transaction count is posted before any other lane's copy can complete
            if (bulk_lists) {
                if (lane < ngraphs) {
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                     agg_smem_u32(s_lst + lane * N * DM)),
                                 "l"(nbr + (size_t)li_mine * N * DM), "r"((uint32_t)(N * DM) * 4u), "r"(bar)
                                 : "memory");
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                     agg_smem_u32(s_deg + lane * N)),
                                 "l"(deg + (size_t)li_mine * N), "r"((uint32_t)N * 4u), "r"(bar)
                                 : "memory");
                }
            } else {
                for (int g = 0; g < ngraphs; g++) {
                    const int li = __shfl_sync(FULL, li_mine, g);
                    const int* src = nbr + (size_t)li * N * DM;
                    for (int t = lane; t < N * DM; t += 32) s_lst[g * N * DM + t] = src[t];
                    for (int t = lane; t < N; t += 32) s_deg[g * N + t] = deg[(size_t)li * N + t];
                }
            }
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");  // release: the lists are visible
        }
        return;
    }
    // ---- consumers ----
    // A task = one 8-row group x `kc` consecutive k-blocks: the row's list, degree, graph base and tile address are formed
    // once per row and reused for every k-block, divisions are replaced by shifts / a multiply-high, all shared-memory
    // offsets are 32-bit (the first form of this loop issued ~380 instructions per 8x32 unit, 66 % issue-slot utilisation).
    const int cw = warp - 1;
    const int r4 = lane >> 3, c = lane & 7;
    const int kc = (kbs & 1) == 0 ? 2 : 1;
    const int kgroups = kbs / kc;
    const unsigned n_magic = (unsigned)((0x100000000ull + (unsigned)N - 1u) / (unsigned)N);  // rl / N = umulhi(rl, magic), rl < 2^16
    for (int blk = blockIdx.x; blk < n_blocks; blk += (int)gridDim.x, it++) {
        const int st = it % AGG_STAGES;
        const uint32_t ph = (uint32_t)(it / AGG_STAGES) & 1u;
        const uint8_t* base = agg_sm + 128 + (size_t)st * stage_bytes;
        const float* s_h = (const float*)base;
        const int* s_lst = (const int*)(base + (size_t)rows_per_block * H * 4);
        const int* s_deg = s_lst + rows_per_block * DM;
        const int64_t row0 = (int64_t)blk * rows_per_block;
        const int nrows = (int)min((int64_t)rows_per_block, R - row0);
        const int tasks = ((nrows + 7) >> 3) * kgroups;
        agg_mbar_wait(full0 + 8 * st, ph);
        for (int t = cw; t < tasks; t += n_cons) {
            const int grp = t / kgroups;
            const int kb0 = (t - grp * kgroups) * kc;
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int rl = grp * 8 + 4 * j + r4;
                if (rl >= nrows) continue;
                const int dg = s_deg[rl];
                const int gbase = (N == 1 ? rl : (int)__umulhi((unsigned)rl, n_magic)) * N;  // first row of this row's graph
                const int64_t row = row0 + rl;
                const int r = (int)(row & (TC_BM - 1));
                uint8_t* drow = Mpk + (size_t)(row / TC_BM) * kbs * TC_PK_BLOCK + (r >> 3) * (TC_BK * 16) + (c >> 1) * 128 +
                                (r & 7) * 16 + (c & 1) * 8;
                const bool four = DM == 4 && dg == 4;
                int4 l4 = make_int4(0, 0, 0, 0);
                if (four) l4 = *(const int4*)(s_lst + rl * 4);
                for (int kk = 0; kk < kc; kk++) {
                    const int kb = kb0 + kk;
                    const float* hb = s_h + (gbase * H + kb * TC_BK + c * 4);
                    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (four) {  // ascending list order = the reference's bmm row order
                        const float4 e0 = *(const float4*)(hb + l4.x * H), e1 = *(const float4*)(hb + l4.y * H);
                        const float4 e2 = *(const float4*)(hb + l4.z * H), e3 = *(const float4*)(hb + l4.w * H);
                        x.x = (((x.x + e0.x) + e1.x) + e2.x) + e3.x; x.y = (((x.y + e0.y) + e1.y) + e2.y) + e3.y;
                        x.z = (((x.z + e0.z) + e1.z) + e2.z) + e3.z; x.w = (((x.w + e0.w) + e1.w) + e2.w) + e3.w;
                    } else {
                        const int* lst = s_lst + rl * DM;
                        for (int q = 0; q < dg; q++) {
                            const float4 e = *(const float4*)(hb + lst[q] * H);
                            x.x += e.x; x.y += e.y; x.z += e.z; x.w += e.w;
                        }
                    }
                    if (mean) {
                        const float d = (float)max(dg, 1);
                        x.x = x.x / d; x.y = x.y / d; x.z = x.z / d; x.w = x.w / d;
                    }
                    const uint32_t hi0 = agg_pack2(x.x, x.y), hi1 = agg_pack2(x.z, x.w);
                    uint8_t* dst = drow + (size_t)kb * TC_PK_BLOCK;
                    *(uint2*)dst = make_uint2(hi0, hi1);
                    if (write_lo) {
                        const uint32_t lo0 = agg_pack2(x.x - __uint_as_float(hi0 << 16), x.y - __uint_as_float(hi0 & 0xffff0000u));
                        const uint32_t lo1 = agg_pack2(x.z - __uint_as_float(hi1 << 16), x.w - __uint_as_float(hi1 & 0xffff0000u));
                        *(uint2*)(dst + TC_BM * TC_BK * 2) = make_uint2(lo0, lo1);
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(empty0 + 8 * st) : "memory");
    }
}

// rows a block of the aggregation kernels owns: whole graphs, a multiple of 8 rows, about 40-80 rows
static int aggregate_rows_per_block(int N) {
    int g = N;  // smallest whole-graph row count divisible by 8: N * 8 / gcd(N, 8)
    for (int d = 8; d > 1; d >>= 1) if (N % d == 0) { g = N * (8 / d); break; }
    if (N % 2 != 0) g = N * 8;
    int rows = g;
    while (rows < 40) rows += g;
    return rows;
}

// fp32 rows [R, H] (row stride ld) -> tile-packed bf16 hi/lo (the carried hidden state for the LayerNormLSTM
// rnn_obs cell, which takes tile-packed operands only).  Same thread mapping as aggregate_pk_kernel.
__global__ void __launch_bounds__(256) split_pk_kernel(const float* __restrict__ src, int64_t ld, uint8_t* __restrict__ dst_pk,
                                                       int64_t R, int H, int write_lo) {
    const int lane = threadIdx.x & 31;
    const int kbs = H / TC_BK;
    const int64_t gw = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t row = (gw / kbs) * 8 + (lane >> 2);
    const int kb = (int)(gw % kbs), part = lane & 3;
    if (row >= R) return;
    const float4* s4 = (const float4*)(src + row * ld + kb * TC_BK + part * 8);
    const float4 a = __ldg(s4), c = __ldg(s4 + 1);
    const float x[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        hi[i] = agg_pack2(x[2 * i], x[2 * i + 1]);
        lo[i] = agg_pack2(x[2 * i] - __uint_as_float(hi[i] << 16), x[2 * i + 1] - __uint_as_float(hi[i] & 0xffff0000u));
    }
    const int64_t mt = row / TC_BM;
    const int r = (int)(row - mt * TC_BM);
    uint8_t* dst = dst_pk + ((size_t)mt * kbs + kb) * TC_PK_BLOCK + (size_t)(r >> 3) * (TC_BK * 16) + part * 128 + (r & 7) * 16;
    *(uint4*)dst = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if (write_lo) *(uint4*)(dst + TC_BM * TC_BK * 2) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// ---------------------------------------------------------------------------------------
// LSTM pointwise (torch.nn.LSTMCell gate math; gate order i,f,g,o)
// ---------------------------------------------------------------------------------------
__global__ void lstm_pointwise_kernel(const float* __restrict__ gates, const float* __restrict__ c_in, int64_t ldc_in,
                                      float* __restrict__ h_out, int64_t ldh_out, float* __restrict__ c_out,
                                      int64_t ldc_out, int64_t R, int H) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * H) return;
    int64_t r = idx / H;
    int j = (int)(idx - r * H);
    const float* g = gates + r * 4 * H;
    float i_ = sigmoidf_(g[j]), f_ = sigmoidf_(g[H + j]), g_ = tanhf(g[2 * H + j]), o_ = sigmoidf_(g[3 * H + j]);
    float c = f_ * c_in[r * ldc_in + j] + i_ * g_;
    float hh = o_ * tanhf(c);
    h_out[r * ldh_out + j] = hh;
    c_out[r * ldc_out + j] = c;
}

// ---------------------------------------------------------------------------------------
// LayerNormLSTM pointwise (layernormlstm.py:28-42): one warp per row.
//   gates = LN(gi) + LN(gh) + b_ih ; c' = LN(sig(f)*c + sig(i)*tanh(g)) ; h' = sig(o)*tanh(c')
// ---------------------------------------------------------------------------------------
__global__ void lnlstm_pointwise_kernel(const float* __restrict__ gi, const float* __restrict__ gh, gm_cell_params cp,
                                        const float* __restrict__ c_in, int64_t ldc_in, float* __restrict__ h_out,
                                        int64_t ldh_out, float* __restrict__ c_out, int64_t ldc_out, int64_t R, int H) {
    int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (r >= R) return;
    const int G = 4 * H;
    const float* a = gi + r * G;
    const float* b = gh + r * G;
    // two-pass mean / biased variance over the 4H gate pre-activations (eps 1e-5)
    float sa = 0.f, sb = 0.f;
    for (int c = lane; c < G; c += 32) { sa += a[c]; sb += b[c]; }
    float ma = warp_sum(sa) / (float)G, mb = warp_sum(sb) / (float)G;
    float va = 0.f, vb = 0.f;
    for (int c = lane; c < G; c += 32) {
        float da = a[c] - ma, db = b[c] - mb;
        va += da * da; vb += db * db;
    }
    float ra = (1.f / sqrtf(warp_sum(va) / (float)G + 1e-5f)), rb = (1.f / sqrtf(warp_sum(vb) / (float)G + 1e-5f));
    auto gate = [&](int c) {
        return (a[c] - ma) * ra * cp.ln_in_w[c] + cp.ln_in_b[c] + ((b[c] - mb) * rb * cp.ln_hid_w[c] + cp.ln_hid_b[c]) +
               cp.b_ih[c];
    };
    // pre-LN cell state for this lane's hidden units (H <= 32*8 handled by a strided loop, kept in registers)
    float cpre[8];
    float og[8];
    float sc = 0.f;
    int nj = 0;
    for (int j = lane; j < H; j += 32, nj++) {
        float i_ = sigmoidf_(gate(j)), f_ = sigmoidf_(gate(H + j)), g_ = tanhf(gate(2 * H + j));
        og[nj] = sigmoidf_(gate(3 * H + j));
        cpre[nj] = f_ * c_in[r * ldc_in + j] + i_ * g_;
        sc += cpre[nj];
    }
    float mc = warp_sum(sc) / (float)H;
    float vc = 0.f;
    for (int q = 0; q < nj; q++) { float dlt = cpre[q] - mc; vc += dlt * dlt; }
    float rc = (1.f / sqrtf(warp_sum(vc) / (float)H + 1e-5f));
    nj = 0;
    for (int j = lane; j < H; j += 32, nj++) {
        float c = (cpre[nj] - mc) * rc * cp.ln_cell_w[j] + cp.ln_cell_b[j];
        float hh = og[nj] * tanhf(c);
        h_out[r * ldh_out + j] = hh;
        c_out[r * ldc_out + j] = c;
    }
}

// GRU pointwise (torch.nn.GRUCell; gate order r,z,n)
__global__ void gru_pointwise_kernel(const float* __restrict__ gi, const float* __restrict__ gh,
                                     const float* __restrict__ h_in, int64_t ldh_in, float* __restrict__ h_out,
                                     int64_t ldh_out, int64_t R, int H) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * H) return;
    int64_t r = idx / H;
    int j = (int)(idx - r * H);
    const float* a = gi + r * 3 * H;
    const float* b = gh + r * 3 * H;
    float rg = sigmoidf_(a[j] + b[j]);
    float z = sigmoidf_(a[H + j] + b[H + j]);
    float n = tanhf(a[2 * H + j] + rg * b[2 * H + j]);
    float hh = (1.f - z) * n + z * h_in[r * ldh_in + j];
    h_out[r * ldh_out + j] = hh;
}

__global__ void copy_rows_kernel(const float* __restrict__ src, int64_t lds, float* __restrict__ dst, int64_t ldd,
                                 int64_t R, int W) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= R * W) return;
    int64_t r = idx / W;
    int j = (int)(idx - r * W);
    dst[r * ldd + j] = src[r * lds + j];
}

// per-graph mean of h over nodes (model.py:624-627) -> gmean [B,H]
__global__ void global_mean_kernel(const float* __restrict__ h, int64_t ldh, float* __restrict__ gmean, int B, int N,
                                   int H) {
    int b = blockIdx.x;
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
        float s = 0.f;
        for (int v = 0; v < N; v++) s += h[((size_t)b * N + v) * ldh + j];
        gmean[(size_t)b * H + j] = s / (float)N;
    }
}

// ---------------------------------------------------------------------------------------
// readout (model.py:458-469, 582-631): out row = [h_v | gmean_b | last[n_1] .. last[n_maxdeg]]
// neighbours in ascending id order without self, zero padded.  Rows are either all nodes
// (node_out) or the node under each agent (agent_out = node_out[agent_node], the gather form
// of bmm with a one-hot node-agent matrix).  One warp per output row.
// ---------------------------------------------------------------------------------------
__global__ void readout_kernel(const float* __restrict__ h, int64_t ldh, const float* __restrict__ last,
                               int64_t ldl, const float* __restrict__ gmean, const int* __restrict__ nbr,
                               const int* __restrict__ deg, int DM, const int* __restrict__ list_index,
                               const int* __restrict__ agent_node, int rows_per_graph, int B, int N, int H,
                               int use_nbr, int use_glob, int max_degree, float* __restrict__ out, int64_t ldo) {
    int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= (int64_t)B * rows_per_graph) return;
    int b = (int)(row / rows_per_graph);
    int v = agent_node ? agent_node[row] : (int)(row - (int64_t)b * rows_per_graph);
    float* o = out + row * ldo;
    const float* hv = h + ((size_t)b * N + v) * ldh;
    for (int c = lane; c < H; c += 32) o[c] = hv[c];
    int off = H;
    if (use_glob) {
        for (int c = lane; c < H; c += 32) o[off + c] = gmean[(size_t)b * H + c];
        off += H;
    }
    if (use_nbr) {
        int li = list_index ? list_index[b] : b;
        const int* lst = nbr + ((size_t)li * N + v) * DM;
        int dg = deg[(size_t)li * N + v];
        int slot = 0;
        for (int q = 0; q < dg && slot < max_degree; q++) {
            int u = lst[q];
            if (u == v) continue;
            const float* lu = last + ((size_t)b * N + u) * ldl;
            for (int c = lane; c < H; c += 32) o[off + slot * H + c] = lu[c];
            slot++;
        }
        for (; slot < max_degree; slot++)
            for (int c = lane; c < H; c += 32) o[off + slot * H + c] = 0.f;
    }
}

// Agent readout for the tensor-core DQN: the same rows as readout_kernel(agent_node != NULL), written as fp32 rows
// (optional) and / or tile-packed bf16 hi/lo (gemm_sm100.cuh) so the DQN's first layer pulls the graph observation
// with bulk copies.  One warp = 8 agent rows x one H-wide SEGMENT of the row ([h_v | gmean_b | last[n_1] | ...]):
// lane = (r8, part) resolves its segment's source row once (agent_node -> list -> degree is a dependent chain of
// three loads) and then moves the segment's H / 32 k-blocks, 32 bytes in and 2 x 16 bytes out each, all in flight
// together.  A warp instruction reads 8 rows x one 128-byte line and fills 512 contiguous bytes of each plane.
// Measured at config 2 (event time per launch): one warp per (8 rows, ONE k-block) 60 us (the chain is repeated for
// every k-block; issue slots 68 % busy), one warp per 8 WHOLE rows 75 us (too few warps to cover the gather latency).
__global__ void __launch_bounds__(256) readout_agents_pk_kernel(
    const float* __restrict__ h, int64_t ldh, const float* __restrict__ last, int64_t ldl, const float* __restrict__ gmean,
    const int* __restrict__ nbr, const int* __restrict__ deg, int DM, const int* __restrict__ list_index,
    const int* __restrict__ agent_node, int A, int B, int N, int H, int use_nbr, int use_glob, int max_degree,
    float* __restrict__ out, int64_t ldo, uint8_t* __restrict__ out_pk, int write_lo) {
    const int lane = threadIdx.x & 31;
    const int n_seg = 1 + (use_glob ? 1 : 0) + (use_nbr ? max_degree : 0);
    const int kb_per_seg = H / TC_BK, kbs = n_seg * kb_per_seg;
    const unsigned gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const unsigned rg = gw / (unsigned)n_seg;
    const int sg = (int)(gw - rg * (unsigned)n_seg);
    const unsigned rows = (unsigned)B * (unsigned)A;
    const unsigned row = rg * 8 + (lane >> 2);
    const int part = lane & 3;
    if (row >= rows) return;
    const int b = (int)(row / (unsigned)A);
    const int v = agent_node[row];
    const float* src = nullptr;
    if (sg == 0) {
        src = h + ((size_t)b * N + v) * ldh;
    } else if (use_glob && sg == 1) {
        src = gmean + (size_t)b * H;
    } else {
        int slot = sg - 1 - (use_glob ? 1 : 0);
        const int li = list_index ? list_index[b] : b;
        const int* lst = nbr + ((size_t)li * N + v) * DM;
        const int dg = deg[(size_t)li * N + v];
        for (int q = 0; q < dg; q++) {
            const int u = lst[q];
            if (u == v) continue;
            if (slot-- == 0) { src = last + ((size_t)b * N + u) * ldl; break; }
        }
    }
    const unsigned mt = row / TC_BM;
    const int r = (int)(row - mt * TC_BM);
    uint8_t* dst_row = out_pk ? out_pk + ((size_t)mt * kbs + (size_t)sg * kb_per_seg) * TC_PK_BLOCK + (size_t)(r >> 3) * (TC_BK * 16) + part * 128 + (r & 7) * 16 : nullptr;
    float* out_row = out ? out + (int64_t)row * ldo + sg * H + part * 8 : nullptr;
#pragma unroll 4
    for (int k = 0; k < kb_per_seg; k++) {
        float x[8];
        if (src) {
            const float4 a = __ldg((const float4*)(src + k * TC_BK + part * 8)), c = __ldg((const float4*)(src + k * TC_BK + part * 8) + 1);
            x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = c.x; x[5] = c.y; x[6] = c.z; x[7] = c.w;
        } else {
#pragma unroll
            for (int i = 0; i < 8; i++) x[i] = 0.f;
        }
        if (out_row) {
            float4* o = (float4*)(out_row + k * TC_BK);
            o[0] = make_float4(x[0], x[1], x[2], x[3]);
            o[1] = make_float4(x[4], x[5], x[6], x[7]);
        }
        if (dst_row) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                hi[i] = agg_pack2(x[2 * i], x[2 * i + 1]);
                lo[i] = agg_pack2(x[2 * i] - __uint_as_float(hi[i] << 16), x[2 * i + 1] - __uint_as_float(hi[i] & 0xffff0000u));
            }
            uint8_t* dst = dst_row + (size_t)k * TC_PK_BLOCK;
            *(uint4*)dst = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            if (write_lo) *(uint4*)(dst + TC_BM * TC_BK * 2) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
    }
}

// general node->agent mapping (model.py:629-631) for a non-one-hot matrix
__global__ void map_to_agents_kernel(const float* __restrict__ node_out, const float* __restrict__ nam, int B, int N,
                                     int A, int O, float* __restrict__ agent_out) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)B * A * O) return;
    int o = (int)(idx % O);
    int a = (int)((idx / O) % A);
    int b = (int)(idx / ((int64_t)O * A));
    float s = 0.f;
    for (int n = 0; n < N; n++) s += node_out[((size_t)b * N + n) * O + o] * nam[((size_t)b * N + n) * A + a];
    agent_out[idx] = s;
}

int aggregate_rows(const float* h, int64_t ldh, float* M, int B, int N, int H, const int* nbr, const int* deg, int DM,
                   const int* list_index, int mean, cudaStream_t s) {
    aggregate_kernel<<<(unsigned)(((int64_t)B * N + 3) / 4), 128, 0, s>>>(h, ldh, M, B, N, H, nbr, deg, DM, list_index, mean);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int readout_rows(const float* h, int64_t ldh, const float* last, int64_t ldl, const float* gmean, const int* nbr,
                 const int* deg, int DM, const int* list_index, const int* agent_node, int rows_per_graph, int B, int N,
                 int H, int use_nbr, int use_glob, int max_degree, float* out, int64_t ldo, cudaStream_t s) {
    readout_kernel<<<(unsigned)(((int64_t)B * rows_per_graph + 3) / 4), 128, 0, s>>>(
        h, ldh, last, ldl, gmean, nbr, deg, DM, list_index, agent_node, rows_per_graph, B, N, H, use_nbr, use_glob,
        max_degree, out, ldo);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int copy_rows(const float* src, int64_t lds, float* dst, int64_t ldd, int64_t R, int W, cudaStream_t s) {
    copy_rows_kernel<<<(unsigned)((R * W + 255) / 256), 256, 0, s>>>(src, lds, dst, ldd, R, W);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

// ---------------------------------------------------------------------------------------
// packed tensor-core weights: encoder layers, then [W_ih | W_hh] of rnn_obs and rnn_update with
// the gate rows interleaved per 64 hidden units (fused LSTM epilogue)
struct NetmonPack {
    int64_t enc[GM_MAX_LAYERS];
    int64_t obs, upd, total;
    bool fused_cells;
    int cell_epi;  // EPI_LSTM, or EPI_LNLSTM (LayerNormLSTM with hidden 128)
    bool enc_fused;   // encoder layers 1 + 2 can run as one kernel for sparse input rows (gemm_sm100_encfused.inc)
    int64_t w1t;      // offset of layer 1's W^T chunks for that kernel
};

// rows of the fused encoder's W1^T chunks: the input columns (unless the caller's rows index the static rows alone) + static rows
static int chunk_rows(const gm_netmon_params* p) {
    const int n_static = p->static_rows ? p->n_static_rows : 0;
    return (p->static_only ? 0 : p->in_features) + n_static;
}

static NetmonPack pack_layout(const gm_netmon_params* p) {
    NetmonPack L{};
    int64_t off = 0;
    int kin = p->in_features;
    const int H = p->hidden;
    L.cell_epi = p->rnn_type == GM_RNN_LNLSTM ? EPI_LNLSTM : EPI_LSTM;
    L.fused_cells = p->rnn_carryover && ((p->rnn_type == GM_RNN_LSTM && (H % 64) == 0) || (p->rnn_type == GM_RNN_LNLSTM && H == 128));
    for (int l = 0; l < p->n_enc_layers; l++) {
        L.enc[l] = off;
        off += tc_shape(p->enc_units[l], kin, 0, EPI_LINEAR, 0).packed_bytes;
        kin = p->enc_units[l];
    }
    L.obs = L.upd = off;
    if (L.fused_cells) {
        int64_t cell = tc_shape(4 * H, H, H, L.cell_epi, H).packed_bytes;
        L.obs = off;
        L.upd = off + cell;
        off += 2 * cell;
    }
    // fused encoder L1 + L2 (sparse input rows): layer 1 additionally as W^T chunks; layer 2's pack is the normal one
    L.enc_fused = L.fused_cells && p->n_enc_layers >= 2 && p->activation == GM_ACT_LEAKY_RELU &&
                  enc_fused_ok(chunk_rows(p), p->enc_units[0], p->enc_units[1], p->math == GM_MATH_BF16 ? -1 : p->math) &&
                  tc_shape(p->enc_units[1], p->enc_units[0], 0, EPI_LINEAR, 0).n_tiles == 1;
    L.w1t = off;
    if (L.enc_fused) off += round_up(enc_fused_w1t_bytes(p->enc_units[0], chunk_rows(p)), 256);
    L.total = off;
    return L;
}

static int netmon_pack(const gm_netmon_params* p, void* out, cudaStream_t s) {
    GM_CHECK_ARG(!p->static_only || (p->static_rows && p->n_static_rows > 0), "static_only needs static_rows");
    NetmonPack L = pack_layout(p);
    int kin = p->in_features, rc;
    for (int l = 0; l < p->n_enc_layers; l++) {
        if ((rc = tc_pack_weights(p->enc_w[l], kin, nullptr, 0, p->enc_b[l], nullptr, p->enc_units[l], kin, 0, EPI_LINEAR, 0,
                                  (char*)out + L.enc[l], s)))
            return rc;
        kin = p->enc_units[l];
    }
    if (L.enc_fused && (rc = enc_fused_pack_w1t(p->enc_w[0], p->enc_b[0], p->enc_units[0], p->in_features, p->static_rows,
                                                p->static_rows ? p->n_static_rows : 0, p->static_only, (char*)out + L.w1t, s)))
        return rc;
    if (L.fused_cells && L.cell_epi == EPI_LNLSTM) {
        const gm_cell_params* cells[2] = {&p->rnn_obs, &p->rnn_update};
        const int64_t offs[2] = {L.obs, L.upd};
        for (int i = 0; i < 2; i++) {
            const gm_cell_params& c = *cells[i];
            if ((rc = tc_pack_lnlstm(c.w_ih, c.w_hh, c.b_ih, c.ln_in_w, c.ln_in_b, c.ln_hid_w, c.ln_hid_b, c.ln_cell_w, c.ln_cell_b,
                                     p->hidden, (char*)out + offs[i], s)))
                return rc;
        }
    } else if (L.fused_cells) {
        const int H = p->hidden;
        if ((rc = tc_pack_weights(p->rnn_obs.w_ih, H, p->rnn_obs.w_hh, H, p->rnn_obs.b_ih, p->rnn_obs.b_hh, 4 * H, H, H, EPI_LSTM, H,
                                  (char*)out + L.obs, s)))
            return rc;
        if ((rc = tc_pack_weights(p->rnn_update.w_ih, H, p->rnn_update.w_hh, H, p->rnn_update.b_ih, p->rnn_update.b_hh, 4 * H, H, H,
                                  EPI_LSTM, H, (char*)out + L.upd, s)))
            return rc;
    }
    return GM_OK;
}

struct NetmonWs {
    float *act0, *act1, *g0, *g1, *hA, *hB, *cA, *cB, *M, *gmean;
    float* ln_scratch;  // LayerNormLSTM cell: [SMs][128 units x 128 rows] sig(o) of the M tile a CTA works on
    uint8_t *pk0, *pk1, *e_pk, *m_pk, *h_pk0, *h_pk1;  // tile-packed activations of the tensor-core path
    int64_t bytes;
};

static bool tc_math(int math) { return math == GM_MATH_BF16X3 || math == GM_MATH_BF16; }

static NetmonWs carve(const gm_netmon_params* p, int64_t R, int B, void* base) {
    NetmonWs w;
    int H = p->hidden;
    int maxw = H;
    for (int i = 0; i < p->n_enc_layers; i++) maxw = max(maxw, p->enc_units[i]);
    int G = p->rnn_type == GM_RNN_GRU ? 3 * H : 4 * H;
    char* c = (char*)base;
    int64_t off = 0;
    auto take = [&](int64_t floats) {
        float* ptr = (float*)(c + off);
        off += round_up(floats * 4, 256);
        return ptr;
    };
    w.act0 = take(R * maxw); w.act1 = take(R * maxw);
    w.g0 = take(R * G); w.g1 = take(R * G);
    w.hA = take(R * H); w.hB = take(R * H);
    w.cA = take(tc_blocked_floats(R, H)); w.cB = take(tc_blocked_floats(R, H));  // the fused cells keep c blocked (gemm_sm100.cuh)
    w.M = take(R * H);
    w.gmean = take((int64_t)max(B, 1) * H);
    w.pk0 = w.pk1 = w.e_pk = w.m_pk = w.h_pk0 = w.h_pk1 = nullptr;
    w.ln_scratch = nullptr;
    if (tc_math(p->math)) {
        auto take_pk = [&](int width) { return (uint8_t*)take(tc_pk_bytes(R, (int)round_up(width, TC_BK)) / 4 + 64); };
        w.pk0 = take_pk(maxw); w.pk1 = take_pk(maxw);
        w.e_pk = take_pk(H); w.m_pk = take_pk(H); w.h_pk0 = take_pk(H); w.h_pk1 = take_pk(H);
        // LayerNormLSTM cell: one M tile of sig(o) per CTA, parked between the gate tiles and the LN_H pass
        if (p->rnn_type == GM_RNN_LNLSTM) w.ln_scratch = take((int64_t)kNumSMs * TC_BM * 128);
    }
    w.bytes = off + (32 << 20);  // + room for per-call packed weights of the unfused tensor-core layers
    return w;
}

}  // namespace gm

using namespace gm;

extern "C" {

int64_t gm_netmon_workspace_bytes(const gm_netmon_params* p, int64_t rows) {
    if (!p) return 0;
    NetmonWs w = carve(p, rows, (int)rows, nullptr);
    return w.bytes + (tc_math(p->math) ? round_up(pack_layout(p).total, 256) + 256 : 0);
}

int64_t gm_netmon_packed_bytes(const gm_netmon_params* p) { return p ? pack_layout(p).total : 0; }

int gm_netmon_pack_weights(const gm_netmon_params* p, void* packed, int64_t packed_bytes, void* stream) {
    GM_CHECK_ARG(p && packed && ((uintptr_t)packed & 255) == 0, "packed buffer must be a 256-byte aligned device pointer");
    GM_CHECK_ARG(packed_bytes >= pack_layout(p).total, "packed buffer too small");
    return netmon_pack(p, packed, (cudaStream_t)stream);
}

int gm_adj_to_lists(const float* mask, int32_t B, int32_t N, int32_t DM, int32_t* nbr_all, int32_t* deg,
                    int32_t* overflow, void* stream) {
    GM_CHECK_ARG(mask && nbr_all && deg && overflow && B > 0 && N > 0 && DM > 0, "bad adj_to_lists args");
    int rows = B * N;
    adj_to_lists_kernel<<<ceil_div(rows, 4), 128, 0, (cudaStream_t)stream>>>(mask, B, N, DM, nbr_all, deg, overflow);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int gm_netmon_map_to_agents(const float* node_out, const float* node_agent, int32_t B, int32_t N, int32_t A,
                            int32_t O, float* agent_out, void* stream) {
    GM_CHECK_ARG(node_out && node_agent && agent_out, "null pointer");
    int64_t tot = (int64_t)B * A * O;
    map_to_agents_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(node_out, node_agent, B, N, A,
                                                                                         O, agent_out);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

int gm_netmon_forward(const gm_netmon_params* p, int32_t B, int32_t N, const float* node_obs, const int32_t* nbr_all,
                      const int32_t* deg, int32_t DM, const int32_t* list_index, const float* state_in,
                      float* state_out, int32_t max_degree, float* node_out, const int32_t* agent_node, int32_t A,
                      float* agent_out, int64_t agent_out_ld, void* agent_out_pk, const void* state_h_pk_in, void* state_h_pk_out,
                      void* workspace, int64_t workspace_bytes, void* stream) {
    GM_CHECK_ARG(p && node_obs && nbr_all && deg && state_out && workspace, "null pointer");
    GM_CHECK_ARG(B > 0 && N > 0 && DM > 0, "bad sizes");
    const int H = p->hidden, K = p->iterations, L = p->n_enc_layers;
    GM_CHECK_ARG(H > 0 && H <= 256, "hidden size %d: need 1..256", H);
    GM_CHECK_ARG(L >= 1 && L <= GM_MAX_LAYERS && p->enc_units[L - 1] == H, "encoder must end in %d units", H);
    GM_CHECK_ARG(p->rnn_type >= GM_RNN_LSTM && p->rnn_type <= GM_RNN_NONE, "rnn_type %d", p->rnn_type);
    GM_CHECK_ARG(K >= 1 || p->rnn_type == GM_RNN_NONE, "iterations must be >= 1 (model.py:564 fails for 0)");
    GM_CHECK_ARG(max_degree <= DM, "max_degree %d > DM %d", max_degree, DM);
    const bool lstm_like = p->rnn_type == GM_RNN_LSTM || p->rnn_type == GM_RNN_LNLSTM;
    const int ns = lstm_like ? (p->rnn_carryover ? 2 : 4) : (p->rnn_type == GM_RNN_GRU ? (p->rnn_carryover ? 1 : 2) : 1);
    const int S = ns * H;
    const int64_t R = (int64_t)B * N;
    GM_CHECK_ARG(workspace_bytes >= gm_netmon_workspace_bytes(p, R), "workspace too small");
    cudaStream_t s = (cudaStream_t)stream;
    NetmonWs w = carve(p, R, B, workspace);
    void* lin_ws = (char*)workspace + w.bytes - (32 << 20);
    int64_t lin_ws_bytes = workspace_bytes - (w.bytes - (32 << 20));
    const NetmonPack PL = pack_layout(p);
    // LayerNormLSTM amplifies rounding (SURVEY 7.4): its fused tensor-core cell always forms the three-pass product;
    // shapes the fused cell is not built for run in fp32
    const int math = (p->rnn_type == GM_RNN_LNLSTM && !PL.fused_cells) ? GM_MATH_FP32
                     : (p->rnn_type == GM_RNN_LNLSTM && p->math == GM_MATH_BF16) ? GM_MATH_BF16X3 : p->math;
    const bool tc = tc_math(math);
    const char* packed = (const char*)p->packed;
    if (tc && packed == nullptr) {  // no cached pack: build it in the workspace tail
        char* dst = (char*)round_up((int64_t)((char*)workspace + w.bytes), 256);
        int rc = netmon_pack(p, dst, s);
        if (rc) return rc;
        packed = dst;
    }
    GM_CHECK_ARG(!tc || ((uintptr_t)packed & 255) == 0, "packed weights must be 256-byte aligned");

    // zero state when none is given (model.py:480-484)
    const float* st_in = state_in;
    if (!st_in) {
        GM_CUDA(cudaMemsetAsync(state_out, 0, (size_t)R * S * 4, s));
        st_in = state_out;  // read as zeros before it is overwritten (all readers finish first: same stream)
    }

    // ---- encoder MLP (model.py:489): activation after every layer incl. the last ----------
    // Tensor-core path with fused cells: layer outputs stay tile-packed (bf16 hi/lo) and are pulled
    // by the next layer with bulk copies; the last layer feeds the rnn_obs cell the same way.
    const bool fused = tc && PL.fused_cells;
    GM_CHECK_ARG(fused || (state_h_pk_in == nullptr && state_h_pk_out == nullptr),
                 "a tile-packed hidden state is only carried by the fused tensor-core cells");
    GM_CHECK_ARG((((uintptr_t)state_h_pk_in | (uintptr_t)state_h_pk_out) & 127) == 0, "tile-packed state must be 128-byte aligned");
    const float* x = node_obs;
    const uint8_t* xpk = nullptr;
    int64_t ldx = p->in_features;
    int kin = p->in_features;
    int l_first = 0;
    // supplied rows of at most 6 entries (e.g. a static part named as one entry + the dynamic fields) run the fused kernel;
    // with more entries per row it is slower than the two separate layers
    const bool six = p->sparse_input_nnz > 0 && p->sparse_input_nnz <= 6 && p->sparse_rows != nullptr;
    GM_CHECK_ARG(!p->static_only || p->sparse_rows != nullptr, "static_only: the rows must be supplied in sparse form");
    if (fused && PL.enc_fused && six) {
        // layers 1 + 2 in one launch: layer 1 on the CUDA cores inside the producer warps, layer 2 on tcgen05
        uint8_t* ypk = (L == 2) ? w.e_pk : w.pk1;
        int rc = enc_fused_launch(p->sparse_rows, R, chunk_rows(p), packed + PL.w1t, packed + PL.enc[1], p->enc_units[0],
                                  p->enc_units[1], p->activation, ypk, s);
        if (rc) return rc;
        xpk = ypk;
        x = nullptr;
        kin = p->enc_units[1];
        ldx = kin;
        l_first = 2;
    }
    for (int l = l_first; l < L; l++) {
        float* y = (l & 1) ? w.act1 : w.act0;
        int rc;
        if (tc) {
            const int U = p->enc_units[l];
            const bool out_pk = fused && (U % TC_BK) == 0;
            uint8_t* ypk = (l == L - 1) ? w.e_pk : ((l & 1) ? w.pk1 : w.pk0);
            TcArgs a{};
            if (xpk) a.A0pk = xpk; else { a.A0 = x; a.lda0 = ldx; }
            a.K0 = kin;
            a.Wp = (const uint8_t*)packed + PL.enc[l];
            if (out_pk) a.Cpk = ypk; else { a.C = y; a.ldc = U; }
            a.act = p->activation;
            a.M = R; a.N = U;
            rc = tc_launch(a, math, EPI_LINEAR, s);
            xpk = out_pk ? ypk : nullptr;
        } else {
            LinearArgs a{x, ldx, p->enc_w[l], kin, p->enc_b[l], nullptr, y, p->enc_units[l], R, p->enc_units[l], kin,
                         p->activation, 0};
            rc = linear_dispatch(a, math, lin_ws, lin_ws_bytes, s);
        }
        if (rc) return rc;
        x = y; ldx = p->enc_units[l]; kin = p->enc_units[l];
    }
    const float* e = x;  // [R,H] (fp32 path) / xpk (tile-packed path)

    const float* h = e;
    int64_t ldh_cur = H;
    const float* c = nullptr;
    const float* last = nullptr;  // value of h before the final iteration's aggregation (:510-519)
    float* hbuf[2] = {w.hA, w.hB};
    float* cbuf[2] = {w.cA, w.cB};

    if (fused) {
        // ===== fused tensor-core path: one launch per cell.  Gate GEMM [x | h] x [W_ih | W_hh]^T on
        // tcgen05 with the LSTM pointwise as epilogue (gates never touch HBM); x and h arrive
        // tile-packed by bulk copy, the new h leaves both as fp32 (state, readout, aggregation) and
        // tile-packed (next cell). =====
        uint8_t* hpk[2] = {w.h_pk0, w.h_pk1};
        // ldcp / ldcn < 0: that cell-state buffer is one of the workspace's blocked buffers (cA / cB)
        auto cell = [&](int64_t woff, const uint8_t* xin_pk, const float* xin, const uint8_t* hp_pk, const float* hp, int64_t ldhp,
                        const float* cprev, int64_t ldcp, float* hn, int64_t ldhn, float* cn, int64_t ldcn, uint8_t* hn_pk) -> int {
            TcArgs a{};
            if (xin_pk) a.A0pk = xin_pk; else { a.A0 = xin; a.lda0 = H; }
            a.K0 = H;
            if (hp_pk) a.A1pk = hp_pk; else { a.A1 = hp; a.lda1 = ldhp; }
            a.K1 = H;
            a.Wp = (const uint8_t*)packed + woff;
            a.c_in = cprev; a.ldc_in = ldcp < 0 ? H : ldcp; a.c_in_blocked = ldcp < 0;
            a.h_out = hn; a.ldh = ldhn; a.c_out = cn; a.ldco = ldcn < 0 ? H : ldcn; a.c_out_blocked = ldcn < 0;
            a.Hpk = hn_pk;
            a.ln_scratch = w.ln_scratch;
            a.H = H; a.M = R; a.N = 4 * H;
            return tc_launch(a, math, PL.cell_epi, s);
        };
        // rnn_obs (:491): x = encoder output, (h, c) = carried state.  The LayerNormLSTM cell takes
        // tile-packed operands only, so the carried h is split once by a small kernel; otherwise the
        // producer warps split it on the fly.
        const int kbs = H / TC_BK;
        int rc;
        // the carried h as the previous step's last cell left it, tile-packed (state_h_pk_in): the cell then runs with
        // every operand pulled by bulk copies (16 epilogue warps, no producer work); only valid with a given state
        const uint8_t* hpk_in = state_in ? (const uint8_t*)state_h_pk_in : nullptr;
        if (hpk_in && xpk) {
            rc = cell(PL.obs, xpk, e, hpk_in, nullptr, 0, st_in + H, S, hbuf[0], H, cbuf[0], -1, hpk[0]);
        } else if (PL.cell_epi == EPI_LNLSTM) {
            GM_CHECK_ARG(xpk != nullptr, "LayerNormLSTM cells need a tile-packed encoder output");
            const unsigned blocks = (unsigned)((((R + 7) / 8) * kbs + 7) / 8);
            split_pk_kernel<<<blocks, 256, 0, s>>>(st_in, S, hpk[1], R, H, math != GM_MATH_BF16);
            GM_LAUNCH_CHECK();
            rc = cell(PL.obs, xpk, e, hpk[1], nullptr, 0, st_in + H, S, hbuf[0], H, cbuf[0], -1, hpk[0]);
        } else {
            rc = cell(PL.obs, xpk, e, nullptr, st_in, S, st_in + H, S, hbuf[0], H, cbuf[0], -1, hpk[0]);
        }
        if (rc) return rc;
        h = hbuf[0]; c = cbuf[0];
        int cur = 0;
        for (int it = 0; it < K; it++) {  // :509-554
            const bool final_it = it == K - 1;
            if (final_it) last = h;
            {
                ProfileScope prof(PROF_AGG, s);
                const int rpb = aggregate_rows_per_block(N);
                const unsigned agg_blocks = (unsigned)((R + rpb - 1) / rpb);
                const int mean = p->agg_type == GM_AGG_MEAN, write_lo = math != GM_MATH_BF16;
                const int pipe_stage = (int)round_up((int64_t)rpb * H * 4 + (int64_t)rpb * (DM + 1) * (int64_t)sizeof(int), 128);
                const size_t pipe_smem = 128 + (size_t)AGG_STAGES * pipe_stage;
                if (rpb % N == 0 && rpb / N <= 32 && pipe_smem <= 72 * 1024 && ((uintptr_t)h & 15) == 0) {
                    static bool configured = false;
                    if (!configured) {
                        GM_CUDA(cudaFuncSetAttribute(aggregate_pk_pipe_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024));
                        GM_CUDA(cudaFuncSetAttribute(aggregate_pk_pipe_kernel<128, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024));
                        configured = true;
                    }
                    int sms = 148;
                    {
                        int dev = 0;
                        cudaGetDevice(&dev);
                        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
                    }
                    const unsigned grid = std::min<unsigned>(agg_blocks, (unsigned)(sms * AGG_PIPE_CTAS));
                    auto kern = (H == 128 && DM == 4) ? aggregate_pk_pipe_kernel<128, 4> : aggregate_pk_pipe_kernel<0, 0>;
                    kern<<<grid, AGG_PIPE_THREADS, pipe_smem, s>>>(h, H, w.m_pk, B, N, H, nbr_all, deg, DM, list_index, mean, write_lo, rpb,
                                                                  (int)agg_blocks, pipe_stage);
                } else {
                    aggregate_pk_kernel<<<agg_blocks, AGG_THREADS, (size_t)rpb * (DM + 1) * sizeof(int), s>>>(
                        h, H, w.m_pk, B, N, H, nbr_all, deg, DM, list_index, mean, write_lo, rpb);
                }
            }
            GM_LAUNCH_CHECK();
            float* hn = final_it ? state_out : hbuf[cur ^ 1];  // the last cell writes the new state in place (:562-564)
            float* cn = final_it ? state_out + H : cbuf[cur ^ 1];
            int64_t ldn = final_it ? S : H;
            rc = cell(PL.upd, w.m_pk, nullptr, hpk[cur], nullptr, 0, c, -1, hn, ldn, cn, final_it ? ldn : -1,
                      final_it ? (uint8_t*)state_h_pk_out : hpk[cur ^ 1]);
            if (rc) return rc;
            h = hn; c = cn; ldh_cur = ldn; cur ^= 1;
        }
    } else {
    // one recurrent cell: (xin [R,H], h_prev, c_prev) -> (h_new, c_new)
    auto run_cell = [&](const gm_cell_params& cp, const float* xin, int64_t ldxin, const float* hp, int64_t ldhp,
                        const float* cprev, int64_t ldcp, float* hn, int64_t ldhn, float* cn, int64_t ldcn) -> int {
        int rc;
        if (p->rnn_type == GM_RNN_LSTM) {
            LinearArgs a{xin, ldxin, cp.w_ih, H, cp.b_ih, cp.b_hh, w.g0, 4 * H, R, 4 * H, H, -1, 0};
            if ((rc = linear_dispatch(a, math, lin_ws, lin_ws_bytes, s))) return rc;
            LinearArgs b{hp, ldhp, cp.w_hh, H, nullptr, nullptr, w.g0, 4 * H, R, 4 * H, H, -1, 1};
            if ((rc = linear_dispatch(b, math, lin_ws, lin_ws_bytes, s))) return rc;
            int64_t tot = R * H;
            lstm_pointwise_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(w.g0, cprev, ldcp, hn, ldhn, cn, ldcn, R, H);
            GM_LAUNCH_CHECK();
        } else if (p->rnn_type == GM_RNN_LNLSTM) {
            LinearArgs a{xin, ldxin, cp.w_ih, H, nullptr, nullptr, w.g0, 4 * H, R, 4 * H, H, -1, 0};
            if ((rc = linear_dispatch(a, math, lin_ws, lin_ws_bytes, s))) return rc;
            LinearArgs b{hp, ldhp, cp.w_hh, H, nullptr, nullptr, w.g1, 4 * H, R, 4 * H, H, -1, 0};
            if ((rc = linear_dispatch(b, math, lin_ws, lin_ws_bytes, s))) return rc;
            lnlstm_pointwise_kernel<<<(unsigned)((R + 3) / 4), 128, 0, s>>>(w.g0, w.g1, cp, cprev, ldcp, hn, ldhn, cn, ldcn, R, H);
            GM_LAUNCH_CHECK();
        } else {  // GRU
            LinearArgs a{xin, ldxin, cp.w_ih, H, cp.b_ih, nullptr, w.g0, 3 * H, R, 3 * H, H, -1, 0};
            if ((rc = linear_dispatch(a, math, lin_ws, lin_ws_bytes, s))) return rc;
            LinearArgs b{hp, ldhp, cp.w_hh, H, cp.b_hh, nullptr, w.g1, 3 * H, R, 3 * H, H, -1, 0};
            if ((rc = linear_dispatch(b, math, lin_ws, lin_ws_bytes, s))) return rc;
            int64_t tot = R * H;
            gru_pointwise_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(w.g0, w.g1, hp, ldhp, hn, ldhn, R, H);
            GM_LAUNCH_CHECK();
        }
        return GM_OK;
    };

    // ---- rnn_obs (model.py:490-495) -------------------------------------------------------
    int cur = 0, rc;
    if (p->rnn_type != GM_RNN_NONE) {
        // no-carryover keeps (h0,c0) in state columns [0,2H) (model.py:566); those columns of
        // state_out are written at the very end from the ping-pong copy to stay alias-safe.
        if ((rc = run_cell(p->rnn_obs, e, H, st_in, S, lstm_like ? st_in + H : nullptr, S, hbuf[0], H, cbuf[0], H))) return rc;
        h = hbuf[0]; c = cbuf[0]; cur = 0;
    }
    // h0/c0 for the no-carry state live in hbuf[0]/cbuf[0]; keep them untouched in that mode
    const bool nocarry = lstm_like && !p->rnn_carryover;
    const bool gru_nocarry = p->rnn_type == GM_RNN_GRU && !p->rnn_carryover;
    float* h0_keep = nullptr; float* c0_keep = nullptr;
    if (nocarry || gru_nocarry) {
        h0_keep = w.act0; c0_keep = w.act1;  // encoder buffers are free now (e was consumed)
        if ((rc = copy_rows(hbuf[0], H, h0_keep, H, R, H, s))) return rc;
        if (nocarry && (rc = copy_rows(cbuf[0], H, c0_keep, H, R, H, s))) return rc;
    }

    // ---- K x (aggregate, rnn_update) (model.py:509-554) ----------------------------------
    float* none_buf[2] = {w.hA, w.hB};
    for (int it = 0; it < K; it++) {
        if (it == K - 1) last = h;
        if ((rc = aggregate_rows(h, H, w.M, B, N, H, nbr_all, deg, DM, list_index, p->agg_type == GM_AGG_MEAN, s))) return rc;
        if (p->rnn_type == GM_RNN_NONE) {
            // h = M; `last` may alias the previous h buffer, so ping-pong
            float* dst = none_buf[it & 1];
            if ((rc = copy_rows(w.M, H, dst, H, R, H, s))) return rc;
            h = dst;
            continue;
        }
        const float* hp = h; int64_t ldhp = H;
        const float* cpv = c; int64_t ldcp = H;
        if (nocarry && it == 0) { hp = st_in + 2 * H; ldhp = S; cpv = st_in + 3 * H; ldcp = S; }  // :538-539
        if (gru_nocarry && it == 0) { hp = st_in + H; ldhp = S; }                                  // :546-547
        int nxt = cur ^ 1;
        if ((rc = run_cell(p->rnn_update, w.M, H, hp, ldhp, cpv, ldcp, hbuf[nxt], H, cbuf[nxt], H))) return rc;
        h = hbuf[nxt]; c = cbuf[nxt]; cur = nxt;
    }

    // ---- new state (model.py:562-578) ------------------------------------------------------
    if (lstm_like) {
        int o = nocarry ? 2 * H : 0;
        if (nocarry) {
            if ((rc = copy_rows(h0_keep, H, state_out, S, R, H, s))) return rc;
            if ((rc = copy_rows(c0_keep, H, state_out + H, S, R, H, s))) return rc;
        }
        if ((rc = copy_rows(h, H, state_out + o, S, R, H, s))) return rc;
        if ((rc = copy_rows(c, H, state_out + o + H, S, R, H, s))) return rc;
    } else if (gru_nocarry) {
        // model.py:571 stacks (h0, h1) as [2,1,R,H]; _state_reshape_out (:449) then transposes the two LEADING
        // axes only, so the flat state buffer is all of h0 followed by all of h1 (not interleaved per row).
        // Reproduced, not fixed: the next step reads row r as [state0 | state1] = flat[r*2H : (r+1)*2H].
        if ((rc = copy_rows(h0_keep, H, state_out, H, R, H, s))) return rc;
        if ((rc = copy_rows(h, H, state_out + R * H, H, R, H, s))) return rc;
    } else {
        if ((rc = copy_rows(h, H, state_out, S, R, H, s))) return rc;
    }
    }  // unfused path

    // ---- readout (model.py:458-474) ---------------------------------------------------------
    const int use_nbr = p->output_neighbor_hidden, use_glob = p->output_global_hidden;
    if (use_glob) {
        global_mean_kernel<<<B, 128, 0, s>>>(h, ldh_cur, w.gmean, B, N, H);
        GM_LAUNCH_CHECK();
    }
    if (use_nbr && last == nullptr) {  // K <= 0 with rnn none: zeros (:498-499)
        GM_CUDA(cudaMemsetAsync(w.M, 0, (size_t)R * H * 4, s));
        last = w.M;
    }
    const int O = H + (use_glob ? H : 0) + (use_nbr ? max_degree * H : 0);
    if (node_out) {
        int rc = readout_rows(h, ldh_cur, last, H, w.gmean, nbr_all, deg, DM, list_index, nullptr, N, B, N, H, use_nbr,
                              use_glob, max_degree, node_out, O, s);
        if (rc) return rc;
    }
    if (agent_out_pk) {
        GM_CHECK_ARG(agent_node && A > 0 && (H % TC_BK) == 0 && ((uintptr_t)agent_out_pk & 127) == 0 &&
                         (agent_out == nullptr || (agent_out_ld >= O && (agent_out_ld & 3) == 0 && ((uintptr_t)agent_out & 15) == 0)) &&
                         (ldh_cur & 3) == 0,
                     "tile-packed agent readout needs agent_node, hidden %% 32 == 0 and 16-byte aligned rows");
        GM_CHECK_ARG((int64_t)B * A * (O / TC_BK) < (1ll << 31) && (int64_t)B * N < (1ll << 31), "batch too large for the 32-bit row arithmetic of the readout / aggregation kernels");
        int64_t rows = (int64_t)B * A;
        const int n_seg = 1 + (use_glob ? 1 : 0) + (use_nbr ? max_degree : 0);
        const unsigned blocks = (unsigned)((((rows + 7) / 8) * n_seg + 7) / 8);
        {
            ProfileScope prof(PROF_READOUT, s);
            readout_agents_pk_kernel<<<blocks, 256, 0, s>>>(h, ldh_cur, last, (int64_t)H, w.gmean, nbr_all, deg, DM, list_index, agent_node, A,
                                                            B, N, H, use_nbr, use_glob, max_degree, agent_out, agent_out_ld,
                                                            (uint8_t*)agent_out_pk, (int)(math != GM_MATH_BF16));
        }
        GM_LAUNCH_CHECK();
    } else if (agent_out) {
        GM_CHECK_ARG(agent_node && A > 0 && agent_out_ld >= O, "agent readout needs agent_node, A, ld >= %d", O);
        return readout_rows(h, ldh_cur, last, H, w.gmean, nbr_all, deg, DM, list_index, agent_node, A, B, N, H, use_nbr,
                            use_glob, max_degree, agent_out, agent_out_ld, s);
    }
    return GM_OK;
}

}  // extern "C"
