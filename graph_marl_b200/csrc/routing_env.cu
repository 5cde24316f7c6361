// routing_env.cu -- batched Routing environment for sm_100a.
//
// One warp owns one environment instance: it pulls the packed env record from HBM into
// shared memory, replays the reference's two order-dependent packet loops with
// warp-level "ordered by key" rounds (lanes = packets; per-edge / per-node fp64 running
// sums are accumulated in packet-id order so every load, congestion decision and
// observation field is bit-identical to the Python reference), writes the record back,
// and then builds the dense agent / node observations in a shared-memory staging tile
// that is zero-filled, scattered with the few non-zero fields per row and pushed to HBM
// with one cp.async.bulk (TMA bulk) store per tile.
//
// Reference semantics: src/env/routing.py:119-144 (reset_packet), :160-178 (reset),
// :187-235 (node obs), :256-267 (node-agent matrix), :269-358 (agent obs), :360-520 (step),
// :522-539 (agent adjacency).  SURVEY.md Appendix A is the distilled spec.
#include "common.cuh"

#include <algorithm>

namespace gm {

struct RoutingLayout {
    int off_load, off_i32, off_vis, off_mask, stride, VW;
    // per-warp shared memory carve-up
    int sm_scratch, sm_stage, sm_per_warp, stage_floats;
};

static RoutingLayout make_layout(int N, int A, int E, int stage_bytes, int stages = 1) {
    RoutingLayout L;
    L.VW = (N + 31) / 32;
    L.off_load = 8 * A;
    L.off_i32 = L.off_load + 8 * E;
    L.off_vis = L.off_i32 + 4 * 8 * A;
    L.off_mask = L.off_vis + 4 * A * L.VW;
    L.stride = (int)round_up(L.off_mask + 4 * A, 16);
    // scratch: tl f64[N] | cnt i32[N] | rew f32[A] | looped u8[A]
    L.sm_scratch = L.stride;
    int scratch = 8 * N + 4 * N + 4 * A + A;
    L.sm_stage = (int)round_up(L.sm_scratch + scratch, 16);
    L.stage_floats = stage_bytes / 4;
    L.sm_per_warp = (int)round_up(L.sm_stage + stages * (stage_bytes + 32), 16);  // per env: record + scratch + staging tile(s)
    return L;
}

enum { MODE_RESET = 0, MODE_STEP = 1, MODE_OBSERVE = 2 };

// -DGM_ROUTING_PROBES=1 (GM_NVCC_EXTRA): per-env SM-clock stamps at the phase boundaries of the step kernel, read back
// with gm_routing_probe_read (tools/env_only.py).  The default build contains none of this.
#ifdef GM_ROUTING_PROBES
constexpr int PROBE_ENVS = 16384, PROBE_N = 10;
__device__ long long g_probe[PROBE_ENVS][PROBE_N];
#define GM_PROBE(k)                                                                      \
    do {                                                                                 \
        if (MODE == MODE_STEP && lane == 0 && b < PROBE_ENVS) g_probe[b][k] = clock64(); \
    } while (0)
#else
#define GM_PROBE(k) do {} while (0)
#endif
#ifndef GM_ROUTING_MIN_CTAS
#define GM_ROUTING_MIN_CTAS 7
#endif
constexpr int WARPS_PER_CTA = 4;

// Lanes with `valid` run fn() in ascending lane order among lanes that share `key`
// (different keys proceed in the same round).  This reproduces the sequential
// "for i in range(n_data)" update order of routing.py for state that is keyed by edge
// or node id, without serialising independent keys.
template <class F>
__device__ __forceinline__ void ordered_by_key(bool valid, int key, int lane, F fn) {
    unsigned any = __ballot_sync(FULL, valid);
    if (any == 0) return;
    unsigned grp = __match_any_sync(FULL, valid ? key : (-1 - lane));
    int rank = __popc(grp & ((1u << lane) - 1u));
    int maxrank = __reduce_max_sync(FULL, valid ? rank : 0);
    for (int r = 0; r <= maxrank; r++) {
        if (valid && rank == r) fn();
        __syncwarp();
    }
}

struct EnvView {
    double* size;
    double* load;
    int *now, *target, *edge, *time, *ttl, *spw, *start, *steps;
    uint32_t* vis;
    uint8_t* mask;
    double* tl;
    int* cnt;
    float* rew;
    uint8_t* looped;
};

__device__ __forceinline__ EnvView make_view(uint8_t* sm, const RoutingLayout& L, int A, int N) {
    EnvView v;
    v.size = (double*)sm;
    v.load = (double*)(sm + L.off_load);
    v.now = (int*)(sm + L.off_i32);
    v.target = v.now + A; v.edge = v.now + 2 * A; v.time = v.now + 3 * A; v.ttl = v.now + 4 * A;
    v.spw = v.now + 5 * A; v.start = v.now + 6 * A; v.steps = v.now + 7 * A;
    v.vis = (uint32_t*)(sm + L.off_vis);
    v.mask = sm + L.off_mask;
    v.tl = (double*)(sm + L.sm_scratch);
    v.cnt = (int*)(sm + L.sm_scratch + 8 * N);
    v.rew = (float*)(sm + L.sm_scratch + 12 * N);
    v.looped = sm + L.sm_scratch + 12 * N + 4 * A;
    return v;
}

// routing.py:119-144 (the load release of :126-127 is done by the caller in id order)
__device__ __forceinline__ void spawn_packet(const EnvView& v, const RoutingLayout& L, int i, int start,
                                             int target, double size, const gm_routing_desc& d,
                                             const int* apsp) {
    v.now[i] = start; v.target[i] = target; v.size[i] = size; v.start[i] = start;
    v.time[i] = 0; v.edge[i] = -1; v.ttl[i] = d.ttl;
    v.spw[i] = apsp[start * d.N + target];
    for (int w = 0; w < L.VW; w++) v.vis[i * L.VW + w] = (w == (start >> 5)) ? (1u << (start & 31)) : 0u;
    if (d.action_mask) {
        *(uint32_t*)(v.mask + 4 * i) = (start != target) ? 1u : 0u;  // [idle forbidden?,0,0,0]
    }
}

// ---- staged dense-row emitter ------------------------------------------------------
// The env's block of `total` floats starting at g (4-byte aligned) is produced tile by
// tile in `stage` (16-byte aligned shared memory, congruent to the global address mod 16
// so that the interior of every tile moves as 16-byte units).
template <class ScatterRows>
__device__ __forceinline__ void emit_f32_block(float* g, int total, int W, float* stage, int stage_floats,
                                               int lane, ScatterRows scatter_rows) {
    int tile_cap = stage_floats - 4;
    for (int f0 = 0; f0 < total; f0 += tile_cap) {
        int nfl = min(tile_cap, total - f0);
        float* gt = g + f0;
        int shift = (int)(((uintptr_t)gt & 15u) >> 2);  // floats
        int span4 = (shift + nfl + 3) >> 2;             // float4 units touched
        float4* st4 = (float4*)stage;
        for (int q = lane; q < span4; q += 32) st4[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        __syncwarp();
        float* s = stage + shift;
        int r0 = f0 / W, r1 = (f0 + nfl - 1) / W;
        // put(): write one value of row r / column c if it falls into this tile
        scatter_rows(r0, r1, [&](int r, int c, float val) {
            int idx = r * W + c - f0;
            if (idx >= 0 && idx < nfl) s[idx] = val;
        });
        // copy out: head (unaligned floats), 16-byte interior, tail
        int head = (4 - shift) & 3;
        if (head > nfl) head = nfl;
        int body4 = (nfl - head) >> 2;
        int tail = nfl - head - 4 * body4;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane < head) gt[lane] = s[lane];
        if (lane < tail) gt[head + 4 * body4 + lane] = s[head + 4 * body4 + lane];
        if (body4 > 0 && lane == 0) {
            uint32_t saddr = (uint32_t)__cvta_generic_to_shared(s + head);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gt + head),
                         "r"(saddr), "r"(body4 * 16)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
        __syncwarp();
    }
}

// ---- int8 matrices with rows of A bytes; a lane owns whole rows, four bytes per store when rows are 4-byte aligned ----
// (a flat per-byte form with a division and three table lookups per byte cost 37 % of the kernel's issue samples).
// Separate functions: they run last, nothing of the kernel's state is live across them, and inlining them pushed
// the step kernel over its 72-register budget.
__device__ __forceinline__ void put_row4(int8_t* row, bool aligned, int A, int j0, uint32_t w) {
    if (aligned) {
        *(uint32_t*)(row + j0) = w;
    } else {
#pragma unroll
        for (int u = 0; u < 4; u++)
            if (j0 + u < A) row[j0 + u] = (int8_t)((w >> (8 * u)) & 0xffu);
    }
}

// agent adjacency (routing.py:522-539): adj[i,j] = node_adj[now_i, now_j]; the lane keeps now_i and its three
// neighbours in registers, now_j comes from shared memory as a broadcast
__device__ __noinline__ void emit_adj_rows(const int* now, const int* __restrict__ nb, int8_t* g, int N, int A, int lane) {
    const bool aligned = (A & 3) == 0 && ((uintptr_t)g & 3u) == 0;
    if (aligned && N <= 32 && ((uintptr_t)now & 15u) == 0) {
        // small graphs: the row's node set {now_i} + neighbours as a 32-bit mask, now_j four at a time (LDS.128)
#pragma unroll 1
        for (int i = lane; i < A; i += 32) {
            const int ni = now[i];
            const uint32_t m = (1u << ni) | (1u << nb[ni * 3]) | (1u << nb[ni * 3 + 1]) | (1u << nb[ni * 3 + 2]);
            uint32_t* gr = (uint32_t*)(g + (size_t)i * A);
#pragma unroll 1
            for (int j0 = 0; j0 < A; j0 += 4) {
                const int4 nj = *(const int4*)(now + j0);
                gr[j0 >> 2] = ((m >> nj.x) & 1u) | (((m >> nj.y) & 1u) << 8) | (((m >> nj.z) & 1u) << 16) | (((m >> nj.w) & 1u) << 24);
            }
        }
        return;
    }
#pragma unroll 1
    for (int i = lane; i < A; i += 32) {
        const int ni = now[i];
        const int n0 = nb[ni * 3], n1 = nb[ni * 3 + 1], n2 = nb[ni * 3 + 2];
#pragma unroll 1
        for (int j0 = 0; j0 < A; j0 += 4) {
            uint32_t w = 0;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int nj = now[min(j0 + u, A - 1)];
                w |= (uint32_t)((nj == ni) | (nj == n0) | (nj == n1) | (nj == n2)) << (8 * u);
            }
            put_row4(g + (size_t)i * A, aligned, A, j0, w);
        }
    }
}

// node-agent matrix (routing.py:256-267): M[n,a] = (now_a == n), lane = node
__device__ __noinline__ void emit_node_agent_rows(const int* now, int8_t* g, int N, int A, int lane) {
    const bool aligned = (A & 3) == 0 && ((uintptr_t)g & 3u) == 0;
    if (aligned && ((uintptr_t)now & 15u) == 0) {
#pragma unroll 1
        for (int n = lane; n < N; n += 32) {
            uint32_t* gr = (uint32_t*)(g + (size_t)n * A);
#pragma unroll 1
            for (int a0 = 0; a0 < A; a0 += 4) {
                const int4 na = *(const int4*)(now + a0);
                gr[a0 >> 2] = (uint32_t)(na.x == n) | ((uint32_t)(na.y == n) << 8) | ((uint32_t)(na.z == n) << 16) | ((uint32_t)(na.w == n) << 24);
            }
        }
        return;
    }
#pragma unroll 1
    for (int n = lane; n < N; n += 32) {
#pragma unroll 1
        for (int a0 = 0; a0 < A; a0 += 4) {
            uint32_t w = 0;
#pragma unroll
            for (int u = 0; u < 4; u++) w |= (uint32_t)(now[min(a0 + u, A - 1)] == n) << (8 * u);
            put_row4(g + (size_t)n * A, aligned, A, a0, w);
        }
    }
}

// WPE = warps per env.  1: one warp owns the env from record load to the last observation byte.  2 (batches that
// leave half of an SM's warp slots empty): the pair shares the env's shared-memory record; warp 0 advances it, then --
// after a 64-thread named barrier -- emits the agent observations and adjacency while warp 1 builds the waiting-packet
// sums, the node observations and the node-agent matrix (each warp has its own staging tile).
// SIMPLE: the common configuration (env_var 1, no action mask, no evaluation extras) compiled
// without the other variants' code: the general kernel is 5.4 K SASS instructions and 16 % of its stall samples were
// instruction fetches (ncu, profiles/r2_env_step_ncu.md).
template <int MODE, int WPE, bool SIMPLE>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, GM_ROUTING_MIN_CTAS)
routing_kernel(const gm_routing_desc d, const gm_routing_io io, const RoutingLayout L) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int role = WPE == 2 ? (warp & 1) : 0;
    const int slot_in_cta = WPE == 2 ? (warp >> 1) : warp;
    const int b = blockIdx.x * (WARPS_PER_CTA / WPE) + slot_in_cta;
    if (b >= d.B) return;  // the env's warp(s) exit together; only pair-wide named barriers are used below
    if (MODE == MODE_RESET && io.env_mask != nullptr && io.env_mask[b] == 0) return;

    const int N = d.N, A = d.A, E = d.E;
    const int env_var = SIMPLE ? 1 : d.env_var;
    const bool use_mask = SIMPLE ? false : (d.action_mask != 0);
    const bool eval_info = SIMPLE ? false : (io.eval_f64 != nullptr);
    const int topo = d.topo_index ? d.topo_index[b] : 0;
    const int* __restrict__ ne = d.node_edges + (size_t)topo * N * 3;
    const int* __restrict__ nb = d.node_nbrs + (size_t)topo * N * 3;
    const int4* __restrict__ ed = (const int4*)d.edges + (size_t)topo * E;
    const int* __restrict__ apsp = d.apsp + (size_t)topo * N * N;

    uint8_t* sm = smem + (size_t)slot_in_cta * L.sm_per_warp;
    EnvView v = make_view(sm, L, A, N);
    uint8_t* gstate = d.state + (size_t)b * L.stride;

    GM_PROBE(0);
    int n_resets = 0;
    // compact replay transition written by this launch (gm_routing_io.ring_*): the env's slot in the ring
    size_t ring_slot = 0;
    if (MODE == MODE_STEP && io.ring_rec)
        ring_slot = (size_t)((io.ring_index + (io.ring_index_dev ? *io.ring_index_dev : 0) + b) % io.ring_capacity);
    if (role == 0) {  // ======== warp 0 of the env: record load, reset / step, write-back ========
    // ---- load the env record ------------------------------------------------------
    // (the first chunk of actions is requested before the record so that both DRAM round trips overlap; every record
    // load of a 128-unit group is in flight before the first store waits -- the plain copy loop serialised three round
    // trips: 3.6 K of a warp's 32 K clocks, tools/env_only.py with the probe build)
    int act_first = 0;
    if (MODE == MODE_STEP && lane < A) act_first = __ldg(io.actions + (size_t)b * A + lane);
    if (MODE != MODE_RESET) {
        const uint4* src = (const uint4*)gstate;
        uint4* dst = (uint4*)sm;
        uint4* ring = (MODE == MODE_STEP && io.ring_rec) ? (uint4*)(io.ring_rec + ring_slot * (size_t)L.stride) : nullptr;
        const int n16 = L.stride / 16;
        for (int q0 = 0; q0 < n16; q0 += 128) {
            uint4 t[4];
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (q0 + 32 * k + lane < n16) t[k] = src[q0 + 32 * k + lane];
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (q0 + 32 * k + lane < n16) {
                    dst[q0 + 32 * k + lane] = t[k];
                    if (ring) ring[q0 + 32 * k + lane] = t[k];  // the transition's record before the step
                }
        }
    } else {
        uint4* dst = (uint4*)sm;
        for (int q = lane; q < L.stride / 16; q += 32) dst[q] = make_uint4(0, 0, 0, 0);
    }
    __syncwarp();
    GM_PROBE(1);

    const bool host_draws = io.draw_start != nullptr;
    const uint64_t pstep = io.philox_step + (io.philox_step_dev ? *io.philox_step_dev : 0ull);
    auto draw = [&](int slot, int& s, int& t, double& z) {
        if (host_draws) {
            s = io.draw_start[(size_t)b * A + slot];
            t = io.draw_target[(size_t)b * A + slot];
            z = io.draw_size[(size_t)b * A + slot];
        } else {
            Philox p((uint32_t)slot, (uint32_t)b, (uint32_t)pstep, (uint32_t)(pstep >> 32),
                     io.philox_seed);
            s = (int)__umulhi(p.r[0], (uint32_t)N);
            t = (int)__umulhi(p.r[1], (uint32_t)N);
            z = u53(p.r[2], p.r[3]);
        }
    };

    if (MODE == MODE_RESET) {
        // routing.py:160-178: agent_steps = 0, every edge load = 0 (record already zeroed),
        // packets 0..A-1 spawned from draw slots 0..A-1
        for (int i = lane; i < A; i += 32) {
            int s, t; double z;
            draw(i, s, t, z);
            spawn_packet(v, L, i, s, t, z, d, apsp);
        }
        n_resets = A;
        __syncwarp();
    }

    if (MODE == MODE_STEP) {
        const int* act = io.actions + (size_t)b * A;
        int blocked = 0, n_looped = 0, n_success = 0, n_dropped = 0;
        if (!SIMPLE && io.sum_packets_per_node) {  // routing.py:384-386: waiting packets seen at the start of the step
            for (int i = lane; i < A; i += 32)
                if (v.edge[i] == -1) atomicAdd(io.sum_packets_per_node + (size_t)b * N + v.now[i], 1);
        }
        // ---- loop 1 (routing.py:380-412): edge admission in packet-id order -------
        for (int c0 = 0; c0 < A; c0 += 32) {
            int i = c0 + lane;
            bool in = i < A;
            int a = in ? (c0 == 0 ? act_first : act[i]) : 0;
            float rew = 0.f;
            uint8_t lp = 0;
            bool want = in && v.edge[i] == -1 && a != 0;
            int t = -1, dst = -1;
            if (want) {
                int nw = v.now[i];
                t = ne[nw * 3 + a - 1];
                dst = nb[nw * 3 + a - 1];
            }
            ordered_by_key(want, t, lane, [&]() {
                double l = v.load[t], s = v.size[i];
                if (d.congestion && (l + s > 1.0)) {
                    rew = -0.2f;  // np.float32(0) - 0.2
                    blocked++;
                } else {
                    v.edge[i] = t;
                    v.time[i] = ed[t].z;
                    v.load[t] = l + s;
                    v.now[i] = dst;
                    uint32_t* w = &v.vis[i * L.VW + (dst >> 5)];
                    uint32_t bit = 1u << (dst & 31);
                    if (*w & bit) lp = 1; else *w |= bit;
                }
            });
            if (in) { v.rew[i] = rew; v.looped[i] = lp; v.steps[i] += 1; }  // :371 agent_steps += 1
        }
        __syncwarp();
        GM_PROBE(2);
        if (eval_info) {  // routing.py:414-441, between the two loops
            for (int i = lane; i < A; i += 32) {
                if (v.edge[i] != -1 && io.sum_packets_per_edge) atomicAdd(io.sum_packets_per_edge + (size_t)b * E + v.edge[i], 1);
                if (io.packet_sizes) io.packet_sizes[(size_t)b * A + i] = v.size[i];
                if (io.packet_dist) io.packet_dist[(size_t)b * A + i] = apsp[v.now[i] * N + v.target[i]];
            }
            if (lane == 0) {  // sequential fp64 sums in edge / packet id order, like the python loops
                double tel = 0.0, tps = 0.0;
                int occ = 0, on_edges = 0;
                for (int e = 0; e < E; e++) { tel += v.load[e]; occ += v.load[e] > 0.0; }
                for (int i = 0; i < A; i++) { tps += v.size[i]; on_edges += v.edge[i] != -1; }
                io.eval_f64[2 * (size_t)b] = tel; io.eval_f64[2 * (size_t)b + 1] = tps;
                if (io.eval_i32) { io.eval_i32[2 * (size_t)b] = occ; io.eval_i32[2 * (size_t)b + 1] = on_edges; }
            }
            __syncwarp();
        }
        // ---- loop 2 (routing.py:444-491): timers, arrival, drop, delivery, respawn --
        int slot_base = 0;
        for (int c0 = 0; c0 < A; c0 += 32) {
            int i = c0 + lane;
            bool in = i < A;
            int e = -1, nw = 0;
            bool arrive = false, drop = false, reached = false, dn = false;
            if (in) {
                int tt = v.ttl[i] - 1;
                v.ttl[i] = tt;
                e = v.edge[i];
                nw = v.now[i];
                if (e != -1) {
                    int tm = v.time[i] - 1;
                    v.time[i] = tm;
                    arrive = tm <= 0;
                }
                drop = (d.ttl > 0) && (tt <= 0);
                bool on_edge_after = (e != -1) && !arrive;
                if (use_mask) {  // :456-469
                    uint32_t m = 0;
                    if (!on_edge_after) {
                        m = 1u;
                        int all = 1;
                        for (int q = 0; q < 3; q++) {
                            int o = nb[nw * 3 + q];
                            uint32_t seen = (v.vis[i * L.VW + (o >> 5)] >> (o & 31)) & 1u;
                            m |= seen << (8 * (q + 1));
                            all += (int)seen;
                        }
                        if (all == 4) drop = true;
                    }
                    *(uint32_t*)(v.mask + 4 * i) = m;
                }
                reached = !on_edge_after && (nw == v.target[i]);
                dn = reached || drop;
            }
            // load release: arrival (:451-453) or reset of a packet that is still in flight (:126-127)
            bool sub = in && (e != -1) && (arrive || dn);
            ordered_by_key(sub, e, lane, [&]() { v.load[e] -= v.size[i]; });
            if (in && (arrive || dn)) v.edge[i] = -1;
            unsigned dmask = __ballot_sync(FULL, dn);
            if (in) {
                float rew = v.rew[i];
                int dl = 0;
                double sp = 0.0;
                if (dn) {
                    rew += reached ? 10.f : -10.f;  // float32 add, :474
                    int st = v.steps[i];
                    dl = st;
                    if (reached) {
                        int opt = max(v.spw[i], 1);
                        sp = (double)st / (double)opt;
                        n_success++;
                    } else {
                        n_dropped++;
                    }
                    v.steps[i] = 0;
                    int slot = slot_base + __popc(dmask & ((1u << lane) - 1u));
                    int s, t; double z;
                    draw(slot, s, t, z);
                    spawn_packet(v, L, i, s, t, z, d, apsp);
                }
                n_looped += v.looped[i];
                size_t o = (size_t)b * A + i;
                if (io.reward) io.reward[o] = rew;
                if (io.done) io.done[o] = dn ? 1 : 0;
                if (io.ring_rec) {
                    const size_t ro = ring_slot * A + i;
                    if (io.ring_reward) io.ring_reward[ro] = rew;
                    if (io.ring_done) io.ring_done[ro] = dn ? 1 : 0;
                    if (io.ring_action) io.ring_action[ro] = (int8_t)act[i];
                }
                if (io.delays) io.delays[o] = dl;
                if (io.arrived) io.arrived[o] = (dn && reached) ? 1 : 0;
                if (io.spr) io.spr[o] = sp;
            }
            slot_base += __popc(dmask);
        }
        n_resets = slot_base;
        __syncwarp();
        if (io.info) {
            int v0 = __reduce_add_sync(FULL, n_looped), v1 = __reduce_add_sync(FULL, n_success);
            int v2 = __reduce_add_sync(FULL, n_dropped), v3 = __reduce_add_sync(FULL, blocked);
            if (lane == 0) {
                int4 w = make_int4(v0, v1, v2, v3);
                *((int4*)io.info + b) = w;
            }
        }
    }

    GM_PROBE(3);
    }  // role 0

    if (WPE == 2) {  // hand the advanced record (shared memory) to the env's second warp
        __syncwarp();
        if (slot_in_cta == 0) asm volatile("bar.sync 1, 64;" ::: "memory");  // literal ids: a register id reserves all 16 barriers
        else asm volatile("bar.sync 2, 64;" ::: "memory");
    }
    const bool do_agent = WPE == 1 || role == 0, do_node = WPE == 1 || role == 1;

    // While the observations are emitted the SM writes at the rate the L2 / HBM write path takes (27 B/clk per SM at
    // config 2, all 28 warps in the same phase); everything below that is pure latency -- the record write-back, the
    // small outputs, the waiting-packet sums -- is therefore issued BETWEEN the bulk stores of the two observation
    // blocks, where it costs nothing, instead of in front of them (probe build: 2.5 K of a warp's 32 K clocks).
    // ---- write the record back + small per-agent outputs (the env's first warp) ----------------------------------
    auto finish_record = [&]() {
    if (MODE != MODE_OBSERVE) {
        uint4* dst = (uint4*)gstate;
        const uint4* src = (const uint4*)sm;
        uint4* ring = (MODE == MODE_STEP && io.ring_rec && io.ring_next_rec) ? (uint4*)(io.ring_next_rec + ring_slot * (size_t)L.stride) : nullptr;
        for (int q = lane; q < L.stride / 16; q += 32) {
            const uint4 t = src[q];
            dst[q] = t;
            if (ring) ring[q] = t;  // the transition's record after the step
        }
        if (MODE == MODE_STEP && io.ring_rec && lane == 0) {
            if (io.ring_topo) io.ring_topo[ring_slot] = topo;
            if (io.ring_episode_done) io.ring_episode_done[ring_slot] = (uint8_t)(io.ring_episode_flag != 0);
        }
        if (io.n_resets && lane == 0) io.n_resets[b] = n_resets;
    }
    if (MODE == MODE_RESET) {  // outputs that only step produces are cleared on reset
        for (int i = lane; i < A; i += 32) {
            size_t o = (size_t)b * A + i;
            if (io.reward) io.reward[o] = 0.f;
            if (io.done) io.done[o] = 0;
            if (io.delays) io.delays[o] = 0;
            if (io.arrived) io.arrived[o] = 0;
            if (io.spr) io.spr[o] = 0.0;
        }
        if (io.info && lane == 0) *((int4*)io.info + b) = make_int4(0, 0, 0, 0);
    }

    // ---- small per-agent outputs --------------------------------------------------------
    if (io.agent_node)
        for (int i = lane; i < A; i += 32) io.agent_node[(size_t)b * A + i] = v.now[i];
    if (!SIMPLE && io.action_mask_out)
        for (int i = lane; i < A; i += 32)
            *((uint32_t*)io.action_mask_out + (size_t)b * A + i) = *(uint32_t*)(v.mask + 4 * i);
    };

    float* stage = (float*)(sm + L.sm_stage + (WPE == 2 && role == 1 ? L.stage_floats * 4 + 32 : 0));

    // waiting packets per node: count and fp64 size sum in packet-id order (routing.py:200-205); needed by
    // the node observations and by the GLOBAL agent observation
    const bool need_wait = ((io.node_obs != nullptr || io.node_sparse != nullptr) && do_node) || (io.obs != nullptr && env_var == 3);
    auto waiting_sums = [&]() {
        for (int j = lane; j < N; j += 32) { v.tl[j] = 0.0; v.cnt[j] = 0; }
        __syncwarp();
        for (int c0 = 0; c0 < A; c0 += 32) {
            int i = c0 + lane;
            bool waiting = (i < A) && v.edge[i] == -1;
            int nw = waiting ? v.now[i] : -1;
            ordered_by_key(waiting, nw, lane, [&]() {
                v.cnt[nw] += 1;
                v.tl[nw] += v.size[i];
            });
        }
        __syncwarp();
    };
    // the node rows once more in sparse form (12 (column, value) slots in a fixed order) for NetMon's fused encoder.
    // An env's block is N x 6 16-byte pieces (3 of columns, 3 of values per row): consecutive lanes write consecutive
    // pieces, so every store instruction of the warp covers 512 contiguous bytes.
    auto emit_node_sparse = [&]() {
        if (!(io.node_sparse && do_node)) return;
        int4* const out = (int4*)(io.node_sparse + (size_t)b * N * 24);
        const int mode = d.node_sparse_static;
        const int dyn = d.T * N;  // mode 2: first dictionary row of the five dynamic fields
        // slot t of row j: (column, value)
        auto slot = [&](int j, int t, int& col, float& val) {
            col = 0;
            val = 0.f;
            if (mode) {
                // the constant part of the row (one-hots, lengths) as ONE entry: column 4N+8 + topology*N + node (mode 1),
                // or everything as indices into the T*N + 5 row dictionary (mode 2)
                if (t == 0) { col = (mode == 2 ? 0 : 4 * N + 8) + topo * N + j; val = 1.f; }
                else if (t == 1) { col = mode == 2 ? dyn : N; val = (float)v.cnt[j]; }
                else if (t == 2) { col = mode == 2 ? dyn + 1 : N + 1; val = (float)v.tl[j]; }
                else if (t < 6) {
                    const int q = t - 3;
                    col = mode == 2 ? dyn + 2 + q : N + 2 + q * (N + 2) + N + 1;
                    val = (float)v.load[ne[j * 3 + q]];
                }
            } else {
                if (t == 0) { col = j; val = 1.f; }
                else if (t == 1) { col = N; val = (float)v.cnt[j]; }
                else if (t == 2) { col = N + 1; val = (float)v.tl[j]; }
                else {
                    const int q = (t - 3) / 3, f = (t - 3) % 3;
                    const int k = ne[j * 3 + q], b2 = N + 2 + q * (N + 2);
                    if (f == 0) { col = b2 + nb[j * 3 + q]; val = 1.f; }
                    else if (f == 1) { col = b2 + N; val = (float)ed[k].z; }
                    else { col = b2 + N + 1; val = (float)v.load[k]; }
                }
            }
        };
        for (int q = lane; q < N * 6; q += 32) {
            const int j = q / 6, part = q % 6, t0 = (part % 3) * 4;
            int c[4];
            float x[4];
#pragma unroll
            for (int i = 0; i < 4; i++) slot(j, t0 + i, c[i], x[i]);
            out[q] = part < 3 ? make_int4(c[0], c[1], c[2], c[3])
                              : make_int4(__float_as_int(x[0]), __float_as_int(x[1]), __float_as_int(x[2]), __float_as_int(x[3]));
        }
    };
    // the GLOBAL agent observation embeds node rows: it needs the sums (and, to keep one code path, the record
    // write-back) first
    const bool early = !SIMPLE && env_var == 3;
    if (early) {
        if (role == 0) finish_record();
        if (need_wait) waiting_sums();
    }
    // non-zero fields of node row j (routing.py:193-234) placed at column offset `base` of row r.  The row's 12
    // fields are split over four lanes: part 0..2 = the node's q-th edge (one-hot, length, load), part 3 = the node's
    // own fields; part < 0 = everything (the GLOBAL agent observation embeds whole node rows).
    auto node_row = [&](int r, int base, int j, int part, auto put) {
        if (part < 0 || part == 3) {
            put(r, base + j, 1.f);
            put(r, base + N, (float)v.cnt[j]);
            put(r, base + N + 1, (float)v.tl[j]);
        }
        for (int q = (part < 0 || part == 3) ? 0 : part; q < ((part < 0) ? 3 : (part == 3 ? 0 : part + 1)); q++) {
            int k = ne[j * 3 + q], o = nb[j * 3 + q];
            int b2 = base + N + 2 + q * (N + 2);
            put(r, b2 + o, 1.f);
            put(r, b2 + N, (float)ed[k].z);
            put(r, b2 + N + 1, (float)v.load[k]);
        }
    };

    // ---- agent observations (routing.py:277-358) ------------------------------------------
    // row = 6N+10 packet/edge fields | env_var 2: 5 fields of up to k neighbouring agents (:328-348)
    //                                | env_var 3: flattened node adjacency + node observations (:271-275,353-354)
    if (io.obs && do_agent) {
        const int W0 = 6 * N + 10;
        const int W = W0 + (env_var == 2 ? 5 * d.k : 0) + (env_var == 3 ? N * N + N * (4 * N + 8) : 0);
        emit_f32_block(io.obs + (size_t)b * A * W, A * W, W, stage, L.stage_floats, lane,
                       [&](int r0, int r1, auto put) {
                           // four lanes per row (8 rows per pass): the ~16 fields of a row are written by four lanes
                           // side by side instead of one lane after the other (a tile holds 7-9 rows at N = 20)
                           const int part = lane & 3;
                           for (int i = r0 + (lane >> 2); i <= r1; i += 8) {
                               const int nw = v.now[i];
                               if (part == 3) {
                                   const int e = v.edge[i];
                                   put(i, nw, 1.f);
                                   put(i, N + v.target[i], 1.f);
                                   if (e != -1) {
                                       put(i, 2 * N, 1.f);
                                       int4 ee = ed[e];
                                       int prev = (ee.x == nw) ? ee.y : ee.x;
                                       put(i, 2 * N + 1 + prev, 1.f);
                                   }
                                   put(i, 3 * N + 3, (float)i);
                               } else {
                                   const int q = part;
                                   int k = ne[nw * 3 + q], o = nb[nw * 3 + q];
                                   int base = 3 * N + 4 + q * (N + 2);
                                   put(i, base + o, 1.f);
                                   put(i, base + N, (float)ed[k].z);
                                   put(i, base + N + 1, (float)v.load[k]);
                                   if (q == 0) put(i, 3 * N + 1, (float)v.time[i]);
                                   if (q == 1) put(i, 3 * N + 2, (float)v.size[i]);
                               }
                               if (env_var == 2 && part == 3) {
                                   int count = 0;
                                   for (int j = 0; j < A && count < d.k; j++) {
                                       if (j == i) continue;
                                       int nj = v.now[j];
                                       if (nj == nw || nb[nw * 3] == nj || nb[nw * 3 + 1] == nj || nb[nw * 3 + 2] == nj) {
                                           int base = W0 + 5 * count;
                                           put(i, base, (float)nj);
                                           put(i, base + 1, (float)v.target[j]);
                                           put(i, base + 2, (float)v.edge[j]);
                                           put(i, base + 3, (float)v.size[j]);
                                           put(i, base + 4, (float)i);
                                           count++;
                                       }
                                   }
                                   for (; count < d.k; count++)
                                       for (int q = 0; q < 5; q++) put(i, W0 + 5 * count + q, -1.f);
                               } else if (env_var == 3) {
                                   for (int j = part; j < N; j += 4) {
                                       put(i, W0 + j * N + j, 1.f);
                                       for (int q = 0; q < 3; q++) put(i, W0 + j * N + nb[j * 3 + q], 1.f);
                                       node_row(i, W0 + N * N + j * (4 * N + 8), j, -1, put);
                                   }
                               }
                           }
                       });
    }

    if (do_agent) GM_PROBE(4);
    if (!early) {
        if (role == 0) finish_record();
        GM_PROBE(5);
        if (need_wait) waiting_sums();
    }
    emit_node_sparse();
    if (do_node) GM_PROBE(6);
    // ---- node observations (routing.py:193-234), row width 4N+8 ------------------------
    if (io.node_obs && do_node) {
        const int W = 4 * N + 8;
        emit_f32_block(io.node_obs + (size_t)b * N * W, N * W, W, stage, L.stage_floats, lane,
                       [&](int r0, int r1, auto put) {
                           for (int j = r0 + (lane >> 2); j <= r1; j += 8) node_row(j, 0, j, lane & 3, put);
                       });
    }

    if (do_node) GM_PROBE(7);
    if (io.adj && do_agent) emit_adj_rows(v.now, nb, io.adj + (size_t)b * A * A, N, A, lane);
    if (io.node_agent && do_node) emit_node_agent_rows(v.now, io.node_agent + (size_t)b * N * A, N, A, lane);
    if (do_agent) GM_PROBE(8);
    if (do_node) GM_PROBE(9);
}

static int launch_routing(int mode, const gm_routing_desc* d, const gm_routing_io* io, void* stream) {
    GM_CHECK_ARG(d && io, "null descriptor");
    GM_CHECK_ARG(d->B > 0 && d->N > 0 && d->A > 0, "bad sizes B=%d N=%d A=%d", d->B, d->N, d->A);
    GM_CHECK_ARG(d->E * 2 == d->N * 3, "E must be 3N/2 (3-regular graph), got N=%d E=%d", d->N, d->E);
    GM_CHECK_ARG(d->env_var >= 1 && d->env_var <= 3, "env_var %d", d->env_var);
    GM_CHECK_ARG(d->env_var != 2 || (d->k >= 0 && d->k <= d->A), "k = %d", d->k);
    GM_CHECK_ARG(d->state && d->node_edges && d->node_nbrs && d->edges && d->apsp, "null device table");
    GM_CHECK_ARG(((uintptr_t)d->state & 15) == 0 && ((uintptr_t)d->edges & 15) == 0, "state/edges must be 16-byte aligned");
    GM_CHECK_ARG((io->draw_start == nullptr) == (io->draw_target == nullptr) &&
                     (io->draw_start == nullptr) == (io->draw_size == nullptr),
                 "draw tables must be all set or all NULL");
    GM_CHECK_ARG(mode != MODE_STEP || io->actions, "step needs actions");
    GM_CHECK_ARG(io->info == nullptr || ((uintptr_t)io->info & 15) == 0, "info must be 16-byte aligned");

    // staging tile: 4 KiB per warp keeps >= 7 CTAs (28 warps) resident per SM, so 4096 envs run as ONE wave
    // (measured: 30.8 us vs 37.9 us with 16 KiB tiles; double-buffered tiles were slower, they halve residency)
    const int64_t W_obs = 6 * d->N + 10 + (d->env_var == 2 ? 5 * d->k : 0) + (d->env_var == 3 ? d->N * d->N + d->N * (4 * d->N + 8) : 0);
    int64_t need = 4ll * (int64_t)std::max((int64_t)d->A * W_obs, (int64_t)d->N * (4 * d->N + 8)) + 32;
    int stage_bytes = (int)std::min<int64_t>(4096, round_up(need, 256));
    // the common configuration runs the specialised instance; batches that would leave at least half of the warp slots
    // of every SM empty (2 B <= SMs x 28) give each env two warps (inside the bench step: 23.0 vs 27.1 us per launch at
    // cfg3's 2048 envs, 0.33 vs 0.42 ms at cfg4's 1024 envs against one warp per env)
    const bool simple = d->env_var == 1 && !d->action_mask && io->eval_f64 == nullptr &&
                        io->sum_packets_per_node == nullptr && io->action_mask_out == nullptr;
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = kNumSMs;
    }
    const int wpe = (simple && 2ll * d->B <= (int64_t)sms * WARPS_PER_CTA * GM_ROUTING_MIN_CTAS) ? 2 : 1;
    RoutingLayout L = make_layout(d->N, d->A, d->E, stage_bytes, wpe);
    GM_CHECK_ARG(d->state_stride == L.stride, "state_stride %d != %d", d->state_stride, L.stride);
    while (L.sm_per_warp * (WARPS_PER_CTA / wpe) > 200 * 1024 && stage_bytes > 2048) {
        stage_bytes /= 2;
        L = make_layout(d->N, d->A, d->E, stage_bytes, wpe);
    }
    size_t smem = (size_t)L.sm_per_warp * (WARPS_PER_CTA / wpe);
    GM_CHECK_ARG(smem <= 227 * 1024, "env too large for shared memory (%zu bytes)", smem);

    dim3 grid(ceil_div(d->B, WARPS_PER_CTA / wpe)), block(WARPS_PER_CTA * 32);
    cudaStream_t s = (cudaStream_t)stream;
#define GM_ROUTING_LAUNCH(MODE_, WPE_, SIMPLE_)                                                                              \
    do {                                                                                                                     \
        GM_CUDA(cudaFuncSetAttribute(routing_kernel<MODE_, WPE_, SIMPLE_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        routing_kernel<MODE_, WPE_, SIMPLE_><<<grid, block, smem, s>>>(*d, *io, L);                                          \
    } while (0)
#define GM_ROUTING_VARIANT(MODE_)                                 \
    do {                                                          \
        if (wpe == 2) GM_ROUTING_LAUNCH(MODE_, 2, true);          \
        else if (simple) GM_ROUTING_LAUNCH(MODE_, 1, true);       \
        else GM_ROUTING_LAUNCH(MODE_, 1, false);                  \
    } while (0)
    switch (mode) {
        case MODE_RESET: GM_ROUTING_VARIANT(MODE_RESET); break;
        case MODE_STEP: {
            ProfileScope prof(PROF_ENV, s);
            GM_ROUTING_VARIANT(MODE_STEP);
            break;
        }
        default: GM_ROUTING_VARIANT(MODE_OBSERVE); break;
    }
#undef GM_ROUTING_VARIANT
#undef GM_ROUTING_LAUNCH
    GM_LAUNCH_CHECK();
    return GM_OK;
}

}  // namespace gm

extern "C" {

int gm_routing_state_layout(int32_t N, int32_t A, int32_t E, int32_t* out) {
    GM_CHECK_ARG(out && N > 0 && A > 0 && E > 0, "bad layout query");
    gm::RoutingLayout L = gm::make_layout(N, A, E, 16384);
    out[0] = 0; out[1] = L.off_load; out[2] = L.off_i32; out[3] = L.off_vis; out[4] = L.off_mask;
    out[5] = L.stride; out[6] = L.VW; out[7] = 0;
    return GM_OK;
}

int gm_routing_reset(const gm_routing_desc* d, const gm_routing_io* io, void* stream) {
    return gm::launch_routing(gm::MODE_RESET, d, io, stream);
}
int gm_routing_step(const gm_routing_desc* d, const gm_routing_io* io, void* stream) {
    return gm::launch_routing(gm::MODE_STEP, d, io, stream);
}
int gm_routing_observe(const gm_routing_desc* d, const gm_routing_io* io, void* stream) {
    return gm::launch_routing(gm::MODE_OBSERVE, d, io, stream);
}

#ifdef GM_ROUTING_PROBES
GM_API int gm_routing_probe_read(long long* out, int n_envs) {  // out[n_envs][PROBE_N], synchronises
    GM_CUDA(cudaDeviceSynchronize());
    GM_CUDA(cudaMemcpyFromSymbol(out, gm::g_probe, sizeof(long long) * gm::PROBE_N * n_envs));
    return GM_OK;
}
#endif

}  // extern "C"
