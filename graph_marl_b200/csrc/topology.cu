// topology.cu -- the random 3-regular geometric graph generator of host_topology.cpp (network.py:122-272) for B envs in
// one launch, writing each topology straight into a slot of the device topology pool (gm_topology_generate_device), and
// the pool's next-hop tables in networkx's tie-breaking order (gm_topology_next_hops, further down).
//
// One warp per env.  Lane 0 runs everything that is sequential in the reference -- the env's private legacy MT19937
// stream (shared memory), the node positions, the edge rule, the validity check and the reseed loop -- and the warp
// does the rest: the distances from node i, the next candidate in (distance, id) order (a stable sort by distance
// visits the nodes in exactly that order), the exclusion-list scan and the output tables.  The candidates of node i are
// produced one at a time by a warp arg-min above the previous one, so only as many as the edge rule looks at are ranked.
//
// Every table is bit-identical to the host generator's: the distances and edge lengths use explicitly rounded double
// operations (nvcc would otherwise contract dx*dx + dy*dy and sqrt(d)*10 into FMAs), and the shortest-path weights are
// integers, so Floyd-Warshall gives the host's Dijkstra table exactly.
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace gm {
namespace {

constexpr int kTopoMaxWarps = 4;
constexpr int kTopoSmemBudget = 48 * 1024;
constexpr int kApspInf = 1 << 29;  // INF + INF stays below INT_MAX

// per-warp shared memory: MT state (625 words, padded to 8 bytes), x, y, distances (doubles), then int tables; a
// multiple of 16 bytes, so that the doubles of every warp's slice stay aligned (3E ints is odd for odd E)
__host__ __device__ inline int topo_warp_bytes(int N) {
    const int E = 3 * N / 2;
    return (int)round_up(626 * 4 + 3 * N * 8 + (3 * N + 3 * N + N + 3 * E) * 4, 16);
}

struct WarpMT {  // LegacyMT of host_topology.cpp on a shared-memory state; lane 0 only
    uint32_t* key;
    __device__ void seed(uint32_t s) {
        for (uint32_t i = 0; i < 624; ++i) {
            key[i] = s;
            s = 1812433253u * (s ^ (s >> 30)) + i + 1u;
        }
        key[624] = 624;
    }
    __device__ uint32_t next() {
        if (key[624] >= 624) {
            for (int i = 0; i < 624; ++i) {
                const uint32_t y = (key[i] & 0x80000000u) | (key[(i + 1) % 624] & 0x7fffffffu);
                key[i] = key[(i + 397) % 624] ^ (y >> 1) ^ (0x9908b0dfu & (0u - (y & 1u)));
            }
            key[624] = 0;
        }
        uint32_t y = key[key[624]++];
        y ^= y >> 11;
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        return y ^ (y >> 18);
    }
    __device__ double uniform() {  // genrand_res53
        const uint32_t hi = next() >> 5, lo = next() >> 6;
        return __ddiv_rn(__dadd_rn(__dmul_rn((double)hi, 67108864.0), (double)lo), 9007199254740992.0);
    }
    __device__ uint32_t below_int31() {  // bounded(2^31 - 2): masked rejection with mask 0x7fffffff
        for (;;) {
            const uint32_t v = next() & 0x7fffffffu;
            if (v <= 2147483646u) return v;
        }
    }
};

__device__ inline bool key_less(double da, int ja, double db, int jb) { return da < db || (da == db && ja < jb); }

__global__ void __launch_bounds__(kTopoMaxWarps * 32) topology_generate_kernel(
    gm_topology_tables t, int B, const int64_t* __restrict__ seeds, const int32_t* __restrict__ slot,
    const int64_t* __restrict__ exclude, int n_exclude, int max_attempts, int64_t* __restrict__ seed_used,
    int32_t* __restrict__ repetitions, int32_t* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char topo_smem[];
    const int N = t.N, E = 3 * N / 2;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * (blockDim.x >> 5) + w;
    if (b >= B) return;  // whole warps leave together
    unsigned char* base = topo_smem + (size_t)w * topo_warp_bytes(N);
    WarpMT rng{(uint32_t*)base};
    double* x = (double*)(base + 626 * 4);
    double* y = x + N;
    double* dist = y + N;
    int* nbr = (int*)(dist + N);   // [N][3] neighbours in creation order
    int* inc = nbr + 3 * N;        // [N][3] incident edge ids in creation order
    int* cnt = inc + 3 * N;        // [N] degree so far
    int* ea = cnt + N;             // [E] edges in creation order, ea < eb
    int* eb = ea + E;
    int* elen = eb + E;
    __shared__ int n_edges_sh[kTopoMaxWarps];

    const int s = slot[b];
    if (s < 0 || s >= t.P) {
        if (lane == 0) atomicCAS(status, 0, -(b + 1));
        return;
    }
    int64_t topo_seed = seeds[b];
    if (lane == 0) rng.seed((uint32_t)topo_seed);
    int reps = 0;
    bool valid = false;
    while (!valid && reps < max_attempts) {
        // ---- Graph::build (network.py:122-195) ----
        if (lane == 0) {
            for (int i = 0; i < N; ++i) {
                x[i] = rng.uniform();
                y[i] = rng.uniform();
            }
            n_edges_sh[w] = 0;
        }
        for (int i = lane; i < N; i += 32) cnt[i] = 0;
        __syncwarp();
        for (int i = 0; i < N; ++i) {
            if (cnt[i] >= 3) continue;  // warp-uniform: cnt is only written by lane 0 before a __syncwarp
            const double xi = x[i], yi = y[i];
            for (int j = lane; j < N; j += 32) {
                const double dx = __dsub_rn(x[j], xi), dy = __dsub_rn(y[j], yi);
                dist[j] = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
            }
            __syncwarp();
            double last_d = -1.0;
            int last_j = -1;
            // candidate positions 0..N-1 of the stable order; position 0 is skipped like the host's `j = 1`
            for (int pos = 0; pos < N && cnt[i] < 3; ++pos) {
                double bd = INFINITY;
                int bj = 0x7fffffff;
                for (int j = lane; j < N; j += 32) {
                    const double d = dist[j];
                    if (key_less(last_d, last_j, d, j) && key_less(d, j, bd, bj)) bd = d, bj = j;
                }
#pragma unroll
                for (int o = 16; o; o >>= 1) {
                    const double od = __shfl_xor_sync(FULL, bd, o);
                    const int oj = __shfl_xor_sync(FULL, bj, o);
                    if (key_less(od, oj, bd, bj)) bd = od, bj = oj;
                }
                last_d = bd, last_j = bj;
                if (pos >= 1 && lane == 0) {  // host_topology.cpp:99-108
                    const int c = bj;
                    bool linked = false;
                    for (int q = 0; q < cnt[c]; ++q) linked |= nbr[3 * c + q] == i;
                    if (cnt[c] < 3 && !linked && n_edges_sh[w] < E) {  // (E caps the edge list only for coincident points)
                        const int len = __double2int_rz(__dmul_rn(__dsqrt_rn(bd), 10.0)) / 2 + 1;
                        const int id = n_edges_sh[w]++;
                        ea[id] = min(i, c), eb[id] = max(i, c), elen[id] = len;
                        // the host appends to nbr[i] before nbr[c] and to inc[c] before inc[i]; for c == i (two nodes at
                        // the same point) both land in node i's lists in that order
                        nbr[3 * i + cnt[i]] = c;
                        if (c == i) {
                            inc[3 * i + cnt[i]] = id;
                            ++cnt[i];
                            if (cnt[i] < 3) nbr[3 * i + cnt[i]] = i, inc[3 * i + cnt[i]] = id, ++cnt[i];
                        } else {
                            nbr[3 * c + cnt[c]] = i;
                            inc[3 * c + cnt[c]] = id;
                            inc[3 * i + cnt[i]] = id;
                            ++cnt[i], ++cnt[c];
                        }
                    }
                }
                __syncwarp();
            }
        }
        ++reps;
        // ---- validity (network.py:197-213): degree 3 everywhere, connected from node 0 ----
        bool ok = true;
        for (int i = lane; i < N; i += 32) ok &= cnt[i] >= 3;
        ok = __all_sync(FULL, ok);
        if (ok) {
            int* seen = (int*)dist;  // the distances are no longer needed: N seen flags + an N-entry stack
            int* stack = seen + N;
            if (lane == 0) {
                for (int i = 0; i < N; ++i) seen[i] = 0;
                int top = 0, n_seen = 1;
                stack[top++] = 0;
                seen[0] = 1;
                while (top > 0) {
                    const int u = stack[--top];
                    for (int q = 0; q < cnt[u]; ++q) {
                        const int v = nbr[3 * u + q];
                        if (!seen[v]) seen[v] = 1, ++n_seen, stack[top++] = v;
                    }
                }
                ok = n_seen == N;
            }
            ok = __shfl_sync(FULL, ok, 0);
        }
        valid = ok;
        if (!valid && reps < max_attempts) {  // reseed from the topology stream, skipping excluded seeds (:252-255)
            for (;;) {
                uint32_t cand = 0;
                if (lane == 0) cand = rng.below_int31();
                cand = __shfl_sync(FULL, cand, 0);
                bool hit = false;
                for (int k = lane; k < n_exclude; k += 32) hit |= exclude[k] == (int64_t)cand;
                if (!__any_sync(FULL, hit)) {
                    topo_seed = cand;
                    break;
                }
            }
            if (lane == 0) rng.seed((uint32_t)topo_seed);
            __syncwarp();
        }
    }
    if (!valid) {
        if (lane == 0) atomicCAS(status, 0, b + 1);
        return;
    }
    // ---- outputs ----
    if (lane == 0) seed_used[b] = topo_seed, repetitions[b] = reps;
    int32_t* edges = t.edges + (size_t)s * E * 4;
    for (int e = lane; e < E; e += 32) {
        edges[4 * e] = ea[e], edges[4 * e + 1] = eb[e], edges[4 * e + 2] = elen[e], edges[4 * e + 3] = 0;
    }
    for (int i = lane; i < N; i += 32) {
        // network.py:191-195: a node's edges ordered by the neighbour's id (stable insertion sort of three)
        int ord[3] = {inc[3 * i], inc[3 * i + 1], inc[3 * i + 2]}, oth[3];
        for (int q = 0; q < 3; ++q) oth[q] = ea[ord[q]] == i ? eb[ord[q]] : ea[ord[q]];
        for (int q = 1; q < 3; ++q)
            for (int r = q; r > 0 && oth[r] < oth[r - 1]; --r) {
                int tmp = oth[r]; oth[r] = oth[r - 1]; oth[r - 1] = tmp;
                tmp = ord[r]; ord[r] = ord[r - 1]; ord[r - 1] = tmp;
            }
        int32_t* ne = t.node_edges + ((size_t)s * N + i) * 3;
        int32_t* nn = t.node_nbrs + ((size_t)s * N + i) * 3;
        int all[4] = {i, oth[0], oth[1], oth[2]};
        for (int q = 0; q < 3; ++q) ne[q] = ord[q], nn[q] = oth[q];
        for (int q = 1; q < 4; ++q)  // lists_from_tables: self + neighbours, ascending
            for (int r = q; r > 0 && all[r] < all[r - 1]; --r) {
                const int tmp = all[r]; all[r] = all[r - 1]; all[r - 1] = tmp;
            }
        int32_t* na = t.nbr_all + ((size_t)s * N + i) * 4;
        for (int q = 0; q < 4; ++q) na[q] = all[q];
        t.deg[(size_t)s * N + i] = 4;
    }
    // all-pairs shortest-path weights: Floyd-Warshall in place in the slot's table (row and column k do not change
    // during round k, so every lane may update its own entries without further ordering)
    int32_t* d = t.apsp + (size_t)s * N * N;
    for (int p = lane; p < N * N; p += 32) d[p] = (p / N == p % N) ? 0 : kApspInf;
    __syncwarp();
    for (int e = lane; e < E; e += 32)
        if (ea[e] != eb[e]) d[ea[e] * N + eb[e]] = elen[e], d[eb[e] * N + ea[e]] = elen[e];
    __syncwarp();
    for (int k = 0; k < N; ++k) {
        const int32_t* dk = d + (size_t)k * N;
        for (int p = lane; p < N * N; p += 32) {
            const int i = p / N, j = p - i * N;
            const int via = d[i * N + k] + dk[j];
            if (via < d[p]) d[p] = via;
        }
        __syncwarp();
    }
}

// ---- next-hop tables: networkx's single-source Dijkstra paths, tie for tie ----
//
// nx.shortest_path(G, weight=...) runs _dijkstra_multisource from every source: neighbours in G._adj order (edge
// creation order, the order G.add_edge inserted them), a heap popped by (distance, push counter), a push and
// pred[u] = [v] only on a strictly shorter distance, and paths[u] = paths[pred[u][0]] + [u].  The entry popped next is
// always the current entry of an unsettled node -- an older entry of a node has a larger distance than its current one
// -- so keeping one (distance, counter) per node and taking the warp arg-min over the unsettled nodes pops in the heap's
// order without a heap.  The first hop of u is u itself when its predecessor is the source and its predecessor's first
// hop otherwise; a settled node's predecessor no longer changes, so it is final when u is relaxed from it.
constexpr int kHopWarps = 8;
constexpr int kHopSmemBudget = 48 * 1024;
constexpr int kHopUnseen = 0x7fffffff;

__global__ void __launch_bounds__(kHopWarps * 32) topology_next_hops_kernel(gm_topology_tables t, int n,
                                                                          const int32_t* __restrict__ slots,
                                                                          int8_t* __restrict__ next_hop) {
    extern __shared__ __align__(16) int hop_smem[];
    const int N = t.N, E = 3 * N / 2;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + w;  // (listed slot, source) pair of this warp
    if (g >= (int64_t)n * N) return;  // whole warps leave together
    const int i = (int)(g / N), src = (int)(g - (int64_t)i * N);
    const int s = slots[i];
    int8_t* out = next_hop + ((size_t)i * N + src) * N;
    if (s < 0 || s >= t.P) {  // a slot outside the pool: the row is marked, nothing is read
        for (int v = lane; v < N; v += 32) out[v] = -1;
        return;
    }
    int* dist = hop_smem + (size_t)w * 3 * N;  // tentative or final distance; kHopUnseen before the first push
    int* cnt = dist + N;                       // push counter of the current entry; -1 once settled
    int* hop = cnt + N;                        // first hop of the current predecessor's path
    for (int v = lane; v < N; v += 32) dist[v] = kHopUnseen, cnt[v] = 0, hop[v] = -1;
    __syncwarp();
    if (lane == 0) dist[src] = 0;
    __syncwarp();
    const int32_t* node_edges = t.node_edges + (size_t)s * N * 3;
    const int32_t* edges = t.edges + (size_t)s * E * 4;
    int counter = 1;  // the source's entry took counter 0
    for (;;) {
        // pop: the unsettled node of least (distance, counter)
        int bd = kHopUnseen, bc = 0x7fffffff, bv = -1;
        for (int v = lane; v < N; v += 32) {
            const int d = dist[v], c = cnt[v];
            if (c >= 0 && d != kHopUnseen && (d < bd || (d == bd && c < bc))) bd = d, bc = c, bv = v;
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const int od = __shfl_xor_sync(FULL, bd, o), oc = __shfl_xor_sync(FULL, bc, o), ov = __shfl_xor_sync(FULL, bv, o);
            if (od < bd || (od == bd && oc < bc)) bd = od, bc = oc, bv = ov;
        }
        if (bv < 0) break;
        const int v = bv;
        // relax v's three edges in creation (edge id) order: lane q takes the q-th smallest incident edge id
        bool improve = false;
        int u = 0, nd = 0;
        if (lane < 3) {
            const int e0 = node_edges[3 * v], e1 = node_edges[3 * v + 1], e2 = node_edges[3 * v + 2];
            const int lo = min(e0, min(e1, e2)), hi = max(e0, max(e1, e2));
            const int e = lane == 0 ? lo : lane == 2 ? hi : e0 + e1 + e2 - lo - hi;
            const int a = edges[4 * e], b = edges[4 * e + 1];
            u = a == v ? b : a;
            nd = bd + edges[4 * e + 2];
            improve = cnt[u] >= 0 && nd < dist[u];  // (u == v, the self-loop of two coincident nodes, never improves)
        }
        const unsigned mask = __ballot_sync(FULL, improve);
        __syncwarp();
        if (lane == 0) cnt[v] = -1;  // settled
        if (improve) {
            dist[u] = nd;
            cnt[u] = counter + __popc(mask & ((1u << lane) - 1));
            hop[u] = v == src ? u : hop[v];
        }
        counter += __popc(mask);
        __syncwarp();
    }
    // the entry of (src, t): 1 + the index in node_edges[src] of the edge towards hop[t]
    const int32_t* nb = t.node_nbrs + ((size_t)s * N + src) * 3;
    const int n0 = nb[0], n1 = nb[1], n2 = nb[2];
    for (int v = lane; v < N; v += 32) {
        const int h = hop[v];
        out[v] = (int8_t)(v == src || h < 0 ? 0 : h == n0 ? 1 : h == n1 ? 2 : h == n2 ? 3 : 0);
    }
}

}  // namespace
}  // namespace gm

extern "C" int gm_topology_next_hops(const gm_topology_tables* tables, int32_t P, const int32_t* slots, int32_t n,
                                     int8_t* next_hop, void* stream) {
    using namespace gm;
    GM_CHECK_ARG(tables, "null topology tables");
    gm_topology_tables t = *tables;
    GM_CHECK_ARG(t.N >= 4 && t.N % 2 == 0 && t.N <= GM_TOPOLOGY_MAX_NODES,
                 "n_nodes must be even and in [4, %d] for the next-hop tables, got %d", GM_TOPOLOGY_MAX_NODES, t.N);
    GM_CHECK_ARG(P > 0 && P <= t.P && t.edges && t.node_edges && t.node_nbrs, "bad topology tables");
    GM_CHECK_ARG(n >= 0 && (n == 0 || (slots && next_hop)), "bad next-hop arguments");
    if (n == 0) return GM_OK;
    t.P = P;
    const int per_warp = 3 * t.N * (int)sizeof(int);
    const int warps = std::min(kHopWarps, kHopSmemBudget / per_warp);
    const int64_t blocks = ((int64_t)n * t.N + warps - 1) / warps;
    GM_CHECK_ARG(blocks < (int64_t)1 << 31, "too many next-hop tables in one launch: %d", n);
    topology_next_hops_kernel<<<(unsigned)blocks, warps * 32, (size_t)warps * per_warp,
                                (cudaStream_t)stream>>>(t, n, slots, next_hop);
    GM_LAUNCH_CHECK();
    return GM_OK;
}

extern "C" int gm_topology_generate_device(const gm_topology_tables* tables, int32_t B, const int64_t* seeds,
                                           const int32_t* slot, const int64_t* exclude, int32_t n_exclude,
                                           int32_t max_attempts, int64_t* seed_used, int32_t* repetitions,
                                           int32_t* status, void* stream) {
    using namespace gm;
    GM_CHECK_ARG(tables, "null topology tables");
    const gm_topology_tables& t = *tables;
    GM_CHECK_ARG(t.N >= 4 && t.N % 2 == 0 && t.N <= GM_TOPOLOGY_MAX_NODES,
                 "n_nodes must be even and in [4, %d] for the device generator, got %d", GM_TOPOLOGY_MAX_NODES, t.N);
    GM_CHECK_ARG(t.P > 0 && t.edges && t.node_edges && t.node_nbrs && t.apsp && t.nbr_all && t.deg, "bad topology tables");
    GM_CHECK_ARG(B > 0 && seeds && slot && seed_used && repetitions && status, "bad generator arguments");
    GM_CHECK_ARG(n_exclude >= 0 && (n_exclude == 0 || exclude), "bad exclusion list");
    GM_CHECK_ARG(max_attempts >= 1, "max_attempts must be >= 1, got %d", max_attempts);
    const int per_warp = topo_warp_bytes(t.N);
    const int warps = per_warp * kTopoMaxWarps <= kTopoSmemBudget ? kTopoMaxWarps : std::max(1, kTopoSmemBudget / per_warp);
    topology_generate_kernel<<<ceil_div(B, warps), warps * 32, (size_t)warps * per_warp, (cudaStream_t)stream>>>(
        t, B, seeds, slot, exclude, n_exclude, max_attempts, seed_used, repetitions, status);
    GM_LAUNCH_CHECK();
    return GM_OK;
}
