// host_topology.cpp -- host-side (CPU) pieces of the rollout path that the reference runs
// once per episode, written natively so that thousands of topologies per second can feed
// the device-resident topology pool (SURVEY.md 7.6, 8f-2):
//
//   * numpy's legacy MT19937 stream (np.random.seed / random / randint), which drives the
//     topology generator (src/env/network.py:122-258), packet respawns
//     (src/env/routing.py:130-135) and epsilon-greedy draws (src/policy.py:46-47);
//   * the random 3-regular geometric graph generator with validity check and reseed loop
//     (network.py:122-272);
//   * integer all-pairs shortest path WEIGHTS (network.py:274-290; Dijkstra per source).
//
// No device code here; compiled by nvcc as plain C++ into the same shared library.
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <queue>
#include <utility>
#include <vector>

#include "common.cuh"

namespace {

// -------- legacy numpy generator ----------------------------------------------------------
class LegacyMT {
  public:
    explicit LegacyMT(uint32_t* st) : key_(st), pos_(st + 624) {}
    void seed(uint32_t s) {  // init_genrand
        for (uint32_t i = 0; i < 624; ++i) {
            key_[i] = s;
            s = 1812433253u * (s ^ (s >> 30)) + i + 1u;
        }
        *pos_ = 624;
    }
    uint32_t next() {
        if (*pos_ >= 624) refill();
        uint32_t y = key_[(*pos_)++];
        y ^= y >> 11;
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        return y ^ (y >> 18);
    }
    double uniform() {  // genrand_res53
        uint32_t hi = next() >> 5, lo = next() >> 6;
        return (hi * 67108864.0 + lo) / 9007199254740992.0;
    }
    // value in [0, span] by masked rejection; span == 0 draws nothing (numpy legacy bounded ints)
    uint32_t bounded(uint32_t span) {
        if (span == 0) return 0;
        if (span == 0xffffffffu) return next();
        uint32_t m = span;
        for (int sh = 1; sh < 32; sh <<= 1) m |= m >> sh;
        for (;;) {
            uint32_t v = next() & m;
            if (v <= span) return v;
        }
    }
    uint32_t below(uint32_t high) { return bounded(high - 1); }

  private:
    void refill() {
        for (int i = 0; i < 624; ++i) {
            uint32_t y = (key_[i] & 0x80000000u) | (key_[(i + 1) % 624] & 0x7fffffffu);
            key_[i] = key_[(i + 397) % 624] ^ (y >> 1) ^ (0x9908b0dfu & (0u - (y & 1u)));
        }
        *pos_ = 0;
    }
    uint32_t* key_;
    uint32_t* pos_;
};

// -------- topology ---------------------------------------------------------------------------
struct Graph {
    int n = 0;
    std::vector<double> x, y;
    std::vector<std::vector<int>> nbr;     // creation order
    std::vector<std::vector<int>> inc;     // incident edge ids, creation order
    std::vector<int> ea, eb, elen;         // edges in creation order, ea < eb

    int other(int e, int v) const { return ea[e] == v ? eb[e] : ea[e]; }

    // network.py:122-195
    void build(LegacyMT& rng, int nodes) {
        n = nodes;
        x.assign(n, 0); y.assign(n, 0);
        nbr.assign(n, {}); inc.assign(n, {});
        ea.clear(); eb.clear(); elen.clear();
        for (int i = 0; i < n; ++i) { x[i] = rng.uniform(); y[i] = rng.uniform(); }
        std::vector<std::pair<double, int>> cand(n);
        for (int i = 0; i < n; ++i) {
            for (int j = 0; j < n; ++j) {
                double dx = x[j] - x[i], dy = y[j] - y[i];
                cand[j] = {dx * dx + dy * dy, j};
            }
            // list.sort(key=dist) is stable; (dist, j) lexicographic order is the same permutation
            std::stable_sort(cand.begin(), cand.end(),
                             [](const std::pair<double, int>& a, const std::pair<double, int>& b) { return a.first < b.first; });
            for (int j = 1; j < n && nbr[i].size() < 3; ++j) {
                int c = cand[j].second;
                if (nbr[c].size() >= 3) continue;
                if (std::find(nbr[c].begin(), nbr[c].end(), i) != nbr[c].end()) continue;
                int len = (int)(sqrt(cand[j].first) * 10.0) / 2 + 1;  // int(int(sqrt(d)*10)/2+1), :173
                int id = (int)ea.size();
                ea.push_back(std::min(i, c)); eb.push_back(std::max(i, c)); elen.push_back(len);
                nbr[i].push_back(c); nbr[c].push_back(i);
                inc[c].push_back(id); inc[i].push_back(id);
            }
        }
    }
    // network.py:197-213
    bool valid() const {
        for (int i = 0; i < n; ++i)
            if (nbr[i].size() < 3) return false;
        std::vector<char> seen(n, 0);
        std::vector<int> stack{0};
        seen[0] = 1;
        int cnt = 1;
        while (!stack.empty()) {
            int u = stack.back();
            stack.pop_back();
            for (int v : nbr[u])
                if (!seen[v]) { seen[v] = 1; ++cnt; stack.push_back(v); }
        }
        return cnt == n;
    }
};

bool excluded(int64_t s, const int64_t* ex, int n) {
    for (int i = 0; i < n; ++i)
        if (ex[i] == s) return true;
    return false;
}

void dijkstra_all(int n, int n_edges, const int32_t* edges4, int32_t* apsp) {
    std::vector<std::vector<std::pair<int, int>>> adj(n);
    for (int e = 0; e < n_edges; ++e) {
        int a = edges4[4 * e], b = edges4[4 * e + 1], w = edges4[4 * e + 2];
        adj[a].push_back({b, w});
        adj[b].push_back({a, w});
    }
    const int INF = 1 << 30;
    for (int src = 0; src < n; ++src) {
        int32_t* d = apsp + (size_t)src * n;
        for (int i = 0; i < n; ++i) d[i] = INF;
        d[src] = 0;
        using QE = std::pair<int, int>;
        std::priority_queue<QE, std::vector<QE>, std::greater<QE>> pq;
        pq.push({0, src});
        while (!pq.empty()) {
            auto [du, u] = pq.top();
            pq.pop();
            if (du > d[u]) continue;
            for (auto [v, w] : adj[u])
                if (du + w < d[v]) { d[v] = du + w; pq.push({d[v], v}); }
        }
    }
}

}  // namespace

extern "C" {

void gm_mt_seed(uint32_t* state, uint32_t seed) { LegacyMT(state).seed(seed); }
uint32_t gm_mt_u32(uint32_t* state) { return LegacyMT(state).next(); }
double gm_mt_random(uint32_t* state) { return LegacyMT(state).uniform(); }
uint32_t gm_mt_randint(uint32_t* state, uint32_t high) { return LegacyMT(state).below(high); }

void gm_mt_packet_draws(uint32_t* state, int32_t n_nodes, int32_t n, int32_t* start, int32_t* target, double* size) {
    LegacyMT r(state);
    for (int i = 0; i < n; ++i) {
        start[i] = (int32_t)r.below((uint32_t)n_nodes);
        target[i] = (int32_t)r.below((uint32_t)n_nodes);
        size[i] = r.uniform();
    }
}

int gm_mt_reset_draws(uint32_t* state, int32_t seed_mode, const int64_t* seed_list, int32_t n_seeds,
                      const int64_t* exclude, int32_t n_exclude, int32_t n_nodes, int32_t S, int32_t A, int64_t* seeds,
                      int32_t* start, int32_t* target, double* size) {
    GM_CHECK_ARG(state && S >= 0 && A >= 0 && n_nodes > 0 && (S == 0 || seeds), "bad reset-draw arguments");
    GM_CHECK_ARG(A == 0 || S == 0 || (start && target && size), "null packet-draw output");
    GM_CHECK_ARG(seed_mode >= 0 && seed_mode <= 2, "seed_mode must be 0, 1 or 2, got %d", seed_mode);
    GM_CHECK_ARG(seed_mode == 0 || (seed_list && n_seeds > 0), "seed_mode %d needs a seed list", seed_mode);
    GM_CHECK_ARG(n_exclude >= 0 && (n_exclude == 0 || exclude), "bad exclusion list");
    std::vector<int64_t> ex(exclude, exclude + n_exclude);
    std::sort(ex.begin(), ex.end());
    LegacyMT r(state);
    for (int s = 0; s < S; ++s) {
        if (seed_mode == 0) {  // pick_seed without a seed list: randint(2**31 - 1), redrawn on excluded seeds
            int64_t v;
            do v = r.below(2147483647u); while (std::binary_search(ex.begin(), ex.end(), v));
            seeds[s] = v;
        } else if (seed_mode == 1) {  // the sample's seed is given: no draw
            seeds[s] = seed_list[s];
        } else {  // np.random.choice(seed_list): randint(len); a one-seed list draws nothing
            seeds[s] = seed_list[r.below((uint32_t)n_seeds)];
        }
        const size_t o = (size_t)s * A;
        for (int i = 0; i < A; ++i) {  // routing.py:130-135
            start[o + i] = (int32_t)r.below((uint32_t)n_nodes);
            target[o + i] = (int32_t)r.below((uint32_t)n_nodes);
            size[o + i] = r.uniform();
        }
    }
    return GM_OK;
}

void gm_mt_policy_draws(uint32_t* state, int32_t n_actions, int32_t n, int32_t* rand_action, double* rand_u) {
    LegacyMT r(state);
    for (int i = 0; i < n; ++i) rand_action[i] = (int32_t)r.below((uint32_t)n_actions);
    for (int i = 0; i < n; ++i) rand_u[i] = r.uniform();
}

int gm_topology_apsp(int32_t n_nodes, int32_t n_edges, const int32_t* edges, int32_t* apsp) {
    GM_CHECK_ARG(n_nodes > 0 && n_edges > 0 && edges && apsp, "bad apsp arguments");
    dijkstra_all(n_nodes, n_edges, edges, apsp);
    return GM_OK;
}

int gm_topology_generate(uint32_t* global_state, int32_t n_nodes, int32_t seed_mode, int64_t seed,
                         const int64_t* exclude, int32_t n_exclude, int32_t* edges, int32_t* node_edges,
                         int32_t* node_nbrs, int32_t* nbr_creation, int32_t* apsp, double* xy, int32_t* repetitions,
                         int64_t* seed_used) {
    GM_CHECK_ARG(n_nodes >= 4 && n_nodes % 2 == 0, "n_nodes must be even and >= 4 for a 3-regular graph, got %d", n_nodes);
    GM_CHECK_ARG(edges && node_edges && node_nbrs && apsp && repetitions && seed_used, "null output");
    GM_CHECK_ARG(seed_mode != 0 || global_state, "seed_mode 0 needs the caller's random stream");
    int64_t topo_seed = seed;
    if (seed_mode == 0) {  // network.py:229-232
        LegacyMT g(global_state);
        do topo_seed = g.below(2147483647u); while (excluded(topo_seed, exclude, n_exclude));
    }
    // network.py:241-258 saves the global state, reseeds, and restores afterwards: a private
    // stream has the same effect without touching the caller's state.
    std::vector<uint32_t> priv(GM_MT_STATE_WORDS);
    LegacyMT rng(priv.data());
    rng.seed((uint32_t)topo_seed);
    Graph g;
    int reps = 0;
    for (;;) {
        g.build(rng, n_nodes);
        ++reps;
        if (g.valid()) break;
        if (seed_mode == 1) {
            gm::set_error("Provided seed %lld is invalid.", (long long)topo_seed);
            return GM_ERR_SEED;
        }
        do topo_seed = rng.below(2147483647u); while (excluded(topo_seed, exclude, n_exclude));  // :252-254
        rng.seed((uint32_t)topo_seed);
    }
    *repetitions = reps;
    *seed_used = topo_seed;
    const int E = (int)g.ea.size();
    for (int e = 0; e < E; ++e) {
        edges[4 * e] = g.ea[e]; edges[4 * e + 1] = g.eb[e]; edges[4 * e + 2] = g.elen[e]; edges[4 * e + 3] = 0;
    }
    for (int i = 0; i < n_nodes; ++i) {
        // network.py:191-195: a node's edges ordered by the neighbour's node id
        std::vector<int> order = g.inc[i];
        std::sort(order.begin(), order.end(), [&](int a, int b) { return g.other(a, i) < g.other(b, i); });
        for (int q = 0; q < 3; ++q) {
            node_edges[3 * i + q] = order[q];
            node_nbrs[3 * i + q] = g.other(order[q], i);
            if (nbr_creation) nbr_creation[3 * i + q] = g.nbr[i][q];
        }
        if (xy) { xy[2 * i] = g.x[i]; xy[2 * i + 1] = g.y[i]; }
    }
    dijkstra_all(n_nodes, E, edges, apsp);
    return GM_OK;
}

}  // extern "C"
