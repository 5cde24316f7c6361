/*
 * graphmarl_b200.h -- C ABI of libgraphmarl_b200.so, the B200 (sm_100a) implementation
 * of graph-marl's data-parallel rollout hot path.
 *
 * The reference (jw3il/graph-marl) is pure Python and has no FFI: its boundary is the
 * Python class surface called by src/main.py, src/sl.py and src/eval.py (SURVEY.md 8b).
 * Each entry point below names the reference interface it replaces (file:line under
 * /root/reference).  The thin Python classes in graph_marl_b200/ bind these with ctypes
 * and keep the reference's names / signatures.
 *
 * Conventions
 *   - every function returns 0 on success, a negative gm_status on failure;
 *     gm_last_error() returns a thread-local message. No C++ exception crosses.
 *   - "device" pointers are caller-owned device memory (torch tensors' data_ptr());
 *     the library allocates nothing persistent. "host" pointers are plain host memory.
 *   - `stream` is a cudaStream_t passed as void*; all device work is asynchronous on it.
 *   - no torch types, no C++ types in any signature.
 */
#ifndef GRAPHMARL_B200_H
#define GRAPHMARL_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define GM_API __attribute__((visibility("default")))
#else
#define GM_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    GM_OK = 0,
    GM_ERR_INVALID = -1,   /* bad argument / unsupported configuration */
    GM_ERR_CUDA = -2,      /* a CUDA runtime call failed (message has the string) */
    GM_ERR_NO_DEVICE = -3, /* no sm_100 device: the library has NO CPU fallback */
    GM_ERR_SEED = -4       /* provided topology seed is invalid (network.py:251) */
} gm_status;

GM_API const char* gm_last_error(void);
/* ABI version, bumped on any signature/struct change. */
GM_API int gm_abi_version(void);   /* currently 6 */
/* 0 if a CUDA device with compute capability 10.x is present, else GM_ERR_NO_DEVICE. */
GM_API int gm_device_check(void);

/* ======================================================================== */
/* Host-side topology + legacy RNG (replaces src/env/network.py:122-290 and  */
/* numpy's legacy MT19937 stream used by network.py / routing.py / policy.py)*/
/* ======================================================================== */

/* np.random legacy stream. `state` is 625 uint32 (624 key words + position). */
#define GM_MT_STATE_WORDS 625
GM_API void gm_mt_seed(uint32_t* state, uint32_t seed);                  /* np.random.seed(int)        */
GM_API uint32_t gm_mt_u32(uint32_t* state);
GM_API double gm_mt_random(uint32_t* state);                             /* np.random.random()         */
GM_API uint32_t gm_mt_randint(uint32_t* state, uint32_t high);           /* np.random.randint(high)    */
/* packet draws of Routing.reset_packet (routing.py:130-135): n triples
 * (randint(N), randint(N), random()) in that order. */
GM_API void gm_mt_packet_draws(uint32_t* state, int32_t n_nodes, int32_t n, int32_t* start,
                        int32_t* target, double* size);
/* S sequential compat Routing.reset() calls (Network.reset()'s seed choice, then A packet triples as above) on the
 * caller's stream, which is left where the S-th call leaves it.  seed_mode 0: pick_seed without a seed list,
 * randint(2**31 - 1) redrawn while it is in exclude[n_exclude]; 1: the sample's seed is seed_list[s] (n_seeds >= S:
 * sequential provided seeds, no draw); 2: np.random.choice(seed_list[n_seeds]), one randint(n_seeds), none when
 * n_seeds == 1.  Outputs (host): seeds[S], start/target/size[S*A].  The topology generator draws from a private stream,
 * so nothing else is consumed. */
GM_API int gm_mt_reset_draws(uint32_t* state, int32_t seed_mode, const int64_t* seed_list, int32_t n_seeds,
                             const int64_t* exclude, int32_t n_exclude, int32_t n_nodes, int32_t S, int32_t A,
                             int64_t* seeds, int32_t* start, int32_t* target, double* size);
/* policy draws of EpsilonGreedy.__call__ (policy.py:46-47): randint(n_act,size=n) then rand(n) */
GM_API void gm_mt_policy_draws(uint32_t* state, int32_t n_actions, int32_t n, int32_t* rand_action,
                        double* rand_u);

/* Network._create_valid_network + _update_shortest_paths + _update_nodes_adjacency
 * (network.py:215-290, 385-389) for one topology.
 *   global_state : caller's MT19937 stream (may be NULL when seed_mode == 1)
 *   seed_mode    : 0 draw the seed from global_state (network.py:229-232); 1 use `seed`,
 *                  fail if it is invalid (:251); 2 start from `seed` (drawn by the caller from
 *                  its own stream) and reseed from the topology stream while invalid (:252-255)
 *   exclude      : seeds that must not be used (EVAL_SEEDS), may be NULL
 * Outputs (host): edges[E*4] = (start,end,length,0) in creation order, E = 3N/2;
 *   node_edges[N*3] edge ids sorted by neighbour id; node_nbrs[N*3] those neighbours;
 *   nbr_creation[N*3] neighbours in creation order; apsp[N*N] shortest-path weights;
 *   xy[N*2] node positions; *repetitions; *seed_used.
 * Returns GM_ERR_SEED if seed_mode==1 and the first attempt is not a valid graph. */
GM_API int gm_topology_generate(uint32_t* global_state, int32_t n_nodes, int32_t seed_mode, int64_t seed,
                         const int64_t* exclude, int32_t n_exclude, int32_t* edges,
                         int32_t* node_edges, int32_t* node_nbrs, int32_t* nbr_creation,
                         int32_t* apsp, double* xy, int32_t* repetitions, int64_t* seed_used);
/* apsp only, after edge lengths changed (network.py:292-329 randomize_edge_weights) */
GM_API int gm_topology_apsp(int32_t n_nodes, int32_t n_edges, const int32_t* edges, int32_t* apsp);

/* Device-resident topology tables of P pool slots (all int32, device pointers), the layout Routing reads. */
#define GM_TOPOLOGY_MAX_NODES 512
typedef struct gm_topology_tables {
    int32_t P, N;          /* slots, nodes (E = 3N/2 edges) */
    int32_t* edges;        /* [P,E,4] (start, end, length, 0) in creation order, start < end */
    int32_t* node_edges;   /* [P,N,3] incident edge ids ordered by neighbour id */
    int32_t* node_nbrs;    /* [P,N,3] those neighbours */
    int32_t* apsp;         /* [P,N,N] shortest-path weights */
    int32_t* nbr_all;      /* [P,N,4] the node and its three neighbours, ascending (NetMon's adjacency lists) */
    int32_t* deg;          /* [P,N]   4 */
} gm_topology_tables;
/* B topologies in one launch: env b's topology is gm_topology_generate(seed_mode 2, seeds[b], exclude) -- bit-identical
 * tables, seed_used[b] and repetitions[b] -- written into pool slot slot[b] (device arrays seeds i64[B], slot i32[B],
 * exclude i64[n_exclude], seed_used i64[B], repetitions i32[B]).  Each env builds at most `max_attempts` graphs; *status
 * (device i32, zeroed by the caller) is left 0 on success, else set to b + 1 for an env b that ran out of attempts or
 * -(b + 1) for one whose slot lies outside [0, P) (nothing is written for that env).  N even,
 * 4 <= N <= GM_TOPOLOGY_MAX_NODES.  Asynchronous on `stream`. */
GM_API int gm_topology_generate_device(const gm_topology_tables* tables, int32_t B, const int64_t* seeds,
                                       const int32_t* slot, const int64_t* exclude, int32_t n_exclude,
                                       int32_t max_attempts, int64_t* seed_used, int32_t* repetitions, int32_t* status,
                                       void* stream);
/* Next-hop tables of the pool slots slots[0..n) (device i32[n]) into next_hop (device i8[n,N,N]): next_hop[i,v,t] is 0
 * for v == t, else 1 + the index in node_edges[v] of the edge that carries the first hop of nx.shortest_path(G)[v][t] --
 * networkx's Dijkstra with its tie-breaking (neighbours in edge creation order, pops by (distance, push counter), a
 * predecessor only on a strictly shorter distance).  A slot outside [0, P) (P <= tables->P) gets rows of -1.  One warp
 * per (slot, source), 4 <= N <= GM_TOPOLOGY_MAX_NODES.  Asynchronous on `stream`. */
GM_API int gm_topology_next_hops(const gm_topology_tables* tables, int32_t P, const int32_t* slots, int32_t n,
                                 int8_t* next_hop, void* stream);

/* ======================================================================== */
/* Routing environment (replaces src/env/routing.py:119-178, 187-235,        */
/* 256-358, 360-539 for B independent env instances advanced in place)       */
/* ======================================================================== */

typedef struct gm_routing_desc {
    int32_t B, N, A, E, T;       /* envs, nodes, agents(=packets), edges=3N/2, pool size */
    int32_t env_var;             /* EnvironmentVariant 1 (independent), 2 (with k neighbours), 3 (global) */
    int32_t k;                   /* neighbours in obs for env_var 2 */
    int32_t congestion;          /* enable_congestion (routing.py:61) */
    int32_t action_mask;         /* enable_action_mask (routing.py:62) */
    int32_t ttl;                 /* ttl, 0 = disabled (routing.py:63) */
    int32_t state_stride;        /* bytes per env in `state`, from gm_routing_state_layout */
    int32_t node_sparse_static;  /* 0: node_sparse rows list all 12 fields; 1: 6 entries -- (4N+8 + topology*N + node, 1)
                                    for the constant part of the row, then #waiting, size sum and the three edge loads;
                                    2: the same 6 entries as indices into a dictionary of T*N + 5 rows: topology*N + node,
                                    then T*N + 0..4 for #waiting, size sum and the three loads (static_only packs) */
    /* topology pool (device, int32) */
    const int32_t* node_edges;   /* [T,N,3] edge ids of node n sorted by neighbour id */
    const int32_t* node_nbrs;    /* [T,N,3] the neighbour reached by action 1..3 */
    const int32_t* edges;        /* [T,E,4] start,end,length,0 */
    const int32_t* apsp;         /* [T,N,N] shortest-path weights */
    const int32_t* topo_index;   /* [B] env -> topology, NULL = all use topology 0 */
    uint8_t* state;              /* [B,state_stride] packed env state, advanced in place */
} gm_routing_desc;

typedef struct gm_routing_io {
    /* inputs */
    const int32_t* actions;      /* [B,A] in {0..3}; step only */
    const uint8_t* env_mask;     /* [B]; reset only; NULL = reset every env */
    const int32_t* draw_start;   /* [B,A] host-supplied draws; slot s feeds the s-th reset */
    const int32_t* draw_target;  /*        packet in id order (routing.py:130-135).        */
    const double* draw_size;     /*        All three NULL => device Philox4x32-10 draws.    */
    uint64_t philox_seed, philox_step;
    /* optional device counter added to philox_step (u64): lets a captured CUDA graph replay the call with a
     * step that advances between replays (the host updates the counter, the baked argument is the offset) */
    const uint64_t* philox_step_dev;
    /* outputs (device); any may be NULL and is then not produced */
    float* obs;                  /* [B,A,W] routing.py:269-358; W = 6N+10 (+5k for env_var 2, +N*N+N*(4N+8) for 3) */
    int8_t* adj;                 /* [B,A,A]      routing.py:522-539 */
    float* node_obs;             /* [B,N,4N+8]   routing.py:187-235 */
    int8_t* node_agent;          /* [B,N,A]      routing.py:256-267 */
    int32_t* agent_node;         /* [B,A] node of each agent (= argmax of node_agent column) */
    int32_t* node_sparse;        /* [B,N,24] the node observation rows in sparse form: 12 column indices then 12 fp32
                                    values (bit patterns) in the fixed slot order node, #waiting, size sum, 3 x (neighbour,
                                    length, load); consumed by gm_netmon_params.sparse_rows */
    float* reward;               /* [B,A] f32    routing.py:361,398,474 */
    uint8_t* done;               /* [B,A]        routing.py:475 */
    int32_t* delays;             /* [B,A] agent_steps at done else 0 (routing.py:488) */
    uint8_t* arrived;            /* [B,A] success (routing.py:476) */
    double* spr;                 /* [B,A] agent_steps/max(spw,1) where arrived (routing.py:484) */
    int32_t* info;               /* [B,4] looped, throughput, dropped, blocked (routing.py:499-508) */
    int32_t* n_resets;           /* [B] draw slots consumed by this call */
    uint8_t* action_mask_out;    /* [B,A,4] env.action_mask after the call (routing.py:106) */
    /* set_eval_info(True) extras (routing.py:384-386, 414-441); enabled by eval_f64 != NULL, step only */
    double* eval_f64;            /* [B,2] total_edge_load, total_packet_size (sequential fp64 sums) */
    int32_t* eval_i32;           /* [B,2] occupied_edges, packets_on_edges */
    int32_t* packet_dist;        /* [B,A] shortest-path weight now->target of every packet */
    double* packet_sizes;        /* [B,A] packet sizes before respawns */
    int32_t* sum_packets_per_node; /* [B,N] cumulative: += 1 per waiting packet per step (routing.py:384-386) */
    int32_t* sum_packets_per_edge; /* [B,E] cumulative: += 1 per in-flight packet per step (routing.py:428-429) */
    /* Optional, step only: the step kernel itself writes this step's transition in the compact replay format
     * (what ReplayBuffer.add stores, replaybuffer.py:243-287, restated by CompactReplayBuffer: the env record before and
     * after the step instead of the dense observation rows) into ring slot (ring_index + *ring_index_dev + env) %
     * ring_capacity.  Enabled by ring_rec != NULL; any other ring pointer may be NULL.  The record is in the kernel's
     * shared memory at both moments, so the two separate insert launches of a rollout step disappear. */
    uint8_t* ring_rec;           /* [capacity, state_stride] env record BEFORE the step */
    uint8_t* ring_next_rec;      /* [capacity, state_stride] env record AFTER the step */
    int32_t* ring_topo;          /* [capacity] topology index of the env (0 without a pool) */
    int8_t* ring_action;         /* [capacity, A] the actions of this call */
    float* ring_reward;          /* [capacity, A] */
    uint8_t* ring_done;          /* [capacity, A] */
    uint8_t* ring_episode_done;  /* [capacity] = ring_episode_flag */
    int64_t ring_capacity, ring_index;
    const int64_t* ring_index_dev; /* optional device counter added to ring_index (CUDA-graph replays), may be NULL */
    int32_t ring_episode_flag, ring_pad;
} gm_routing_io;

/* byte offsets inside one env's state record; out[8] =
 * {size f64[A], load f64[E], i32 block [8][A] (now,target,edge,time,ttl,spw,start,agent_steps),
 *  visited u32[A][ceil(N/32)], mask u8[A][4], stride, VW, 0} */
GM_API int gm_routing_state_layout(int32_t N, int32_t A, int32_t E, int32_t* out);
/* Routing.reset (routing.py:160-178) for envs selected by io->env_mask */
GM_API int gm_routing_reset(const gm_routing_desc* d, const gm_routing_io* io, void* stream);
/* Routing.step (routing.py:360-520) + observations */
GM_API int gm_routing_step(const gm_routing_desc* d, const gm_routing_io* io, void* stream);
/* observations of the current state without advancing it (get_node_observation etc.) */
GM_API int gm_routing_observe(const gm_routing_desc* d, const gm_routing_io* io, void* stream);

/* ======================================================================== */
/* SimpleEnvironment (replaces src/env/simple_environment.py:217-315)        */
/* ======================================================================== */
/* B instances. Device arrays: scores i32[B,3], edges i32[B,2,2], start_node i32[B],
 * start_edges i32[B,2]; actions i32[B] in {0,1}; env_var 1 or 3.
 * Outputs: obs f32[B,1,W] (W = 1 or 1+9+3), node_obs f32[B,3,1], node_agent i8[B,3,1],
 * node_adj i8[B,3,3], reward f32[B] (step only; NULL for reset). */
GM_API int gm_simple_step(int32_t B, int32_t env_var, const int32_t* scores, const int32_t* edges,
                   const int32_t* start_node, const int32_t* start_edges, const int32_t* actions,
                   float* obs, float* node_obs, int8_t* node_agent, int8_t* node_adj,
                   float* reward, void* stream);

/* ======================================================================== */
/* NetMon forward (replaces src/model.py:451-631, src/layernormlstm.py:24-42,*/
/* src/env/wrapper.py:66-109)                                                */
/* ======================================================================== */
#define GM_MAX_LAYERS 8
enum { GM_RNN_LSTM = 0, GM_RNN_LNLSTM = 1, GM_RNN_GRU = 2, GM_RNN_NONE = 3 };
enum { GM_AGG_SUM = 0, GM_AGG_MEAN = 1 };
enum { GM_ACT_LEAKY_RELU = 0, GM_ACT_RELU = 1, GM_ACT_TANH = 2, GM_ACT_SIGMOID = 3, GM_ACT_ELU = 4 };
/* GEMM arithmetic: FP32 = CUDA-core FFMA; BF16X3 = tcgen05 bf16 hi/lo split, 3 products,
 * fp32 accumulate (rel. error ~2^-17 per product); BF16 = single tcgen05 pass. */
enum { GM_MATH_FP32 = 0, GM_MATH_BF16X3 = 1, GM_MATH_BF16 = 2 };

typedef struct gm_cell_params {     /* nn.LSTMCell / nn.GRUCell / LayerNormLSTMCell */
    const float *w_ih, *w_hh;       /* [G*H, H] */
    const float *b_ih, *b_hh;       /* [G*H]; b_hh NULL for lnlstm (layernormlstm.py:19) */
    const float *ln_in_w, *ln_in_b, *ln_hid_w, *ln_hid_b; /* [4H] lnlstm only */
    const float *ln_cell_w, *ln_cell_b;                    /* [H]  lnlstm only */
} gm_cell_params;

typedef struct gm_netmon_params {
    int32_t in_features, hidden;            /* D_n, H */
    int32_t n_enc_layers;                   /* encoder MLP layers incl. the last (-> H) */
    int32_t enc_units[GM_MAX_LAYERS];       /* output width of each encoder layer */
    int32_t iterations;                     /* K (model.py:278) */
    int32_t rnn_type, agg_type, activation; /* enums above */
    int32_t rnn_carryover;                  /* model.py:281 */
    int32_t output_neighbor_hidden, output_global_hidden; /* model.py:279-280 */
    int32_t math;                           /* GM_MATH_* */
    /* > 0: the caller guarantees that every node observation row has at most this many (<= 12) non-zero entries (the
     * one-hot layout of routing.py:193-234 has 12): the tensor-core path then runs encoder layers 1 + 2 as one kernel
     * (layer 1 as 12 weight-column gathers, SURVEY 8d "one-hot layer-1 gathers").  0 = dense rows. */
    int32_t sparse_input_nnz;
    const float* enc_w[GM_MAX_LAYERS];      /* [out,in] row-major, nn.Linear layout */
    const float* enc_b[GM_MAX_LAYERS];
    gm_cell_params rnn_obs, rnn_update;
    /* tensor-core modes only: weights packed by gm_netmon_pack_weights (device, 256-byte aligned),
     * or NULL = pack into the workspace on every forward call */
    const void* packed;
    /* per call, optional (with sparse_input_nnz > 0): the rows already in sparse form, i32[ceil(B*N/128)*128][24] = 12
     * column indices then 12 fp32 values per row (gm_routing_io.node_sparse writes them in a fixed slot order, which
     * lets the kernel's shared-memory gathers of the fixed columns broadcast); NULL = the library derives them from
     * node_obs.  Rows behind B*N are never read as data. */
    const int32_t* sparse_rows;
    /* optional: S dense rows f32[S, D_n] holding per-(topology, node) CONSTANT parts of the observation rows (one-hot of
     * the node and of its neighbours, edge lengths).  gm_netmon_pack_weights appends layer 1 applied to each of them to
     * its weight pack, and a supplied sparse row may then name its constant part as ONE entry (column D_n + s, value 1)
     * next to its dynamic entries: with sparse_input_nnz <= 6 the fused encoder runs 6 terms per row instead of 12.
     * static_only = 1: the supplied sparse rows index the static rows ALONE (entry s = static row s; dynamic fields name
     * unit rows among them): the weight pack then holds S instead of D_n + S rows per chunk, which buys the fused kernel
     * a deeper weight ring.  The pack depends on these rows: repack when they change. */
    const float* static_rows;
    int32_t n_static_rows, static_only;
} gm_netmon_params;

/* Packed tensor-core weights (GM_MATH_BF16X3 / GM_MATH_BF16): the fp32 parameters split into bf16
 * hi/lo tiles in the shared-memory layout the tcgen05 kernels stream with bulk copies.  Pack once
 * per parameter update and pass the buffer in params.packed. */
GM_API int64_t gm_netmon_packed_bytes(const gm_netmon_params* p);
GM_API int gm_netmon_pack_weights(const gm_netmon_params* p, void* packed, int64_t packed_bytes, void* stream);

/* bytes of device scratch gm_netmon_forward needs for R = B*N rows */
GM_API int64_t gm_netmon_workspace_bytes(const gm_netmon_params* p, int64_t rows);

/* Dense adjacency mask -> padded neighbour lists (model.py:213-229 sums over mask!=0
 * columns; :597-614 orders neighbours by ascending node id).
 *   mask f32[B,N,N]; out: nbr_all i32[B,N,DM] (ascending ids with mask!=0, incl. self if
 *   set, -1 padded), deg i32[B,N]. Rows with more than DM entries set *overflow (device int). */
GM_API int gm_adj_to_lists(const float* mask, int32_t B, int32_t N, int32_t DM, int32_t* nbr_all,
                    int32_t* deg, int32_t* overflow, void* stream);

/* One NetMon step for B graphs of N nodes.
 *   node_obs f32[B,N,D_n]
 *   nbr_all  i32[L,N,DM], deg i32[L,N]: adjacency lists (from gm_adj_to_lists or built from
 *            the topology pool); list_index i32[B] maps env -> list (NULL: env b uses list b)
 *   state_in f32[B,N,S] or NULL (= zeros, model.py:480-484); state_out f32[B,N,S]
 *   max_degree: neighbour slots in the readout (model.py:588-589), <= DM
 *   node_out f32[B,N,O] or NULL; agent_node i32[B,A] + agent_out f32[B,A,O] (row stride
 *   agent_out_ld floats) or NULL: graph observation of each agent = node_out[agent_node]
 *   (model.py:629-631 with a one-hot node-agent matrix).
 *   agent_out_pk: optional (tensor-core modes) copy of agent_out as tile-packed bf16 hi/lo blocks
 *   (gm_packed_activation_bytes(B*A, O) bytes, 128-byte aligned) that gm_dqn_act can consume as
 *   obs_g_pk instead of re-reading the fp32 rows.
 *   state_h_pk_in / state_h_pk_out: optional (fused tensor-core cells only; NULL otherwise) tile-packed copy of
 *   the hidden half of the state (gm_packed_activation_bytes(B*N, H) bytes, 128-byte aligned).  The last cell of a
 *   step writes state_h_pk_out next to state_out; handing it back as state_h_pk_in with the same state lets the next
 *   step's rnn_obs cell pull h with bulk copies instead of re-splitting the fp32 rows.
 *   workspace: device scratch of gm_netmon_workspace_bytes (256-byte aligned). */
GM_API int64_t gm_packed_activation_bytes(int64_t rows, int32_t width);
GM_API int gm_netmon_forward(const gm_netmon_params* p, int32_t B, int32_t N, const float* node_obs,
                      const int32_t* nbr_all, const int32_t* deg, int32_t DM,
                      const int32_t* list_index, const float* state_in, float* state_out,
                      int32_t max_degree, float* node_out, const int32_t* agent_node, int32_t A,
                      float* agent_out, int64_t agent_out_ld, void* agent_out_pk, const void* state_h_pk_in,
                      void* state_h_pk_out, void* workspace, int64_t workspace_bytes, void* stream);
/* general node->agent mapping with an arbitrary (not one-hot) node_agent matrix f32[B,N,A]
 * (NetMon.output_to_network_obs, model.py:629-631; frozen wrapper path wrapper.py:67-75) */
GM_API int gm_netmon_map_to_agents(const float* node_out, const float* node_agent, int32_t B, int32_t N,
                            int32_t A, int32_t O, float* agent_out, void* stream);

/* ======================================================================== */
/* DQN forward + epsilon-greedy (replaces src/model.py:199-203,              */
/* src/policy.py:20-51)                                                      */
/* ======================================================================== */
typedef struct gm_dqn_params {
    int32_t in_features;                    /* D_j = D_a + D_g */
    int32_t n_layers;                       /* encoder MLP layers */
    int32_t units[GM_MAX_LAYERS];
    int32_t n_actions, activation, math;
    const float* w[GM_MAX_LAYERS];
    const float* b[GM_MAX_LAYERS];
    const float *q_w, *q_b;                 /* [n_actions, units[last]] */
    /* tensor-core modes only: weights packed by gm_dqn_pack_weights for input rows split as
     * [packed_split | in_features - packed_split] (0 = one segment); NULL = pack every call */
    const void* packed;
    int32_t packed_split, pad;
} gm_dqn_params;

GM_API int64_t gm_dqn_packed_bytes(const gm_dqn_params* p, int32_t split);
GM_API int gm_dqn_pack_weights(const gm_dqn_params* p, int32_t split, void* packed, int64_t packed_bytes, void* stream);

GM_API int64_t gm_dqn_workspace_bytes(const gm_dqn_params* p, int64_t rows);
/* rows = B*A agents. Input row r = [obs_a[r, 0:Da] | obs_g[r, 0:Dg]] (the concat of
 * wrapper.py:50 without materialising it); obs_g may be NULL with Dg = 0.
 *   obs_g_pk: optional tile-packed copy of obs_g written by gm_netmon_forward (same math mode).
 *   action_mask u8[rows,n_actions] or NULL: masked actions get Q = -inf (policy.py:42-43)
 *   rand_action i32[rows], rand_u f64[rows]: host-supplied draws (policy.py:46-47), both NULL
 *   => device Philox(seed, step + *philox_step_dev) (philox_step_dev: optional device counter, see
 *   gm_routing_io).  act[r] = rand_u<eps ? rand_action : argmax (first max).
 *   q_out f32[rows,n_actions] or NULL; act_out i32[rows]. */
GM_API int gm_dqn_act(const gm_dqn_params* p, int64_t rows, const float* obs_a, int32_t Da, int64_t lda,
               const float* obs_g, int32_t Dg, int64_t ldg, const void* obs_g_pk, const uint8_t* action_mask,
               double epsilon, const int32_t* rand_action, const double* rand_u,
               uint64_t philox_seed, uint64_t philox_step, const uint64_t* philox_step_dev, float* q_out, int32_t* act_out,
               void* workspace, int64_t workspace_bytes, void* stream);

/* ======================================================================== */
/* Replay ring (replaces src/replaybuffer.py:243-287 add, :132-187 gather)   */
/* ======================================================================== */
#define GM_REPLAY_MAX_FIELDS 24
typedef struct gm_replay_field {
    void* ring;            /* device [capacity, elem_bytes] */
    const void* src;       /* device source for insert; unused for sample */
    void* dst;             /* device [n, elems] for sample; unused for insert */
    int64_t elem_bytes;    /* bytes of one transition of this field in the ring */
    int32_t convert;       /* sample: 0 raw copy, 1 u8/bool->f32, 2 i8->i64, 3 f16->f32;
                              insert: 0 raw copy, 4 i32 source elements -> i8 ring elements */
    int32_t broadcast;     /* insert: src holds ONE transition that is written to all n slots */
    /* insert, optional 2-D sub-block: per transition the source holds `rows` contiguous rows of
     * `row_bytes`, written at byte offset ring_offset + row * ring_pitch inside the transition
     * (e.g. the agent part and the graph part of the joint observation, wrapper.py:50, land in
     * one ring row without a concat).  rows = 0: plain contiguous copy of elem_bytes. */
    int32_t rows, pad;
    int64_t row_bytes, ring_pitch, ring_offset;
} gm_replay_field;
/* copy n consecutive transitions into ring slots (index + *index_dev + i) % capacity
 * (index_dev: optional device counter for CUDA-graph replays, may be NULL) */
GM_API int gm_replay_insert(const gm_replay_field* fields, int32_t n_fields, int64_t capacity,
                     int64_t index, const int64_t* index_dev, int64_t n, void* stream);
/* gather n transitions ring[indices[i]] -> dst[i] with the dtype conversions of
 * ReplayBuffer._get_transition_batch; indices i64[n] on device */
GM_API int gm_replay_sample(const gm_replay_field* fields, int32_t n_fields, const int64_t* indices,
                     int64_t n, void* stream);

/* Index streams of ReplayBuffer.get_batch (src/replaybuffer.py:101, :111-130): numpy's
 * default_rng(seed) (PCG64 seeded through SeedSequence) and Generator.choice(n, size, replace=True),
 * restated bit-exactly.  `state` is GM_PCG64_STATE_WORDS uint64 (128-bit LCG state hi/lo, increment
 * hi/lo, "has buffered uint32" flag, buffered uint32). */
#define GM_PCG64_STATE_WORDS 6
GM_API void gm_pcg64_seed(uint64_t* state, uint64_t seed);                             /* host: default_rng(seed) */
GM_API void gm_pcg64_choice(uint64_t* state, int64_t n, int64_t size, int64_t* out);   /* host: rng.choice(n, size) */
/* device-side sampler: the generator state lives in HBM (state_dev, seeded on the host and copied) and
 * advances there; out i64[max(seq_len,1), batch] (device) receives the ring slots of get_batch:
 * seq_len <= 1: choice(count, batch); else start = (index % count + choice(count - seq_len, batch)) % count
 * and row o = (start + o) % count.  No host round trip. */
GM_API int gm_replay_sample_indices(uint64_t* state_dev, int64_t count, int64_t index, int32_t batch,
                             int32_t seq_len, int64_t* out, void* stream);
/* Per-env sequences on a ring that each batched step fills with num_envs consecutive slots (one per env), for the
 * batched learner: with S = steps_stored, start_i = (head_step % S + choice(S - seq_len)) % S for i < batch (the rule
 * above counted in steps), then env_i = choice(num_envs) for i < batch, both from the same device PCG64 state;
 * out i64[seq_len, batch] row o = ((start_i + o) % S) * num_envs + env_i. */
GM_API int gm_replay_sample_env_sequences(uint64_t* state_dev, int64_t steps_stored, int64_t head_step, int32_t num_envs,
                                   int32_t batch, int32_t seq_len, int64_t* out, void* stream);

/* ======================================================================== */
/* Training path: forward with a tape + backward (replaces the torch autograd */
/* of the learner, src/main.py:830-1006, src/sl.py:366-428, over               */
/* src/model.py:32-42, 199-203, 213-229, 476-631)                              */
/* ======================================================================== */
/* An MLP (model.py:13-42; the DQN of :187-203 = its encoder layers + the Q head as a last layer without
 * activation).  act[l] = GM_ACT_* or -1 for identity. */
typedef struct gm_mlp_desc {
    int32_t n_layers, in_features;
    int32_t units[GM_MAX_LAYERS];
    int32_t act[GM_MAX_LAYERS];
    int32_t math, pad;                  /* GM_MATH_FP32 | GM_MATH_BF16X3 (forward GEMMs; the backward GEMMs are fp32) */
    const float* w[GM_MAX_LAYERS];      /* [units[l], in_l] row-major */
    const float* b[GM_MAX_LAYERS];
} gm_mlp_desc;
typedef struct gm_mlp_grads {           /* device outputs, written (not accumulated); NULL = not wanted */
    float* w[GM_MAX_LAYERS];
    float* b[GM_MAX_LAYERS];
} gm_mlp_grads;
/* tape = the post-activation output of every layer, layer l at float offset rows * sum(units[0..l-1]); the last
 * block is the module's output */
GM_API int64_t gm_mlp_tape_floats(const gm_mlp_desc* m, int64_t rows);
GM_API int64_t gm_mlp_train_workspace_bytes(const gm_mlp_desc* m, int64_t rows);
GM_API int gm_mlp_forward_train(const gm_mlp_desc* m, int64_t rows, const float* x, int64_t ldx, float* tape,
                         void* workspace, int64_t workspace_bytes, void* stream);
/* d_out f32[rows, units[last]] (row stride ldd) -> parameter gradients and, if d_x != NULL, d_x f32[rows, in_features] */
GM_API int gm_mlp_backward(const gm_mlp_desc* m, int64_t rows, const float* x, int64_t ldx, const float* tape,
                    const float* d_out, int64_t ldd, float* d_x, const gm_mlp_grads* grads, void* workspace,
                    int64_t workspace_bytes, void* stream);

typedef struct gm_cell_grads {
    float *w_ih, *w_hh, *b_ih, *b_hh;                                           /* b_hh: nn.LSTMCell only */
    float *ln_in_w, *ln_in_b, *ln_hid_w, *ln_hid_b, *ln_cell_w, *ln_cell_b;     /* LayerNormLSTMCell only */
} gm_cell_grads;
typedef struct gm_netmon_grads {
    float* enc_w[GM_MAX_LAYERS];
    float* enc_b[GM_MAX_LAYERS];
    gm_cell_grads rnn_obs, rnn_update;
} gm_netmon_grads;
/* One NetMon step with a tape (rnn_type lstm or lnlstm with carry-over, agg sum | mean, K >= 1, no global readout;
 * anything else returns GM_ERR_INVALID).  Arguments as gm_netmon_forward; node_out f32[B,N,O] (O = H (1 + max_degree) with the
 * neighbour readout) or NULL; state_in f32[B,N,2H] or NULL (= zeros). */
GM_API int64_t gm_netmon_tape_floats(const gm_netmon_params* p, int64_t rows);
GM_API int64_t gm_netmon_train_workspace_bytes(const gm_netmon_params* p, int64_t rows);
GM_API int gm_netmon_forward_train(const gm_netmon_params* p, int32_t B, int32_t N, const float* node_obs,
                            const int32_t* nbr_all, const int32_t* deg, int32_t DM, const int32_t* list_index,
                            const float* state_in, float* state_out, int32_t max_degree, float* node_out, float* tape,
                            void* workspace, int64_t workspace_bytes, void* stream);
/* Backward of that step: d_node_out f32[B,N,O] and / or d_state_out f32[B,N,2H] (gradients of the step's two outputs;
 * either may be NULL = zero) -> d_state_in f32[B,N,2H] (may be NULL) and the parameter gradients (written, not
 * accumulated: a sequence of steps sums them outside, as autograd does). */
GM_API int gm_netmon_backward(const gm_netmon_params* p, int32_t B, int32_t N, const float* node_obs, const int32_t* nbr_all,
                       const int32_t* deg, int32_t DM, const int32_t* list_index, const float* state_in,
                       int32_t max_degree, const float* tape, const float* d_node_out, const float* d_state_out,
                       float* d_state_in, const gm_netmon_grads* grads, void* workspace, int64_t workspace_bytes,
                       void* stream);

/* ======================================================================== */
/* Optional learner collective (hook between loss.backward() and             */
/* optimizer.step(), src/main.py:1002-1004; SURVEY 8e): one fused NCCL        */
/* all-reduce of the flat fp32 gradient.  The rollout path has no collective. */
/* ======================================================================== */
#define GM_NCCL_UNIQUE_ID_BYTES 128
/* NCCL is bound at run time (the libnccl.so.2 already mapped into the process, else the system one); 0 = unavailable */
GM_API int gm_nccl_version(void);
/* rank 0 creates the id (host bytes) and the host code hands it to every rank (any transport) */
GM_API int gm_nccl_unique_id(uint8_t* id128);
GM_API int gm_nccl_comm_create(int32_t world_size, int32_t rank, const uint8_t* id128, void** comm);
GM_API int gm_nccl_comm_destroy(void* comm);
/* flat f32[n] (device) <- sum (average = 0) or mean (average = 1) over the ranks, in place, asynchronous on stream */
GM_API int gm_allreduce_grads(void* comm, float* flat, int64_t n, int32_t average, void* stream);
/* start-up: every rank's flat parameter buffer <- rank root's */
GM_API int gm_broadcast_weights(void* comm, float* flat, int64_t n, int32_t root, void* stream);

/* ======================================================================== */
/* Batched DQN learner (graph_marl_b200/learner.py): TD gradient + optimizer */
/* tail.  Fixed-order reductions (no float atomics): eager calls and CUDA-   */
/* graph replays agree bit for bit.  `partials` is a device workspace of     */
/* GM_LEARNER_PARTIALS doubles.                                              */
/* ======================================================================== */
#define GM_LEARNER_PARTIALS 296
/* q, q_next f32[rows, n_actions] (online / target network), action i64[rows], reward f32[rows], done bool[rows]:
 * y = reward + (!done) * gamma * max_a q_next (a NaN in a q_next row propagates, like torch.max); dq = 2 * scale * (q - y)
 * at the taken action, 0 elsewhere;
 * *loss (device f32) += scale * sum_rows (q[action] - y)^2 */
GM_API int gm_td_grad(const float* q, const float* q_next, const int64_t* action, const float* reward, const uint8_t* done,
               int64_t rows, int32_t n_actions, float gamma, float scale, float* dq, float* loss, double* partials,
               void* stream);
/* sl.py:395-400 (NetMonSL's all-pairs loss): pred f32[B*N, N] (row stride ldp), targets_all i32[S, N, N], index i64[B]
 * (NULL: sample b = row block b): y = (float)targets_all[index[b], v, u] for row b*N+v, column u;
 * d_pred (may be NULL: evaluation) = 2 * scale * (pred - y);  *loss (device f32) += scale * sum (pred - y)^2 */
GM_API int gm_sl_mse_grad(const float* pred, int64_t ldp, const int32_t* targets_all, const int64_t* index,
                          int32_t B, int32_t N, float scale, float* d_pred, float* loss, double* partials, void* stream);
typedef struct gm_opt_entry {           /* one optimised tensor (device pointers) */
    float *param, *grad, *exp_avg, *exp_avg_sq;
    int64_t numel;
} gm_opt_entry;
typedef struct gm_opt_pair {            /* one tensor of the target network and its online counterpart */
    const float* online;
    float* target;
    int64_t numel;
} gm_opt_pair;
typedef struct gm_opt_hparams {
    double lr, beta1, beta2, eps, weight_decay, tau;
    float clip_value, max_norm;
} gm_opt_hparams;
/* One update over the device tables: grads clamped to +-clip_value in place; their global L2 norm; grads scaled by
 * min(1, max_norm / (norm + 1e-6)) in place; *step_dev += 1; AdamW in the operation order of
 * torch.optim.AdamW(foreach=False); then target = tau * online + (1 - tau) * target for every pair. */
GM_API int gm_optimizer_step(const gm_opt_entry* table_dev, int32_t n_entries, const gm_opt_pair* pairs_dev,
                      int32_t n_pairs, int64_t* step_dev, const gm_opt_hparams* h, double* partials, void* stream);

/* ======================================================================== */
/* Batched evaluation (graph_marl_b200/evaluation.py): per-env sums of the   */
/* episode metrics, one row of GM_EVAL_FIELDS doubles per env.  No atomics:  */
/* repeated and captured launches agree bit for bit.                         */
/* ======================================================================== */
#define GM_EVAL_REWARD_SUM 0         /* sum of rewards over agents and steps */
#define GM_EVAL_AGENT_STEPS 1        /* agents x steps */
#define GM_EVAL_DELAY_SUM 2          /* sum of delays of done packets */
#define GM_EVAL_DELAY_COUNT 3        /* done packets */
#define GM_EVAL_ARRIVED_DELAY_SUM 4  /* sum of delays of arrived packets */
#define GM_EVAL_ARRIVED_COUNT 5      /* arrived packets */
#define GM_EVAL_SPR_SUM 6            /* sum of spr of arrived packets */
#define GM_EVAL_LOOPED 7             /* sums of info[:, 0..3] */
#define GM_EVAL_THROUGHPUT 8
#define GM_EVAL_DROPPED 9
#define GM_EVAL_BLOCKED 10
#define GM_EVAL_STEPS 11             /* env steps */
#define GM_EVAL_FIELDS 12
/* One env step's outputs (gm_routing_io: reward f32[B,A], done u8[B,A], arrived u8[B,A], delays i32[B,A], spr f64[B,A],
 * info i32[B,4]) added into acc f64[B, GM_EVAL_FIELDS]. */
GM_API int gm_eval_accumulate(const float* reward, const uint8_t* done, const uint8_t* arrived, const int32_t* delays,
                              const double* spr, const int32_t* info, int32_t B, int32_t A, double* acc, void* stream);

/* ======================================================================== */
/* building blocks exposed for tests / profiling                             */
/* ======================================================================== */
/* C[M,N] = act(A[M,K] * W[N,K]^T + bias) in the requested math mode */
GM_API int gm_linear(const float* A, int64_t lda, const float* W, const float* bias, float* C,
              int64_t ldc, int64_t M, int32_t N, int32_t K, int32_t activation, int32_t math,
              void* workspace, int64_t workspace_bytes, void* stream);
GM_API int64_t gm_linear_workspace_bytes(int64_t M, int32_t N, int32_t K, int32_t math);
/* Per-launch timing with CUDA events recorded on the launching stream: enable, run, then collect the
 * summed device time ms[8] and the launch count launches[8] per kernel category (collect synchronises on
 * the recorded events and clears them).  Categories: 0 tensor-core linear/cell/Q-head kernels, 1 routing
 * env step, 2 aggregation, 3 agent readout, 4 replay insert. */
#define GM_PROFILE_CATEGORIES 8
GM_API void gm_profile_enable(int on);
GM_API int gm_profile_collect(double* ms, int32_t* launches);
/* number of kernels this library launched since load (all streams), for bench accounting */
GM_API int64_t gm_kernel_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* GRAPHMARL_B200_H */
