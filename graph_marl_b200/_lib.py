"""ctypes binding of libgraphmarl_b200.so (include/graphmarl_b200.h).

The product has NO CPU fallback: device entry points raise `GraphMarlError` when the
library is missing or no sm_100 device is present.  Host-only entry points (legacy
MT19937 stream, topology generator) work without a GPU.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GM_LIB_PATH: a probe / experiment build of the same sources (tools/env_only.py, tools/tc_trace.py); default in-tree
LIB_PATH = os.environ.get("GM_LIB_PATH") or os.path.join(_HERE, "lib", "libgraphmarl_b200.so")

GM_MAX_LAYERS = 8
GM_REPLAY_MAX_FIELDS = 24
GM_MT_STATE_WORDS = 625
GM_TOPOLOGY_MAX_NODES = 512
GM_PCG64_STATE_WORDS = 6
GM_NCCL_UNIQUE_ID_BYTES = 128
RNN_TYPES = {"lstm": 0, "lnlstm": 1, "gru": 2, "none": 3}
AGG_TYPES = {"sum": 0, "mean": 1}
ACTIVATIONS = {"leaky_relu": 0, "relu": 1, "tanh": 2, "sigmoid": 3, "elu": 4}
MATH_MODES = {"fp32": 0, "bf16x3": 1, "bf16": 2}


class GraphMarlError(RuntimeError):
    pass


class RoutingDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "N", "A", "E", "T", "env_var", "k", "congestion",
                                         "action_mask", "ttl", "state_stride", "node_sparse_static")] + \
               [(n, C.c_void_p) for n in ("node_edges", "node_nbrs", "edges", "apsp", "topo_index", "state")]


class RoutingIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("actions", "env_mask", "draw_start", "draw_target", "draw_size")] + \
               [("philox_seed", C.c_uint64), ("philox_step", C.c_uint64), ("philox_step_dev", C.c_void_p)] + \
               [(n, C.c_void_p) for n in ("obs", "adj", "node_obs", "node_agent", "agent_node", "node_sparse", "reward",
                                          "done", "delays", "arrived", "spr", "info", "n_resets",
                                          "action_mask_out", "eval_f64", "eval_i32", "packet_dist", "packet_sizes",
                                          "sum_packets_per_node", "sum_packets_per_edge")] + \
               [(n, C.c_void_p) for n in ("ring_rec", "ring_next_rec", "ring_topo", "ring_action", "ring_reward", "ring_done",
                                          "ring_episode_done")] + \
               [("ring_capacity", C.c_int64), ("ring_index", C.c_int64), ("ring_index_dev", C.c_void_p),
                ("ring_episode_flag", C.c_int32), ("ring_pad", C.c_int32)]


class TopologyTables(C.Structure):
    _fields_ = [("P", C.c_int32), ("N", C.c_int32)] + \
               [(n, C.c_void_p) for n in ("edges", "node_edges", "node_nbrs", "apsp", "nbr_all", "deg")]


class CellParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("w_ih", "w_hh", "b_ih", "b_hh", "ln_in_w", "ln_in_b",
                                          "ln_hid_w", "ln_hid_b", "ln_cell_w", "ln_cell_b")]


class NetmonParams(C.Structure):
    _fields_ = [("in_features", C.c_int32), ("hidden", C.c_int32), ("n_enc_layers", C.c_int32),
                ("enc_units", C.c_int32 * GM_MAX_LAYERS), ("iterations", C.c_int32),
                ("rnn_type", C.c_int32), ("agg_type", C.c_int32), ("activation", C.c_int32),
                ("rnn_carryover", C.c_int32), ("output_neighbor_hidden", C.c_int32),
                ("output_global_hidden", C.c_int32), ("math", C.c_int32), ("sparse_input_nnz", C.c_int32),
                ("enc_w", C.c_void_p * GM_MAX_LAYERS), ("enc_b", C.c_void_p * GM_MAX_LAYERS),
                ("rnn_obs", CellParams), ("rnn_update", CellParams), ("packed", C.c_void_p), ("sparse_rows", C.c_void_p),
                ("static_rows", C.c_void_p), ("n_static_rows", C.c_int32), ("static_only", C.c_int32)]


class DqnParams(C.Structure):
    _fields_ = [("in_features", C.c_int32), ("n_layers", C.c_int32), ("units", C.c_int32 * GM_MAX_LAYERS),
                ("n_actions", C.c_int32), ("activation", C.c_int32), ("math", C.c_int32),
                ("w", C.c_void_p * GM_MAX_LAYERS), ("b", C.c_void_p * GM_MAX_LAYERS),
                ("q_w", C.c_void_p), ("q_b", C.c_void_p), ("packed", C.c_void_p),
                ("packed_split", C.c_int32), ("pad", C.c_int32)]


class ReplayField(C.Structure):
    _fields_ = [("ring", C.c_void_p), ("src", C.c_void_p), ("dst", C.c_void_p),
                ("elem_bytes", C.c_int64), ("convert", C.c_int32), ("broadcast", C.c_int32),
                ("rows", C.c_int32), ("pad", C.c_int32), ("row_bytes", C.c_int64), ("ring_pitch", C.c_int64),
                ("ring_offset", C.c_int64)]


class MlpDesc(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("in_features", C.c_int32), ("units", C.c_int32 * GM_MAX_LAYERS),
                ("act", C.c_int32 * GM_MAX_LAYERS), ("math", C.c_int32), ("pad", C.c_int32),
                ("w", C.c_void_p * GM_MAX_LAYERS), ("b", C.c_void_p * GM_MAX_LAYERS)]


class MlpGrads(C.Structure):
    _fields_ = [("w", C.c_void_p * GM_MAX_LAYERS), ("b", C.c_void_p * GM_MAX_LAYERS)]


class CellGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("w_ih", "w_hh", "b_ih", "b_hh", "ln_in_w", "ln_in_b", "ln_hid_w", "ln_hid_b",
                                          "ln_cell_w", "ln_cell_b")]


class NetmonGrads(C.Structure):
    _fields_ = [("enc_w", C.c_void_p * GM_MAX_LAYERS), ("enc_b", C.c_void_p * GM_MAX_LAYERS),
                ("rnn_obs", CellGrads), ("rnn_update", CellGrads)]


GM_LEARNER_PARTIALS = 296
# gm_eval_accumulate's row layout (GM_EVAL_* in the header), in field order
EVAL_FIELDS = ("reward_sum", "agent_steps", "delay_sum", "delay_count", "arrived_delay_sum", "arrived_count", "spr_sum",
               "looped", "throughput", "dropped", "blocked", "steps")


class OptEntry(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("param", "grad", "exp_avg", "exp_avg_sq")] + [("numel", C.c_int64)]


class OptPair(C.Structure):
    _fields_ = [("online", C.c_void_p), ("target", C.c_void_p), ("numel", C.c_int64)]


class OptHparams(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("lr", "beta1", "beta2", "eps", "weight_decay", "tau")] + \
               [("clip_value", C.c_float), ("max_norm", C.c_float)]


_lib = None

_SIGS = {
    "gm_last_error": (C.c_char_p, []),
    "gm_abi_version": (C.c_int, []),
    "gm_device_check": (C.c_int, []),
    "gm_kernel_launch_count": (C.c_int64, []),
    "gm_profile_enable": (None, [C.c_int]),
    "gm_profile_collect": (C.c_int, [C.c_void_p, C.c_void_p]),  # double ms[8], int32 launches[8]
    "gm_mt_seed": (None, [C.c_void_p, C.c_uint32]),
    "gm_mt_u32": (C.c_uint32, [C.c_void_p]),
    "gm_mt_random": (C.c_double, [C.c_void_p]),
    "gm_mt_randint": (C.c_uint32, [C.c_void_p, C.c_uint32]),
    "gm_mt_packet_draws": (None, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_mt_reset_draws": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_mt_policy_draws": (None, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "gm_topology_generate": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_topology_apsp": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "gm_topology_generate_device": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                              C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_topology_next_hops": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "gm_routing_state_layout": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "gm_routing_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_routing_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_routing_observe": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_simple_step": (C.c_int, [C.c_int32, C.c_int32] + [C.c_void_p] * 11),
    "gm_netmon_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "gm_adj_to_lists": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]),
    "gm_netmon_forward": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                    C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_packed_activation_bytes": (C.c_int64, [C.c_int64, C.c_int32]),
    "gm_netmon_map_to_agents": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_void_p]),
    "gm_dqn_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "gm_netmon_packed_bytes": (C.c_int64, [C.c_void_p]),
    "gm_netmon_pack_weights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_dqn_packed_bytes": (C.c_int64, [C.c_void_p, C.c_int32]),
    "gm_dqn_pack_weights": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_dqn_act": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int32,
                             C.c_int64, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_uint64,
                             C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_replay_insert": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_replay_sample": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_pcg64_seed": (None, [C.c_void_p, C.c_uint64]),
    "gm_pcg64_choice": (None, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "gm_replay_sample_indices": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "gm_replay_sample_env_sequences": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                                 C.c_void_p]),
    "gm_td_grad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float,
                             C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_sl_mse_grad": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "gm_eval_accumulate": (C.c_int, [C.c_void_p] * 6 + [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "gm_optimizer_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    "gm_mlp_tape_floats": (C.c_int64, [C.c_void_p, C.c_int64]),
    "gm_mlp_train_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "gm_mlp_forward_train": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_void_p]),
    "gm_mlp_backward": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_netmon_tape_floats": (C.c_int64, [C.c_void_p, C.c_int64]),
    "gm_netmon_train_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "gm_netmon_forward_train": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_netmon_backward": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_nccl_version": (C.c_int, []),
    "gm_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "gm_nccl_comm_create": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "gm_nccl_comm_destroy": (C.c_int, [C.c_void_p]),
    "gm_allreduce_grads": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "gm_broadcast_weights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "gm_linear": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                            C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "gm_linear_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32, C.c_int32]),
}

EXPORTS = sorted(_SIGS)


def lib():
    """Loads the library or raises (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GraphMarlError(
                f"{LIB_PATH} is missing: build it with `python -m graph_marl_b200.build` "
                "(graph_marl_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise GraphMarlError(f"libgraphmarl_b200 error {rc}: {lib().gm_last_error().decode()}")


_device_ok = None


def require_device():
    """Fails loudly when the CUDA path cannot run."""
    global _device_ok
    if _device_ok is None:
        check(lib().gm_device_check())
        _device_ok = True


def ptr(t):
    """data_ptr of a torch tensor / numpy array (or None)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def current_stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


class DeviceCounter:
    """A 64-bit device scalar that shadows a host counter so that a captured CUDA graph can replay calls
    whose step / ring index advances between replays: kernels read `*ptr + offset`, where `offset` (baked
    into the graph) is the host value at capture time minus `base`, and `set()` moves the base."""

    def __init__(self, device):
        import torch

        self.t = torch.zeros((1,), dtype=torch.int64, device=device)
        self.base = 0

    def set(self, value):
        self.base = int(value)
        self.t.fill_(self.base)

    def offset(self, value):
        return int(value) - self.base

    def ptr(self):
        return self.t.data_ptr()
