"""The supervised shortest-path dataset of the reference's src/sl.py (BASELINE config 5), built on the device.

sl.py builds it one sample at a time: a compat `Routing.reset()` per sample (a new topology from `Network.reset()`
and A packets from the global numpy stream), then networkx's shortest paths on the host for the next-hop label of
every node (sl.py:174-286).  `build_sl_dataset` builds the same samples chunk by chunk:

* the seeds and packet draws of the chunk's resets are replayed natively from the global stream
  (`gm_mt_reset_draws`), which is left exactly where the compat resets leave it;
* the chunk's topologies are generated into a `TopologyPool.slots` pool (`gm_topology_generate_device`);
* one batched `Routing` resets on that pool with those draws, which gives the node observations;
* labels come from the pool's next-hop tables (`gm_topology_next_hops`, networkx's tie-breaking), targets from its
  shortest-path weights.
"""
import numpy as np
import torch

from . import _lib
from .env.environment import EnvironmentVariant
from .env.network import Network, generate_tables
from .env.routing import Routing, TopologyPool

FIELDS = ("node_obs", "node_adj", "labels", "targets", "targets_all", "seeds")


def _seed_mode(net):
    """How Network.reset() picks its seed: 0 fresh draws, 1 sequential provided seeds (no draw), 2 np.random.choice."""
    if len(net.seeds) == 0:
        return 0
    return 1 if net.next_topology_seed_index(advance_index=False) is not None else 2


def reset_draws(net, n, n_data):
    """What n compat `Routing(net, n_data, ...).reset()` calls draw from the global numpy stream: the topology seeds
    Network.reset() picks (int64 [n]) and the packet triples (start, target int32 [n, n_data], size float64
    [n, n_data]).  Advances the global stream and the Network's sequential seed index as those calls do."""
    mode, N = _seed_mode(net), net.n_nodes
    seed_list = None
    if mode == 1:
        k, idx = len(net.seeds), net.sequential_topology_index
        if net.sequential_topology_seeds_frozen:
            pos = np.full(n, idx)
        else:
            pos = (idx + np.arange(n)) % k
            net.sequential_topology_index = (idx + n) % k
        seed_list = np.asarray(net.seeds, dtype=np.int64)[pos]
    elif mode == 2:
        seed_list = np.asarray(net.seeds, dtype=np.int64)
    ex = None
    if mode == 0 and net.exclude_seeds:
        ex = np.fromiter(net.exclude_seeds, np.int64, len(net.exclude_seeds))
    name, key, pos_, has_gauss, gauss = np.random.get_state()
    st = np.zeros(_lib.GM_MT_STATE_WORDS, np.uint32)
    st[:624], st[624] = key, pos_
    seeds = np.zeros(max(n, 1), np.int64)
    start, target = np.zeros((max(n, 1), n_data), np.int32), np.zeros((max(n, 1), n_data), np.int32)
    size = np.zeros((max(n, 1), n_data), np.float64)
    _lib.check(_lib.lib().gm_mt_reset_draws(_lib.ptr(st), mode, _lib.ptr(seed_list),
                                            0 if seed_list is None else seed_list.size, _lib.ptr(ex),
                                            0 if ex is None else ex.size, N, n, n_data, _lib.ptr(seeds),
                                            _lib.ptr(start), _lib.ptr(target), _lib.ptr(size)))
    np.random.set_state((name, st[:624].copy(), int(st[624]), has_gauss, gauss))
    return seeds[:n], start[:n], target[:n], size[:n]


def build_sl_dataset(network: Network, n_samples, n_data=20, chunk=4096, device="cuda"):
    """sl.py's dataset of `n_samples` samples as device tensors, bit-identical to n_samples compat resets of
    `Routing(network, n_data, INDEPENDENT)` with the labels and targets of get_sl_sample (sl.py:174-219):

        node_obs f32 [S, N, 4N+8]   node observations after the reset
        node_adj i8  [S, N, N]      adjacency with self loops
        labels   i8  [S, N]         1 + index in nodes[v].edges of the first hop towards node 0 (0 at node 0)
        targets  i32 [S, N]         shortest-path weight to node 0
        targets_all i32 [S, N, N]   all shortest-path weights
        seeds    i64 [S]            the topology seed each sample used

    The global numpy stream and the Network (seed index, sampled seeds, current topology and its host views) end as
    after those resets.  A provided seed that is not a valid topology raises AssertionError as Network.reset() does."""
    _lib.require_device()
    net, S, A = network, int(n_samples), int(n_data)
    if S < 1 or int(chunk) < 1:
        raise ValueError(f"build_sl_dataset needs n_samples >= 1 and chunk >= 1, got {S}, {chunk}")
    N, dev = net.n_nodes, torch.device(device)
    mode = _seed_mode(net)
    e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)
    out = dict(node_obs=e((S, N, 4 * N + 8), torch.float32), node_adj=e((S, N, N), torch.int8),
               labels=e((S, N), torch.int8), targets=e((S, N), torch.int32), targets_all=e((S, N, N), torch.int32),
               seeds=e((S,), torch.int64))
    P = min(int(chunk), S)
    pool = TopologyPool.slots(P, N, dev)
    exclude = None
    if mode == 0 and net.exclude_seeds:
        exclude = torch.from_numpy(np.array(sorted(net.exclude_seeds), np.int64)).to(dev)
    envs = {}
    last_seed = None
    for lo in range(0, S, P):
        c = min(P, S - lo)
        seeds, start, target, size = reset_draws(net, c, A)
        slot = torch.arange(c, dtype=torch.int32, device=dev)
        used, _ = pool.generate(seeds, slot, exclude)
        if mode != 0 and not np.array_equal(used, seeds):  # the device generator reseeds; a provided seed must not
            bad = int(np.flatnonzero(used != seeds)[0])
            raise AssertionError(f"Provided seed {int(seeds[bad])} is invalid.")
        if c not in envs:
            envs[c] = Routing(net, A, EnvironmentVariant.INDEPENDENT, num_envs=c, device=dev, batched=True)
        env = envs[c]
        env.set_draws(start, target, size)
        env.reset_on_pool(pool, slot)
        hi = lo + c
        out["node_obs"][lo:hi] = env.get_node_observation()
        out["node_adj"][lo:hi] = env.get_nodes_adjacency()
        out["labels"][lo:hi] = pool.next_hop[:c, :, 0]
        out["targets_all"][lo:hi] = pool.apsp[:c]
        out["targets"][lo:hi] = pool.apsp[:c, :, 0]
        out["seeds"][lo:hi] = torch.from_numpy(used)
        net.sampled_topology_seeds.extend(int(s) for s in used)
        last_seed = int(seeds[-1])
    # the last sample's topology once more on the host, for the Network's attribute views (nodes, edges, adj_matrix)
    used_last = net.sampled_topology_seeds[-1]
    net._install(generate_tables(N, last_seed, allow_reseed=mode == 0, exclude=net.exclude_seeds if mode == 0 else None))
    if net.current_topology_seed != used_last:
        raise _lib.GraphMarlError(f"device topology from seed {last_seed} ended on seed {used_last}, "
                                  f"the host generator on {net.current_topology_seed}")
    return out
