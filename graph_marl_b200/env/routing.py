"""Routing environment, mirrors src/env/routing.py of the reference over the batched CUDA
kernel in csrc/routing_env.cu.

    Routing(network, n_data, env_var, k=3, enable_congestion=True,
            enable_action_mask=False, ttl=0)                      # reference signature
    ... , num_envs=B, device="cuda", seed=0)                       # batched extension

* num_envs == 1 (default, "compat"): `reset()` / `step()` return numpy arrays of the
  reference's shapes and dtypes and consume the global legacy `np.random` stream exactly
  like routing.py:130-135 (three draws per respawned packet, in packet-id order), so the
  class drops into src/main.py / src/eval.py unchanged.
* num_envs  > 1 ("batched"): every returned object is a CUDA tensor with a leading num_envs
  dimension; nothing leaves the device.  Packet draws come from a device Philox stream unless
  `set_draws()` supplies tables.

All state lives in one packed record per env in HBM and is advanced in place.
"""
import ctypes as C
import textwrap
from collections import defaultdict
from types import SimpleNamespace

import numpy as np
import torch

from .. import _lib
from .environment import EnvironmentVariant, NetworkEnv
from .network import Network, generate_tables, lists_from_tables


class Discrete:
    """Minimal stand-in for gymnasium.spaces.Discrete (only `.n`/`.start`/`.sample()` are used,
    routing.py:108, policy.py:150)."""

    def __init__(self, n, start=0):
        self.n = int(n)
        self.start = int(start)

    def sample(self):
        return self.start + int(np.random.randint(self.n))


class TopologyPool:
    """Device-resident tables of T topologies (SURVEY.md 7.2)."""

    def __init__(self, tables, device):
        self.T = len(tables)
        st = lambda k: torch.from_numpy(np.ascontiguousarray(np.stack([t[k] for t in tables]))).to(device)
        self.node_edges = st("node_edges")
        self.node_nbrs = st("node_nbrs")
        self.edges = st("edges")
        self.apsp = st("apsp")
        lists = [lists_from_tables(t) for t in tables]
        self.nbr_all = torch.from_numpy(np.stack([l[0] for l in lists])).to(device)
        self.deg = torch.from_numpy(np.stack([l[1] for l in lists])).to(device)
        self.seeds = [t.get("seed") for t in tables]
        self.edges_host = np.array(tables[0]["edges"], copy=True) if self.T == 1 else None
        self.fresh = False  # slots() pools: filled by generate()
        # The constant part of every node observation row (routing.py:193-234: one-hot of the node, of its three
        # neighbours, the three edge lengths) as dense rows, for small pools: NetMon folds layer 1 applied to them into
        # its weight pack and the env then names that part of a row as ONE sparse entry (model.NetMon).  The five
        # dynamic fields (#waiting, size sum, three edge loads) follow as unit rows, so that a row is six indices into
        # this [T*N + 5, 4N+8] dictionary and nothing else (gm_netmon_params.static_only).
        self.static_rows = None
        N = tables[0]["node_edges"].shape[0]
        if self.T * N + 5 <= 73:  # four weight-ring slots in the fused encoder (gemm_sm100_encfused.inc: ef_plan)
            rows = np.zeros((self.T * N + 5, 4 * N + 8), np.float32)
            for t, tab in enumerate(tables):
                for j in range(N):
                    r = rows[t * N + j]
                    r[j] = 1.0
                    for q in range(3):
                        b2 = N + 2 + q * (N + 2)
                        r[b2 + int(tab["node_nbrs"][j, q])] = 1.0
                        r[b2 + N] = float(tab["edges"][int(tab["node_edges"][j, q])][2])
            dyn = self.T * N
            rows[dyn, N] = 1.0
            rows[dyn + 1, N + 1] = 1.0
            for q in range(3):
                rows[dyn + 2 + q, N + 2 + q * (N + 2) + N + 1] = 1.0
            self.static_rows = torch.from_numpy(rows).to(device)

    @classmethod
    def slots(cls, P, n_nodes, device):
        """P empty slots at fixed device addresses, filled by generate() (Routing's fresh-topology mode).  Such a pool has
        no static rows: its slots change from episode to episode, NetMon's weight pack could not fold them in."""
        pool = cls.__new__(cls)
        N, E = int(n_nodes), 3 * int(n_nodes) // 2
        z = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=device)
        pool.T = int(P)
        pool.node_edges, pool.node_nbrs, pool.edges, pool.apsp = z(P, N, 3), z(P, N, 3), z(P, E, 4), z(P, N, N)
        pool.nbr_all, pool.deg = z(P, N, 4), z(P, N)
        pool.seeds = [None] * pool.T
        pool.edges_host = None
        pool.static_rows = None
        pool.fresh = True
        return pool

    def generate(self, seeds, slot, exclude=None, max_attempts=10000):
        """Generate topology b from seeds[b] (gm_topology_generate_device: what generate_tables(N, seeds[b],
        allow_reseed=True, exclude) builds) into slot slot[b] (device int32 [B]), in place, and refresh the lazily built
        caches of those slots.  exclude: device int64 tensor of seeds a reseed must skip.  Returns the host arrays
        (seed_used int64 [B], repetitions int32 [B]); raises GraphMarlError when an env found no valid topology within
        `max_attempts` graphs."""
        _lib.require_device()
        dev, N, B = self.apsp.device, self.apsp.shape[-1], len(seeds)
        seeds = np.ascontiguousarray(seeds, dtype=np.int64)
        seeds_d = torch.from_numpy(seeds).to(dev)
        used = torch.empty((B,), dtype=torch.int64, device=dev)
        reps = torch.empty((B,), dtype=torch.int32, device=dev)
        status = torch.zeros((1,), dtype=torch.int32, device=dev)
        t = _lib.TopologyTables(P=self.T, N=N, edges=self.edges.data_ptr(), node_edges=self.node_edges.data_ptr(),
                                node_nbrs=self.node_nbrs.data_ptr(), apsp=self.apsp.data_ptr(), nbr_all=self.nbr_all.data_ptr(),
                                deg=self.deg.data_ptr())
        n_ex = 0 if exclude is None else exclude.numel()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gm_topology_generate_device(C.byref(t), B, seeds_d.data_ptr(), slot.data_ptr(),
                                                              _lib.ptr(exclude) if n_ex else None, n_ex, int(max_attempts),
                                                              used.data_ptr(), reps.data_ptr(), status.data_ptr(),
                                                              _lib.current_stream()))
        st = int(status.item())
        if st > 0:
            raise _lib.GraphMarlError(f"no valid {N}-node topology within {max_attempts} attempts from seed {int(seeds[st - 1])}")
        if st < 0:
            raise _lib.GraphMarlError(f"env {-st - 1}: topology slot outside the pool's {self.T} slots")
        sl = slot.long()
        if getattr(self, "_next_hop", None) is not None:
            self._next_hop[sl] = self.next_hops(slot)
        if getattr(self, "apsp_f32", None) is not None:
            self.apsp_f32[sl] = self.apsp[sl].float()
        if getattr(self, "node_adj", None) is not None:
            adj = torch.zeros((B, N, N), dtype=torch.int8, device=dev)
            adj.scatter_(2, self.nbr_all[sl].long(), 1)
            self.node_adj[sl] = adj
        used, reps = used.cpu().numpy(), reps.cpu().numpy()
        for s_, u in zip(slot.cpu().tolist(), used.tolist()):
            self.seeds[s_] = u
        return used, reps

    def next_hops(self, slot):
        """Next-hop tables of the slots slot[i] (device int32 [n]) as int8 [n, N, N] (gm_topology_next_hops): entry
        [i, v, t] is 0 for v == t, else 1 + the index in nodes[v].edges of the edge towards the first hop of
        Network.shortest_paths[v][t] -- networkx's path, ties included."""
        _lib.require_device()
        dev, N, n = self.apsp.device, self.apsp.shape[-1], slot.numel()
        out = torch.empty((n, N, N), dtype=torch.int8, device=dev)
        t = _lib.TopologyTables(P=self.T, N=N, edges=self.edges.data_ptr(), node_edges=self.node_edges.data_ptr(),
                                node_nbrs=self.node_nbrs.data_ptr(), apsp=self.apsp.data_ptr(), nbr_all=self.nbr_all.data_ptr(),
                                deg=self.deg.data_ptr())
        slot = slot.to(device=dev, dtype=torch.int32).contiguous()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gm_topology_next_hops(C.byref(t), self.T, slot.data_ptr(), n, out.data_ptr(),
                                                        _lib.current_stream()))
        return out

    @property
    def next_hop(self):
        """int8 [T, N, N] next-hop tables of every slot (next_hops), built on first use; generate() refreshes the
        regenerated slots once it exists."""
        if getattr(self, "_next_hop", None) is None:
            self._next_hop = self.next_hops(torch.arange(self.T, dtype=torch.int32, device=self.apsp.device))
        return self._next_hop


class Routing(NetworkEnv):
    """Packet routing on a random 3-regular graph (routing.py:43-552)."""

    def __init__(self, network: Network, n_data, env_var, k=3, enable_congestion=True,
                 enable_action_mask=False, ttl=0, num_envs=1, device=None, seed=0, batched=None):
        super().__init__()
        assert isinstance(network, Network)
        self.network = network
        self.n_data = n_data
        self.env_var = EnvironmentVariant(env_var)
        self.k = k
        self.num_random_targets = self.network.n_nodes
        self.distance_map = defaultdict(list)
        self.enable_ttl = ttl > 0
        self.enable_congestion = enable_congestion
        self.ttl = ttl
        self.sum_packets_per_node = None
        self.sum_packets_per_edge = None
        self.enable_action_mask = enable_action_mask
        self.action_space = Discrete(4, start=0)
        self.eval_info_enabled = False
        # a node observation row (routing.py:193-234) has at most 12 non-zero entries: one-hot(node), #waiting, their
        # size sum, 3 x (one-hot(neighbour), length, load); NetMon's tensor-core encoder exploits that
        self._node_obs_nnz = 12

        self.num_envs = int(num_envs)
        self.batched = (self.num_envs > 1) if batched is None else bool(batched)
        self.device = torch.device(device if device is not None else "cuda")
        self._seed = int(seed)
        self._calls = 0
        N, A = network.n_nodes, n_data
        self._N, self._A, self._E = N, A, 3 * N // 2
        lay = np.zeros(8, np.int32)
        _lib.check(_lib.lib().gm_routing_state_layout(N, A, self._E, _lib.ptr(lay)))
        self._layout = dict(size=int(lay[0]), load=int(lay[1]), i32=int(lay[2]), vis=int(lay[3]),
                            mask=int(lay[4]), stride=int(lay[5]), VW=int(lay[6]))
        self._state = None
        self._pool = None
        self._topo_index = None
        self._topo_episodes = 1  # fresh-topology mode: episodes whose pool slots are kept (set_topology_episodes)
        self._episode = 0
        self._exclude_dev = None
        self._draws = None
        self._ring = None  # set_ring(): the next step writes its compact replay transition itself
        self._out = {}
        self._sum_node = self._sum_edge = None
        self._dev_step = None
        self.action_mask = np.zeros((n_data, 4), dtype=bool)
        self.agent_steps = np.zeros(n_data)

    # ------------------------------------------------------------------------------------------
    @property
    def node_obs_nnz(self):
        """Entries per row of the `node_sparse` output: 12, or 6 when the pool is small enough for static rows."""
        return 6 if (self._pool is not None and self._pool.static_rows is not None) else self._node_obs_nnz

    @property
    def node_static_rows(self):
        return None if self._pool is None else self._pool.static_rows

    def set_eval_info(self, val):
        """Whether step() returns the evaluation extras (routing.py:111-117, 384-386, 414-441)."""
        self.eval_info_enabled = bool(val)

    def obs_width(self):
        N = self._N
        W = 6 * N + 10
        if self.env_var == EnvironmentVariant.WITH_K_NEIGHBORS:
            W += 5 * self.k
        elif self.env_var == EnvironmentVariant.GLOBAL:
            W += N * N + N * (4 * N + 8)
        return W

    def __str__(self) -> str:
        return textwrap.dedent(
            f"""\
            Routing environment with parameters
            > Network: {self.network.n_nodes} nodes
            > Number of packets: {self.n_data}
            > Environment variant: {self.env_var.name}
            > Number of considered neighbors (k): {self.k if self.env_var == EnvironmentVariant.WITH_K_NEIGHBORS else "disabled"}
            > Congestion: {self.enable_congestion}
            > Action mask: {self.enable_action_mask}
            > TTL: {self.ttl if self.enable_ttl else "disabled"}
            > Instances: {self.num_envs} on {self.device} (libgraphmarl_b200)\
            """
        )

    # ---- device plumbing -----------------------------------------------------------------------
    def set_topology_pool(self, pool: TopologyPool, topo_index=None):
        self._pool = pool
        self._topo_index = topo_index

    def set_topology_episodes(self, S):
        """Fresh-topology mode (batched, Network(random_topology=True) without a seed list): the pool keeps the topologies
        of the last S episodes, B * S slots at fixed addresses; env b's topology of episode e lives in slot
        (e mod S) * B + b.  A compact replay ring names a transition's topology by its slot, so S must exceed the number
        of episodes whose transitions the ring can still hold.  Default 1: a reset overwrites the previous episode's
        topologies.  Takes effect at the next reset (a pool of another size is allocated then)."""
        S = int(S)
        if S < 1:
            raise ValueError(f"set_topology_episodes needs S >= 1, got {S}")
        self._topo_episodes = S

    def set_draws(self, start, target, size):
        """Host-supplied packet draws for the NEXT reset/step: arrays [B,A] (or [A]); slot s
        feeds the s-th respawn in packet-id order."""
        B, A = self.num_envs, self._A

        def mk(a, dt, tdt):
            if torch.is_tensor(a):
                return a.to(device=self.device, dtype=tdt).reshape(B, A).contiguous()
            return torch.from_numpy(np.array(np.broadcast_to(np.asarray(a, dtype=dt), (B, A)), dtype=dt, order="C", copy=True)).to(self.device)

        self._draws = (mk(start, np.int32, torch.int32), mk(target, np.int32, torch.int32),
                       mk(size, np.float64, torch.float64))

    def _desc(self):
        p = self._pool
        d = _lib.RoutingDesc()
        d.B, d.N, d.A, d.E, d.T = self.num_envs, self._N, self._A, self._E, p.T
        d.env_var, d.k = self.env_var.value, self.k
        d.congestion, d.action_mask, d.ttl = int(self.enable_congestion), int(self.enable_action_mask), int(self.ttl)
        d.state_stride = self._layout["stride"]
        d.node_sparse_static = 2 if p.static_rows is not None else 0
        d.node_edges, d.node_nbrs, d.edges, d.apsp = (p.node_edges.data_ptr(), p.node_nbrs.data_ptr(),
                                                      p.edges.data_ptr(), p.apsp.data_ptr())
        d.topo_index = None if self._topo_index is None else self._topo_index.data_ptr()
        d.state = self._state.data_ptr()
        return d

    def _alloc_outputs(self, step):
        B, N, A, dev = self.num_envs, self._N, self._A, self.device
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)
        o = dict(obs=e((B, A, self.obs_width()), torch.float32), adj=e((B, A, A), torch.int8),
                 node_obs=e((B, N, 4 * N + 8), torch.float32), node_agent=e((B, N, A), torch.int8),
                 agent_node=e((B, A), torch.int32), n_resets=e((B,), torch.int32),
                 node_sparse=self._sparse_rows_buffer(B))
        if step:
            o.update(reward=e((B, A), torch.float32), done=e((B, A), torch.uint8), delays=e((B, A), torch.int32),
                     arrived=e((B, A), torch.uint8), spr=e((B, A), torch.float64), info=e((B, 4), torch.int32))
        if self.enable_action_mask:
            o["action_mask_out"] = e((B, A, 4), torch.uint8)
        if step and self.eval_info_enabled:
            o.update(eval_f64=e((B, 2), torch.float64), eval_i32=e((B, 2), torch.int32),
                     packet_dist=e((B, A), torch.int32), packet_sizes=e((B, A), torch.float64))
            if self._sum_node is None:
                self._sum_node = torch.zeros((B, N), dtype=torch.int32, device=dev)
                self._sum_edge = torch.zeros((B, self._E), dtype=torch.int32, device=dev)
            o.update(sum_packets_per_node=self._sum_node, sum_packets_per_edge=self._sum_edge)
        return o

    def _sparse_rows_buffer(self, n):
        """[n, N, 24] int32 view for the node observation rows in sparse form (12 column indices + 12 fp32 bit patterns
        per row, csrc/routing_env.cu) on an allocation rounded up to whole 128-row tiles: NetMon's fused encoder pulls
        the rows tile by tile with bulk copies (rows behind n * N are never used as data)."""
        N = self._N
        rows = -(-(n * N) // 128) * 128
        flat = torch.empty((rows * 24,), dtype=torch.int32, device=self.device)
        return flat[:n * N * 24].view(n, N, 24)

    def _io(self, out, actions=None, env_mask=None):
        io = _lib.RoutingIO()
        io.actions = None if actions is None else actions.data_ptr()
        io.env_mask = None if env_mask is None else env_mask.data_ptr()
        if self._draws is not None:
            io.draw_start, io.draw_target, io.draw_size = (t.data_ptr() for t in self._draws)
        io.philox_seed, io.philox_step = self._seed, self._calls
        if self._dev_step is not None:  # CUDA-graph mode: the device counter carries the base
            io.philox_step, io.philox_step_dev = self._dev_step.offset(self._calls), self._dev_step.ptr()
        for k, v in out.items():
            setattr(io, k, v.data_ptr())
        if self._ring is not None and actions is not None:  # this step also writes its compact replay transition
            for k, v in self._ring.items():
                setattr(io, k, v)
        return io

    def set_ring(self, ring):
        """One-shot: the next step() writes its transition (records before / after, actions, reward, done) straight into
        the compact replay ring described by `ring` (gm_routing_io.ring_* fields, CompactReplayBuffer.ring_io)."""
        self._ring = ring

    def _launch(self, fn, out, actions=None, env_mask=None):
        _lib.require_device()
        d, io = self._desc(), self._io(out, actions, env_mask)
        with torch.cuda.device(self.device):
            _lib.check(fn(C.byref(d), C.byref(io), _lib.current_stream()))
        self._keep = (d, io, actions, env_mask, self._draws)  # keep inputs alive until the next launch
        self._draws = None
        if actions is not None:
            self._ring = None
        self._calls += 1
        self._out = out

    # ---- reference API ---------------------------------------------------------------------------
    def _new_topologies(self):
        """network.reset() semantics (routing.py:162) for 1 or B instances."""
        net = self.network
        if not self.batched or not net.random_topology:
            net.reset()
            # a fixed topology keeps its device tables (and their addresses: captured CUDA graphs hold them)
            same = (self._pool is not None and not net.random_topology and self._pool.T == 1
                    and self._pool.seeds == [net.tables.get("seed")]
                    and np.array_equal(self._pool.edges_host, net.tables["edges"]))  # edge weights may be re-randomised
            if not same:
                self._pool = TopologyPool([net.tables], self.device)
            self._topo_index = None
            return
        B = self.num_envs
        if len(net.seeds) > 0:  # finite pool (--num-topologies-train): upload once, draw an index per env
            if self._pool is None or self._pool.seeds != list(net.seeds):
                self._pool = TopologyPool([generate_tables(net.n_nodes, s) for s in net.seeds], self.device)
            idx = np.random.randint(len(net.seeds), size=B).astype(np.int32)
            net.reset()
        else:  # a fresh random topology per env and episode, generated on the device into this episode's slots
            P = B * self._topo_episodes
            if self._pool is None or not self._pool.fresh or self._pool.T != P:
                self._pool = TopologyPool.slots(P, net.n_nodes, self.device)
                self._episode = 0
            idx = np.arange(B, dtype=np.int32) + (self._episode % self._topo_episodes) * B
            self._episode += 1
        if self._topo_index is not None and self._topo_index.shape[0] == B:
            self._topo_index.copy_(torch.from_numpy(idx))  # same device address: captured CUDA graphs keep reading it
        else:
            self._topo_index = torch.from_numpy(idx).to(self.device)
        if len(net.seeds) == 0:
            self._generate_fresh(B)

    def _generate_fresh(self, B):
        """B calls of network.reset() without a seed list, on the device: the seeds come from the global stream as
        pick_seed draws them, the topologies are built into the slots _topo_index names, and the Network ends as after
        those calls (sampled_topology_seeds extended by the B seeds used, its tables the last env's topology)."""
        net = self.network
        ex = net.exclude_seeds
        if ex and self._exclude_dev is None:
            self._exclude_dev = torch.from_numpy(np.array(sorted(ex), np.int64)).to(self.device)
        seeds = net.pick_fresh_seeds(B)
        used, _ = self._pool.generate(seeds, self._topo_index, self._exclude_dev if ex else None)
        net.sampled_topology_seeds.extend(int(s) for s in used[:-1])
        # the last env's topology once more on the host, for the Network's attribute views (nodes, edges, adj_matrix)
        net._install(generate_tables(net.n_nodes, int(seeds[-1]), allow_reseed=True, exclude=ex))
        if net.current_topology_seed != int(used[-1]):
            raise _lib.GraphMarlError(f"device topology from seed {int(seeds[-1])} ended on seed {int(used[-1])}, "
                                      f"the host generator on {net.current_topology_seed}")
        net.sampled_topology_seeds.append(net.current_topology_seed)

    def reset(self):
        _lib.require_device()
        self._new_topologies()
        return self._reset_envs()

    def reset_on_pool(self, pool: TopologyPool, topo_index):
        """reset() onto topologies already in `pool`: env b starts on slot topo_index[b] (device int32 [B]).  The
        Network is neither reset nor read, so no topology seed is drawn; packets come from set_draws() as in reset()."""
        _lib.require_device()
        self.set_topology_pool(pool, topo_index)
        return self._reset_envs()

    def _reset_envs(self):
        B = self.num_envs
        if self._state is None:
            self._state = torch.zeros((B, self._layout["stride"]), dtype=torch.uint8, device=self.device)
        if not self.batched and self._draws is None:
            # routing.py:130-135: start, target, size per packet from the global stream, id order
            A, N = self._A, self._N
            ds, dt, dz = np.zeros(A, np.int32), np.zeros(A, np.int32), np.zeros(A, np.float64)
            for i in range(A):
                ds[i] = np.random.randint(N)
                dt[i] = np.random.randint(self.num_random_targets)
                dz[i] = np.random.random()
            self.set_draws(ds, dt, dz)
        if self.eval_info_enabled:  # routing.py:167-169
            self._sum_node = self._sum_edge = None
            self.sum_packets_per_node = np.zeros(self._N)
            self.sum_packets_per_edge = np.zeros(self._E)
        out = self._alloc_outputs(step=False)
        self._launch(_lib.lib().gm_routing_reset, out)
        self.agent_steps = np.zeros(self.n_data)
        return self._ret(out["obs"]), self._ret(out["adj"])

    def step(self, act):
        B, A = self.num_envs, self._A
        if not torch.is_tensor(act):
            act = torch.as_tensor(np.ascontiguousarray(np.asarray(act, dtype=np.int32)))
        act = act.to(device=self.device, dtype=torch.int32).reshape(B, A).contiguous()
        rng_state = None
        if not self.batched and self._draws is None:
            # Speculatively draw A respawn triples from a COPY of the global stream; after the
            # step the real stream is advanced by exactly the triples the env consumed.
            rng_state = np.random.get_state()
            ds, dt, dz, _ = self._native_draws(rng_state, A)
            self.set_draws(ds, dt, dz)
        out = self._alloc_outputs(step=True)
        self._launch(_lib.lib().gm_routing_step, out, actions=act)
        if self.batched:
            info = dict(looped=out["info"][:, 0], throughput=out["info"][:, 1], dropped=out["info"][:, 2],
                        blocked=out["info"][:, 3], delays=out["delays"], arrived=out["arrived"], spr=out["spr"])
            if self.eval_info_enabled:
                info.update(total_edge_load=out["eval_f64"][:, 0], total_packet_size=out["eval_f64"][:, 1],
                            occupied_edges=out["eval_i32"][:, 0], packets_on_edges=out["eval_i32"][:, 1],
                            packet_sizes=out["packet_sizes"], packet_distances=out["packet_dist"])
            return out["obs"], out["adj"], out["reward"], out["done"].view(torch.bool), info
        n = int(out["n_resets"][0].item())
        if rng_state is not None and n > 0:
            _, _, _, new_state = self._native_draws(rng_state, n)
            np.random.set_state(new_state)
        done = out["done"][0].cpu().numpy().astype(bool)
        delays = out["delays"][0].cpu().numpy()
        arrived = out["arrived"][0].cpu().numpy().astype(bool)
        spr = out["spr"][0].cpu().numpy()
        inf = out["info"][0].cpu().numpy()
        info = {
            "delays": [float(x) for x in delays[done]],
            "delays_arrived": [float(x) for x in delays[arrived]],
            "spr": [float(x) for x in spr[arrived]],
            "looped": np.float32(inf[0]),
            "throughput": np.int64(inf[1]),
            "dropped": np.int64(inf[2]),
            "blocked": int(inf[3]),
        }
        if self.eval_info_enabled:  # routing.py:509-519, 484-486
            ef, ei = out["eval_f64"][0].cpu().numpy(), out["eval_i32"][0].cpu().numpy()
            info.update(total_edge_load=float(ef[0]) if ef[0] != 0 else 0, occupied_edges=int(ei[0]),
                        packets_on_edges=int(ei[1]), total_packet_size=float(ef[1]),
                        packet_sizes=[float(x) for x in out["packet_sizes"][0].cpu().numpy()],
                        packet_distances=[int(x) for x in out["packet_dist"][0].cpu().numpy()])
            self.sum_packets_per_node = self._sum_node[0].cpu().numpy().astype(np.float64)
            self.sum_packets_per_edge = self._sum_edge[0].cpu().numpy().astype(np.float64)
            for st, sp in zip(delays[arrived], spr[arrived]):
                opt = int(round(st / sp)) if sp > 0 else 1
                self.distance_map[opt].append(float(st))
        self.agent_steps = np.where(done, 0, self.agent_steps + 1)
        if self.enable_action_mask:
            self.action_mask = out["action_mask_out"][0].cpu().numpy().astype(bool)
        return (self._ret(out["obs"]), self._ret(out["adj"]), out["reward"][0].cpu().numpy(), done, info)

    def _native_draws(self, np_state, n):
        st = np.zeros(_lib.GM_MT_STATE_WORDS, np.uint32)
        st[:624] = np_state[1]
        st[624] = np_state[2]
        ds, dt, dz = np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.float64)
        _lib.lib().gm_mt_packet_draws(_lib.ptr(st), self._N, n, _lib.ptr(ds), _lib.ptr(dt), _lib.ptr(dz))
        new_state = (np_state[0], st[:624].copy(), int(st[624]), np_state[3], np_state[4])
        return ds[:n], dt[:n], dz[:n], new_state

    def observe(self):
        """Rebuild every observation from the current state without advancing it."""
        out = self._alloc_outputs(step=False)
        out.pop("n_resets")
        self._launch(_lib.lib().gm_routing_observe, out)
        self._calls -= 1
        return out

    def observe_records(self, records, topo_index=None):
        """Observations of ARBITRARY packed env records (uint8 [n, state_stride], e.g. gathered from the compact
        replay ring) on this env's topology pool: the same emitters as reset()/step(), nothing is advanced.
        Returns dict(obs, adj, node_obs, node_agent, agent_node)."""
        _lib.require_device()
        n = records.shape[0]
        assert records.dtype == torch.uint8 and records.shape[1] == self._layout["stride"] and records.is_contiguous()
        N, A, dev = self._N, self._A, self.device
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)
        out = dict(obs=e((n, A, self.obs_width()), torch.float32), adj=e((n, A, A), torch.int8),
                   node_obs=e((n, N, 4 * N + 8), torch.float32), node_agent=e((n, N, A), torch.int8),
                   agent_node=e((n, A), torch.int32), node_sparse=self._sparse_rows_buffer(n))
        d = self._desc()
        d.B, d.state = n, records.data_ptr()
        d.topo_index = None if topo_index is None else topo_index.data_ptr()
        io = _lib.RoutingIO()
        for k, v in out.items():
            setattr(io, k, v.data_ptr())
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gm_routing_observe(C.byref(d), C.byref(io), _lib.current_stream()))
        return out

    def _ret(self, t):
        return t if self.batched else t[0].cpu().numpy()

    def render(self):
        self.network.render()

    def get_nodes_adjacency(self):
        if not self.batched:
            return self.network.adj_matrix
        p = self._pool
        N = self._N
        if getattr(p, "node_adj", None) is None:
            eye = torch.zeros((p.T, N, N), dtype=torch.int8, device=self.device)
            eye.scatter_(2, p.nbr_all.long(), 1)
            p.node_adj = eye
        if self._topo_index is not None:
            return p.node_adj[self._topo_index.long()]
        return p.node_adj.expand(self.num_envs, N, N)

    def get_node_observation(self):
        return self._ret(self._out["node_obs"])

    def get_node_agent_matrix(self):
        return self._ret(self._out["node_agent"])

    def get_agent_nodes(self):
        """[B,A] int32 node index of every agent (batched readout gather)."""
        return self._out["agent_node"]

    def get_adjacency_lists(self):
        """(nbr_all i32[T,N,4], deg i32[T,N], list_index i32[B] or None) for NetMon."""
        idx = self._topo_index
        if idx is None and self.num_envs > 1:  # shared topology: every env reads list 0
            if getattr(self, "_zero_index", None) is None:
                self._zero_index = torch.zeros((self.num_envs,), dtype=torch.int32, device=self.device)
            idx = self._zero_index
        return self._pool.nbr_all, self._pool.deg, idx

    def get_node_aux(self):
        """Shortest-path weights as float32 (routing.py:237-254)."""
        if not self.batched:
            return np.asarray(self.network.shortest_paths_weights, dtype=np.float32)
        if getattr(self._pool, "apsp_f32", None) is None:
            self._pool.apsp_f32 = self._pool.apsp.float()
        a = self._pool.apsp_f32
        return a[self._topo_index.long()] if self._topo_index is not None else a.expand(self.num_envs, -1, -1)

    def get_state(self):
        """Read back the packed env records as named host arrays (parity tests, heuristics)."""
        raw = self._state.cpu().numpy()
        L, A, E, B = self._layout, self._A, self._E, self.num_envs
        i32 = raw[:, L["i32"]:L["i32"] + 32 * A].copy().view(np.int32).reshape(B, 8, A)
        names = ["now", "target", "edge", "time", "ttl", "spw", "start", "agent_steps"]
        s = {n: i32[:, j] for j, n in enumerate(names)}
        s["size"] = raw[:, L["size"]:L["size"] + 8 * A].copy().view(np.float64).reshape(B, A)
        s["load"] = raw[:, L["load"]:L["load"] + 8 * E].copy().view(np.float64).reshape(B, E)
        s["visited"] = raw[:, L["vis"]:L["vis"] + 4 * A * L["VW"]].copy().view(np.uint32).reshape(B, A, L["VW"])
        s["mask"] = raw[:, L["mask"]:L["mask"] + 4 * A].copy().reshape(B, A, 4)
        return s

    @property
    def data(self):
        """Packets of env 0 as objects with the reference's attribute names (routing.py:12-40)."""
        s = self.get_state()
        return [SimpleNamespace(id=i, now=int(s["now"][0, i]), target=int(s["target"][0, i]),
                                size=float(s["size"][0, i]), start=int(s["start"][0, i]),
                                time=int(s["time"][0, i]), edge=int(s["edge"][0, i]), ttl=int(s["ttl"][0, i]),
                                shortest_path_weight=int(s["spw"][0, i]))
                for i in range(self._A)]

    def get_final_info(self, info: dict):
        """routing.py:541-546 (single env)."""
        steps = self.get_state()["agent_steps"][0] if self._state is not None else []
        for agent_step in steps:
            if agent_step != 0:
                info["delays"].append(float(agent_step))
        return info

    def get_num_agents(self):
        return self.n_data

    def get_num_nodes(self):
        return self.network.n_nodes
