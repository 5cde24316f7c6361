"""Device-resident rollout loop: the reference's rollout section (src/main.py:673-737) for B
environment instances at once, built only from the public classes of this package.

    policy(obs, adj) -> env.step(actions) [Routing step + NetMon step] -> buff.add(...)

Nothing crosses the host per step unless `host_draws=True`, in which case the step's random
draws (policy.py:46-47 and routing.py:130-135) are supplied from pinned host memory, the
mode used for bit-exact replays and for the end-to-end measurement.
"""
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn.functional as F

from .env.network import Network
from .env.routing import Routing
from .env.wrapper import NetMonWrapper
from .model import DQN, NetMon, PackedRows
from .policy import EpsilonGreedy
from .replaybuffer import CompactReplayBuffer, ReplayBuffer

CONFIGS = {
    # BASELINE.json configs[1]: routing single graph, seed 923430603, DQN + NetMon, 4096 envs
    "cfg2": dict(n_nodes=20, n_data=20, topo_seed=923430603, congestion=True, K=3, rnn="lstm", H=128,
                 enc=(512, 256), dqn=(512, 256), episode_steps=300),
    # configs[1] with the LayerNormLSTM cell BASELINE.json's north_star names (src/layernormlstm.py)
    "cfg2ln": dict(n_nodes=20, n_data=20, topo_seed=923430603, congestion=True, K=3, rnn="lnlstm", H=128,
                   enc=(512, 256), dqn=(512, 256), episode_steps=300),
    # BASELINE.json configs[2]: no congestion, a random topology per env and episode out of a pool built with the
    # reference generator (network.py:100-120), 50-step episodes, K=1 (16384 envs over 8 GPUs = 2048 per GPU)
    "cfg3": dict(n_nodes=20, n_data=20, topo_seed=476, random_topology=True, n_topologies=4096, congestion=False, K=1,
                 rnn="lstm", H=128, enc=(512, 256), dqn=(512, 256), episode_steps=50),
    # configs[2] as the reference trains it without a seed list (Network(random_topology=True)): a fresh topology per env
    # and episode, generated on the device into the env's topology pool (Routing.set_topology_episodes)
    "cfg3fresh": dict(n_nodes=20, n_data=20, topo_seed=476, random_topology=True, n_topologies=None, congestion=False,
                      K=1, rnn="lstm", H=128, enc=(512, 256), dqn=(512, 256), episode_steps=50),
    # BASELINE.json configs[3]: synthetic large graph 200 nodes / 100 agents, lnlstm, K=4
    "cfg4": dict(n_nodes=200, n_data=100, topo_seed=476, congestion=True, K=4, rnn="lnlstm", H=128,
                 enc=(512, 256), dqn=(512, 256), episode_steps=300),
}


def shard_envs(total_envs, world_size, rank):
    """Contiguous block of env instances owned by `rank` (SURVEY 8e): [lo, hi).  Independent
    environments shard across the GPUs of one box with no collective on the rollout path."""
    base, rem = divmod(int(total_envs), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def aggregate_throughput(units_per_rank, ms_local, world_size):
    """Whole-job throughput from per-rank device times: all ranks' units / the MAX time over ranks
    (all-reduced over the default process group when world_size > 1)."""
    import torch.distributed as dist

    t = torch.tensor([float(ms_local)], dtype=torch.float64,
                     device="cuda" if (dist.is_initialized() and dist.get_backend() == "nccl") else "cpu")
    n = torch.tensor([float(units_per_rank)], dtype=torch.float64, device=t.device)
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(n, op=dist.ReduceOp.SUM)
    return float(n.item()) / (float(t.item()) * 1e-3), float(t.item())


class Rollout:
    def __init__(self, cfg="cfg2", num_envs=4096, device="cuda", math="fp32", replay_capacity=None,
                 epsilon=1.0, seed=0, with_replay=True, host_draws=False, overlap_replay=True, host_draw_steps=64,
                 graph_steps=0, replay="compact", device_sampler=False, state_ring=True, fused_insert=True):
        """replay: "compact" (default; replaybuffer.CompactReplayBuffer: env records + NetMon state, dense fields are
        rebuilt when sampled) or "dense" (the reference's 17 dense fields per transition, replaybuffer.ReplayBuffer)."""
        c = dict(CONFIGS[cfg]) if isinstance(cfg, str) else dict(cfg)
        self.cfg, self.B, self.device = c, num_envs, torch.device(device)
        N, A = c["n_nodes"], c["n_data"]
        torch.manual_seed(seed)
        np.random.seed(seed)
        if c.get("random_topology"):
            net = Network(N, random_topology=True, n_random_seeds=c.get("n_topologies"), topology_init_seed=c["topo_seed"])
        else:
            net = Network(N, random_topology=False, topology_init_seed=c["topo_seed"])
        self.base_env = Routing(net, A, 1, enable_congestion=c["congestion"], num_envs=num_envs, device=device,
                                seed=seed, batched=True)
        Dn, Da = 4 * N + 8, 6 * N + 10
        self.netmon = NetMon(Dn, c["H"], c["enc"], c["K"], F.leaky_relu, rnn_type=c["rnn"], agg_type="sum",
                             output_neighbor_hidden=True, math=math).to(device).eval()
        assert replay in ("compact", "dense")
        self.compact = bool(with_replay) and replay == "compact"
        self.state_ring = False
        # the compact ring does not store the graph observation (it is recomputed when sampled): on the tensor-core
        # path it then exists only tile-packed, written once by the readout and pulled by the DQN's bulk copies
        lean_graph_obs = (self.compact or not with_replay) and math != "fp32" and c["H"] % 32 == 0
        self.env = NetMonWrapper(self.base_env, self.netmon, 1, split_obs=True, graph_obs_fp32=not lean_graph_obs)
        Dj = Da + self.netmon.get_out_features()
        self.model = DQN(Dj, c["dqn"], 4, F.leaky_relu, math=math).to(device).eval()
        args = SimpleNamespace(epsilon=epsilon, step_before_train=10**9, epsilon_update_freq=100, epsilon_decay=0.996)
        self.policy = EpsilonGreedy(self.env, self.model, 4, args, seed=seed)
        self.buff = None
        if with_replay:
            # default ring: 8 batched steps, capped at ~48 GB of HBM (a cfg4 transition is ~3 MB), never below 2 steps
            per_transition = 4 * (2 * A * Dj + 2 * N * Dn + N * self.netmon.get_state_size() + N * N) + 2 * (A * A + N * N + N * A)
            steps_fit = max(2, min(8, int(48e9 // (per_transition * num_envs))))
            cap = replay_capacity or steps_fit * num_envs
            if self.compact:
                # state ring: NetMon reads / writes its carried state directly in the ring's node_state field
                ring = state_ring and cap % num_envs == 0 and cap // num_envs >= 1
                self.buff = CompactReplayBuffer(seed, cap, self.env, device_sampler=device_sampler, state_ring=ring,
                                                ring_align=max(int(graph_steps), 1))
            else:
                self.buff = ReplayBuffer(seed, cap, A, Dj, 0, N, Dn, self.netmon.get_state_size(), N, device=device,
                                         device_sampler=device_sampler)
        self.state_ring = self.compact and self.buff.state_ring
        if c.get("random_topology") and not c.get("n_topologies") and self.buff is not None:
            # fresh topologies: keep the pool slots of every episode the ring can still hold transitions of, plus the
            # current one (the compact ring names a transition's topology by its pool slot)
            cap_steps = -(-self.buff.buffer_size // num_envs)
            self.base_env.set_topology_episodes(-(-cap_steps // c["episode_steps"]) + 1)
        # state-ring mode: the env's step kernel writes the transition into the ring itself (gm_routing_io.ring_*)
        self.fused_insert = bool(fused_insert) and self.state_ring and hasattr(self.base_env, "set_ring")
        self.sizes = dict(N=N, A=A, Dn=Dn, Da=Da, Dj=Dj, H=c["H"], K=c["K"])
        self.host_draws = host_draws
        if host_draws:
            # a table of `host_draw_steps` steps of host-generated draws in pinned memory (policy.py:46-47 and
            # routing.py:130-135 consume host randomness in the reference); every step copies ITS slice H2D
            B, T = num_envs, int(host_draw_steps)
            pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
            self._h = dict(ra=pin((T, B, A), torch.int32), ru=pin((T, B, A), torch.float64), ds=pin((T, B, A), torch.int32),
                           dt=pin((T, B, A), torch.int32), dz=pin((T, B, A), torch.float64))
            self._rng = np.random.default_rng(seed)
            self._h_reward = pin((B, A), torch.float32)
            self._h_steps, self._h_cursor = T, 0
            self.refresh_host_draws()
        # the dense insert (141 kB per transition) is worth a side stream; the compact one is two small launches
        self.overlap_replay = overlap_replay and with_replay and not self.compact
        self._replay_stream = torch.cuda.Stream(device=self.device) if self.overlap_replay else None
        self.graph_steps = int(graph_steps)
        self._graphs, self._graph_pool, self._static, self._graph_tables = {}, None, None, None
        self.graph_launches = 0  # kernels of this library launched through graph replays
        self._h_trace = None     # optional list: indices of the host draw table consumed so far (tests)
        self._draw_bufs, self._copy_stream = None, None  # static per-step draw buffers of the captured units
        self._d2h_stream, self._capture_keep = None, []  # reward read-back stream of the captured units
        if host_draws and self.graph_steps > 0:
            assert host_draw_steps % self.graph_steps == 0, "host draw table must hold whole graph units"
        self.episode_step = None
        self._marks = None
        self.obs = self.adj = None
        self.node_aux = None
        self.total_reward = torch.zeros((), dtype=torch.float64, device=device)

    def h2d_bytes_per_step(self):
        return sum(t[0].numel() * t.element_size() for t in self._h.values()) if self.host_draws else 0

    def d2h_bytes_per_step(self):
        return self._h_reward.numel() * 4 if self.host_draws else 0

    def join_streams(self):
        """Make the current stream wait for the side-stream replay insert (end of a timed region)."""
        if self._replay_stream is not None:
            torch.cuda.current_stream().wait_stream(self._replay_stream)

    def refresh_host_draws(self):
        """Regenerate the host draw table (call outside a timed region, with the device idle)."""
        T, B, A, N = self._h_steps, self.B, self.sizes["A"], self.sizes["N"]
        r = self._rng
        self._h["ra"].numpy()[...] = r.integers(0, 4, (T, B, A), dtype=np.int32)
        self._h["ru"].numpy()[...] = r.random((T, B, A))
        self._h["ds"].numpy()[...] = r.integers(0, N, (T, B, A), dtype=np.int32)
        self._h["dt"].numpy()[...] = r.integers(0, N, (T, B, A), dtype=np.int32)
        self._h["dz"].numpy()[...] = r.random((T, B, A))

    def _ring_states(self):
        """State-ring mode: point the wrapper's carried states at their ring blocks (T = committed steps: the state that
        produced the current observations is the node_state of transition T, the current one that of T + 1)."""
        T, env = self.buff.steps_total, self.env
        hpk = getattr(env.current_netmon_state, "_gm_hpk", None)
        env.last_netmon_state = self.buff.state_block(T)
        env.current_netmon_state = self.buff.state_block(T + 1)
        if hpk is not None:
            env.current_netmon_state._gm_hpk = hpk
        env.netmon.state = env.current_netmon_state

    def reset(self):
        if self.state_ring:
            T = self.buff.steps_total
            self.buff.state_block(T).zero_()  # the state before an episode's first NetMon step (wrapper.py:40-41)
            self.env._state_sink = self.buff.state_block(T + 1)
        self.obs, self.adj = self.env.reset()
        if self.state_ring:
            self._ring_states()
        aux = self.env.get_node_aux()
        if (self.node_aux is not None and self.node_aux.shape == aux.shape and self.node_aux.is_contiguous()
                and aux.data_ptr() != self.node_aux.data_ptr()):
            self.node_aux.copy_(aux)  # per-env topologies: refresh in place, captured graph units hold this address
        else:
            self.node_aux = aux
        # the state "before the first step" is all zeros (wrapper.py:40-41, main.py:692-696 store 0 then): keep it as a
        # tensor so that an episode's first step is not a special case for the captured graph units
        if self.env.last_netmon_state is None and self.env.current_netmon_state is not None:
            self.env.last_netmon_state = torch.zeros_like(self.env.current_netmon_state)
        self.episode_step = 0

    def _mark(self, name):
        if self._marks is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self._marks.append((name, e))

    def _step_eager(self, draws=None):
        """One batched rollout step (main.py:673-737).  draws: device copies of this step's slice of the host draw table
        that a copy stream already fetched (captured graph units prefetch all their slices, see _capture_unit)."""
        env, c = self.env, self.cfg
        if self.episode_step is None or self.episode_step >= c["episode_steps"]:
            self.reset()
        last_state = env.last_netmon_state
        netmon_info = env.get_netmon_info()
        obs, adj = self.obs, self.adj
        self._mark("start")
        if self.host_draws:
            i = self._h_cursor % self._h_steps
            self._h_cursor += 1
            if self._h_trace is not None and not torch.cuda.is_current_stream_capturing():
                self._h_trace.append(i)
            d = draws if draws is not None else {k: v[i].to(self.device, non_blocking=True) for k, v in self._h.items()}
            with torch.no_grad():
                _, actions = self.model.act(obs[0], obs[1], epsilon=self.policy._epsilon, rand_action=d["ra"].reshape(-1),
                                            rand_u=d["ru"].reshape(-1), want_q=False)
            self.base_env.set_draws(d["ds"], d["dt"], d["dz"])
        else:
            actions = self.policy(obs, adj)
        self._mark("dqn_act")
        fused_insert = self.compact and self.fused_insert
        if fused_insert:
            # the step kernel writes the transition itself (records before / after, actions, reward, done): no insert launch
            self.base_env.set_ring(self.buff.ring_io(self.episode_step + 1 >= c["episode_steps"]))
        elif self.compact:
            self.buff.stage(self.B)  # the env records are advanced in place: snapshot them into the ring first
        next_obs_a, next_adj, reward, done, info = self.base_env.step(actions)
        self._mark("env_step")
        if self.state_ring:
            env._state_sink = self.buff.state_block(self.buff.steps_total + 2)
        next_obs = env._with_graph_obs(next_obs_a)
        self._mark("netmon")
        next_info = env.get_netmon_info()
        self.episode_step += 1
        episode_done = self.episode_step >= c["episode_steps"]
        if fused_insert:
            self.buff.advance(self.B)
            self._ring_states()
        elif self.compact:
            self.buff.commit(actions, reward, done, episode_done, last_state, num=self.B)
            if self.state_ring:
                self._ring_states()
        elif self.buff is not None:
            node_state = last_state if last_state is not None else 0
            if self.overlap_replay:
                # the insert is off the critical path (nothing in the next step reads the ring): run it on a
                # side stream so its HBM-bound copies overlap the next step's tensor-core kernels
                main = torch.cuda.current_stream()
                self._replay_stream.wait_stream(main)
                with torch.cuda.stream(self._replay_stream):
                    self.buff.add(obs, actions, reward, next_obs, adj, next_adj, done, episode_done, 0, node_state,
                                  self.node_aux, *netmon_info, *next_info, num=self.B)
            else:
                self.buff.add(obs, actions, reward, next_obs, adj, next_adj, done, episode_done, 0, node_state,
                              self.node_aux, *netmon_info, *next_info, num=self.B)
        self._mark("replay_insert")
        self.obs, self.adj = next_obs, next_adj
        if self.host_draws:
            if draws is not None and self._d2h_stream is not None and torch.cuda.is_current_stream_capturing():
                # captured unit: the read-back of this step's reward runs on its own stream, so the next step's kernels
                # do not queue behind a PCIe copy; the unit joins that stream at its end.  The reward tensor stays
                # referenced until the capture ends (its block must not be handed to a later allocation of the unit).
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream())
                self._d2h_stream.wait_event(ev)
                with torch.cuda.stream(self._d2h_stream):
                    self._h_reward.copy_(reward, non_blocking=True)
                self._capture_keep.append(reward)
            else:
                self._h_reward.copy_(reward, non_blocking=True)
        return reward, done, info

    # ---- CUDA-graph execution ----------------------------------------------------------------------
    # A rollout step launches ~25 kernels from ~0.8 ms of Python; on a busy host that issue time, not the
    # GPU, bounds the throughput.  `run(k)` therefore replays captured units of `graph_steps` consecutive
    # steps.  Everything a step hands to the next one (observations, adjacency, NetMon states, node tables)
    # lives in static tensors that the unit reads first and refreshes last; the three host counters that
    # change between replays (env / policy Philox steps, replay ring index) are shadowed by device scalars.
    def _carried(self):
        env, be = self.env, self.base_env
        obs_a, obs_g = self.obs
        d = dict(obs_a=obs_a, adj=self.adj, node_obs=be._out["node_obs"], node_agent=be._out["node_agent"])
        if not self.state_ring:  # (ring mode: the carried states live in ring blocks that a captured unit addresses directly)
            d["cur"] = env.current_netmon_state
        if isinstance(obs_g, PackedRows):  # graph observation exists only tile-packed
            d["pk"] = obs_g.buf
            self._pk_shape = obs_g.shape
            pk = (obs_g.buf, obs_g.math)
        else:
            d["obs_g"] = obs_g
            pk = getattr(obs_g, "_gm_pk", None)
            if pk is not None:
                d["pk"] = pk[0]
        if env.last_netmon_state is not None and not self.state_ring:
            d["last"] = env.last_netmon_state
        hpk = getattr(env.current_netmon_state, "_gm_hpk", None)  # tile-packed hidden half of the carried state
        if hpk is not None:
            d["cur_hpk"] = hpk[0]
        return d, (pk[1] if pk is not None else None)

    def _adopt(self, t, math):
        """Point every cross-step reference at the tensors in `t`."""
        env, be = self.env, self.base_env
        if "obs_g" not in t:
            obs_g = PackedRows(t["pk"], self._pk_shape, math)
        else:
            obs_g = t["obs_g"]
            if "pk" in t:
                obs_g._gm_pk = (t["pk"], math)
        self.obs, self.adj = (t["obs_a"], obs_g), t["adj"]
        if self.state_ring:
            self._ring_states()
            if "cur_hpk" in t:
                env.current_netmon_state._gm_hpk = (t["cur_hpk"], env.netmon.math)
        else:
            if "cur_hpk" in t:
                t["cur"]._gm_hpk = (t["cur_hpk"], env.netmon.math)
            env.current_netmon_state = t["cur"]
            env.netmon.state = t["cur"]
            if "last" in t:
                env.last_netmon_state = t["last"]
        be._out["node_obs"], be._out["node_agent"] = t["node_obs"], t["node_agent"]

    def _counters(self):
        return (self.episode_step, self.base_env._calls, self.policy._step,
                (self.buff.index, self.buff.count, getattr(self.buff, "steps_total", 0)) if self.buff is not None else None)

    def _set_counters(self, c):
        self.episode_step, self.base_env._calls, self.policy._step = c[0], c[1], c[2]
        if self.buff is not None:
            self.buff.index, self.buff.count = c[3][0], c[3][1]
            if hasattr(self.buff, "steps_total"):
                self.buff.steps_total = c[3][2]

    def _sync_device_counters(self):
        # a replay insert still pending on the side stream reads the ring-index counter (and the static
        # observation tensors): the main stream must not overwrite either before that insert has run
        self.join_streams()
        self.base_env._dev_step.set(self.base_env._calls)
        self.policy._dev_step.set(self.policy._step)
        if self.buff is not None:
            self.buff._dev_index.set(self.buff.index)

    def _ring_phase(self):
        """A captured unit addresses fixed blocks of the state ring: it can be replayed whenever the step counter sits at
        the same position of the ring (the ring length is a multiple of the unit length)."""
        return self.buff.steps_total % self.buff.M if self.state_ring else 0

    def _capture_unit(self, n, slot=None):
        """Capture n consecutive steps (from the current, static state) into a CUDA graph."""
        from . import _lib

        if self.base_env._dev_step is None:
            self.base_env._dev_step = _lib.DeviceCounter(self.device)
            self.policy._dev_step = _lib.DeviceCounter(self.device)
            if self.buff is not None:
                self.buff._dev_index = _lib.DeviceCounter(self.device)
        cur, math = self._carried()
        if self._static is None:  # static copies of the carried state; from now on the rollout lives in them
            self._static = {k: v.clone() for k, v in cur.items()}
            self._adopt(self._static, math)
        saved = self._counters()
        saved_cursor = self._h_cursor if self.host_draws else 0
        if slot is not None:
            self._h_cursor = slot * n  # this unit consumes the host draw slices [slot*n, slot*n + n)
        self._sync_device_counters()
        torch.cuda.synchronize()
        launches0 = _lib.lib().gm_kernel_launch_count()
        g = torch.cuda.CUDAGraph()
        if self.host_draws and (self._draw_bufs is None or len(self._draw_bufs) < n):
            self._draw_bufs = [{k: torch.empty_like(v[0], device=self.device) for k, v in self._h.items()} for _ in range(n)]
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._d2h_stream = torch.cuda.Stream(device=self.device)
        with torch.cuda.graph(g, pool=self._graph_pool):
            fetched = None
            if self.host_draws:
                # every step still copies ITS slice of the pinned host table, but on a copy stream that runs ahead of
                # the compute: slice k lands in its own static buffer while steps < k execute; step k waits for event k
                main, cs = torch.cuda.current_stream(), self._copy_stream
                cs.wait_stream(main)
                fetched = []
                with torch.cuda.stream(cs):
                    for k in range(n):
                        i = (self._h_cursor + k) % self._h_steps
                        for name, buf in self._draw_bufs[k].items():
                            buf.copy_(self._h[name][i], non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(cs)
                        fetched.append(ev)
            for k in range(n):
                if fetched is not None:
                    torch.cuda.current_stream().wait_event(fetched[k])
                    self._step_eager(draws=self._draw_bufs[k])
                else:
                    self._step_eager()
            if fetched is not None:
                torch.cuda.current_stream().wait_stream(self._copy_stream)
                torch.cuda.current_stream().wait_stream(self._d2h_stream)
            self.join_streams()
            out, _ = self._carried()
            for k, v in self._static.items():
                v.copy_(out[k])
        self._capture_keep = []
        if self._graph_pool is None:
            self._graph_pool = g.pool()
        # capture executes nothing: remember by how much the host bookkeeping moved, then restore it and the
        # static references
        after = self._counters()
        g.gm_delta = (after[0] - saved[0], after[1] - saved[1], after[2] - saved[2])
        g.gm_launches = _lib.lib().gm_kernel_launch_count() - launches0
        self._set_counters(saved)
        if self.host_draws:
            self._h_cursor = saved_cursor
        self._adopt(self._static, math)
        return g

    def _enter_static(self):
        """After eager steps the carried state lives in fresh tensors: move it into the static ones."""
        cur, math = self._carried()
        if cur["obs_a"] is not self._static["obs_a"]:
            self.join_streams()  # pending side-stream inserts may still read the static tensors
            for k, v in self._static.items():
                v.copy_(cur[k])
            self._adopt(self._static, math)

    def _replay_unit(self, g, n):
        self._sync_device_counters()
        g.replay()
        self.graph_launches += g.gm_launches
        c = self._counters()
        buf = None
        if self.buff is not None:
            buf = ((c[3][0] + n * self.B) % self.buff.buffer_size, min(self.buff.buffer_size, c[3][1] + n * self.B), c[3][2] + n)
        d = g.gm_delta
        self._set_counters((c[0] + d[0], c[1] + d[1], c[2], buf))
        # epsilon is a launch argument, i.e. constant inside a captured unit: the decay schedule (policy.py:55-62) is
        # applied here, step by step, and takes effect at the next unit (units are keyed by epsilon)
        for _ in range(d[2]):
            self.policy._step += 1
            self.policy._decay()
        if self.state_ring:  # the carried states moved n blocks along the ring
            self._ring_states()
            if "cur_hpk" in self._static:
                self.env.current_netmon_state._gm_hpk = (self._static["cur_hpk"], self.netmon.math)
        if self.host_draws:
            if self._h_trace is not None:
                self._h_trace.extend((self._h_cursor + k) % self._h_steps for k in range(n))
            self._h_cursor += n

    def run(self, steps):
        """Advance `steps` rollout steps, through captured graph units where an episode allows it.  A unit is n
        consecutive steps of one episode; the unit that ends an episode is its own captured variant (the episode-end flag
        of its last replay insert is part of the captured work).  Resets run eagerly."""
        n = self.graph_steps
        done = 0
        while done < steps:
            if self._graphs and self._graph_tables is not self.base_env._pool:
                self._graphs.clear()  # the topology tables moved (new pool): the captured units are stale
            if self.episode_step is None or self.episode_step >= self.cfg["episode_steps"]:
                self.reset()
            left_in_episode = self.cfg["episode_steps"] - self.episode_step
            usable = n > 0 and steps - done >= n and left_in_episode >= n
            if usable and self.host_draws and self._h_cursor % n != 0:
                # units consume whole, aligned blocks of the host draw table: skip to the next block (the table
                # holds independent draws, skipping some changes nothing statistically)
                self._h_cursor += n - self._h_cursor % n
            if not usable:
                self._step_eager()
                done += 1
                continue
            slot = (self._h_cursor // n) % (self._h_steps // n) if self.host_draws else 0
            key = (slot, left_in_episode == n, float(self.policy._epsilon), self._ring_phase())
            if key not in self._graphs:
                self._graphs[key] = self._capture_unit(n, slot if self.host_draws else None)
                self._graph_tables = self.base_env._pool
            self._enter_static()
            self._replay_unit(self._graphs[key], n)
            done += n

    def precapture(self):
        """Capture every graph unit up front (one per block of the host draw table, or a single one; each as a mid-episode
        and, when the episode length is a multiple of the unit, as an episode-ending variant) so that no capture happens
        inside a timed region."""
        n = self.graph_steps
        if n <= 0:
            return
        E = self.cfg["episode_steps"]
        slots = range(self._h_steps // n) if self.host_draws else [0]

        def advance_until(cond):
            guard = 0
            while not cond():
                if self.episode_step is None or self.episode_step >= E:
                    self.reset()
                    continue
                self._step_eager()
                guard += 1
                assert guard <= 2 * E + 2

        variants = [False] + ([True] if E % n == 0 and E >= 2 * n else [])
        for tail in variants:
            if tail:
                advance_until(lambda: self.episode_step is not None and E - self.episode_step == n)
            else:
                advance_until(lambda: self.episode_step is not None and E - self.episode_step > n)
            for slot in slots:
                key = (slot, tail, float(self.policy._epsilon), self._ring_phase())
                if key not in self._graphs:
                    self._graphs[key] = self._capture_unit(n, slot if self.host_draws else None)
                    self._graph_tables = self.base_env._pool

    def step(self):
        return self._step_eager()

    def profile_stages(self, iters=10):
        """Per-stage device time of one step (CUDA events on the launching stream), plus the time of
        the summed event time of the step's tensor-core GEMM launches."""
        import ctypes as C

        from . import _lib

        if self.episode_step is None or self.episode_step + iters + 1 >= self.cfg["episode_steps"]:
            self.reset()
        overlap, self.overlap_replay = self.overlap_replay, False  # stage times are taken with everything on one stream
        self.join_streams()
        self.step()
        acc = {}
        for _ in range(iters):
            self._marks = []
            self.step()
            torch.cuda.synchronize()
            for (n0, e0), (n1, e1) in zip(self._marks[:-1], self._marks[1:]):
                acc[n1 + "_ms"] = acc.get(n1 + "_ms", 0.0) + e0.elapsed_time(e1) / iters
            self._marks = None
        # device time per kernel category of one step, from CUDA events recorded around every launch inside
        # the library (independent of Python issue time; everything on one stream here)
        math = self.netmon.math
        ms = (C.c_double * 8)()
        cnt = (C.c_int32 * 8)()
        _lib.lib().gm_profile_enable(1)
        for _ in range(iters):
            self._step_eager()
        _lib.lib().gm_profile_enable(0)
        _lib.check(_lib.lib().gm_profile_collect(ms, cnt))
        for i, nm in enumerate(["gemm", "env_kernel", "aggregate_kernel", "readout_kernel", "replay_kernel"]):
            acc[nm + "_ms"] = ms[i] / iters
            acc[nm + "_launches_per_step"] = cnt[i] / iters
        if math == "fp32":
            acc["gemm_ms"] = acc.get("netmon_ms", 0.0) + acc.get("dqn_act_ms", 0.0)  # stage time (SIMT GEMMs dominate it)
        self.overlap_replay = overlap
        acc["gemm_kernel"] = {"fp32": "linear_simt_kernel (fp32 FFMA)", "bf16x3": "linear_tc_kernel (tcgen05, bf16 hi/lo split x3)",
                              "bf16": "linear_tc_kernel (tcgen05, single bf16 pass)"}[math]
        return acc
