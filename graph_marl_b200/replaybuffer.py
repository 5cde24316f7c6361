"""Device-resident replay ring, mirrors src/replaybuffer.py:9-287 of the reference.

Same 17 fields, dtypes and ring arithmetic (`index = (index+1) % size`, `count` saturates),
same `get_batch` index streams (`np.random.default_rng(seed).choice`, contiguous sequences
anchored at the oldest element), but the arrays live in HBM: `add()` takes one transition
(numpy or tensors, reference call shape) or a batch of B transitions (tensors with a leading
env dimension) and lands them with one fused copy kernel; `get_batch()` gathers with one
kernel that also performs the reference's dtype conversions.
"""
import ctypes as C
from collections import namedtuple
from typing import Iterator

import numpy as np
import torch

from . import _lib

TransitionBatch = namedtuple(
    "TransitionBatch",
    ["idx", "obs", "action", "reward", "next_obs", "adj", "next_adj", "done", "episode_done", "agent_state",
     "node_obs", "node_adj", "node_state", "node_aux", "node_agent_matrix", "next_node_obs", "next_node_adj",
     "next_node_agent_matrix"],
)

# add() argument order of the reference (replaybuffer.py:243-262)
ADD_ORDER = ["obs", "action", "reward", "next_obs", "adj", "next_adj", "done", "episode_done", "agent_state",
             "node_state", "node_aux", "node_obs", "node_adj", "node_agent_matrix", "next_node_obs",
             "next_node_adj", "next_node_agent_matrix"]


class _RingSampler(object):
    """Index streams of get_batch (replaybuffer.py:101, 111-130).  Host mode draws from numpy's
    `default_rng(seed)` like the reference; `device_sampler=True` keeps a bit-identical PCG64 stream in HBM
    (csrc/replay_sampler.cu) so that a batch of sequences is sampled without any host round trip (`idx` of the
    returned batches is then a device tensor)."""

    def _init_sampler(self, seed, device_sampler):
        self._random_generator = np.random.default_rng(seed)
        self._pcg_dev = None
        if device_sampler:
            st = np.zeros(_lib.GM_PCG64_STATE_WORDS, np.uint64)
            _lib.lib().gm_pcg64_seed(_lib.ptr(st), int(seed) & (2**64 - 1))
            self._pcg_dev = torch.from_numpy(st.view(np.int64)).to(self.device)

    def _index_rows(self, batch_size, sequence_length):
        """[max(sequence_length, 1), batch_size] ring slots: numpy int64 (host mode) or a device tensor."""
        T = max(int(sequence_length), 1)
        if self._pcg_dev is not None:
            _lib.require_device()
            out = torch.empty((T, batch_size), dtype=torch.int64, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib().gm_replay_sample_indices(self._pcg_dev.data_ptr(), self.count, self.index,
                                                               batch_size, int(sequence_length), out.data_ptr(),
                                                               _lib.current_stream()))
            return out
        if sequence_length <= 1:
            return self._random_generator.choice(self.count, batch_size, replace=True, p=None)[None]
        buffer_start = self.index % self.count
        batch_sequence_start = self._random_generator.choice(self.count - sequence_length, batch_size,
                                                             replace=True, p=None)
        batch_sequence_start = (buffer_start + batch_sequence_start) % self.count
        return np.stack([(batch_sequence_start + offset) % self.count for offset in range(sequence_length)])

    def get_batch(self, batch_size, device, sequence_length=0) -> Iterator[TransitionBatch]:
        rows = self._index_rows(batch_size, sequence_length)
        for offset in range(rows.shape[0]):
            yield self._get_transition_batch(rows[offset], device)

    def _device_indices(self, indices):
        if torch.is_tensor(indices):
            return indices.to(device=self.device, dtype=torch.int64).contiguous()
        return torch.as_tensor(np.ascontiguousarray(indices, dtype=np.int64)).to(self.device)



class ReplayBuffer(_RingSampler):
    def __init__(self, seed, buffer_size, n_agents, observation_size, agent_state_size, n_nodes=0,
                 node_observation_size=0, node_state_size=0, node_aux_size=0, half_precision=False,
                 device="cuda", device_sampler=False):
        self.buffer_size = int(buffer_size)
        self.count = 0
        self.index = 0
        self.device = torch.device(device)
        ft = torch.float16 if half_precision else torch.float32
        A, N = n_agents, n_nodes
        shapes = dict(
            obs=((A, observation_size), ft), action=((A,), torch.int8), reward=((A,), ft),
            next_obs=((A, observation_size), ft), adj=((A, A), torch.bool), next_adj=((A, A), torch.bool),
            done=((A,), torch.bool), episode_done=((), torch.bool), agent_state=((A, agent_state_size), ft),
            node_state=((N, node_state_size), ft), node_aux=((N, node_aux_size), ft),
            node_obs=((N, node_observation_size), ft), next_node_obs=((N, node_observation_size), ft),
            node_adj=((N, N), torch.bool), next_node_adj=((N, N), torch.bool),
            node_agent_matrix=((N, A), torch.bool), next_node_agent_matrix=((N, A), torch.bool))
        self._shapes = shapes
        for name, (shape, dt) in shapes.items():
            setattr(self, name, torch.zeros((self.buffer_size, *shape), dtype=dt, device=self.device))
        self._consts = {}
        self._dev_index = None  # _lib.DeviceCounter in CUDA-graph mode (rollout.Rollout)
        self._init_sampler(seed, device_sampler)
        # dtype conversion of _get_transition_batch (replaybuffer.py:132-187)
        self._out_dtype = {n: torch.float32 for n in shapes}
        self._out_dtype.update(action=torch.int64, done=torch.bool, episode_done=torch.bool)

    # ---- insert ------------------------------------------------------------------------------
    def _source(self, name, value, n):
        """(tensor, convert, broadcast) for one ring field without staging copies where possible:
        0/1 int8/uint8 tensors are reinterpreted as bool, int32 actions are narrowed by the insert
        kernel, python scalars / expanded (stride-0) tensors are written as one broadcast transition."""
        shape, dt = self._shapes[name]
        numel = int(np.prod(shape, dtype=np.int64))
        if isinstance(value, (bool, int, float)):
            key = (name, value)
            if key not in self._consts:  # e.g. the scalar 0 for absent states (main.py:659,695), episode_done
                self._consts[key] = torch.full((1, *shape), value, dtype=dt, device=self.device)
            return self._consts[key], 0, 1
        t = torch.as_tensor(value)
        if name == "agent_state" and t.dim() == len(shape) + 1 and n == 1 and t.shape[0] == 1:
            t = t.squeeze(0)  # replaybuffer.py:272-273
        if t.device != self.device:
            t = t.to(self.device)
        bcast = 0
        if t.dim() == len(shape) + 1 and t.shape[0] == n and n > 1 and t.stride(0) == 0:
            t, bcast = t[:1], 1  # expanded per-topology tensor (node_adj, node_aux): one copy for all envs
        rows = 1 if bcast else n
        convert = 0
        if t.dtype != dt:
            if dt == torch.bool and t.dtype in (torch.int8, torch.uint8):
                t = t.contiguous().view(torch.bool)  # env outputs are exactly 0/1
            elif dt == torch.int8 and t.dtype == torch.int32 and name == "action":
                convert = 4
            else:
                t = (t != 0) if dt == torch.bool else t.to(dt)
        if t.numel() != rows * numel:
            t = torch.broadcast_to(t, (rows, *shape))
        return t.reshape(rows, *shape).contiguous(), convert, bcast

    def add(self, obs, action, reward, next_obs, adj, next_adj, done, episode_done, agent_state, node_state,
            node_aux, node_obs, node_adj, node_agent_matrix, next_node_obs, next_node_adj,
            next_node_agent_matrix, num=1):
        """One transition (reference call, replaybuffer.py:243-287) or `num` transitions whose
        arguments carry a leading dimension of size num (batched rollout).  `obs` / `next_obs` may be
        (agent_obs, graph_obs) pairs: both parts land in the joint ring row without a concat."""
        _lib.require_device()
        vals = dict(zip(ADD_ORDER, (obs, action, reward, next_obs, adj, next_adj, done, episode_done, agent_state,
                                    node_state, node_aux, node_obs, node_adj, node_agent_matrix, next_node_obs,
                                    next_node_adj, next_node_agent_matrix)))
        n = int(num)
        assert n <= self.buffer_size
        fields = (_lib.ReplayField * _lib.GM_REPLAY_MAX_FIELDS)()
        keep = []
        k = 0
        for name in ADD_ORDER:
            ring = getattr(self, name)
            eb = ring[0].numel() * ring.element_size()
            if eb == 0:
                continue
            v = vals[name]
            if name in ("obs", "next_obs") and isinstance(v, (tuple, list)):
                # split joint observation: column blocks of the [A, D] ring element
                (A, D), dt = self._shapes[name]
                col = 0
                for part in v:
                    w = part.shape[-1]
                    t = part if part.dtype == dt else part.to(dt)
                    t = t.reshape(n * A, w).contiguous()
                    keep.append(t)
                    f = fields[k]
                    f.ring, f.src, f.elem_bytes = ring.data_ptr(), t.data_ptr(), eb
                    f.rows, f.row_bytes = A, w * ring.element_size()
                    f.ring_pitch, f.ring_offset = D * ring.element_size(), col * ring.element_size()
                    col += w
                    k += 1
                assert col == D, f"{name}: parts cover {col} of {D} columns"
                continue
            src, convert, bcast = self._source(name, v, n)
            keep.append(src)
            f = fields[k]
            f.ring, f.src, f.elem_bytes, f.convert, f.broadcast = ring.data_ptr(), src.data_ptr(), eb, convert, bcast
            k += 1
        index, index_dev = self.index, None
        if self._dev_index is not None:
            index, index_dev = self._dev_index.offset(self.index) % self.buffer_size, self._dev_index.ptr()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().gm_replay_insert(fields, k, self.buffer_size, index, index_dev, n, _lib.current_stream()))
            cur = torch.cuda.current_stream()
            if cur != torch.cuda.default_stream() and not torch.cuda.is_current_stream_capturing():
                # insert running on a side stream (overlapped with the next rollout step): keep the caching
                # allocator from recycling the sources before the copy has run
                for t in keep:
                    t.record_stream(cur)
        # the sources of the last TWO inserts stay referenced: inside a captured graph unit (no record_stream) the
        # allocator must not hand a source block to step k+2's main-stream work while insert k may still read it on the
        # side stream -- the main stream joins the side stream only at the end of the unit
        self._keep_prev = getattr(self, "_keep", None)
        self._keep = keep
        self.count = min(self.buffer_size, self.count + n)
        self.index = (self.index + n) % self.buffer_size

    # ---- sample ------------------------------------------------------------------------------
    def _get_transition_batch(self, indices, device) -> TransitionBatch:
        _lib.require_device()
        n = len(indices)
        idx = self._device_indices(indices)
        names = [f for f in TransitionBatch._fields if f != "idx"]
        fields = (_lib.ReplayField * len(names))()
        outs = {}
        k = 0
        for name in names:
            ring = getattr(self, name)
            shape, dt = self._shapes[name]
            od = self._out_dtype[name]
            out = torch.empty((n, *shape), dtype=od, device=self.device)
            outs[name] = out
            eb = ring[0].numel() * ring.element_size()
            if eb == 0:
                continue
            if od == torch.float32 and dt == torch.bool:
                conv = 1
            elif od == torch.int64:
                conv = 2
            elif od == torch.float32 and dt == torch.float16:
                conv = 3
            else:
                conv = 0
            fields[k].ring, fields[k].dst, fields[k].elem_bytes, fields[k].convert = (
                ring.data_ptr(), out.data_ptr(), eb, conv)
            k += 1
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().gm_replay_sample(fields, k, idx.data_ptr(), n, _lib.current_stream()))
        dev = torch.device(device)
        return TransitionBatch(indices, *[outs[f].to(dev, non_blocking=True) for f in names])


class CompactReplayBuffer(_RingSampler):
    """Compact replay format for the batched rollout (SURVEY 8f-3): a transition keeps only what cannot be recomputed

        rec / next_rec   the packed Routing env record before / after the step (csrc/routing_env.cu layout)
        topo             topology-pool index of the env
        action i8[A], reward f32[A], done[A], episode_done, node_state f32[N,S]

    (23 kB instead of the reference's 141 kB at BASELINE config 2) and `get_batch` rebuilds all 17 fields of the
    reference's TransitionBatch (replaybuffer.py:132-187) on the device: the dense one-hot `obs` / `node_obs` /
    `adj` / `node_agent_matrix` rows of both sides of the transition come from the env's own observation emitters
    run on the gathered records (gm_routing_observe), `node_adj` / `node_aux` from the topology pool, and the
    graph-observation tail of `obs` / `next_obs` from two NetMon steps starting at `node_state` -- the same
    recomputation the learner performs anyway before it uses them (main.py:854-880, 909-915).  With unchanged NetMon
    weights every field is bit-identical to what the dense ring returns (tests/test_gpu_rollout.py).

    `env` is the batched NetMonWrapper over Routing that produces the transitions.  Insert is two small launches per
    batched step: `stage()` BEFORE env.step (the records are advanced in place) and `commit()` after it."""

    FIELDS = ("rec", "next_rec", "topo", "action", "reward", "done", "episode_done", "node_state")

    def __init__(self, seed, buffer_size, env, device_sampler=False, state_ring=False, ring_align=1):
        """state_ring: the node_state field doubles as the NetMon state history of the rollout (rollout.Rollout): the
        NetMon step that produces the observations of transition t+1 reads its state from that transition's block and
        writes the next one, so the state is never copied into the ring.  The field then has its own modulus
        (capacity in steps + 2 blocks: two states are always "ahead" of the newest committed transition), rounded up to a
        multiple of `ring_align` steps so that captured CUDA-graph units of that length meet the same blocks again."""
        self.env = env
        be = env.get()
        self.device = be.device
        self.buffer_size = int(buffer_size)
        self.count = 0
        self.index = 0
        A, N = be._A, be._N
        S = env.netmon.get_state_size()
        stride = be._layout["stride"]
        z = lambda shape, dt: torch.zeros((self.buffer_size, *shape), dtype=dt, device=self.device)
        self.rec, self.next_rec = z((stride,), torch.uint8), z((stride,), torch.uint8)
        self.topo = z((), torch.int32)
        self.action, self.reward, self.done = z((A,), torch.int8), z((A,), torch.float32), z((A,), torch.bool)
        self.episode_done = z((), torch.bool)
        self.state_ring = bool(state_ring)
        self.steps_total = 0  # batched steps committed so far (state-ring mode: transition t <-> state block t % M)
        if self.state_ring:
            B = be.num_envs
            assert self.buffer_size % B == 0 and self.buffer_size // B >= 1, "a state ring needs a capacity of whole batched steps"
            self._B, self.cap_steps = B, self.buffer_size // B
            a = max(1, int(ring_align))
            self.M = -(-(self.cap_steps + 2) // a) * a
            self.node_state = torch.zeros((self.M * B, N, S), dtype=torch.float32, device=self.device)
        else:
            self.node_state = z((N, S), torch.float32)
        self._zero_topo = torch.zeros((1,), dtype=torch.int32, device=self.device)
        self._flags = {v: torch.full((1,), v, dtype=torch.bool, device=self.device) for v in (False, True)}
        self._dev_index = None  # _lib.DeviceCounter in CUDA-graph mode (rollout.Rollout)
        self._staged = False
        self._init_sampler(seed, device_sampler)

    def state_block(self, t):
        """State-ring mode: the [B,N,S] block that holds the node_state of transition (batched step) t."""
        b = (int(t) % self.M) * self._B
        return self.node_state[b:b + self._B]

    def _state_slots(self, idx, clock=None):
        """Ring slots (device int64) -> rows of the state ring: slot s was written by step t = T - 1 - age.  clock: the
        (head step, steps_total) pair as device int64 tensors instead of the host counters (captured CUDA graphs)."""
        if not self.state_ring:
            return idx
        B, cap = self._B, self.cap_steps
        j_now, total = clock if clock is not None else ((self.index // B) % cap, self.steps_total)
        age = (j_now - 1 - idx // B) % cap
        t = total - 1 - age
        return (t % self.M) * B + idx % B

    def clock(self):
        """(head step, steps_total): the host counters _state_slots() reads, for a device copy of them."""
        return (self.index // self._B) % self.cap_steps, self.steps_total

    def sample_env_sequences(self, batch_size, seq_len, out=None):
        """[seq_len, batch_size] ring slots (device int64) of per-env sequences in state-ring mode: row k holds the slot
        of row 0's env k batched steps later.  Start steps follow get_batch's sequence rule counted in steps (the whole
        sequence stays behind the ring head), then one env per sample is drawn (csrc/replay_sampler.cu,
        gm_replay_sample_env_sequences).  Needs device_sampler=True; `out` receives the slots in place."""
        assert self.state_ring and self._pcg_dev is not None, "per-env sequences need the state ring and the device sampler"
        _lib.require_device()
        T = int(seq_len)
        if out is None:
            out = torch.empty((T, batch_size), dtype=torch.int64, device=self.device)
        assert out.shape == (T, batch_size) and out.dtype == torch.int64 and out.is_contiguous()
        B = self._B
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().gm_replay_sample_env_sequences(self._pcg_dev.data_ptr(), self.count // B, self.index // B,
                                                                 B, batch_size, T, out.data_ptr(), _lib.current_stream()))
        return out

    def learner_views(self, idx, clock=None):
        """What a learner that recomputes the graph observation needs of the transitions at ring slots `idx` (device
        int64 [n]): the gathered compact fields (rec / next_rec / topo / action / reward / done / episode_done /
        node_state), the agent observations, node observations and agent nodes of both sides (`obs`, `node_obs`,
        `agent_node`, `next_obs`, `next_node_obs`, `next_agent_node`, plus the env's sparse node rows `node_sparse` /
        `next_node_sparse` for NetMon's sparse encoder) -- no NetMon forwards, unlike get_batch.
        clock: see _state_slots."""
        be = self.env.get()
        g = self._gather(idx, clock)
        cur = be.observe_records(g["rec"], g["topo"])
        nxt = be.observe_records(g["next_rec"], g["topo"])
        for k in ("obs", "node_obs", "agent_node", "node_sparse"):
            g[k], g["next_" + k] = cur[k], nxt[k]
        return g

    def bytes_per_transition(self):
        return sum(getattr(self, f)[0].numel() * getattr(self, f).element_size() for f in self.FIELDS)

    def _insert(self, items, n):
        """items: (ring, source tensor [n or 1 rows], convert, broadcast)."""
        fields = (_lib.ReplayField * _lib.GM_REPLAY_MAX_FIELDS)()
        keep = []
        for k, (ring, src, convert, bcast) in enumerate(items):
            f = fields[k]
            f.ring, f.src, f.elem_bytes = ring.data_ptr(), src.data_ptr(), ring[0].numel() * ring.element_size()
            f.convert, f.broadcast = convert, bcast
            keep.append(src)
        index, index_dev = self.index, None
        if self._dev_index is not None:
            index, index_dev = self._dev_index.offset(self.index) % self.buffer_size, self._dev_index.ptr()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().gm_replay_insert(fields, len(items), self.buffer_size, index, index_dev, n,
                                                   _lib.current_stream()))
        return keep

    # ---- fused insert: the env's step kernel writes the transition (state-ring mode) -------------------------------
    def ring_io(self, episode_done):
        """gm_routing_io.ring_* arguments for Routing.set_ring(): the step kernel then writes this step's transition
        (records before / after, topology index, actions, reward, done, episode_done) into the slots at the ring head --
        what stage() + commit() do with two insert launches.  Follow the step with advance()."""
        assert self.state_ring, "the fused insert needs the state ring (node_state is written in place by NetMon)"
        index, index_dev = self.index, None
        if self._dev_index is not None:
            index, index_dev = self._dev_index.offset(self.index) % self.buffer_size, self._dev_index.ptr()
        return dict(ring_rec=self.rec.data_ptr(), ring_next_rec=self.next_rec.data_ptr(), ring_topo=self.topo.data_ptr(),
                    ring_action=self.action.data_ptr(), ring_reward=self.reward.data_ptr(), ring_done=self.done.data_ptr(),
                    ring_episode_done=self.episode_done.data_ptr(), ring_capacity=self.buffer_size, ring_index=index,
                    ring_index_dev=index_dev, ring_episode_flag=int(bool(episode_done)))

    def advance(self, num):
        """Host bookkeeping of the `num` transitions a step kernel wrote through ring_io()."""
        n = int(num)
        self.count = min(self.buffer_size, self.count + n)
        self.index = (self.index + n) % self.buffer_size
        self.steps_total += 1

    def stage(self, num):
        """Before env.step: the records (and topology indices) that produced the current observations."""
        _lib.require_device()
        be = self.env.get()
        n = int(num)
        assert n == be.num_envs and n <= self.buffer_size
        ti = be._topo_index
        items = [(self.rec, be._state, 0, 0), (self.topo, self._zero_topo if ti is None else ti, 0, 1 if ti is None else 0)]
        self._keep0 = self._insert(items, n)
        self._staged = True

    def commit(self, action, reward, done, episode_done, node_state, num):
        """After env.step (+ the NetMon step): completes the `num` transitions staged at the ring head."""
        assert self._staged, "CompactReplayBuffer.commit() without stage()"
        be = self.env.get()
        n = int(num)
        action = action.reshape(n, -1)
        conv = 4 if action.dtype == torch.int32 else 0
        if not conv and action.dtype != torch.int8:
            action = action.to(torch.int8)
        done_b = done.contiguous().view(torch.bool) if done.dtype in (torch.uint8, torch.int8) else done.to(torch.bool).contiguous()
        if torch.is_tensor(episode_done):
            ep, ep_b = episode_done.to(torch.bool).reshape(-1).contiguous(), 0 if episode_done.numel() == n else 1
        else:
            ep, ep_b = self._flags[bool(episode_done)], 1
        items = [(self.next_rec, be._state, 0, 0), (self.action, action.contiguous(), conv, 0),
                 (self.reward, reward.reshape(n, -1).contiguous(), 0, 0), (self.done, done_b.reshape(n, -1), 0, 0),
                 (self.episode_done, ep, 0, ep_b)]
        if not self.state_ring:  # (state-ring mode: the NetMon steps wrote it in place)
            if node_state is None or (isinstance(node_state, (int, float)) and node_state == 0):
                if getattr(self, "_zero_state", None) is None:
                    self._zero_state = torch.zeros_like(self.node_state[:1])  # main.py:692-696 stores 0 before the first step
                ns, ns_b = self._zero_state, 1
            else:
                ns, ns_b = node_state.reshape(n, *self.node_state.shape[1:]).contiguous(), 0
            items.append((self.node_state, ns, 0, ns_b))
        self._keep1 = self._insert(items, n)
        self._staged = False
        self.count = min(self.buffer_size, self.count + n)
        self.index = (self.index + n) % self.buffer_size
        self.steps_total += 1

    # ---- sample: gather the compact fields, rebuild the reference's 17 dense fields ----------------
    def _gather(self, idx, clock=None):
        n = idx.shape[0]
        spec = [("rec", torch.uint8, 0), ("next_rec", torch.uint8, 0), ("topo", torch.int32, 0), ("action", torch.int64, 2),
                ("reward", torch.float32, 0), ("done", torch.bool, 0), ("episode_done", torch.bool, 0),
                ("node_state", torch.float32, 0)]
        fields = (_lib.ReplayField * len(spec))()
        out = {}
        for k, (name, od, conv) in enumerate(spec):
            ring = getattr(self, name)
            out[name] = torch.empty((n, *ring.shape[1:]), dtype=od, device=self.device)
            fields[k].ring, fields[k].dst, fields[k].convert = ring.data_ptr(), out[name].data_ptr(), conv
            fields[k].elem_bytes = ring[0].numel() * ring.element_size()
        with torch.cuda.device(self.device):
            if self.state_ring:  # the state field has its own modulus: gather it with its own row indices
                sidx = self._state_slots(idx, clock).contiguous()
                _lib.check(_lib.lib().gm_replay_sample(fields, len(spec) - 1, idx.data_ptr(), n, _lib.current_stream()))
                last = (_lib.ReplayField * 1)()
                C.memmove(last, C.byref(fields[len(spec) - 1]), C.sizeof(_lib.ReplayField))
                _lib.check(_lib.lib().gm_replay_sample(last, 1, sidx.data_ptr(), n, _lib.current_stream()))
            else:
                _lib.check(_lib.lib().gm_replay_sample(fields, len(spec), idx.data_ptr(), n, _lib.current_stream()))
        return out

    def _get_transition_batch(self, indices, device) -> TransitionBatch:
        _lib.require_device()
        env, be = self.env, self.env.get()
        nm, pool = env.netmon, be._pool
        idx = self._device_indices(indices)
        g = self._gather(idx)
        n = idx.shape[0]
        topo = g["topo"]
        cur = be.observe_records(g["rec"], topo)
        nxt = be.observe_records(g["next_rec"], topo)
        be.get_nodes_adjacency(), be.get_node_aux()  # materialise the pool's dense tables
        tl = topo.long()
        node_adj = pool.node_adj.index_select(0, tl).float()
        node_aux = pool.apsp_f32.index_select(0, tl)
        # graph-observation tails: NetMon from the stored state on the current, then on the next node view
        saved = nm.state
        with torch.no_grad():
            nm.state = g["node_state"]
            md = pool.nbr_all.shape[-1] - 1
            nnz = getattr(be, "node_obs_nnz", 0)  # same encoder path as the rollout that produced the transitions
            _, tail = nm.forward_lists(cur["node_obs"], pool.nbr_all, pool.deg, topo, md, agent_node=cur["agent_node"], sparse_nnz=nnz,
                                       sparse_rows=cur.get("node_sparse"), static_rows=getattr(be, "node_static_rows", None))
            _, ntail = nm.forward_lists(nxt["node_obs"], pool.nbr_all, pool.deg, topo, md, agent_node=nxt["agent_node"], sparse_nnz=nnz,
                                        sparse_rows=nxt.get("node_sparse"), static_rows=getattr(be, "node_static_rows", None))
        nm.state = saved
        A = be._A
        f = dict(
            obs=torch.cat((cur["obs"], tail), -1), action=g["action"], reward=g["reward"],
            next_obs=torch.cat((nxt["obs"], ntail), -1), adj=cur["adj"].float(), next_adj=nxt["adj"].float(),
            done=g["done"], episode_done=g["episode_done"],
            agent_state=torch.empty((n, A, 0), dtype=torch.float32, device=self.device),
            node_obs=cur["node_obs"], node_adj=node_adj, node_state=g["node_state"], node_aux=node_aux,
            node_agent_matrix=cur["node_agent"].float(), next_node_obs=nxt["node_obs"], next_node_adj=node_adj,
            next_node_agent_matrix=nxt["node_agent"].float())
        dev = torch.device(device)
        return TransitionBatch(indices, *[f[k].to(dev, non_blocking=True) for k in TransitionBatch._fields if k != "idx"])
