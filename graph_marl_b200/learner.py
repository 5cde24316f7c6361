"""Batched DQN + NetMon learner on the compact replay ring (the learner of src/main.py:830-1026, restated for sequences
in tools/train_simple.py), with the TD gradient and the optimizer tail in CUDA (csrc/learner.cu).

One update samples per-env sequences from the state ring, runs the device NetMon / DQN forwards with their device
backward (model._NetMonStepFn, model._MlpFn), hands the TD gradient of every element to one autograd backward, and
applies clip_grad_value_ + clip_grad_norm_ + AdamW + the Polyak target update in three launches.  With graph=True the
update, after one eager warm-up, is replayed from a captured CUDA graph.
"""
import copy
import ctypes as C

import torch

from . import _lib
from .model import _NetMonStepFn


class Learner:
    def __init__(self, netmon, model, lr, gamma, tau, clip_value=0.5, max_norm=1.0, graph=True):
        """netmon / model: the online NetMon and DQN (their parameters are updated in place); the target DQN is a deepcopy
        of `model`.  AdamW with torch's defaults (betas 0.9 / 0.999, eps 1e-8, weight_decay 0.01)."""
        self.netmon, self.model = netmon, model
        self.target = copy.deepcopy(model)
        self.target._pack = type(model._pack)()  # its own weight pack (the deepcopy would share the key of model's)
        self.gamma, self.graph = float(gamma), bool(graph)
        self.device = next(model.parameters()).device
        # parameter order of the reference's optimizer (main.py / train_simple.py): DQN, then NetMon
        self.params = list(model.parameters()) + list(netmon.parameters())
        self.opt = FusedOptimizer(self.params, list(zip(model.parameters(), self.target.parameters())), lr, tau,
                                  clip_value, max_norm)
        self.loss = torch.zeros((1,), dtype=torch.float32, device=self.device)   # loss of the latest update
        # the inference workspaces of the next-observation NetMon step and of the target DQN's act(): never the rollout's
        # (captured rollout units hold its address), and one pair per captured update (a graph holds the addresses of the
        # pair it was captured with; a larger batch must not reallocate them)
        self._ws_eager = self._new_workspaces()
        self._static = {}   # (buffer, batch, seq_len) -> static index / clock tensors and workspaces of the captured update
        self._graphs = CapturedUpdates()
        self.updates = 0

    def td_grad(self, q, q_next, action, reward, done, scale):
        """gm_td_grad: returns dq (f32 like q) and adds scale * sum (q[action] - y)^2 into self.loss."""
        nA = q.shape[-1]
        q2, qn2 = q.reshape(-1, nA).contiguous(), q_next.reshape(-1, nA).contiguous()
        act = action.reshape(-1).to(torch.int64).contiguous()
        rew = reward.reshape(-1).float().contiguous()
        dn = done.reshape(-1).to(torch.bool).contiguous().view(torch.uint8)
        dq = torch.empty_like(q2)
        with torch.cuda.device(q.device):
            _lib.check(_lib.lib().gm_td_grad(q2.data_ptr(), qn2.data_ptr(), act.data_ptr(), rew.data_ptr(), dn.data_ptr(),
                                             q2.shape[0], nA, self.gamma, float(scale), dq.data_ptr(), self.loss.data_ptr(),
                                             self.opt.partials.data_ptr(), _lib.current_stream()))
        return dq.view(q.shape)

    def _new_workspaces(self):
        return type(self.netmon._ws)(), type(self.target._ws)()

    def _body(self, buff, idx, clock, ws):
        self.forward_backward(buff, idx, clock, ws)
        self.opt.step()

    def forward_backward(self, buff, idx, clock=None, ws=None):
        """The update on the sampled slots idx [T, batch]: for each element t

          1. state: t = 0 the ring's stored node_state; t > 0 the previous element's output state, zeroed for samples
             whose previous transition ended its episode (episode_done) -- the carried state of main.py's learner
          2. NetMon step with gradient (device forward + backward) on the pool's adjacency lists
          3. its readout gathered at the agents' nodes (equal to the one-hot node-agent bmm)
          4. online Q of [agent obs | graph obs]
          5. no grad: NetMon on the next node view from the detached output state, then the target DQN's Q
          6. TD gradient (gm_td_grad)

        then one backward over all elements into the parameters' .grad tensors (zeroed first, in place).  ws: the
        (NetMon, target DQN) inference workspaces to use (default: the learner's eager pair)."""
        self.opt.check_grads()
        nm, be = self.netmon, buff.env.get()
        pool = be._pool
        nbr, deg = pool.nbr_all, pool.deg
        md = nbr.shape[-1] - 1
        T, n = idx.shape
        A, nA = be._A, self.model.num_actions
        scale = 1.0 / (n * A * nA * T)
        self.loss.zero_()
        torch._foreach_zero_([p.grad for p in self.params])
        params = nm.step_params()
        nnz, static_rows = getattr(be, "node_obs_nnz", 0), getattr(be, "node_static_rows", None)
        qs, dqs = [], []
        state, prev_end = None, None
        saved, saved_ws, saved_tws = nm.state, nm._ws, self.target._ws
        nm._ws, self.target._ws = ws if ws is not None else self._ws_eager
        try:
            for t in range(T):
                v = buff.learner_views(idx[t], clock)
                topo = v["topo"]
                st = v["node_state"] if t == 0 else state * (~prev_end).to(state.dtype).view(-1, 1, 1)
                node_out, state = _NetMonStepFn.apply(nm, v["node_obs"], nbr, deg, topo, md, st, *params)
                an = v["agent_node"].long().unsqueeze(-1).expand(-1, -1, node_out.shape[-1])
                x = torch.cat((v["obs"], torch.gather(node_out, 1, an)), -1)
                q = self.model(x, None)
                with torch.no_grad():
                    nm.state = state.detach()
                    _, g_next = nm.forward_lists(v["next_node_obs"], nbr, deg, topo, md, agent_node=v["next_agent_node"],
                                                 sparse_nnz=nnz, sparse_rows=v.get("next_node_sparse"), static_rows=static_rows)
                    q_next, _ = self.target.act(v["next_obs"], g_next, epsilon=0.0, want_q=True)
                    dqs.append(self.td_grad(q.detach(), q_next, v["action"], v["reward"], v["done"], scale))
                qs.append(q)
                prev_end = v["episode_done"]
        finally:
            nm.state, nm._ws, self.target._ws = saved, saved_ws, saved_tws
        torch.autograd.backward(qs, dqs)

    def refresh_packs(self):
        """The optimizer kernel writes the weights through raw pointers (their version counters do not move): repack the
        online NetMon, online DQN and target DQN into their existing pack buffers, which captured rollout units and the
        next act() read."""
        for m in (self.netmon, self.model, self.target):
            m._pack.refresh()

    def update(self, buff, batch, seq_len):
        """One learner update on `batch` per-env sequences of `seq_len` transitions from `buff` (a state-ring
        CompactReplayBuffer with the device sampler).  Returns the update's loss as a device scalar tensor."""
        _lib.require_device()
        self.opt.check_grads()
        key = (id(buff), int(batch), int(seq_len))
        if not self.graph:
            self._body(buff, buff.sample_env_sequences(batch, seq_len), None, self._ws_eager)
        else:
            s = self._static.get(key)
            if s is None:
                s = self._static[key] = dict(idx=torch.zeros((seq_len, batch), dtype=torch.int64, device=self.device),
                                             clock=torch.zeros((2,), dtype=torch.int64, device=self.device),
                                             ws=self._new_workspaces(), buff=buff)  # (holds buff: its id stays unique)
            buff.sample_env_sequences(batch, seq_len, out=s["idx"])
            for i, c in enumerate(buff.clock()):
                s["clock"][i].fill_(c)
            clock = (s["clock"][0], s["clock"][1])
            pool = buff.env.get()._pool
            if s.get("pool") is not pool:  # new topology tables (random-topology pools): the captured update is stale
                self._graphs.pop(key, None)
                s["pool"] = pool
            self._graphs.run(key, lambda: self._body(buff, s["idx"], clock, s["ws"]))
        self.refresh_packs()
        self.updates += 1
        return self.loss.clone()


class CapturedUpdates(dict):
    """key -> captured CUDA graph of an update, all captured into one shared memory pool.  The first run of a key is
    eager, so that workspaces, weight packs and autograd state exist before capture; the second synchronises, captures
    and replays; later runs replay.  A key popped from the dict is captured again on its next run, without another eager
    run."""

    def __init__(self):
        super().__init__()
        self._warm = set()
        self._pool = None

    def run(self, key, body):
        g = self.get(key)
        if g is None and key not in self._warm:
            body()
            self._warm.add(key)
            return
        if g is None:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=self._pool):
                body()
            if self._pool is None:
                self._pool = g.pool()
            self[key] = g
        g.replay()


class FusedOptimizer:
    """clip_grad_value_ + clip_grad_norm_ + torch.optim.AdamW(foreach=False, betas 0.9 / 0.999, eps 1e-8,
    weight_decay 0.01) over `params`, then target = tau * online + (1 - tau) * target over `pairs` (util.interpolate_model)
    in the three launches of gm_optimizer_step.  Every .grad gets a preallocated tensor whose address the device table
    holds: zero it in place, never replace it."""

    def __init__(self, params, pairs, lr, tau, clip_value=0.5, max_norm=1.0):
        self.params = list(params)
        dev = self.params[0].device
        for p in self.params:
            assert p.dtype == torch.float32 and p.is_contiguous() and p.device == dev
            if p.grad is None:
                p.grad = torch.zeros_like(p)
        self._grads = [p.grad for p in self.params]
        self.exp_avg = [torch.zeros_like(p) for p in self.params]
        self.exp_avg_sq = [torch.zeros_like(p) for p in self.params]
        table = (_lib.OptEntry * len(self.params))()
        for e, p, m, v in zip(table, self.params, self.exp_avg, self.exp_avg_sq):
            e.param, e.grad, e.exp_avg, e.exp_avg_sq, e.numel = p.data_ptr(), p.grad.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel()
        ptab = (_lib.OptPair * max(len(pairs), 1))()
        for e, (on, tg) in zip(ptab, pairs):
            assert on.shape == tg.shape and tg.dtype == torch.float32 and tg.is_contiguous()
            e.online, e.target, e.numel = on.data_ptr(), tg.data_ptr(), on.numel()
        to_dev = lambda arr: torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev)
        self._table, self._pairs, self._n, self._n_pairs = to_dev(table), to_dev(ptab), len(self.params), len(pairs)
        self._keep = [tg for _, tg in pairs]
        self.hparams = _lib.OptHparams(lr=float(lr), beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.01, tau=float(tau),
                                       clip_value=float(clip_value), max_norm=float(max_norm))
        self.step_count = torch.zeros((1,), dtype=torch.int64, device=dev)
        self.partials = torch.empty((_lib.GM_LEARNER_PARTIALS,), dtype=torch.float64, device=dev)
        self.device = dev

    def check_grads(self):
        """Raise when a .grad tensor is no longer the one the device table points at (e.g. after zero_grad(), which sets
        grads to None, or an assignment to .grad): the kernels would read and write memory nothing else uses."""
        for i, (p, g) in enumerate(zip(self.params, self._grads)):
            if p.grad is not g:
                raise _lib.GraphMarlError(f"parameter {i}: .grad was replaced or set to None; the fused optimizer keeps "
                                          "its own .grad tensors (zero them in place, e.g. zero_grad(set_to_none=False))")

    def step(self):
        self.check_grads()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().gm_optimizer_step(self._table.data_ptr(), self._n, self._pairs.data_ptr(), self._n_pairs,
                                                    self.step_count.data_ptr(), C.byref(self.hparams),
                                                    self.partials.data_ptr(), _lib.current_stream()))
