"""Training and evaluation of sl.py's shortest-path NetMon (BASELINE config 5, src/sl.py:366-536) on the device dataset
of `sl_dataset.build_sl_dataset`, with the loss gradient in CUDA (`gm_sl_mse_grad`, csrc/learner.cu).

SURVEY §3.5 describes `sl.py`'s training step:
- state `None` at the start of a sequence;
- the same node observations fed for `sequence_length` NetMon steps;
- the identity node-agent matrix, so NetMon's per-node output is used directly;
- an MSE of the all-pairs prediction ("pred_all") against the shortest-path weights;
- AdamW with default arguments;
- batches drawn uniformly with replacement.

The trainer implements this as follows. Given a batch of sample indices `idx[b]`, with `b < B`, drawn from a dataset of
S samples:

    state = None
    for t in 0 .. T-1:
        node_out_t, state = NetMon step(node_obs[idx], lists[idx], state)      # [B, N, O], O = H (1 + max_degree)
        pred_t = head(node_out_t.view(B*N, O))                                  # [B*N, N], head = model.MLP, last layer N wide, no output activation
        loss  += mean over (b, v, u) of (pred_t[b*N+v, u] - targets_all[idx[b], v, u])^2

The head's output `[b·N + v, u]` predicts the weight from v to u. After the loop comes a backward through all T steps,
then AdamW over the NetMon parameters followed by the head's (torch defaults: betas 0.9/0.999, eps 1e-8,
weight_decay 0.01, `lr` as given), with no gradient clipping. The state is carried from step to step without masking.

One update draws the batch on the device (`gm_replay_sample_indices`: `np.random.default_rng(seed).choice(S, B)` with the
PCG64 state in HBM), runs the device NetMon forward / backward (`model._NetMonStepFn`) over the dataset's adjacency
lists and the head through `model._MlpFn`, takes each step's loss gradient from `gm_sl_mse_grad` (targets read from the
dataset through the sample index), and applies AdamW through `learner.FusedOptimizer` with infinite clip bounds (the
clamp and the norm scale are then exact no-ops).  With graph=True every (batch, seq_len) is, after one eager warm-up,
replayed from a captured CUDA graph, which does not synchronise with the host.
"""
import numpy as np
import torch

from . import _lib
from .learner import CapturedUpdates, FusedOptimizer
from .model import NetMon, _mlp_fn_args, _MlpFn, _NetMonStepFn


def adjacency_lists(node_adj, chunk=4096):
    """Neighbour lists of a dataset's int8 [S, N, N] adjacency (self loops included) through gm_adj_to_lists, `chunk`
    samples at a time (no [S, N, N] float mask exists at once): (nbr i32 [S, N, D], deg i32 [S, N], D), where D is every
    row's entry count.  Raises GraphMarlError when the rows do not all have the same degree (sl.py:211 asserts it).
    One host sync."""
    S, N, _ = node_adj.shape
    deg = torch.empty((S, N), dtype=torch.int32, device=node_adj.device)
    for lo in range(0, S, chunk):
        deg[lo:lo + chunk] = (node_adj[lo:lo + chunk] != 0).sum(-1)
    d_min, d_max = torch.stack(torch.aminmax(deg)).tolist()
    if d_min != d_max:
        raise _lib.GraphMarlError(f"sl.py's NetMon needs one degree for every node of every sample; the dataset's rows "
                                  f"have {d_min} to {d_max} entries (self loop included)")
    nbr = torch.empty((S, N, d_max), dtype=torch.int32, device=node_adj.device)
    for lo in range(0, S, chunk):
        nbr[lo:lo + chunk], deg[lo:lo + chunk], _ = NetMon.lists_from_mask(node_adj[lo:lo + chunk], max_entries=d_max)
    return nbr, deg, d_max


class SLTrainer:
    def __init__(self, netmon, head, data, lr=1e-3, seed=0, graph=True):
        """netmon: a NetMon whose configuration the device backward covers (lstm / lnlstm with carry-over, no global
        readout, >= 1 iteration); head: a model.MLP from NetMon's per-node output to N weights; data: the dict that
        build_sl_dataset returns.  Both modules' parameters are updated in place."""
        _lib.require_device()
        x = data["node_obs"]
        why = netmon._device_backward_reason(x)
        if why is not None:
            raise _lib.GraphMarlError(f"SLTrainer runs the device backward only: {why}")
        self.netmon, self.head, self.graph = netmon, head, bool(graph)
        self.device = x.device
        S, N, _ = x.shape
        self.S, self.N = S, N
        self.x, self.targets_all = x, data["targets_all"]
        if x.dtype != torch.float32 or self.targets_all.dtype != torch.int32:
            raise _lib.GraphMarlError("node_obs must be f32 and targets_all i32, as build_sl_dataset returns them")
        self.nbr, self.deg, entries = adjacency_lists(data["node_adj"])
        self.max_degree = entries - 1  # model.py:588-589
        self._md = self.max_degree if netmon.output_neighbor_hidden else 0
        self.out_width = netmon.out_width(self._md)
        layers = list(head.linear_layers)
        if layers[0].in_features != self.out_width or layers[-1].out_features != N:
            raise _lib.GraphMarlError(f"the head maps {layers[0].in_features} -> {layers[-1].out_features} features; "
                                      f"NetMon's per-node output is {self.out_width} wide and N = {N}")
        self._head_spec, self._head_params = _mlp_fn_args(layers, head.activation_fn, head.activation_on_output, netmon.math)
        self._nm_params = netmon.step_params()
        # AdamW alone: no target pairs, clamp at +-inf and max_norm inf leave every gradient as it is
        self.opt = FusedOptimizer(list(netmon.parameters()) + list(head.parameters()), [], lr, 0.0,
                                  clip_value=float("inf"), max_norm=float("inf"))
        self.params = self.opt.params
        st = np.zeros(_lib.GM_PCG64_STATE_WORDS, np.uint64)
        _lib.lib().gm_pcg64_seed(_lib.ptr(st), int(seed) & (2**64 - 1))
        self._pcg = torch.from_numpy(st.view(np.int64)).to(self.device)
        self.loss = torch.zeros((1,), dtype=torch.float32, device=self.device)  # loss of the latest update
        self._static = {}   # (batch, seq_len) -> static index / observation tensors of that update
        self._graphs = CapturedUpdates()
        self.last_indices = None
        self.updates = 0

    def _mse(self, pred, targets_all, index, B, scale, d_pred, loss):
        _lib.check(_lib.lib().gm_sl_mse_grad(pred.data_ptr(), pred.stride(0), targets_all.data_ptr(), _lib.ptr(index), B,
                                             self.N, float(scale), _lib.ptr(d_pred), loss.data_ptr(),
                                             self.opt.partials.data_ptr(), _lib.current_stream()))

    def _body(self, s, B, T):
        nm, N, O = self.netmon, self.N, self.out_width
        idx, li, xb = s["idx"], s["li"], s["x"]
        _lib.check(_lib.lib().gm_replay_sample_indices(self._pcg.data_ptr(), self.S, 0, B, 1, idx.data_ptr(),
                                                       _lib.current_stream()))
        li.copy_(idx)
        torch.index_select(self.x, 0, idx, out=xb)
        self.loss.zero_()
        torch._foreach_zero_([p.grad for p in self.params])
        scale = 1.0 / (B * N * N)
        preds, d_preds = [], []
        state = None
        for _ in range(T):
            node_out, state = _NetMonStepFn.apply(nm, xb, self.nbr, self.deg, li, self._md, state, *self._nm_params)
            pred = _MlpFn.apply(self._head_spec, node_out.view(B * N, O), *self._head_params)
            d = torch.empty_like(pred)
            self._mse(pred, self.targets_all, idx, B, scale, d, self.loss)
            preds.append(pred)
            d_preds.append(d)
        torch.autograd.backward(preds, d_preds)
        self.opt.step()

    def update(self, batch, seq_len):
        """One update on `batch` samples drawn uniformly with replacement, `seq_len` NetMon steps each.  Returns the
        update's loss (the sum over steps of each step's MSE) as a device scalar tensor."""
        self.opt.check_grads()
        B, T = int(batch), int(seq_len)
        if B < 1 or T < 1:
            raise ValueError(f"SLTrainer.update needs batch >= 1 and seq_len >= 1, got {B}, {T}")
        key = (B, T)
        s = self._static.get(key)
        if s is None:
            dev = self.device
            s = self._static[key] = dict(idx=torch.zeros((B,), dtype=torch.int64, device=dev),
                                         li=torch.zeros((B,), dtype=torch.int32, device=dev),
                                         x=torch.empty((B,) + tuple(self.x.shape[1:]), dtype=torch.float32, device=dev))
        with torch.cuda.device(self.device), torch.enable_grad():
            if self.graph:
                self._graphs.run(key, lambda: self._body(s, B, T))
            else:
                self._body(s, B, T)
        # the optimizer kernel writes the weights through raw pointers: repack them for the inference kernels
        self.netmon._pack.refresh()
        self.last_indices = s["idx"]
        self.updates += 1
        return self.loss.clone()

    def evaluate(self, data, sequence_lengths, chunk=4096):
        """sl.py's test over sequence lengths (sl.py:448-536), restated as the MSE of the all-pairs prediction after T
        steps: for each T, every sample of `data` (a build_sl_dataset dict) runs T inference NetMon steps from state None
        (`forward_lists`, the tensor-core or fp32 kernels) and the head, and the last step's prediction is scored
        against targets_all with gm_sl_mse_grad.  Returns {T: mse}; one host read for all T.  netmon.state is left as
        it was found."""
        x, targets_all = data["node_obs"], data["targets_all"]
        S, N, _ = x.shape
        if N != self.N:
            raise _lib.GraphMarlError(f"the evaluation data has N = {N}, the trainer N = {self.N}")
        nbr, deg, entries = adjacency_lists(data["node_adj"], chunk)
        if entries - 1 != self.max_degree:
            raise _lib.GraphMarlError(f"the evaluation data's degree {entries - 1} differs from the training data's "
                                      f"{self.max_degree}")
        Ts = [int(T) for T in sequence_lengths]
        if any(T < 1 for T in Ts):
            raise ValueError(f"sequence lengths must be >= 1, got {Ts}")
        nm, O = self.netmon, self.out_width
        loss = torch.zeros((len(Ts),), dtype=torch.float32, device=self.device)
        saved = nm.state
        try:
            with torch.no_grad(), torch.cuda.device(self.device):
                for k, T in enumerate(Ts):
                    for lo in range(0, S, chunk):
                        c = min(chunk, S - lo)
                        nm.state = None
                        for _ in range(T):
                            node_out, _ = nm.forward_lists(x[lo:lo + c], nbr[lo:lo + c], deg[lo:lo + c], None, self._md,
                                                           want_node_out=True)
                        pred = _MlpFn.apply(self._head_spec, node_out.view(c * N, O), *self._head_params)
                        self._mse(pred, targets_all[lo:lo + c], None, c, 1.0 / (S * N * N), None, loss[k:k + 1])
        finally:
            nm.state = saved
        return dict(zip(Ts, loss.tolist()))
