"""NetMon graph-observation module and the DQN agent model, mirroring src/model.py of the
reference (MLP :13-42, Q_Net :119-125, DQN :187-203, NetMon :256-650) and
src/layernormlstm.py, with the forward passes executed by libgraphmarl_b200.

The modules stay `nn.Module`s with the reference's parameter names (`encode.linear_layers.i`,
`rnn_obs.weight_ih`, `q_net.fc.weight`, ...) so reference checkpoints load and the learner can
optimise them.  Inference (no grad) always runs the CUDA kernels and fails loudly without
them; when autograd is recording (the learner, src/main.py:830-1006, a scheduled row of
SURVEY 8f) the same math is composed from torch ops so gradients exist.
"""
import ctypes as C

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn import LayerNorm, RNNCellBase

from . import _lib


def _act_name(fn):
    name = getattr(fn, "__name__", str(fn))
    if name not in _lib.ACTIVATIONS:
        raise ValueError(f"activation {name} is not built into libgraphmarl_b200 ({list(_lib.ACTIVATIONS)})")
    return name


class _Workspace:
    def __init__(self):
        self.buf = None

    def get(self, nbytes, device):
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            self.buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        return self.buf


def _rows2d(t):
    """[..., D] tensor -> 2-D row view [rows, D] with unit column stride, without copying when the
    leading dimensions collapse to one uniform row stride (e.g. a column slice of a joint tensor)."""
    D = t.shape[-1]
    if t.dim() == 1:
        t = t.unsqueeze(0)
    if t.stride(-1) == 1 or D == 1:
        ok = all(t.stride(i) == t.stride(i + 1) * t.shape[i + 1] for i in range(t.dim() - 2))
        if ok and t.dtype == torch.float32:
            rows = 1
            for n in t.shape[:-1]:
                rows *= n
            return t.as_strided((rows, D), (t.stride(-2), 1))
    return t.reshape(-1, D).float().contiguous()


class PackedRows:
    """Activation rows that exist ONLY as tile-packed bf16 hi/lo blocks (csrc/gemm_sm100.cuh), i.e. the graph
    observation of the batched rollout when nothing needs its fp32 rows: NetMon's agent readout writes it, the
    tensor-core DQN of the same math mode pulls it with bulk copies."""

    is_cuda = True

    def __init__(self, buf, shape, math):
        self.buf, self.shape, self.math = buf, tuple(shape), math

    @property
    def device(self):
        return self.buf.device

    def float(self):
        """The rows as an fp32 tensor of `shape` (hi + lo; hi alone in single-pass bf16, which writes no lo part)."""
        K = self.shape[-1]
        R = 1
        for n in self.shape[:-1]:
            R *= n
        mt, kb = -(-R // 128), K // 32
        # block (mt, kb) -> [hi|lo] planes of [r>>3][(k&31)>>3][r&7][k&7] bf16 elements (layout in csrc/gemm_sm100.cuh)
        x = self.buf.reshape(-1)[:mt * kb * 16384].view(torch.bfloat16).view(mt, kb, 2, 16, 4, 8, 8).float()
        x = x[:, :, 0] if self.math == "bf16" else x[:, :, 0] + x[:, :, 1]
        return x.permute(0, 2, 4, 1, 3, 5).reshape(mt * 128, K)[:R].reshape(self.shape)


class _PackedWeights:
    """Cache of the tensor-core weight pack (bf16 hi/lo tiles) of a module; rebuilt whenever a
    parameter's storage or version counter changes (optimizer step, load_state_dict, .to())."""

    def __init__(self):
        self.buf, self.key, self._pack_fn = None, None, None

    def get(self, module, extra, nbytes_fn, pack_fn):
        params = list(module.parameters())
        key = (extra,) + tuple((q.data_ptr(), q._version) for q in params)
        if key != self.key:
            dev = params[0].device
            n = int(nbytes_fn())
            if self.buf is None or self.buf.numel() < n or self.buf.device != dev:
                self.buf = torch.empty(max(n, 256), dtype=torch.uint8, device=dev)
            assert self.buf.data_ptr() % 256 == 0
            pack_fn(self.buf)
            self.key, self._pack_fn = key, pack_fn
        return self.buf

    def refresh(self):
        """Repack the current parameter values into the existing buffer, with the layout of the last pack.  For writers
        that change parameters without moving their version counters (the learner's optimizer kernel writes through
        raw pointers): captured CUDA graphs hold this buffer's address and keep reading it."""
        if self._pack_fn is not None:
            self._pack_fn(self.buf)


# ---- training path: device-side backward (csrc/train.cu) behind torch.autograd ---------------------
# `loss.backward()` of the unmodified learner (main.py:1002, sl.py:392) reaches these nodes; each runs ONE C-ABI
# call forward (writes a tape) and one backward (hand-written kernels).  A sequence of NetMon steps (main.py:840-915)
# is a chain of _NetMonStep nodes: the state gradient d_state_in of step t+1 is the d_state_out of step t.
GRAD_PATH_CALLS = {"device": 0, "torch": 0}  # how often grad-mode forwards ran the kernels / the torch-composed path
_warned_torch_path = set()


def _note_torch_path(who, why):
    GRAD_PATH_CALLS["torch"] += 1
    if (who, why) not in _warned_torch_path:
        _warned_torch_path.add((who, why))
        import warnings

        warnings.warn(f"{who}: grad-mode forward runs the torch-composed path, not the CUDA kernels ({why})", stacklevel=3)


def _mlp_fn_args(layers, activation_fn, activation_on_output, math):
    """(spec, params) that _MlpFn takes for the nn.Linear `layers` with activation_fn after every layer but the last,
    and after the last too when activation_on_output."""
    act = _lib.ACTIVATIONS[_act_name(activation_fn)]
    acts = (act,) * (len(layers) - 1) + (act if activation_on_output else -1,)
    return (acts, math), [t for l in layers for t in (l.weight, l.bias)]


class _MlpFn(torch.autograd.Function):
    """y = MLP(x) through gm_mlp_forward_train / gm_mlp_backward.  spec: (activation ids per layer, math mode);
    params: each layer's (weight, bias)."""

    @staticmethod
    def _desc(spec, x, params):
        acts, math = spec
        d = _lib.MlpDesc()
        d.n_layers, d.in_features, d.math = len(acts), x.shape[1], _lib.MATH_MODES["bf16x3" if math == "bf16" else math]
        for l in range(len(acts)):
            w, b = params[2 * l], params[2 * l + 1]
            d.units[l], d.act[l], d.w[l], d.b[l] = w.shape[0], acts[l], w.data_ptr(), b.data_ptr()
        return d

    @staticmethod
    def forward(ctx, spec, x, *params):
        rows = x.shape[0]
        d = _MlpFn._desc(spec, x, params)
        lib = _lib.lib()
        tape = torch.empty(int(lib.gm_mlp_tape_floats(C.byref(d), rows)), dtype=torch.float32, device=x.device)
        ws = torch.empty(int(lib.gm_mlp_train_workspace_bytes(C.byref(d), rows)), dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(lib.gm_mlp_forward_train(C.byref(d), rows, x.data_ptr(), x.stride(0), tape.data_ptr(), ws.data_ptr(),
                                                ws.numel(), _lib.current_stream()))
        ctx.save_for_backward(x, tape, *params)
        ctx.spec = spec
        out_w = params[-2].shape[0]
        return tape[tape.numel() - rows * out_w:].view(rows, out_w).clone()

    @staticmethod
    def backward(ctx, d_out):
        x, tape, *params = ctx.saved_tensors
        rows = x.shape[0]
        d = _MlpFn._desc(ctx.spec, x, params)
        g = _lib.MlpGrads()
        grads = []
        for l in range(len(ctx.spec[0])):
            gw = torch.empty_like(params[2 * l]) if ctx.needs_input_grad[2 + 2 * l] else None
            gb = torch.empty_like(params[2 * l + 1]) if ctx.needs_input_grad[3 + 2 * l] else None
            g.w[l], g.b[l] = _lib.ptr(gw), _lib.ptr(gb)
            grads += [gw, gb]
        d_out = d_out.float().contiguous()
        dx = torch.empty_like(x) if ctx.needs_input_grad[1] else None
        lib = _lib.lib()
        ws = torch.empty(int(lib.gm_mlp_train_workspace_bytes(C.byref(d), rows)), dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(lib.gm_mlp_backward(C.byref(d), rows, x.data_ptr(), x.stride(0), tape.data_ptr(), d_out.data_ptr(),
                                           d_out.stride(0), _lib.ptr(dx), C.byref(g), ws.data_ptr(), ws.numel(),
                                           _lib.current_stream()))
        return (None, dx, *grads)


class _NetMonStepFn(torch.autograd.Function):
    """One NetMon step (model.py:476-631 without the node->agent bmm) through gm_netmon_forward_train /
    gm_netmon_backward: (node_obs, state_in, parameters) -> (node_out, state_out)."""

    @staticmethod
    def forward(ctx, nm, x, nbr, deg, list_index, max_degree, state_in, *params):
        B, N, _ = x.shape
        dev = x.device
        p = nm._params(packed=False)
        lib = _lib.lib()
        R = B * N
        H = nm.hidden_features
        tape = torch.empty(int(lib.gm_netmon_tape_floats(C.byref(p), R)), dtype=torch.float32, device=dev)
        ws = torch.empty(int(lib.gm_netmon_train_workspace_bytes(C.byref(p), R)), dtype=torch.uint8, device=dev)
        st_out = torch.empty((B, N, 2 * H), dtype=torch.float32, device=dev)
        O = nm.out_width(max_degree)
        node_out = torch.empty((B, N, O), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.gm_netmon_forward_train(
                C.byref(p), B, N, x.data_ptr(), nbr.data_ptr(), deg.data_ptr(), nbr.shape[-1], _lib.ptr(list_index),
                _lib.ptr(state_in), st_out.data_ptr(), max_degree, node_out.data_ptr(), tape.data_ptr(), ws.data_ptr(),
                ws.numel(), _lib.current_stream()))
        ctx.nm, ctx.max_degree, ctx.has_state = nm, max_degree, state_in is not None
        ctx.save_for_backward(x, nbr, deg, list_index if list_index is not None else x.new_empty(0),
                              state_in if state_in is not None else x.new_empty(0), tape, *params)
        return node_out, st_out

    @staticmethod
    def backward(ctx, d_node_out, d_state_out):
        x, nbr, deg, list_index, state_in, tape, *params = ctx.saved_tensors
        nm = ctx.nm
        B, N, _ = x.shape
        dev = x.device
        H = nm.hidden_features
        p = nm._params(packed=False)
        g = _lib.NetmonGrads()
        grads = [torch.empty_like(q) if ctx.needs_input_grad[7 + i] else None for i, q in enumerate(params)]
        L = len(nm.encode.linear_layers)
        for l in range(L):
            g.enc_w[l], g.enc_b[l] = _lib.ptr(grads[2 * l]), _lib.ptr(grads[2 * l + 1])
        names = nm._cell_param_names()
        for k, cell in enumerate((g.rnn_obs, g.rnn_update)):
            base = 2 * L + len(names) * k
            for j, (_, field) in enumerate(names):
                setattr(cell, field, _lib.ptr(grads[base + j]))
        d_state_in = torch.empty((B, N, 2 * H), dtype=torch.float32, device=dev) if (ctx.has_state and ctx.needs_input_grad[6]) else None
        dn = None if d_node_out is None else d_node_out.float().contiguous()
        ds = None if d_state_out is None else d_state_out.float().contiguous()
        lib = _lib.lib()
        ws = torch.empty(int(lib.gm_netmon_train_workspace_bytes(C.byref(p), B * N)), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.gm_netmon_backward(
                C.byref(p), B, N, x.data_ptr(), nbr.data_ptr(), deg.data_ptr(), nbr.shape[-1],
                list_index.data_ptr() if list_index.numel() else None, state_in.data_ptr() if ctx.has_state else None,
                ctx.max_degree, tape.data_ptr(), _lib.ptr(dn), _lib.ptr(ds), _lib.ptr(d_state_in), C.byref(g), ws.data_ptr(),
                ws.numel(), _lib.current_stream()))
        return (None, None, None, None, None, None, d_state_in, *grads)


class MLP(nn.Module):
    """model.py:13-42."""

    def __init__(self, in_features, mlp_units, activation_fn, activation_on_output=True):
        super().__init__()
        self.activation_fn = activation_fn
        self.linear_layers = nn.ModuleList()
        previous_units = in_features
        if isinstance(mlp_units, int):
            mlp_units = [mlp_units]
        for units in mlp_units:
            self.linear_layers.append(nn.Linear(previous_units, units))
            previous_units = units
        self.out_features = previous_units
        self.activation_on_output = activation_on_output

    def forward(self, x):
        for module in self.linear_layers[:-1]:
            x = self.activation_fn(module(x))
        x = self.linear_layers[-1](x)
        if self.activation_on_output:
            x = self.activation_fn(x)
        return x


class Q_Net(nn.Module):
    """model.py:119-125."""

    def __init__(self, in_features, actions):
        super().__init__()
        self.fc = nn.Linear(in_features, actions)

    def forward(self, x):
        return self.fc(x)


class LayerNormLSTMCell(RNNCellBase):
    """layernormlstm.py:8-42 (parameter container + autograd math)."""

    def __init__(self, input_size, hidden_size, bias=True):
        super().__init__(input_size, hidden_size, bias, num_chunks=4)
        del self.bias_hh
        self.ln_input = LayerNorm(4 * hidden_size)
        self.ln_hidden = LayerNorm(4 * hidden_size)
        self.ln_cell = LayerNorm(hidden_size)

    def forward(self, input, state):
        hx, cx = state
        gates = self.ln_input(torch.mm(input, self.weight_ih.t())) + self.ln_hidden(
            torch.mm(hx, self.weight_hh.t())) + self.bias_ih
        i, f, g, o = gates.chunk(4, 1)
        cy = self.ln_cell(torch.sigmoid(f) * cx + torch.sigmoid(i) * torch.tanh(g))
        return torch.sigmoid(o) * torch.tanh(cy), cy


class DQN(nn.Module):
    """model.py:187-203: MLP encoder (activation on every layer) + linear Q head."""

    def __init__(self, in_features, mlp_units, num_actions, activation_fn, math="fp32"):
        super().__init__()
        self.encoder = MLP(in_features, mlp_units, activation_fn)
        self.q_net = Q_Net(self.encoder.out_features, num_actions)
        self.activation_fn = activation_fn
        self.in_features = in_features
        self.num_actions = num_actions
        self.math = math
        self._ws = _Workspace()
        self._pack = _PackedWeights()

    def _params(self, split=0):
        p = _lib.DqnParams()
        layers = list(self.encoder.linear_layers)
        p.in_features, p.n_layers = self.in_features, len(layers)
        for i, l in enumerate(layers):
            p.units[i] = l.out_features
            p.w[i], p.b[i] = l.weight.data_ptr(), l.bias.data_ptr()
        p.n_actions = self.num_actions
        p.activation = _lib.ACTIVATIONS[_act_name(self.activation_fn)]
        p.math = _lib.MATH_MODES[self.math]
        p.q_w, p.q_b = self.q_net.fc.weight.data_ptr(), self.q_net.fc.bias.data_ptr()
        if self.math != "fp32" and layers[0].weight.is_cuda:
            dev = layers[0].weight.device

            def pack(buf):
                with torch.cuda.device(dev):
                    _lib.check(_lib.lib().gm_dqn_pack_weights(C.byref(p), split, buf.data_ptr(), buf.numel(),
                                                              _lib.current_stream()))

            buf = self._pack.get(self, split, lambda: _lib.lib().gm_dqn_packed_bytes(C.byref(p), split), pack)
            p.packed, p.packed_split = buf.data_ptr(), split
        return p

    def act(self, obs_a, obs_g=None, action_mask=None, epsilon=0.0, rand_action=None, rand_u=None,
            seed=0, step=0, want_q=True, step_dev=None):
        """Q-values and epsilon-greedy actions for rows [..., Da] (+ [..., Dg]) on the device.
        Returns (q [..., n_act] or None, actions int32 [...])."""
        _lib.require_device()
        if not obs_a.is_cuda:
            raise _lib.GraphMarlError("DQN.act needs CUDA tensors (no CPU fallback)")
        lead = obs_a.shape[:-1]
        Da = obs_a.shape[-1]
        a2 = _rows2d(obs_a)
        rows = a2.shape[0]
        g2, Dg = None, 0
        g_pk = None
        if isinstance(obs_g, PackedRows):
            if obs_g.math != self.math or self.math == "fp32":
                raise _lib.GraphMarlError(f"graph observation is tile-packed for math={obs_g.math}, the DQN runs {self.math}")
            Dg, g_pk = obs_g.shape[-1], obs_g.buf
        elif obs_g is not None:
            Dg = obs_g.shape[-1]
            g2 = _rows2d(obs_g)
            pk = getattr(obs_g, "_gm_pk", None)  # tile-packed copy written by NetMon's readout (same math mode)
            if pk is not None and pk[1] == self.math and self.math != "fp32":
                g_pk = pk[0]
        dev = obs_a.device
        p = self._params(split=Da if Dg > 0 else 0)
        nbytes = _lib.lib().gm_dqn_workspace_bytes(C.byref(p), rows)
        ws = self._ws.get(nbytes, dev)
        q = torch.empty((rows, self.num_actions), dtype=torch.float32, device=dev) if want_q else None
        act = torch.empty((rows,), dtype=torch.int32, device=dev)
        if action_mask is not None:
            action_mask = action_mask.reshape(rows, self.num_actions).to(torch.uint8).contiguous()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gm_dqn_act(
                C.byref(p), rows, a2.data_ptr(), Da, a2.stride(0), _lib.ptr(g2), Dg, 0 if g2 is None else g2.stride(0),
                _lib.ptr(g_pk), _lib.ptr(action_mask), float(epsilon), _lib.ptr(rand_action), _lib.ptr(rand_u), int(seed), int(step),
                step_dev, _lib.ptr(q), act.data_ptr(), ws.data_ptr(), ws.numel(), _lib.current_stream()))
        return (None if q is None else q.reshape(*lead, self.num_actions)), act.reshape(lead)

    def forward(self, x, mask):
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            # learner path (main.py:917): one autograd node whose forward / backward are gm_mlp_forward_train /
            # gm_mlp_backward (encoder layers + the Q head as a last layer without activation)
            if x.is_cuda and _act_name(self.activation_fn) in _lib.ACTIVATIONS:
                _lib.require_device()
                GRAD_PATH_CALLS["device"] += 1
                spec, params = _mlp_fn_args(list(self.encoder.linear_layers) + [self.q_net.fc], self.activation_fn, False,
                                            self.math)
                x2 = x.reshape(-1, x.shape[-1]).float().contiguous()
                q = _MlpFn.apply(spec, x2, *params)
                return q.reshape(*x.shape[:-1], self.num_actions)
            _note_torch_path("DQN", "CPU tensors")
            return self.q_net(self.encoder(x))
        q, _ = self.act(x.float())
        return q


class SimpleAggregation(nn.Module):
    """model.py:206-229 (autograd path only; inference aggregates over neighbour lists)."""

    def __init__(self, agg: str, mask_eye: bool) -> None:
        super().__init__()
        assert agg in ("mean", "sum")
        self.agg = agg
        self.mask_eye = mask_eye

    def forward(self, node_features, node_adjacency):
        feature_sum = torch.bmm(node_adjacency, node_features)
        if self.agg == "sum":
            return feature_sum
        return feature_sum / torch.clamp(node_adjacency.sum(dim=-1), min=1).unsqueeze(-1)


class NetMon(nn.Module):
    """model.py:256-650 for agg_type in {sum, mean} and rnn_type in {lstm, lnlstm, gru, none}."""

    def __init__(self, in_features, hidden_features: int, encoder_units, iterations, activation_fn,
                 rnn_type="lstm", rnn_carryover=True, agg_type="sum", output_neighbor_hidden=False,
                 output_global_hidden=False, math="fp32"):
        super().__init__()
        assert isinstance(hidden_features, int)
        self.encode = MLP(in_features, (*encoder_units, hidden_features), activation_fn)
        self.state = None
        self.iterations = iterations
        self.output_neighbor_hidden = output_neighbor_hidden
        self.output_global_hidden = output_global_hidden
        self.rnn_carryover = rnn_carryover
        self.agg_type_str = agg_type
        if agg_type not in ("sum", "mean"):
            raise ValueError(
                f"aggregation type {agg_type}: only 'sum' and 'mean' are built (the torch_geometric "
                "variants of model.py:326-375 are out of scope, SURVEY.md 2 #9)")
        self.aggregate = SimpleAggregation(agg=agg_type, mask_eye=False)
        self.aggregation_def_type = 0
        self.rnn_type = rnn_type
        if rnn_type == "lstm":
            self.rnn_obs = nn.LSTMCell(hidden_features, hidden_features)
            self.rnn_update = nn.LSTMCell(hidden_features, hidden_features)
            self.num_states = 2 if rnn_carryover else 4
        elif rnn_type == "lnlstm":
            self.rnn_obs = LayerNormLSTMCell(hidden_features, hidden_features)
            self.rnn_update = LayerNormLSTMCell(hidden_features, hidden_features)
            self.num_states = 2 if rnn_carryover else 4
        elif rnn_type == "gru":
            self.rnn_obs = nn.GRUCell(hidden_features, hidden_features)
            self.rnn_update = nn.GRUCell(hidden_features, hidden_features)
            self.num_states = 1 if rnn_carryover else 2
        elif rnn_type == "none":
            self.num_states = 1
        else:
            raise ValueError(f"Unknown rnn type {rnn_type}")
        self.in_features = in_features
        self.hidden_features = hidden_features
        self.state_size = hidden_features * self.num_states
        self.activation_fn = activation_fn
        self.math = math
        self._ws = _Workspace()
        self._pack = _PackedWeights()

    def get_out_features(self):
        out = self.hidden_features
        if self.output_neighbor_hidden:
            out += self.hidden_features * 3
        if self.output_global_hidden:
            out += self.hidden_features
        return out

    def get_state_size(self):
        return self.state_size

    # ---- kernel path ---------------------------------------------------------------------------
    def _cell(self, mod):
        c = _lib.CellParams()
        if mod is None:
            return c
        c.w_ih, c.w_hh, c.b_ih = mod.weight_ih.data_ptr(), mod.weight_hh.data_ptr(), mod.bias_ih.data_ptr()
        if self.rnn_type == "lnlstm":
            c.ln_in_w, c.ln_in_b = mod.ln_input.weight.data_ptr(), mod.ln_input.bias.data_ptr()
            c.ln_hid_w, c.ln_hid_b = mod.ln_hidden.weight.data_ptr(), mod.ln_hidden.bias.data_ptr()
            c.ln_cell_w, c.ln_cell_b = mod.ln_cell.weight.data_ptr(), mod.ln_cell.bias.data_ptr()
        else:
            c.b_hh = mod.bias_hh.data_ptr()
        return c

    def _params(self, packed=True):
        p = _lib.NetmonParams()
        layers = list(self.encode.linear_layers)
        p.in_features, p.hidden, p.n_enc_layers = self.in_features, self.hidden_features, len(layers)
        for i, l in enumerate(layers):
            p.enc_units[i] = l.out_features
            p.enc_w[i], p.enc_b[i] = l.weight.data_ptr(), l.bias.data_ptr()
        p.iterations = self.iterations
        p.rnn_type, p.agg_type = _lib.RNN_TYPES[self.rnn_type], _lib.AGG_TYPES[self.agg_type_str]
        p.activation = _lib.ACTIVATIONS[_act_name(self.activation_fn)]
        p.rnn_carryover = int(self.rnn_carryover)
        p.output_neighbor_hidden = int(self.output_neighbor_hidden)
        p.output_global_hidden = int(self.output_global_hidden)
        p.math = _lib.MATH_MODES[self.math]
        p.sparse_input_nnz = int(getattr(self, "_sparse_nnz", 0) or 0)
        st = getattr(self, "_static_rows", None)
        if st is not None:
            p.static_rows, p.n_static_rows, p.static_only = st.data_ptr(), st.shape[0], int(getattr(self, "_static_only", True))
        p.rnn_obs = self._cell(getattr(self, "rnn_obs", None))
        p.rnn_update = self._cell(getattr(self, "rnn_update", None))
        if packed and self.math != "fp32" and layers[0].weight.is_cuda:
            dev = layers[0].weight.device

            def pack(buf):
                with torch.cuda.device(dev):
                    _lib.check(_lib.lib().gm_netmon_pack_weights(C.byref(p), buf.data_ptr(), buf.numel(),
                                                                 _lib.current_stream()))

            extra = 0 if st is None else (st.data_ptr(), st._version, st.shape[0], int(p.static_only))  # the pack folds the static rows in
            p.packed = self._pack.get(self, extra, lambda: _lib.lib().gm_netmon_packed_bytes(C.byref(p)), pack).data_ptr()
        return p

    def out_width(self, max_degree):
        H = self.hidden_features
        return H + (H if self.output_global_hidden else 0) + (max_degree * H if self.output_neighbor_hidden else 0)

    def forward_lists(self, x, nbr_all, deg, list_index=None, max_degree=3, agent_node=None,
                      want_node_out=False, agent_out=None, want_agent_pk=False, want_agent_fp32=True, state_out=None,
                      sparse_nnz=0, sparse_rows=None, static_rows=None, static_only=True):
        """One NetMon step from adjacency lists (no dense mask).  x [B,N,Dn] CUDA f32;
        nbr_all i32[L,N,DM], deg i32[L,N], list_index i32[B] | None; agent_node i32[B,A] | None.
        Updates self.state; returns (node_out | None, agent_out | None).  want_agent_fp32=False with
        want_agent_pk (tensor-core modes): the agents' graph observation is written ONCE, tile-packed, and
        returned as PackedRows (no fp32 rows).  state_out: optional f32 [B,N,S] tensor that receives the new state (e.g.
        a block of the replay ring's node_state field, so that the state is never copied).  sparse_nnz > 0: the caller
        guarantees rows of x with at most that many (<= 12) non-zeros (the Routing env's one-hot node observations have 12).
        sparse_rows: those rows already in sparse form (int32 [B,N,24] on a 128-row padded allocation, Routing's
        `node_sparse` output); when they are given with sparse_nnz <= 6, the tensor-core path runs encoder layers 1 + 2 as
        one kernel (other rows take the two-layer path).
        static_rows: f32 [S, Dn] dictionary of row parts (Routing's `node_static_rows`; layer 1 applied to them is folded
        into the weight pack): the supplied sparse rows index it (static_only, Routing's form), or name static row s as
        column Dn + s next to ordinary input columns (static_only=False)."""
        _lib.require_device()
        if not x.is_cuda:
            raise _lib.GraphMarlError("NetMon needs CUDA tensors (no CPU fallback)")
        B, N, _ = x.shape
        dev = x.device
        x = x.float().contiguous()
        S = self.state_size
        self._sparse_nnz = int(sparse_nnz or 0)
        self._static_rows = static_rows if (static_rows is not None and sparse_rows is not None and self._sparse_nnz > 0) else None
        self._static_only = bool(static_only)
        p = self._params()
        self._sparse_nnz, self._static_rows = 0, None
        if sparse_rows is not None and p.sparse_input_nnz > 0:
            assert sparse_rows.dtype == torch.int32 and sparse_rows.shape == (B, N, 24) and sparse_rows.is_contiguous()
            p.sparse_rows = sparse_rows.data_ptr()
        ws = self._ws.get(_lib.lib().gm_netmon_workspace_bytes(C.byref(p), B * N), dev)
        st_in = None
        hpk_in = None
        if self.state is not None and self.state.numel() > 0:
            st_in = self.state.to(dev).float().reshape(B, N, S).contiguous()
            tag = getattr(self.state, "_gm_hpk", None)  # tile-packed h left by the step that produced this very tensor
            if tag is not None and tag[1] == self.math and st_in.data_ptr() == self.state.data_ptr():
                hpk_in = tag[0]
        if state_out is not None:
            assert state_out.shape == (B, N, S) and state_out.dtype == torch.float32 and state_out.is_contiguous() and state_out.device == dev
            st_out = state_out
        else:
            st_out = torch.empty((B, N, S), dtype=torch.float32, device=dev)
        # fused tensor-core cells (same condition as pack_layout() in csrc/netmon.cu) also leave h tile-packed
        H = self.hidden_features
        fused = self.math != "fp32" and self.rnn_carryover and self.iterations >= 1 and (
            (self.rnn_type == "lstm" and H % 64 == 0) or (self.rnn_type == "lnlstm" and H == 128))
        hpk_out = None
        if fused:
            hpk_out = torch.empty(int(_lib.lib().gm_packed_activation_bytes(B * N, H)), dtype=torch.uint8, device=dev)
        else:
            hpk_in = None
        O = self.out_width(max_degree)
        node_out = torch.empty((B, N, O), dtype=torch.float32, device=dev) if want_node_out else None
        A = 0
        ld = O
        agent_pk = None
        if agent_node is not None:
            A = agent_node.shape[-1]
            if want_agent_pk and self.math != "fp32" and self.hidden_features % 32 == 0:
                agent_pk = torch.empty(int(_lib.lib().gm_packed_activation_bytes(B * A, O)), dtype=torch.uint8, device=dev)
            pk_only = agent_pk is not None and not want_agent_fp32 and agent_out is None
            if agent_out is None and not pk_only:
                agent_out = torch.empty((B, A, O), dtype=torch.float32, device=dev)
            if agent_out is not None:
                ld = agent_out.stride(-2)
        DM = nbr_all.shape[-1]
        if list_index is None and nbr_all.shape[0] != B:
            if nbr_all.shape[0] != 1:
                raise ValueError(f"{nbr_all.shape[0]} adjacency lists for {B} graphs need a list_index")
            list_index = torch.zeros((B,), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gm_netmon_forward(
                C.byref(p), B, N, x.data_ptr(), nbr_all.data_ptr(), deg.data_ptr(), DM, _lib.ptr(list_index),
                _lib.ptr(st_in), st_out.data_ptr(), max_degree, _lib.ptr(node_out), _lib.ptr(agent_node), A,
                _lib.ptr(agent_out) if agent_node is not None else None, ld, _lib.ptr(agent_pk), _lib.ptr(hpk_in),
                _lib.ptr(hpk_out), ws.data_ptr(), ws.numel(), _lib.current_stream()))
        self.state = st_out
        if hpk_out is not None:
            st_out._gm_hpk = (hpk_out, self.math)
        if agent_pk is not None:
            if agent_out is None:
                return node_out, PackedRows(agent_pk, (B, A, O), self.math)
            agent_out._gm_pk = (agent_pk, self.math)  # consumed by DQN.act of the same math mode
        return node_out, (agent_out if agent_node is not None else None)

    _LIST_CACHE = {}

    @staticmethod
    def lists_from_mask_cached(mask):
        """lists_from_mask + the readout's max degree (model.py:588-589), remembered for the last few mask tensors
        (same storage, same version counter): a learner sequence that feeds one batch for several steps (sl.py:380-392)
        pays the two host syncs once."""
        key = (mask.data_ptr(), mask._version, tuple(mask.shape), mask.dtype)
        hit = NetMon._LIST_CACHE.get(key)
        if hit is None:
            nbr, deg, dm = NetMon.lists_from_mask(mask)
            max_degree = int(mask.sum(dim=-1).max().long().item()) - 1
            if len(NetMon._LIST_CACHE) >= 8:
                NetMon._LIST_CACHE.pop(next(iter(NetMon._LIST_CACHE)))
            hit = NetMon._LIST_CACHE[key] = (nbr, deg, dm, max_degree, mask)  # keeps the mask alive: the key stays unique
        return hit[:4]

    @staticmethod
    def lists_from_mask(mask, max_entries=None):
        """Dense [B,N,N] mask -> (nbr_all, deg, max rowsum).  One host sync for the row-sum
        maximum, like the reference's `.item()` at model.py:589."""
        B, N, _ = mask.shape
        m = mask.float().contiguous()
        dm = int((m != 0).sum(dim=-1).max().item()) if max_entries is None else int(max_entries)
        dm = max(dm, 1)
        nbr = torch.empty((B, N, dm), dtype=torch.int32, device=m.device)
        deg = torch.empty((B, N), dtype=torch.int32, device=m.device)
        ovf = torch.zeros((1,), dtype=torch.int32, device=m.device)
        with torch.cuda.device(m.device):
            _lib.check(_lib.lib().gm_adj_to_lists(m.data_ptr(), B, N, dm, nbr.data_ptr(), deg.data_ptr(),
                                                  ovf.data_ptr(), _lib.current_stream()))
        return nbr, deg, dm

    def _cell_param_names(self):
        """(attribute path, gm_cell_grads field) of a recurrent cell's parameters, in the order they are handed to the
        autograd node (nn.LSTMCell / layernormlstm.py:15-22)."""
        if self.rnn_type == "lnlstm":
            return [("weight_ih", "w_ih"), ("weight_hh", "w_hh"), ("bias_ih", "b_ih"), ("ln_input.weight", "ln_in_w"),
                    ("ln_input.bias", "ln_in_b"), ("ln_hidden.weight", "ln_hid_w"), ("ln_hidden.bias", "ln_hid_b"),
                    ("ln_cell.weight", "ln_cell_w"), ("ln_cell.bias", "ln_cell_b")]
        return [("weight_ih", "w_ih"), ("weight_hh", "w_hh"), ("bias_ih", "b_ih"), ("bias_hh", "b_hh")]

    def step_params(self):
        """The parameters in the order _NetMonStepFn takes them: the encoder's (weight, bias) pairs, then rnn_obs' and
        rnn_update's in _cell_param_names() order."""
        ps = [t for l in self.encode.linear_layers for t in (l.weight, l.bias)]
        for cell in (self.rnn_obs, self.rnn_update):
            for path, _ in self._cell_param_names():
                obj = cell
                for part in path.split("."):
                    obj = getattr(obj, part)
                ps.append(obj)
        return ps

    def _device_backward_reason(self, x):
        """None when the device-side backward (csrc/train.cu) covers this configuration, else why not."""
        if not x.is_cuda:
            return "CPU tensors"
        if self.rnn_type not in ("lstm", "lnlstm") or not self.rnn_carryover:
            return (f"rnn_type {self.rnn_type} / carryover {self.rnn_carryover}: the device backward is built for lstm and lnlstm "
                    "with carry-over")
        if self.output_global_hidden or self.iterations < 1:
            return "global readout / zero iterations"
        return None

    def forward(self, x, mask, node_agent_matrix, max_degree=None, no_agent_mapping=False):
        if torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters())
                                        or (self.state is not None and self.state.requires_grad)):
            why = self._device_backward_reason(x)
            if why is not None:
                _note_torch_path("NetMon", why)
                return self._forward_autograd(x, mask, node_agent_matrix, max_degree, no_agent_mapping)
            _lib.require_device()
            GRAD_PATH_CALLS["device"] += 1
            B, N, _ = x.shape
            with torch.no_grad():
                nbr, deg, dm, md_mask = self.lists_from_mask_cached(mask)
                if max_degree is None:
                    max_degree = md_mask  # model.py:588-589
            md = max(min(max_degree, dm), 0) if self.output_neighbor_hidden else 0
            st = self.state
            if st is not None:
                st = st.to(x.device).float().reshape(B, N, self.state_size).contiguous()
            node_out, self.state = _NetMonStepFn.apply(self, x.float().contiguous(), nbr, deg, None, md, st,
                                                       *self.step_params())
            if no_agent_mapping:
                return node_out
            return torch.bmm(node_out.transpose(1, 2), node_agent_matrix.to(node_out.dtype)).transpose(1, 2)
        _lib.require_device()
        if not x.is_cuda:
            raise _lib.GraphMarlError("NetMon needs CUDA tensors (no CPU fallback)")
        nbr, deg, dm = self.lists_from_mask(mask)
        if max_degree is None:
            max_degree = int(mask.sum(dim=-1).max().long().item()) - 1  # model.py:588-589
        node_out, _ = self.forward_lists(x, nbr, deg, None, max(min(max_degree, dm), 0), want_node_out=True)
        if no_agent_mapping:
            return node_out
        return NetMon.output_to_network_obs(node_out, node_agent_matrix)

    @staticmethod
    def output_to_network_obs(netmon_out, node_agent_matrix):
        """model.py:629-631."""
        if netmon_out.is_cuda and not (torch.is_grad_enabled() and netmon_out.requires_grad):
            B, N, O = netmon_out.shape
            A = node_agent_matrix.shape[-1]
            out = torch.empty((B, A, O), dtype=torch.float32, device=netmon_out.device)
            nam = node_agent_matrix.to(netmon_out.device).float().contiguous()
            with torch.cuda.device(netmon_out.device):
                _lib.check(_lib.lib().gm_netmon_map_to_agents(netmon_out.contiguous().data_ptr(), nam.data_ptr(), B, N,
                                                              A, O, out.data_ptr(), _lib.current_stream()))
            return out
        return torch.bmm(netmon_out.transpose(1, 2), node_agent_matrix).transpose(1, 2)

    # ---- autograd path (learner; same math from torch ops, model.py:476-631) ---------------------
    def _forward_autograd(self, x, mask, node_agent_matrix, max_degree, no_agent_mapping):
        B, N, _ = x.shape
        H = self.hidden_features
        xs = x.reshape(B * N, -1)
        if self.state is None:
            self.state = torch.zeros((B, N, self.state_size), device=x.device)
        st = self.state.reshape(B * N, self.num_states, -1).transpose(0, 1)
        h = self.encode(xs)
        lstm_like = self.rnn_type in ("lstm", "lnlstm")
        if lstm_like:
            h0, c0 = self.rnn_obs(h, (st[0], st[1]))
            h, c = h0, c0
        elif self.rnn_type == "gru":
            h0 = self.rnn_obs(h, st[0])
            h = h0
        last = torch.zeros_like(h) if (self.iterations <= 0 and self.output_neighbor_hidden) else None
        for it in range(self.iterations):
            if self.output_neighbor_hidden and it == self.iterations - 1:
                last = h
            M = self.aggregate(h.view(B, N, -1), mask).view(B * N, -1)
            if lstm_like:
                inp = (st[2], st[3]) if (not self.rnn_carryover and it == 0) else (h, c)
                h1, c1 = self.rnn_update(M, inp)
                h, c = h1, c1
            elif self.rnn_type == "gru":
                inp = st[1] if (not self.rnn_carryover and it == 0) else h
                h1 = self.rnn_update(M, inp)
                h = h1
            else:
                h = M
        if lstm_like:
            new = torch.stack((h1, c1)) if self.rnn_carryover else torch.stack((h0, c0, h1, c1))
        elif self.rnn_type == "gru":
            new = h1.unsqueeze(0)
        else:
            new = h.unsqueeze(0)
        if self.rnn_type == "gru" and not self.rnn_carryover:
            # model.py:571 + :449: [2,1,R,H] transposed on its two leading axes only -> all of h0, then all of h1
            self.state = torch.cat((h0.reshape(-1), h1.reshape(-1))).reshape(B, N, -1)
        else:
            self.state = new.transpose(0, 1).reshape(B, N, -1)
        hb = h.reshape(B, N, -1)
        parts = [hb]
        if self.output_global_hidden:
            parts.append(hb.mean(dim=1, keepdim=True).expand(B, N, H))
        if self.output_neighbor_hidden:
            lb = last.reshape(B, N, -1)
            if max_degree is None:
                max_degree = int(mask.sum(dim=-1).max().long().item()) - 1
            eye = torch.eye(N, device=mask.device, dtype=torch.bool).unsqueeze(0)
            nm = (mask != 0) & ~eye
            slot = nm.cumsum(dim=-1) - 1
            hn = torch.zeros((B, N, max(max_degree, 0), H), device=x.device, dtype=hb.dtype)
            idx = nm.nonzero()
            hn[idx[:, 0], idx[:, 1], slot[idx[:, 0], idx[:, 1], idx[:, 2]]] = lb[idx[:, 0], idx[:, 2]]
            parts.append(hn.reshape(B, N, -1))
        out = torch.cat(parts, dim=-1)
        if no_agent_mapping:
            return out
        return torch.bmm(out.transpose(1, 2), node_agent_matrix).transpose(1, 2)

    def summarize(self, *args):
        import os

        n = sum(p.numel() for p in self.parameters())
        self.state = None
        readout = "> Readout: local" + (" + last neighbors" if self.output_neighbor_hidden else "") + (
            " + global agg" if self.output_global_hidden else "")
        return os.linesep.join([
            "NetMon Module (libgraphmarl_b200)", f"> Parameters: {n}", f"> Aggregation Type: {self.agg_type_str}",
            f"> RNN Type: {self.rnn_type}", f"> Carryover: {self.rnn_carryover}",
            f"> Iterations: {self.iterations}", readout])
