"""The training kernels of csrc/train.cu, one gradient path at a time, against fp64 torch autograd of the same math.

The learner differentiates NetMon and the DQN with the hand-written backward of csrc/train.cu: the training forward
through linear_dispatch, gemm_nn / gemm_tn, colsum / colsum_prod, act_bwd, the LSTM and LayerNormLSTM cell kernels and
the aggregation / readout scatters.  tests/test_gpu_backward.py checks whole modules against fp32 autograd; this file
goes below that:

- The reference is fp64 autograd of the module math (`NetMon._forward_autograd` of a `.double()` copy, an fp64 nn.Linear
  chain), on the fp32 inputs promoted to fp64.  tests/test_oracle_netmon.py pins that fp64 reference to the recordings.
- MLP (gm_mlp_forward_train / gm_mlp_backward through `_MlpFn`): every built activation, at row counts that give
  gemm_tn one row chunk, two, intermediate counts and the cap of 32 (`_gemm_tn_chunks` restates the library's rule),
  with x a column slice of a wider tensor.  dW and db are also held per element to the fp64 sum of absolute terms
  (|dZ|^T |X| and colsum |dZ|, see `_mlp_ref`), a scale-free bound that a lost or doubled row chunk breaks even in
  small entries.  With relu / leaky_relu, rows that hold a pre-activation within the forward bar of the kink get no
  upstream gradient, since either branch is then a correct result.
- NetMon step (gm_netmon_forward_train / gm_netmon_backward through `_NetMonStepFn`): five gradient probes that feed
  one output slice at a time (h columns of node_out, its neighbour slots, the h and c halves of state_out, all together),
  each checking every parameter gradient and d_state_in.  Shapes cover one row, H = 48, the learner's 640 rows, 5120
  rows (18 gemm_tn chunks), N = 200 with 5 graphs on 2 lists, rows with only a self entry or no entry, no readout and
  a readout of width 0, with and without an incoming state.
- The header's contracts at the C ABI: gradients written, not accumulated (NaN-filled buffers), a subset of gradient
  pointers, NULL upstream gradients.
- relu / tanh / sigmoid / elu at inference: DQN.act Q-values and NetMon.forward_lists.

Error measure: max |device - fp64| over a tensor, relative to the tensor's fp64 maximum.  Bars (NVIDIA B200):
- forward outputs, DESIGN section 2: fp32 2e-5 (LayerNormLSTM 1e-3), bf16x3 1e-4; single-pass bf16 inference 3e-2;
- gradients, fp32 forward: 1e-4, LayerNormLSTM included (worst measured 2.0e-5);
- gradients, bf16x3 forward: 5e-4 for every activation (worst measured 1.3e-5 MLP, 1.1e-5 LSTM, 1.7e-4 LayerNormLSTM);
  relu and leaky_relu stay under it because rows near the kink get no upstream gradient (below);
- per element of dW / db, relative to its absolute-term bound (`_mlp_ref`): the per-tensor bar of the case (worst
  measured 1.2e-7 fp32, 4.0e-6 bf16x3).
The NetMon cases use tanh in the encoder: with leaky_relu, a 512-wide encoder over thousands of rows always holds some
pre-activation within rounding of the kink, which moves a whole row's gradient by a finite step (measured up to 4e-2
of a tensor's maximum, fp32 included).  The MLP cases cover leaky_relu and relu with the near-kink rows masked.
Each case prints its worst error.
"""
import copy
import zlib

import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu

ACTS = {"leaky_relu": F.leaky_relu, "relu": torch.relu, "tanh": torch.tanh, "sigmoid": torch.sigmoid, "elu": F.elu}
FWD_TOL = {"fp32": 2e-5, "bf16x3": 1e-4}
FWD_TOL_LNLSTM = {"fp32": 1e-3, "bf16x3": 1e-3}


GRAD_TOL = {"fp32": 1e-4, "bf16x3": 5e-4}


def _err(dev, ref):
    """max |dev - ref| relative to max |ref| (0 when both are zero)."""
    d = (dev.double() - ref).abs().max()
    s = ref.abs().max()
    return float(d / s) if s > 0 else (0.0 if d == 0 else float("inf"))


def _elem_err(dev, ref, bound):
    """max |dev - ref| / bound per element (bound: the fp64 sum of the absolute values of the summed terms)."""
    d = (dev.double() - ref).abs()
    return float(torch.where(bound > 0, d / bound.clamp_min(1e-300), torch.where(d > 0, torch.inf, 0.0)).max())


def _seed(*parts):
    return zlib.crc32(repr(parts).encode()) & 0x7FFFFFFF


def _report(capsys, what, errs):
    with capsys.disabled():
        print(f"\n[train kernels] {what}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))


# ---- MLP ---------------------------------------------------------------------------------------------------------
def _gemm_tn_chunks(M, N, K):
    """Row chunks of gemm_tn (csrc/train.cu) for G[N,K] = A[M,N]^T X[M,K] on 148 SMs."""
    tiles = -(-K // 64) * -(-N // 64)
    c = min(32, max(1, min(2 * 148 // max(tiles, 1), M // 256)))
    rpc = -(-(-(-M // c)) // 16) * 16
    return -(-M // rpc)


MLP_SHAPES = {"dqn_cfg2": (642, (512, 256, 4)), "13_8_4": (13, (8, 4)), "65_63_1": (65, (63, 1))}
MLP_ROWS = [1, 17, 511, 512, 513, 640, 5120, 81920]


def test_mlp_cases_cover_every_gemm_tn_chunk_regime():
    """The MLP cases give the weight-gradient GEMM one row chunk, 2 to 31 chunks, and the cap of 32."""
    seen = set()
    for D, units in MLP_SHAPES.values():
        for M in MLP_ROWS:
            kin = D
            for U in units:
                seen.add(_gemm_tn_chunks(M, U, kin))
                kin = U
    assert 1 in seen and 32 in seen and len(seen & set(range(2, 32))) >= 3, sorted(seen)
    assert _gemm_tn_chunks(640, 512, 128) == 2 and _gemm_tn_chunks(5120, 512, 128) == 18  # NetMon cell dW_ih, H = 128


def _act64(name, z):
    """(activation, derivative) in fp64."""
    if name == "leaky_relu":
        return torch.where(z >= 0, z, 0.01 * z), torch.where(z > 0, 1.0, 0.01).double()
    if name == "relu":
        return z.clamp_min(0), (z > 0).double()
    if name == "tanh":
        t = torch.tanh(z)
        return t, 1 - t * t
    if name == "sigmoid":
        s = torch.sigmoid(z)
        return s, s * (1 - s)
    return torch.where(z > 0, z, torch.expm1(z)), torch.where(z > 0, 1.0, torch.exp(z)).double()


def _mlp_forward64(x, params, acts):
    """fp64 layer inputs / outputs, pre-activations and activation derivatives of the nn.Linear chain, and the
    absolute-term magnitude of each layer output (|act'(z)| times the sum of absolute terms of z, plus |act(z)|): the
    scale its rounding error is proportional to, also where z cancels to near zero."""
    a, zs, ds, mag = [x.double()], [], [], [x.double().abs()]
    for l, (w, b) in enumerate(params):
        z = a[-1] @ w.double().T + b.double()
        y, d = (z, torch.ones_like(z)) if acts[l] is None else _act64(acts[l], z)
        mag.append(d.abs() * (mag[-1] @ w.double().abs().T + b.double().abs()) + y.abs())
        a.append(y)
        zs.append(z)
        ds.append(d)
    return a, zs, ds, mag


def _mlp_ref(x, params, acts, dy):
    """fp64 forward and backward of the chain, with the absolute-term bounds of dW and db: the sums of the absolute
    terms, where every factor the device computed stands for its own absolute-term magnitude -- a layer input (every
    layer's but the first) for `mag` of `_mlp_forward64`, the gradient for its recursion |dy| through |W| and |act'|,
    with act' widened by 2 mag (the kernel takes it from the layer output, and |d act'/d a| <= 2 for every built
    activation).  Rounding then moves an element by a small multiple of the precision times its bound, also where dy
    or a layer output cancels to near zero."""
    a, _, ds, mag = _mlp_forward64(x, params, acts)
    out = {"y": a[-1]}
    g, gabs = dy.double(), dy.double().abs()
    for l in reversed(range(len(params))):
        dz = g * ds[l]
        dzabs = gabs * (ds[l].abs() + (0 if acts[l] is None else 2 * mag[l + 1]))
        out[f"w{l}"], out[f"w{l}_bound"] = dz.T @ a[l], dzabs.T @ mag[l]
        out[f"b{l}"], out[f"b{l}_bound"] = dz.sum(0), dzabs.sum(0)
        g, gabs = dz @ params[l][0].double(), dzabs @ params[l][0].double().abs()
    out["x"] = g
    return out


def _mlp_device(x, params, acts, math, dy):
    import graph_marl_b200.model as M
    from graph_marl_b200 import _lib

    ids = tuple(_lib.ACTIVATIONS[a] if a else -1 for a in acts)
    flat = [t for wb in params for t in wb]
    y = M._MlpFn.apply((ids, math), x, *flat)
    g = torch.autograd.grad(y, [x] + flat, dy)
    out = {"y": y.detach(), "x": g[0]}
    for l in range(len(params)):
        out[f"w{l}"], out[f"b{l}"] = g[1 + 2 * l], g[2 + 2 * l]
    return out


@gpu
@pytest.mark.parametrize("math", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("act", list(ACTS))
@pytest.mark.parametrize("rows", MLP_ROWS)
@pytest.mark.parametrize("shape", list(MLP_SHAPES))
def test_mlp_train_kernels_match_fp64(shape, rows, act, math, capsys):
    """Forward output, dX, dW and db of gm_mlp_forward_train / gm_mlp_backward against fp64.  Hidden layers carry the
    activation, the last (Q) layer none.  math="bf16" trains with the bf16x3 forward: bit-equal outputs, bf16x3 bars."""
    D, units = MLP_SHAPES[shape]
    gen = torch.Generator(device="cuda").manual_seed(_seed(shape, rows))
    params, kin = [], D
    for U in units:
        bound = kin ** -0.5
        w = ((torch.rand(U, kin, device="cuda", generator=gen) * 2 - 1) * bound).requires_grad_()
        b = ((torch.rand(U, device="cuda", generator=gen) * 2 - 1) * bound).requires_grad_()
        params.append((w, b))
        kin = U
    acts = [act] * (len(units) - 1) + [None]
    wide = torch.randn(rows, D + 5, device="cuda", generator=gen)
    x = wide.requires_grad_()[:, 2:2 + D]  # a column slice: ldx = D + 5, not 16-byte aligned
    dy = torch.randn(rows, units[-1], device="cuda", generator=gen)
    m = "fp32" if math == "fp32" else "bf16x3"
    p64 = [(w.detach(), b.detach()) for w, b in params]
    if act in ("leaky_relu", "relu"):
        # a pre-activation within the forward's rounding of the kink may take either branch: rows holding one get no
        # upstream gradient, so that every compared gradient is a smooth function of the forward's values
        _, zs, _, _ = _mlp_forward64(x.detach(), p64, acts)
        near = torch.zeros(rows, dtype=torch.bool, device="cuda")
        for z in zs[:-1]:
            near |= (z.abs() < FWD_TOL[m] * z.abs().max()).any(1)
        dy[near] = 0.0
    dev = _mlp_device(x, params, acts, math, dy)
    if math == "bf16":
        assert torch.equal(dev["y"], _mlp_device(x, params, acts, "bf16x3", dy)["y"])
    ref = _mlp_ref(x.detach(), p64, acts, dy)
    gtol = GRAD_TOL[m]
    etol = gtol
    errs = {"y": _err(dev["y"], ref["y"]), "dx": _err(dev["x"], ref["x"])}
    elem = {}
    for l in range(len(units)):
        for k in (f"w{l}", f"b{l}"):
            errs["d" + k] = _err(dev[k], ref[k])
            elem["d" + k] = _elem_err(dev[k], ref[k], ref[k + "_bound"])
    chunks = [_gemm_tn_chunks(rows, U, k) for U, k in zip(units, (D,) + units[:-1])]
    _report(capsys, f"mlp {shape} rows={rows} {act} {math} chunks={chunks}",
            {"fwd": errs["y"], "grad": max(v for k, v in errs.items() if k != "y"), "elem": max(elem.values())})
    assert errs["y"] < FWD_TOL[m], errs
    for k, v in errs.items():
        assert v < gtol, (k, errs)
    for k, v in elem.items():
        assert v < etol, (k, elem)


# ---- NetMon --------------------------------------------------------------------------------------------------------
# name: B, N, H, encoder, K, input width, neighbour readout, adjacency lists (None: one per graph), edge probability
NM_CASES = {
    "1x1_self_only": (1, 1, 16, (24,), 1, 24, True, None, 0.0),  # one row, a readout of width 0
    "h48": (12, 20, 48, (64,), 2, 88, True, None, 0.15),
    "learner_640_rows": (32, 20, 128, (512, 256), 2, 88, True, None, 0.15),
    "5120_rows": (256, 20, 128, (512, 256), 2, 88, True, None, 0.15),
    "n200_2_lists": (5, 200, 64, (64,), 3, 40, True, [0, 1, 1, 0, 1], 0.02),
    "no_readout": (12, 20, 32, (40,), 2, 88, False, None, 0.15),
}


def _masks(L, N, p, seed):
    """Random adjacency masks with self entries; in every list node 0 keeps only its self entry and node 1 has no entry
    at all (deg 0), while other nodes may still list them."""
    g = torch.Generator().manual_seed(seed)
    m = (torch.rand(L, N, N, generator=g) < p).float()
    m[:, torch.arange(N), torch.arange(N)] = 1.0
    if N >= 3:
        m[:, 0] = 0.0
        m[:, 0, 0] = 1.0
        m[:, 1] = 0.0
    return m


def _param_list(nm):
    """(name, tensor, (gm_netmon_grads field, index or gm_cell_grads field)) in `_NetMonStepFn`'s parameter order."""
    out = []
    for l, lin in enumerate(nm.encode.linear_layers):
        out += [(f"encode.linear_layers.{l}.weight", lin.weight, ("enc_w", l)),
                (f"encode.linear_layers.{l}.bias", lin.bias, ("enc_b", l))]
    for cname in ("rnn_obs", "rnn_update"):
        for path, field in nm._cell_param_names():
            obj = getattr(nm, cname)
            for part in path.split("."):
                obj = getattr(obj, part)
            out.append((f"{cname}.{path}", obj, (cname, field)))
    return out


class NmCase:
    def __init__(self, name, rnn, agg, math, with_state, act="tanh"):
        import graph_marl_b200.model as M

        B, N, H, enc, K, Dn, nbr, lists, p = NM_CASES[name]
        self.B, self.N, self.H = B, N, H
        seed = _seed(name, rnn, agg)
        torch.manual_seed(seed)
        nm = M.NetMon(Dn, H, enc, K, ACTS[act], rnn_type=rnn, agg_type=agg, output_neighbor_hidden=nbr, math=math)
        if rnn == "lnlstm":  # LayerNorm parameters away from their (1, 0) initial values
            with torch.no_grad():
                for cell in (nm.rnn_obs, nm.rnn_update):
                    for ln in (cell.ln_input, cell.ln_hidden, cell.ln_cell):
                        ln.weight.add_(0.2 * torch.randn_like(ln.weight))
                        ln.bias.add_(0.1 * torch.randn_like(ln.bias))
        self.nm = nm.cuda()
        masks = _masks(len(lists) if lists else B, N, p, seed)
        self.li = None if lists is None else torch.tensor(lists, dtype=torch.int32, device="cuda")
        self.adj = (masks[lists] if lists else masks).cuda()
        self.nbr, self.deg, _ = M.NetMon.lists_from_mask(masks.cuda())
        eye = torch.eye(N, dtype=torch.bool, device="cuda")
        self.md = int(((self.adj != 0) & ~eye).sum(-1).max()) if nbr else 0
        self.O = nm.out_width(self.md)
        self.x = torch.randn(B, N, Dn, device="cuda")
        self.state = 0.5 * torch.randn(B, N, 2 * H, device="cuda") if with_state else None
        g = torch.Generator(device="cuda").manual_seed(seed + 1)
        self.dn = torch.randn(B, N, self.O, device="cuda", generator=g)
        self.ds = torch.randn(B, N, 2 * H, device="cuda", generator=g)
        self.names = [n for n, _, _ in _param_list(nm)]

    def probes(self):
        """name -> (d_node_out, d_state_out): one output slice at a time, then everything."""
        H, z = self.H, torch.zeros_like
        out = {}
        dn = z(self.dn); dn[..., :H] = self.dn[..., :H]
        out["node_out_h"] = (dn, z(self.ds))
        if self.O > H:
            dn = z(self.dn); dn[..., H:] = self.dn[..., H:]
            out["node_out_slots"] = (dn, z(self.ds))
        ds = z(self.ds); ds[..., :H] = self.ds[..., :H]
        out["state_out_h"] = (z(self.dn), ds)
        ds = z(self.ds); ds[..., H:] = self.ds[..., H:]
        out["state_out_c"] = (z(self.dn), ds)
        out["all"] = (self.dn, self.ds)
        return out

    def reference(self):
        """fp64 forward and a function of (d_node_out, d_state_out) -> gradients by name ('state_in' too)."""
        ref = copy.deepcopy(self.nm).double()
        s64 = None if self.state is None else self.state.double().requires_grad_()
        ref.state = s64 if s64 is not None else torch.zeros(self.B, self.N, 2 * self.H, dtype=torch.float64, device="cuda")
        out = ref._forward_autograd(self.x.double(), self.adj.double(), None, self.md, True)
        st = ref.state
        inputs = [t for _, t, _ in _param_list(ref)] + ([s64] if s64 is not None else [])
        names = self.names + (["state_in"] if s64 is not None else [])

        def grads(dn, ds):
            g = torch.autograd.grad([out, st], inputs, [dn.double(), ds.double()], retain_graph=True, allow_unused=True)
            return {n: (torch.zeros_like(t) if v is None else v) for n, t, v in zip(names, inputs, g)}

        return out.detach(), st.detach(), grads

    def device(self):
        """Training forward through `_NetMonStepFn` and a function of the upstream gradients -> gradients by name."""
        import graph_marl_b200.model as M

        params = [t for _, t, _ in _param_list(self.nm)]
        st = None if self.state is None else self.state.clone().requires_grad_()
        node_out, st_out = M._NetMonStepFn.apply(self.nm, self.x, self.nbr, self.deg, self.li, self.md, st, *params)
        inputs = params + ([st] if st is not None else [])
        names = self.names + (["state_in"] if st is not None else [])

        def grads(dn, ds):
            g = torch.autograd.grad([node_out, st_out], inputs, [dn, ds], retain_graph=True)
            return dict(zip(names, g))

        return node_out.detach(), st_out.detach(), grads

    def inference(self):
        self.nm.state = None if self.state is None else self.state.clone()
        with torch.no_grad():
            node_out, _ = self.nm.forward_lists(self.x, self.nbr, self.deg, self.li, self.md, want_node_out=True)
        return node_out, self.nm.state


def _check_netmon(c, rnn, math, capsys, label):
    m = "fp32" if math == "fp32" else "bf16x3"
    ftol = (FWD_TOL_LNLSTM if rnn == "lnlstm" else FWD_TOL)[m]
    itol = 3e-2 if math == "bf16" else ftol  # single-pass bf16 inference (DESIGN section 2)
    gtol = GRAD_TOL[m]
    out_r, st_r, grads_r = c.reference()
    out_d, st_d, grads_d = c.device()
    out_i, st_i = c.inference()
    errs = {"node_out": _err(out_d, out_r), "state_out": _err(st_d, st_r),
            "infer_node_out": _err(out_i, out_r), "infer_state_out": _err(st_i, st_r)}
    worst, bad = {}, {}
    for probe, (dn, ds) in c.probes().items():
        gd, gr = grads_d(dn, ds), grads_r(dn, ds)
        assert set(gd) == set(gr)
        e = {n: _err(gd[n], gr[n]) for n in gr}
        worst[probe] = max(e.values())
        bad.update({(probe, n): v for n, v in e.items() if not v < gtol})
    _report(capsys, label, {**errs, **worst})
    assert not bad, bad
    for k, v in errs.items():
        assert v < (itol if k.startswith("infer") else ftol), (k, errs)
    return out_d, st_d


@gpu
@pytest.mark.parametrize("with_state", [True, False], ids=["state_in", "no_state"])
@pytest.mark.parametrize("math", ["fp32", "bf16x3"])
@pytest.mark.parametrize("agg", ["sum", "mean"])
@pytest.mark.parametrize("rnn", ["lstm", "lnlstm"])
@pytest.mark.parametrize("case", list(NM_CASES))
def test_netmon_step_gradient_probes_match_fp64(case, rnn, agg, math, with_state, capsys):
    """node_out / state_out of the training forward and of the inference kernels (forward_lists) against fp64, and the
    five gradient probes: every parameter gradient and d_state_in within the gradient bar."""
    c = NmCase(case, rnn, agg, math, with_state)
    _check_netmon(c, rnn, math, capsys, f"netmon {case} {rnn} {agg} {math} {'state' if with_state else 'no state'}")


@gpu
@pytest.mark.parametrize("rnn", ["lstm", "lnlstm"])
def test_netmon_bf16_trains_with_the_bf16x3_forward(rnn, capsys):
    """A NetMon of math "bf16" runs its training forward in bf16x3 (single-pass products would cost ~2^-9 relative
    error): outputs bit-equal to the bf16x3 module's, gradients within the bf16x3 bars of fp64."""
    c = NmCase("learner_640_rows", rnn, "sum", "bf16", True)
    out, st = _check_netmon(c, rnn, "bf16", capsys, f"netmon learner_640_rows {rnn} bf16 mode")
    c3 = NmCase("learner_640_rows", rnn, "sum", "bf16x3", True)
    out3, st3, _ = c3.device()
    assert torch.equal(out, out3) and torch.equal(st, st3)


# ---- C ABI contracts of gm_netmon_backward ----------------------------------------------------------------------
def _abi_forward(c):
    from graph_marl_b200 import _lib

    import ctypes as C

    nm, B, N, H = c.nm, c.B, c.N, c.H
    p = nm._params(packed=False)
    lib = _lib.lib()
    R = B * N
    tape = torch.empty(int(lib.gm_netmon_tape_floats(C.byref(p), R)), device="cuda")
    ws = torch.empty(int(lib.gm_netmon_train_workspace_bytes(C.byref(p), R)), dtype=torch.uint8, device="cuda")
    st_out = torch.empty(B, N, 2 * H, device="cuda")
    node_out = torch.empty(B, N, c.O, device="cuda")
    _lib.check(lib.gm_netmon_forward_train(C.byref(p), B, N, c.x.data_ptr(), c.nbr.data_ptr(), c.deg.data_ptr(), c.nbr.shape[-1],
                                           _lib.ptr(c.li), _lib.ptr(c.state), st_out.data_ptr(), c.md, node_out.data_ptr(),
                                           tape.data_ptr(), ws.data_ptr(), ws.numel(), _lib.current_stream()))
    return p, tape, ws


def _abi_backward(c, p, tape, ws, dn, ds, names, want_state_grad):
    """gm_netmon_backward into NaN-filled buffers: gradients of `names` (the others NULL) and d_state_in if asked.
    Returns every buffer, passed or not."""
    from graph_marl_b200 import _lib

    import ctypes as C

    bufs = {n: torch.full_like(t, float("nan")) for n, t, _ in _param_list(c.nm)}
    bufs["state_in"] = torch.full((c.B, c.N, 2 * c.H), float("nan"), device="cuda")
    g = _lib.NetmonGrads()
    for n, _, (kind, idx) in _param_list(c.nm):
        if n not in names:
            continue
        if kind in ("enc_w", "enc_b"):
            getattr(g, kind)[idx] = bufs[n].data_ptr()
        else:
            setattr(getattr(g, kind), idx, bufs[n].data_ptr())
    _lib.check(_lib.lib().gm_netmon_backward(
        C.byref(p), c.B, c.N, c.x.data_ptr(), c.nbr.data_ptr(), c.deg.data_ptr(), c.nbr.shape[-1], _lib.ptr(c.li),
        _lib.ptr(c.state), c.md, tape.data_ptr(), _lib.ptr(dn), _lib.ptr(ds), _lib.ptr(bufs["state_in"]) if want_state_grad else None,
        C.byref(g), ws.data_ptr(), ws.numel(), _lib.current_stream()))
    return bufs


@gpu
@pytest.mark.parametrize("rnn", ["lstm", "lnlstm"])
def test_netmon_backward_abi_contract(rnn, capsys):
    """include/graphmarl_b200.h: gradients are written, not accumulated (every requested buffer, NaN before the call, is
    fully written and matches fp64); a subset of gradient pointers gives the same values and writes nothing else; NULL
    d_node_out / d_state_out equal zeros.  640 rows: the weight-gradient GEMMs split their rows (memset + atomics)."""
    c = NmCase("learner_640_rows", rnn, "mean", "fp32", True)
    tol = GRAD_TOL["fp32"]
    _, _, grads_r = c.reference()
    p, tape, ws = _abi_forward(c)
    everything = set(c.names)
    full = _abi_backward(c, p, tape, ws, c.dn, c.ds, everything, True)
    ref = grads_r(c.dn, c.ds)
    errs = {n: _err(full[n], ref[n]) for n in ref}
    _report(capsys, f"abi contract {rnn}", {"full": max(errs.values())})
    for n, v in errs.items():
        assert torch.isfinite(full[n]).all(), n
        assert v < tol, (n, v)
    upd = {n for n in c.names if n.startswith("rnn_update.")}
    sub = _abi_backward(c, p, tape, ws, c.dn, c.ds, upd, False)
    for n in c.names + ["state_in"]:
        if n in upd:
            assert _err(sub[n], full[n].double()) < 1e-6, n
        else:
            assert torch.isnan(sub[n]).all(), n
    zn, zs = torch.zeros_like(c.dn), torch.zeros_like(c.ds)
    for dn, ds, dn0, ds0 in ((None, c.ds, zn, c.ds), (c.dn, None, c.dn, zs)):
        a = _abi_backward(c, p, tape, ws, dn, ds, everything, True)
        b = _abi_backward(c, p, tape, ws, dn0, ds0, everything, True)
        for n in c.names + ["state_in"]:
            assert torch.isfinite(a[n]).all(), n
            assert _err(a[n], b[n].double()) < 1e-6, n


# ---- activations at inference --------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("rows", [129, 20480])
@pytest.mark.parametrize("math", ["fp32", "bf16x3"])
@pytest.mark.parametrize("act", [a for a in ACTS if a != "leaky_relu"])
def test_inference_activations_match_fp64(act, math, rows, capsys):
    """DQN.act Q-values (tensor-core Q head / SIMT layers) and NetMon.forward_lists (encoder layers, tile-packed for the
    cells) with relu / tanh / sigmoid / elu against fp64 nn modules, at the forward bars."""
    from graph_marl_b200.model import DQN, NetMon

    torch.manual_seed(rows + len(act))
    dqn = DQN(642, (512, 256), 4, ACTS[act], math=math).cuda().eval()
    xa = torch.randn(rows, 642, device="cuda")
    with torch.no_grad():
        q, _ = dqn.act(xa)
        ref = copy.deepcopy(dqn).double()
        q_ref = ref.q_net(ref.encoder(xa.double()))
    N = 3 if rows == 129 else 20
    B = rows // N
    nm = NetMon(88, 128, (256,), 2, ACTS[act], output_neighbor_hidden=True, math=math).cuda()
    masks = _masks(B, N, 0.5 if N == 3 else 0.15, rows)
    nbr, deg, _ = NetMon.lists_from_mask(masks.cuda())
    eye = torch.eye(N, dtype=torch.bool)
    md = int(((masks != 0) & ~eye).sum(-1).max())
    x = torch.randn(B, N, 88, device="cuda")
    st = 0.5 * torch.randn(B, N, 256, device="cuda")
    nm.state = st.clone()
    with torch.no_grad():
        out, _ = nm.forward_lists(x, nbr, deg, None, md, want_node_out=True)
        ref = copy.deepcopy(nm).double()
        ref.state = st.double()
        out_ref = ref._forward_autograd(x.double(), masks.cuda().double(), None, md, True)
    errs = {"q": _err(q, q_ref), "node_out": _err(out, out_ref), "state": _err(nm.state, ref.state)}
    _report(capsys, f"inference {act} {math} rows={rows}", errs)
    for k, v in errs.items():
        assert v < FWD_TOL[math], (k, errs)
