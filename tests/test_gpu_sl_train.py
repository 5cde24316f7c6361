"""sl.py's supervised shortest-path training on the device dataset (graph_marl_b200.sl_trainer, BASELINE config 5):

  - gm_sl_mse_grad against fp64 torch on targets of real build_sl_dataset splits (N = 4, 20, 200, 1-4096 samples,
    repeated indices and none, a row stride wider than N), captured against eager, without d_pred, bad arguments;
  - FusedOptimizer with infinite clip bounds and no target pairs against torch.optim.AdamW(foreach=False);
  - the device sampler against np.random.default_rng(seed).choice(S, B);
  - one update's loss and gradients against torch autograd of the objective (NetMon._forward_autograd, the head as
    plain torch, the summed per-step F.mse_loss) on the same batch;
  - captured updates against eager ones, two (batch, seq_len) keys interleaved, netmon.state untouched, the pack refresh;
  - evaluate() against a torch restatement of the test over sequence lengths;
  - the configurations the trainer refuses, and that a short training run learns.
"""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = a.detach(), b.detach()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-12))


def _dataset(N, S, seed=0, eval_seeds=False, n_data=20):
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.sl_dataset import build_sl_dataset

    np.random.seed(seed)
    if eval_seeds:  # sl.py's test split
        net = Network(N, random_topology=True, sequential_topology_seeds=True, provided_seeds=EVAL_SEEDS)
    else:           # its training split: fresh topologies
        net = Network(N, random_topology=True)
    return build_sl_dataset(net, S, n_data=n_data)


@pytest.fixture(scope="module")
def sl_data():
    """Training splits at N = 4, 20 and 200 and the N = 20 test split, built once for the module."""
    return {4: _dataset(4, 64, n_data=4), 20: _dataset(20, 1024), 200: _dataset(200, 12, n_data=50),
            "eval": _dataset(20, 1000, seed=5, eval_seeds=True)}


def _modules(N, H=32, enc=(48,), K=2, rnn="lstm", math="fp32", head_units=(), act=torch.tanh, seed=2):
    from graph_marl_b200.model import MLP, NetMon

    torch.manual_seed(seed)
    nm = NetMon(4 * N + 8, H, enc, K, act, rnn_type=rnn, output_neighbor_hidden=True, math=math).cuda()
    if rnn == "lnlstm":  # LayerNorm parameters away from their (1, 0) initial values
        with torch.no_grad():
            for cell in (nm.rnn_obs, nm.rnn_update):
                for ln in (cell.ln_input, cell.ln_hidden, cell.ln_cell):
                    ln.weight.add_(0.2 * torch.randn_like(ln.weight))
                    ln.bias.add_(0.1 * torch.randn_like(ln.bias))
    head = MLP(nm.out_width(3), (*head_units, N), act, activation_on_output=False).cuda()
    return nm, head


# ---- 1. gm_sl_mse_grad ---------------------------------------------------------------------------------------------------
def _mse_call(pred, ldp, targets_all, index, B, N, scale, d_pred, loss, partials):
    from graph_marl_b200 import _lib

    return _lib.lib().gm_sl_mse_grad(_lib.ptr(pred), ldp, _lib.ptr(targets_all), _lib.ptr(index), B, N, scale,
                                     _lib.ptr(d_pred), _lib.ptr(loss), _lib.ptr(partials), _lib.current_stream())


@pytest.mark.parametrize("N,B", [(4, 1), (4, 63), (4, 4096), (20, 1), (20, 33), (20, 1000), (20, 4096), (200, 1),
                                 (200, 7), (200, 40)])
@pytest.mark.parametrize("indexed", [True, False])
def test_sl_mse_grad_matches_fp64(sl_data, N, B, indexed):
    """B*N*N elements from 16 to 1.6e6 (13 200 at N = 20, B = 33: not a multiple of the 256-thread block); prediction
    rows 3 floats wider than N; indices with repeats, or none (sample b = row block b, B up to the split's size)."""
    from graph_marl_b200 import _lib

    ta = sl_data[N]["targets_all"]
    S = ta.shape[0]
    g = torch.Generator(device="cuda").manual_seed(N * 7919 + B)
    if indexed:
        index = torch.randint(0, S, (B,), device="cuda", generator=g)
        if B > 1:
            index[1] = index[0]  # a repeat
    else:
        B = min(B, S)
        index = None
    ldp = N + 3
    buf = ta.float().mean() + 5 * torch.randn(B * N, ldp, device="cuda", generator=g)
    pred = buf[:, :N]
    scale = 1.0 / (B * N * N * 3)
    y = (ta[index] if indexed else ta[:B]).reshape(B * N, N).double()
    diff = pred.double() - y
    ref_loss = float(scale * (diff * diff).sum())
    ref_d = 2 * scale * diff
    part = torch.empty(_lib.GM_LEARNER_PARTIALS, dtype=torch.float64, device="cuda")
    d_buf = torch.full((B * N, ldp), 7.0, device="cuda")
    loss = torch.full((1,), 0.25, device="cuda")
    assert _mse_call(pred, ldp, ta, index, B, N, scale, d_buf, loss, part) == 0
    d = d_buf[:, :N]
    assert (d_buf[:, N:] == 7.0).all()  # the stride's padding is not written
    # fp32 q - y (y exact) and one multiply by fl(2 * scale): within 3 roundings of the fp64 value
    assert ((d.double() - ref_d).abs() <= 4 * 2.0 ** -24 * ref_d.abs()).all()
    assert abs(float(loss) - 0.25 - ref_loss) <= 1e-6 * ref_loss + 1e-7
    # the same call captured in a CUDA graph: bit-equal loss and gradient
    loss_g, d_g = torch.zeros((1,), device="cuda"), torch.empty_like(d_buf)
    loss_e, d_e = torch.zeros((1,), device="cuda"), torch.empty_like(d_buf)
    assert _mse_call(pred, ldp, ta, index, B, N, scale, d_e, loss_e, part) == 0
    torch.cuda.synchronize()
    cg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(cg):
        loss_g.zero_()
        _mse_call(pred, ldp, ta, index, B, N, scale, d_g, loss_g, part)
    cg.replay()
    torch.cuda.synchronize()
    assert torch.equal(loss_g, loss_e) and torch.equal(d_g[:, :N], d_e[:, :N])
    # evaluation form: no d_pred, the same loss, the prediction untouched
    before = buf.clone()
    loss_n = torch.zeros((1,), device="cuda")
    assert _mse_call(pred, ldp, ta, index, B, N, scale, None, loss_n, part) == 0
    assert torch.equal(loss_n, loss_e) and torch.equal(buf, before)


def test_sl_mse_grad_rejects_bad_arguments(sl_data):
    from graph_marl_b200 import _lib

    ta = sl_data[20]["targets_all"]
    pred = torch.zeros(40, 20, device="cuda")
    d, loss = torch.empty_like(pred), torch.zeros((1,), device="cuda")
    part = torch.empty(_lib.GM_LEARNER_PARTIALS, dtype=torch.float64, device="cuda")
    ok = dict(pred=pred, ldp=20, targets_all=ta, index=None, B=2, N=20, scale=1.0, d_pred=d, loss=loss, partials=part)
    assert _mse_call(**ok) == 0
    for bad in (dict(B=0), dict(N=0), dict(B=-1), dict(ldp=19), dict(pred=None), dict(targets_all=None), dict(loss=None),
                dict(partials=None)):
        assert _mse_call(**dict(ok, **bad)) == -1, bad  # GM_ERR_INVALID
        assert "gm_sl_mse_grad" in _lib.lib().gm_last_error().decode()


# ---- 2. the optimizer as AdamW alone ---------------------------------------------------------------------------------------
def test_optimizer_with_infinite_bounds_is_adamw(capsys):
    """FusedOptimizer(pairs=[], tau=0, clip_value=inf, max_norm=inf) == torch.optim.AdamW(foreach=False): the clamp and
    the norm scale leave the gradients alone, at gradients far above 1 (where the reference's clips would act) too."""
    from graph_marl_b200.learner import FusedOptimizer

    nm, head = _modules(20, H=128, enc=(512, 256), head_units=(64,), act=F.leaky_relu)
    ref_nm, ref_head = copy.deepcopy(nm), copy.deepcopy(head)
    params = list(nm.parameters()) + list(head.parameters())
    ref_params = list(ref_nm.parameters()) + list(ref_head.parameters())
    lr = 1e-3
    opt = FusedOptimizer(params, [], lr, 0.0, clip_value=float("inf"), max_norm=float("inf"))
    ref_opt = torch.optim.AdamW(ref_params, lr=lr, foreach=False)
    worst = {}
    for k, mag in enumerate([30.0, 1e-4, 3e-3, 0.2, 1e-5]):
        grads = [mag * torch.randn_like(p) for p in params]
        for p, g in zip(params, grads):
            p.grad.copy_(g)
        for p, g in zip(ref_params, grads):
            p.grad = g.clone()
        opt.step()
        ref_opt.step()
        st = ref_opt.state
        pairs = [("grad", [p.grad for p in params], grads), ("param", params, ref_params),
                 ("exp_avg", opt.exp_avg, [st[p]["exp_avg"] for p in ref_params]),
                 ("exp_avg_sq", opt.exp_avg_sq, [st[p]["exp_avg_sq"] for p in ref_params])]
        for name, got, ref in pairs:
            for a, b in zip(got, ref):
                e = _rel(a, b)
                worst[name] = max(worst.get(name, 0.0), e)
                assert e < 1e-6, (k, name, e)
        assert int(opt.step_count) == k + 1
    with capsys.disabled():
        print(f"\n[FusedOptimizer, infinite bounds, {sum(p.numel() for p in params)} parameters] worst relative error over "
              "5 steps against AdamW: " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


# ---- 3. sampler -----------------------------------------------------------------------------------------------------------
def test_update_indices_follow_default_rng_choice(sl_data):
    from graph_marl_b200.sl_trainer import SLTrainer

    data = sl_data[20]
    nm, head = _modules(20)
    tr = SLTrainer(nm, head, data, seed=1234, graph=True)
    rng = np.random.default_rng(1234)
    for B, T in [(24, 1), (24, 1), (24, 1), (40, 2), (24, 1), (40, 2), (40, 2)]:
        tr.update(B, T)
        np.testing.assert_array_equal(tr.last_indices.cpu().numpy(), rng.choice(data["node_obs"].shape[0], B))
    assert len(tr._graphs) == 2


# ---- 4. one update against torch autograd --------------------------------------------------------------------------------
def _reference_loss(nm, head, data, idx, T):
    """The module docstring's objective on torch autograd: _forward_autograd with the dense mask, the head as plain
    torch, the per-step F.mse_loss summed."""
    x = data["node_obs"][idx]
    adj = data["node_adj"][idx].float()
    B, N, _ = x.shape
    y = data["targets_all"][idx].float().reshape(B * N, N)
    nm.state = None
    loss = 0.0
    for _ in range(T):
        out = nm._forward_autograd(x, adj, None, 3, True)
        loss = loss + F.mse_loss(head(out.reshape(B * N, -1)), y)
    return loss


UPDATE_CASES = [(T, math, rnn, head, 20, 24) for T in (1, 4) for math in ("fp32", "bf16x3") for rnn in ("lstm", "lnlstm")
                for head in ((), (40,))] + [(4, "bf16x3", "lstm", (40,), 200, 4)]


@pytest.mark.parametrize("T,math,rnn,head_units,N,B", UPDATE_CASES)
def test_update_matches_torch_autograd(sl_data, T, math, rnn, head_units, N, B):
    import graph_marl_b200.model as M
    from graph_marl_b200.sl_trainer import SLTrainer

    tol = {("fp32", "lstm"): 1e-4, ("bf16x3", "lstm"): 5e-3, ("fp32", "lnlstm"): 2e-3, ("bf16x3", "lnlstm"): 3e-2}[math, rnn]
    data = sl_data[N]
    nm, head = _modules(N, rnn=rnn, math=math, head_units=head_units)
    ref_nm, ref_head = copy.deepcopy(nm), copy.deepcopy(head)
    tr = SLTrainer(nm, head, data, lr=1e-3, seed=9, graph=False)
    n_torch = M.GRAD_PATH_CALLS["torch"]
    loss = float(tr.update(B, T))
    assert M.GRAD_PATH_CALLS["torch"] == n_torch
    ref_loss = _reference_loss(ref_nm, ref_head, data, tr.last_indices, T)
    ref_loss.backward()
    assert abs(loss - float(ref_loss)) <= tol * abs(float(ref_loss)), (loss, float(ref_loss))
    for (name, p), r in zip(list(nm.named_parameters()) + list(head.named_parameters()),
                            list(ref_nm.parameters()) + list(ref_head.parameters())):
        assert r.grad is not None, name
        assert _rel(p.grad, r.grad) < tol, (name, _rel(p.grad, r.grad))


# ---- 5. captured against eager -------------------------------------------------------------------------------------------
def _snapshot(tr):
    ts = [p.data for p in tr.params] + tr.opt.exp_avg + tr.opt.exp_avg_sq + [tr.opt.step_count, tr._pcg]
    return ts, [t.clone() for t in ts]


def _restore(snap, tr):
    with torch.no_grad():
        for t, c in zip(*snap):
            t.copy_(c)
    tr.netmon._pack.refresh()


def _forward(nm, data, md=3):
    with torch.no_grad():
        nm.state = None
        out, _ = nm.forward_lists(data["node_obs"][:64], *_lists(data, 64), None, md, want_node_out=True)
    return out


def _lists(data, n):
    from graph_marl_b200.sl_trainer import adjacency_lists

    nbr, deg, _ = adjacency_lists(data["node_adj"][:n])
    return nbr, deg


def test_captured_updates_match_eager_updates(sl_data, capsys):
    from graph_marl_b200.model import _PackedWeights
    from graph_marl_b200.sl_trainer import SLTrainer

    data = sl_data[20]
    nm, head = _modules(20, H=128, enc=(512, 256), math="bf16x3", head_units=(64,), act=F.leaky_relu)
    out0 = _forward(nm, data)  # the weight pack exists before any update
    sentinel = torch.zeros(1, device="cuda")
    graph = SLTrainer(nm, head, data, lr=1e-3, seed=3, graph=True)
    eager = SLTrainer(nm, head, data, lr=1e-3, seed=3, graph=False)
    snap = _snapshot(graph)
    runs = {}
    order = [(32, 2), (32, 2), (96, 1), (96, 1), (32, 2), (96, 1), (32, 2)]
    for name, tr in (("graph", graph), ("eager", eager)):
        nm.state = sentinel
        if name == "graph":
            tr.update(32, 2)  # warm-up (eager), then from the same start as the eager run
            _restore(snap, tr)
        losses = [float(tr.update(32, 2))]
        grads = [p.grad.clone() for p in tr.params]
        losses += [float(tr.update(32, 2)) for _ in range(2)]
        params = [p.detach().clone() for p in tr.params]
        losses += [float(tr.update(b, t)) for b, t in order]
        assert nm.state is sentinel
        runs[name] = (losses, grads, params)
        if name == "graph":
            assert len(tr._graphs) == 2
            # the inference kernels read the refreshed pack: equal to a pack built fresh from the updated weights
            out = _forward(nm, data)
            fresh = copy.deepcopy(nm)
            fresh._pack = _PackedWeights()
            assert not torch.equal(out, out0)
            assert torch.equal(out, _forward(fresh, data))
        _restore(snap, tr)
    (lg, gg, pg), (le, ge, pe) = runs["graph"], runs["eager"]
    assert lg[0] == le[0]  # same inputs, same forward kernels: bit-equal
    worst_g = max(_rel(a, b) for a, b in zip(gg, ge))
    assert worst_g < 1e-5
    # the bars of test_gpu_learner.py::test_captured_updates_match_eager_updates: AdamW's sign-like step on gradients
    # that are ~0 may move an element by up to 2 lr per update, and such elements stay rare
    worst_p = max(float((a - b).abs().max()) for a, b in zip(pg, pe))
    assert worst_p <= 3 * 2 * 1e-3
    far = sum(int(((a - b).abs() > 1e-5 * b.abs().max()).sum()) for a, b in zip(pg, pe))
    total = sum(b.numel() for b in pe)
    assert far <= 0.05 * total
    worst_l = max(abs(a - b) / abs(b) for a, b in zip(lg[1:], le[1:]))
    assert worst_l <= 1e-3, (lg, le)
    with capsys.disabled():
        print(f"\n[SLTrainer captured vs eager] losses {lg[:3]} vs {le[:3]}; first gradients within {worst_g:.2e}; after 3 "
              f"updates worst parameter difference {worst_p:.2e}, {far} of {total} beyond 1e-5 of their tensor's max; "
              f"worst later loss {worst_l:.2e} over {len(lg)} updates")


# ---- 6. evaluate ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("math,bar,mse_bar", [("fp32", 1e-4, 1e-5), ("bf16x3", 3e-4, 1e-4)])
def test_evaluate_matches_torch_restatement(sl_data, math, bar, mse_bar, capsys):
    """1000 test-split samples in chunks of 384 (not a multiple): per-T MSE after T steps from state None."""
    from graph_marl_b200.model import _MlpFn
    from graph_marl_b200.sl_trainer import SLTrainer

    nm, head = _modules(20, math=math, head_units=(40,))
    tr = SLTrainer(nm, head, sl_data[20], seed=4, graph=True)
    for _ in range(3):
        tr.update(32, 2)
    data = sl_data["eval"]
    sentinel = torch.zeros(1, device="cuda")
    nm.state = sentinel
    got = tr.evaluate(data, [1, 3], chunk=384)
    assert nm.state is sentinel and list(got) == [1, 3]
    x, adj = data["node_obs"], data["node_adj"].float()
    S, N, _ = x.shape
    y = data["targets_all"].double().reshape(S * N, N)
    nbr, deg, _ = _lists_all(data)
    ref = copy.deepcopy(nm)
    worst = {}
    for T in (1, 3):
        with torch.no_grad():
            ref.state = None
            nm.state = None
            for _ in range(T):
                out = ref._forward_autograd(x, adj, None, 3, True)
                dev_out, _ = nm.forward_lists(x, nbr, deg, None, 3, want_node_out=True)
            pred = head(out.reshape(S * N, -1))
            dev_pred = _MlpFn.apply(tr._head_spec, dev_out.view(S * N, -1), *tr._head_params)
        nm.state = sentinel
        err = float((dev_pred - pred).abs().max()) / max(1.0, float(pred.abs().max()))
        ref_mse = float(((pred.double() - y) ** 2).mean())
        mse_err = abs(got[T] - ref_mse) / ref_mse
        worst[T] = (err, mse_err)
        assert err < bar, (T, err)
        assert mse_err < mse_bar, (T, got[T], ref_mse)
    with capsys.disabled():
        print(f"\n[SLTrainer.evaluate {math}] prediction / MSE relative errors per T: {worst}")


def _lists_all(data):
    from graph_marl_b200.sl_trainer import adjacency_lists

    return adjacency_lists(data["node_adj"])


# ---- 7. refusals ---------------------------------------------------------------------------------------------------------
def test_trainer_refuses_what_it_cannot_run(sl_data):
    from graph_marl_b200 import _lib
    from graph_marl_b200.model import MLP, NetMon
    from graph_marl_b200.sl_trainer import SLTrainer

    data = sl_data[20]
    Dn = data["node_obs"].shape[-1]
    for kw in (dict(rnn_type="gru"), dict(rnn_type="lstm", rnn_carryover=False)):
        nm = NetMon(Dn, 32, (48,), 2, torch.tanh, output_neighbor_hidden=True, **kw).cuda()
        head = MLP(nm.out_width(3), 20, torch.tanh, activation_on_output=False).cuda()
        with pytest.raises(_lib.GraphMarlError, match="device backward"):
            SLTrainer(nm, head, data)
    nm, _ = _modules(20)
    for head in (MLP(nm.out_width(3) - 1, 20, torch.tanh, activation_on_output=False).cuda(),
                 MLP(nm.out_width(3), (40, 19), torch.tanh, activation_on_output=False).cuda()):
        with pytest.raises(_lib.GraphMarlError, match="head"):
            SLTrainer(nm, head, data)
    _, head = _modules(20)
    bad = dict(data, node_adj=data["node_adj"].clone())
    bad["node_adj"][5, 3] = 1  # one row: every node a neighbour
    with pytest.raises(_lib.GraphMarlError, match="degree"):
        SLTrainer(nm, head, bad)


# ---- 8. learning ---------------------------------------------------------------------------------------------------------
# about half the gain over the constant predictor that this run measured on one NVIDIA B200 at a 1000 W power limit
# (1.70, 1.48, 1.75 and 1.72 in four runs, DESIGN.md section 5)
LEARNING_MARGIN = 0.8


def test_trainer_learns(capsys):
    from graph_marl_b200.model import MLP, NetMon
    from graph_marl_b200.sl_trainer import SLTrainer

    train, test = _dataset(20, 2048, seed=1), _dataset(20, 256, seed=5, eval_seeds=True)
    torch.manual_seed(0)
    nm = NetMon(88, 32, (64,), 2, F.leaky_relu, rnn_type="lstm", output_neighbor_hidden=True).cuda()
    head = MLP(nm.out_width(3), (64, 20), F.leaky_relu, activation_on_output=False).cuda()
    tr = SLTrainer(nm, head, train, lr=1e-3, seed=0)
    before = tr.evaluate(test, [2])[2]
    losses = [tr.update(32, 2) for _ in range(3000)]
    after = tr.evaluate(test, [2])[2]
    mean = train["targets_all"].double().mean()
    const = float(((test["targets_all"].double() - mean) ** 2).mean())
    first, last = float(losses[0]), float(torch.stack(losses[-100:]).mean())
    with capsys.disabled():
        print(f"\n[SLTrainer learns, 3000 updates of 32 x 2 steps] test MSE {after:.4f} (untrained {before:.4f}) against "
              f"{const:.4f} for the training split's mean weight (gain {const - after:.4f}); training loss first "
              f"{first:.4g}, last 100 {last:.4g}")
    assert np.isfinite(after) and after < const - LEARNING_MARGIN
