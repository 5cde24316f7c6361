"""The batched learner (graph_marl_b200/learner.py, trainer.py, csrc/learner.cu, the per-env sequence sampler of
csrc/replay_sampler.cu) against restatements of the reference's learner:

  - the sampler against numpy's default_rng(seed) restating its rule;
  - gm_td_grad against an fp64 torch restatement of tools/train_simple.py:107-110;
  - gm_optimizer_step against clip_grad_value_ + clip_grad_norm_ + AdamW(foreach=False) + util.interpolate_model;
  - the gradients of one learner update against torch autograd of the composed reference math (_forward_autograd +
    nn.Linear chain + the same loss) on the same sampled batch, with the bars of test_gpu_backward.py;
  - captured updates against eager ones, the weight-pack refresh, and that a short training run learns.
"""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-12))


def _cfg(**kw):
    from graph_marl_b200.rollout import CONFIGS

    return dict(CONFIGS["cfg2"], **kw)


# ---- 1. per-env sequence sampler ---------------------------------------------------------------------------------------
def _sample(seed, S, head, B, batch, T, calls=1):
    from graph_marl_b200 import _lib

    st = np.zeros(_lib.GM_PCG64_STATE_WORDS, np.uint64)
    _lib.lib().gm_pcg64_seed(_lib.ptr(st), seed)
    dev = torch.from_numpy(st.view(np.int64)).cuda()
    outs = []
    for _ in range(calls):
        out = torch.empty((T, batch), dtype=torch.int64, device="cuda")
        _lib.check(_lib.lib().gm_replay_sample_env_sequences(dev.data_ptr(), S, head, B, batch, T, out.data_ptr(),
                                                             _lib.current_stream()))
        outs.append(out.cpu().numpy())
    return outs


def _sample_np(rng, S, head, B, batch, T):
    first = head % S
    start = (first + rng.choice(S - T, batch, replace=True)) % S
    env = rng.choice(B, batch, replace=True)
    return np.stack([((start + o) % S) * B + env for o in range(T)])


@pytest.mark.parametrize("S,head,B,batch,T", [(8, 8, 64, 32, 1), (8, 8, 64, 32, 4), (10, 3, 16, 33, 4), (64, 17, 4096, 256, 8),
                                              (5, 0, 7, 1, 4)])
def test_env_sequence_sampler_matches_numpy_and_keeps_sequences_in_one_env(S, head, B, batch, T):
    """head = S: a ring not yet wrapped (oldest step 0); head < S: a full ring whose oldest step is `head`."""
    outs = _sample(1234, S, head, B, batch, T, calls=3)
    rng = np.random.default_rng(1234)
    for out in outs:  # the device generator state carries over from call to call like numpy's
        np.testing.assert_array_equal(out, _sample_np(rng, S, head, B, batch, T))
        steps, env = out // B, out % B
        assert (env == env[0]).all()                                        # one env per sequence
        np.testing.assert_array_equal(steps, (steps[0] + np.arange(T)[:, None]) % S)  # row k = row 0 + k*B mod the ring
        age = (steps - head % S) % S                                        # 0 = oldest stored step, S - 1 = newest
        assert age.max() <= S - 2 and (np.diff(age, axis=0) == 1).all()      # never wraps past the newest into the head


def test_env_sequence_sampler_covers_every_env_and_start():
    S, head, B, batch, T = 12, 5, 24, 4096, 3
    out = _sample(7, S, head, B, batch, T)[0]
    starts = set(((out[0] // B - head) % S).tolist())
    assert starts == set(range(S - T))
    assert set((out[0] % B).tolist()) == set(range(B))


def test_env_sequence_sampler_rejects_short_rings():
    from graph_marl_b200 import _lib

    out = torch.empty((4, 2), dtype=torch.int64, device="cuda")
    st = torch.zeros(_lib.GM_PCG64_STATE_WORDS, dtype=torch.int64, device="cuda")
    with pytest.raises(_lib.GraphMarlError):
        _lib.check(_lib.lib().gm_replay_sample_env_sequences(st.data_ptr(), 4, 4, 8, 2, 4, out.data_ptr(),
                                                             _lib.current_stream()))


# ---- 2. gm_td_grad -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("R", [1, 127, 128, 129, 81920])
@pytest.mark.parametrize("done_mode", ["off", "on", "mixed"])
def test_td_grad_matches_fp64_restatement(R, done_mode):
    from graph_marl_b200 import _lib

    g = torch.Generator(device="cuda").manual_seed(R)
    nA, gamma, T = 4, 0.98, 3
    q = torch.randn(R, nA, device="cuda", generator=g)
    qn = torch.randn(R, nA, device="cuda", generator=g)
    qn[::3, 1] = qn[::3, 2] = qn[::3].max(-1).values + 0.5  # ties of the maximum
    action = torch.randint(0, nA, (R,), device="cuda", generator=g)
    reward = torch.randn(R, device="cuda", generator=g)
    done = {"off": torch.zeros(R, dtype=torch.bool, device="cuda"), "on": torch.ones(R, dtype=torch.bool, device="cuda"),
            "mixed": torch.rand(R, device="cuda", generator=g) < 0.4}[done_mode]
    scale = 1.0 / (R * nA * T)
    loss = torch.full((1,), 0.25, device="cuda")
    dq = torch.empty_like(q)
    part = torch.empty(_lib.GM_LEARNER_PARTIALS, dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().gm_td_grad(q.data_ptr(), qn.data_ptr(), action.data_ptr(), reward.data_ptr(),
                                     done.view(torch.uint8).data_ptr(), R, nA, gamma, scale, dq.data_ptr(), loss.data_ptr(),
                                     part.data_ptr(), _lib.current_stream()))
    # train_simple.py:107-110 in fp64 (the element's mean over R x nA and the / sequence_length)
    qd, qnd = q.double().requires_grad_(True), qn.double()
    target = reward.double() + (~done) * gamma * qnd.max(dim=1)[0]
    q_target = torch.scatter(qd.detach(), -1, action.unsqueeze(-1), target.unsqueeze(-1))
    ref_loss = torch.mean((qd - q_target).pow(2)) / T
    ref_loss.backward()
    ref_loss = ref_loss.detach()
    assert abs(float(loss) - 0.25 - float(ref_loss)) <= 1e-6 * float(ref_loss) + 1e-7
    ref_dq = qd.grad
    # fp32 rounding of y (one add, one multiply) and of q - y, scaled
    bar = 2 * scale * (q.abs() + target.abs().float().unsqueeze(-1) + 1) * 4 * 2.0 ** -24
    assert ((dq.double() - ref_dq).abs() <= bar.double()).all()
    assert (dq.ne(0).sum(-1) <= 1).all()


def test_td_grad_propagates_nan_like_torch_max():
    """A NaN anywhere in a q_next row (first column included) makes that row's target NaN, as torch's max does: the loss
    and the row's dq at the taken action become NaN; the other rows are unaffected."""
    from graph_marl_b200 import _lib

    R, nA = 129, 4
    g = torch.Generator(device="cuda").manual_seed(3)
    q = torch.randn(R, nA, device="cuda", generator=g)
    qn = torch.randn(R, nA, device="cuda", generator=g)
    qn[5, 0] = qn[17, 2] = qn[40, 3] = float("nan")
    action = torch.randint(0, nA, (R,), device="cuda", generator=g)
    reward = torch.randn(R, device="cuda", generator=g)
    done = torch.zeros(R, dtype=torch.bool, device="cuda")
    done[40] = True  # (~done) * gamma * NaN is NaN in torch too
    loss = torch.zeros((1,), device="cuda")
    dq = torch.empty_like(q)
    part = torch.empty(_lib.GM_LEARNER_PARTIALS, dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().gm_td_grad(q.data_ptr(), qn.data_ptr(), action.data_ptr(), reward.data_ptr(),
                                     done.view(torch.uint8).data_ptr(), R, nA, 0.98, 1.0 / (R * nA), dq.data_ptr(),
                                     loss.data_ptr(), part.data_ptr(), _lib.current_stream()))
    target = reward + (~done) * 0.98 * qn.max(dim=1)[0]
    assert torch.isnan(target).nonzero().flatten().tolist() == [5, 17, 40]
    assert torch.isnan(loss).all()
    rows = torch.arange(R, device="cuda")
    assert torch.isnan(dq[rows, action]).nonzero().flatten().tolist() == [5, 17, 40]
    assert not torch.isnan(dq).any(dim=1)[torch.tensor([i not in (5, 17, 40) for i in range(R)], device="cuda")].any()


# ---- 3. gm_optimizer_step ----------------------------------------------------------------------------------------------
class _Tiny(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.a = torch.nn.Parameter(torch.randn(3))
        self.b = torch.nn.Parameter(torch.randn(7, 5))
        self.c = torch.nn.Parameter(torch.randn(1))
        self.d = torch.nn.Parameter(torch.randn(129, 3))


def _cfg2_modules():
    from graph_marl_b200.model import DQN, NetMon

    nm = NetMon(88, 128, (512, 256), 3, F.leaky_relu, rnn_type="lstm", output_neighbor_hidden=True).cuda()
    dqn = DQN(130 + nm.get_out_features(), (512, 256), 4, F.leaky_relu).cuda()
    return dqn, nm


@pytest.mark.parametrize("which", ["cfg2", "tiny"])
def test_optimizer_step_matches_torch_tail(which, capsys):
    from graph_marl_b200.learner import FusedOptimizer
    from graph_marl_b200.util import interpolate_model

    torch.manual_seed(5)
    if which == "cfg2":
        model, other = _cfg2_modules()
    else:
        model, other = _Tiny().cuda(), _Tiny().cuda()
    target = copy.deepcopy(model)
    with torch.no_grad():
        for p in target.parameters():
            p.add_(0.1 * torch.randn_like(p))
    ref_m, ref_o, ref_t = copy.deepcopy(model), copy.deepcopy(other), copy.deepcopy(target)
    params = list(model.parameters()) + list(other.parameters())
    ref_params = list(ref_m.parameters()) + list(ref_o.parameters())
    lr, tau = 1e-3, 0.01
    opt = FusedOptimizer(params, list(zip(model.parameters(), target.parameters())), lr, tau)
    ref_opt = torch.optim.AdamW(ref_params, lr=lr, foreach=False)
    n = sum(p.numel() for p in params)
    worst = {}
    # gradient magnitudes: norm after clamping far above max_norm, then below it, then around it
    for k, mag in enumerate([1.0, 1e-4, 3e-3, 0.2, 1e-5]):
        grads = [mag * torch.randn_like(p) for p in params]
        for p, g in zip(params, grads):
            p.grad.copy_(g)
        for p, g in zip(ref_params, grads):
            p.grad = g.clone()
        opt.step()
        torch.nn.utils.clip_grad_value_(ref_params, 0.5)
        norm = float(torch.nn.utils.clip_grad_norm_(ref_params, 1.0))
        ref_opt.step()
        interpolate_model(ref_m, ref_t, tau, ref_t)
        st = ref_opt.state
        pairs = [("param", params, ref_params)]
        pairs += [("exp_avg", opt.exp_avg, [st[p]["exp_avg"] for p in ref_params])]
        pairs += [("exp_avg_sq", opt.exp_avg_sq, [st[p]["exp_avg_sq"] for p in ref_params])]
        pairs += [("target", list(target.parameters()), list(ref_t.parameters()))]
        for name, got, ref in pairs:
            for a, b in zip(got, ref):
                e = _rel(a, b)  # relative to the tensor's largest magnitude
                worst[name] = max(worst.get(name, 0.0), e)
                assert e < 1e-6, (k, name, e, norm)
        assert int(opt.step_count) == k + 1
    with capsys.disabled():
        print(f"\n[gm_optimizer_step {which}: {n} parameters] worst relative error over 5 steps: "
              + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


# ---- 4.-7. the learner on a live rollout ---------------------------------------------------------------------------------
def _trainer(math="fp32", envs=64, episode_steps=300, seed=3, **kw):
    from graph_marl_b200.trainer import Trainer

    kw.setdefault("graph_learner", False)
    return Trainer(_cfg(episode_steps=episode_steps), envs, math=math, batch_size=kw.pop("batch_size", 24), seed=seed,
                   capacity_steps=kw.pop("capacity_steps", 16), step_before_train=10**9, **kw)


def _reference_grads(tr, idx, ref_nm, ref_model, ref_target, gamma):
    """train_simple.py's learner body (sequences: state carried and masked at episode ends) on torch autograd of the
    composed reference math, dense adjacency and one-hot node-agent matrices."""
    buff, be = tr.rollout.buff, tr.rollout.base_env
    T, n = idx.shape
    md = be._pool.nbr_all.shape[-1] - 1
    be.get_nodes_adjacency()
    node_adj_all = be._pool.node_adj.float()
    N, A = be._N, be._A

    def nam(agent_node):
        m = torch.zeros((agent_node.shape[0], N, A), device="cuda")
        m.scatter_(1, agent_node.long().unsqueeze(1), 1.0)
        return m

    loss = 0.0
    state = None
    for t in range(T):
        v = buff.learner_views(idx[t])
        adj = node_adj_all[v["topo"].long()]
        ref_nm.state = v["node_state"] if t == 0 else state * (~prev_end).float().view(-1, 1, 1)
        g_obs = ref_nm._forward_autograd(v["node_obs"], adj, nam(v["agent_node"]), md, False)
        state = ref_nm.state
        q = ref_model.q_net(ref_model.encoder(torch.cat((v["obs"], g_obs), -1)))
        with torch.no_grad():
            ref_nm.state = state.detach()
            g_next = ref_nm._forward_autograd(v["next_node_obs"], adj, nam(v["next_agent_node"]), md, False)
            qn = ref_target.q_net(ref_target.encoder(torch.cat((v["next_obs"], g_next), -1)))
            target = v["reward"] + (~v["done"]) * gamma * qn.max(dim=2)[0]
            q_target = torch.scatter(q.detach(), -1, v["action"].unsqueeze(-1), target.unsqueeze(-1))
        loss = loss + torch.mean((q - q_target).pow(2)) / T
        prev_end = v["episode_done"]
    loss.backward()
    return float(loss)


@pytest.mark.parametrize("math,tol", [("fp32", 1e-4), ("bf16x3", 5e-3)])
@pytest.mark.parametrize("T", [1, 4])
def test_learner_gradients_match_torch_autograd(math, tol, T):
    import graph_marl_b200.model as M

    # 3-step episodes: every 4-step sequence crosses an episode end
    tr = _trainer(math, episode_steps=3 if T > 1 else 300)
    tr.train(12)
    buff, ln = tr.rollout.buff, tr.learner
    idx = buff.sample_env_sequences(24, T)
    if T > 1:
        ends = torch.stack([buff.learner_views(idx[t])["episode_done"] for t in range(T - 1)])
        assert bool(ends.any())
    ref_nm, ref_model, ref_target = copy.deepcopy(ln.netmon), copy.deepcopy(ln.model), copy.deepcopy(ln.target)
    n_torch = M.GRAD_PATH_CALLS["torch"]
    ln.forward_backward(buff, idx)
    assert M.GRAD_PATH_CALLS["torch"] == n_torch
    ref_loss = _reference_grads(tr, idx, ref_nm, ref_model, ref_target, ln.gamma)
    assert abs(float(ln.loss) - ref_loss) <= tol * abs(ref_loss)
    for (name, p), r in zip(list(ln.model.named_parameters()) + list(ln.netmon.named_parameters()),
                            list(ref_model.parameters()) + list(ref_nm.parameters())):
        assert r.grad is not None, name
        assert _rel(p.grad, r.grad) < tol, (name, _rel(p.grad, r.grad))


def _snapshot(ln, buff):
    ts = [p.data for p in ln.params] + list(ln.target.parameters()) + ln.opt.exp_avg + ln.opt.exp_avg_sq
    ts += [ln.opt.step_count, buff._pcg_dev]
    return ts, [t.clone() for t in ts]


def _restore(snap, ln):
    with torch.no_grad():
        for t, c in zip(*snap):
            t.copy_(c)
    ln.refresh_packs()


def test_captured_updates_match_eager_updates(capsys):
    """Three updates replayed from a captured graph against three eager updates from the same start (weights, target,
    moments, step count, sampler state)."""
    from graph_marl_b200.learner import Learner

    tr = _trainer("bf16x3", envs=128, episode_steps=5)
    tr.train(10)
    buff, r = tr.rollout.buff, tr.rollout
    eager = tr.learner
    graph = Learner(r.netmon, r.model, 1e-3, 0.98, 0.01, graph=True)
    graph.target.load_state_dict(eager.target.state_dict())
    runs = {}
    for name, ln in (("graph", graph), ("eager", eager)):
        snap = _snapshot(ln, buff)
        if name == "graph":
            ln.update(buff, 32, 2)  # warm-up (eager), then from the same start as the eager run
            _restore(snap, ln)
        losses = [ln.update(buff, 32, 2)]
        grads = [p.grad.clone() for p in ln.params]  # the first update's gradients as the optimizer left them
        losses += [ln.update(buff, 32, 2) for _ in range(2)]
        runs[name] = ([float(x) for x in losses], grads, [p.detach().clone() for p in ln.params],
                      [p.detach().clone() for p in ln.target.parameters()])
        _restore(snap, ln)
    assert len(graph._graphs) == 1
    (lg, gg, pg, tg), (le, ge, pe, te) = runs["graph"], runs["eager"]
    assert lg[0] == le[0]  # same inputs, same forward kernels: bit-equal
    # the device backward accumulates some weight gradients with atomics: the first update's gradients agree to rounding,
    # later updates start from weights that differ in their last bits
    worst_g = max(_rel(a, b) for a, b in zip(gg, ge))
    assert worst_g < 1e-5
    for a, b in zip(lg[1:], le[1:]):
        assert abs(a - b) <= 1e-4 * abs(b)
    # AdamW's step is ~lr * sign(gradient) wherever |gradient| >> eps: where a gradient is ~0 its rounding can flip that
    # sign, so an element may move apart by up to 2 * lr per update -- the bar for every parameter and target element
    worst_p = max(float((a - b).abs().max()) for a, b in zip(pg + tg, pe + te))
    assert worst_p <= 3 * 2 * 1e-3
    # and such flips stay rare: measured 0 %, 0.9 %, 1.9 % and 2.4 % of the elements beyond 1e-5 of their tensor's max
    far = sum(int(((a - b).abs() > 1e-5 * b.abs().max()).sum()) for a, b in zip(pg + tg, pe + te))
    total = sum(b.numel() for b in pe + te)
    assert far <= 0.05 * total
    with capsys.disabled():
        print(f"\n[captured vs eager, 3 updates] losses {lg} vs {le}; first gradients within {worst_g:.2e}; worst parameter "
              f"difference {worst_p:.2e}, {far} of {total} elements beyond 1e-5 of their tensor's max")


def test_captured_updates_of_two_batch_sizes_match_eager_updates():
    """Captured updates of two batch sizes, interleaved, against the same sequence of eager updates: each captured graph
    keeps the inference workspaces it was captured with (warming up the larger batch must not move them)."""
    from graph_marl_b200.learner import Learner

    tr = _trainer("bf16x3", envs=128, episode_steps=5)
    tr.train(10)
    buff, r = tr.rollout.buff, tr.rollout
    eager = tr.learner
    graph = Learner(r.netmon, r.model, 1e-3, 0.98, 0.01, graph=True)
    graph.target.load_state_dict(eager.target.state_dict())
    order = [32, 32, 256, 256, 32, 256, 32]  # warm-up 32, capture 32, warm-up 256, capture 256, replays
    runs = {}
    for name, ln in (("graph", graph), ("eager", eager)):
        snap = _snapshot(ln, buff)
        losses, ws = [], None
        for k, b in enumerate(order):
            losses.append(float(ln.update(buff, b, 2)))
            if name == "graph" and k == 1:
                ws = [w.buf.data_ptr() for w in graph._static[(id(buff), 32, 2)]["ws"]]
        runs[name] = losses
        if name == "graph":
            assert len(graph._graphs) == 2
            assert [w.buf.data_ptr() for w in graph._static[(id(buff), 32, 2)]["ws"]] == ws
        _restore(snap, ln)
    lg, le = runs["graph"], runs["eager"]
    assert lg[0] == le[0]
    for a, b in zip(lg[1:], le[1:]):  # later updates: the backward's atomics reorder sums (see above)
        assert abs(a - b) <= 1e-4 * abs(b), (lg, le)


def test_update_rejects_replaced_grads():
    """The fused optimizer's device table points at the .grad tensors it allocated: zero_grad() (which sets them to None)
    or a new .grad must raise, not let the kernels write memory nothing reads."""
    from graph_marl_b200 import _lib

    tr = _trainer("fp32", envs=32)
    tr.train(6)
    buff, ln = tr.rollout.buff, tr.learner
    ln.update(buff, 8, 1)
    ln.model.zero_grad()
    with pytest.raises(_lib.GraphMarlError, match="grad"):
        ln.update(buff, 8, 1)
    for p, g in zip(ln.params, ln.opt._grads):
        p.grad = g
    p = ln.params[-1]
    p.grad = torch.zeros_like(p)
    with pytest.raises(_lib.GraphMarlError, match="grad"):
        ln.opt.step()
    p.grad = ln.opt._grads[-1]
    assert torch.isfinite(ln.update(buff, 8, 1)).all()


def test_update_refreshes_the_weight_packs_that_captured_work_reads():
    """A CUDA graph captured before an update (like a rollout unit) keeps reading the pack buffers: after the update its
    Q-values (and NetMon's graph observation) equal eager calls on freshly built packs of the new weights."""
    from graph_marl_b200.model import PackedRows, _PackedWeights

    tr = _trainer("bf16x3", envs=64)
    tr.train(10)
    r, buff, ln = tr.rollout, tr.rollout.buff, tr.learner
    be, nm, model = r.base_env, r.netmon, r.model
    obs_a, obs_g = r.obs
    nbr, deg, li = be.get_adjacency_lists()
    kw = dict(agent_node=be.get_agent_nodes(), sparse_nnz=be.node_obs_nnz, sparse_rows=be._out.get("node_sparse"),
              static_rows=be.node_static_rows)
    st0 = r.env.current_netmon_state.clone()
    x = be._out["node_obs"].clone()
    ga = obs_g.float() if isinstance(obs_g, PackedRows) else obs_g.clone()

    def unit():
        nm.state = st0
        _, g = nm.forward_lists(x, nbr, deg, li, nbr.shape[-1] - 1, **kw)
        q, _ = model.act(obs_a, ga, epsilon=0.0, want_q=True)
        qt, _ = ln.target.act(obs_a, ga, epsilon=0.0, want_q=True)
        return g, q, qt

    ln.update(buff, 16, 1)  # the target's pack exists from here on
    with torch.no_grad():
        unit()
        torch.cuda.synchronize()
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            out = unit()
        cg.replay()
        before = [t.clone() for t in out]
    ln.update(buff, 16, 1)
    with torch.no_grad():
        cg.replay()
        torch.cuda.synchronize()
        fresh = []
        for m in (nm, model, ln.target):
            c = copy.deepcopy(m)
            c._pack = _PackedWeights()
            fresh.append(c)
        fresh[0].state = st0
        _, g = fresh[0].forward_lists(x, nbr, deg, li, nbr.shape[-1] - 1, **kw)
        q, _ = fresh[1].act(obs_a, ga, epsilon=0.0, want_q=True)
        qt, _ = fresh[2].act(obs_a, ga, epsilon=0.0, want_q=True)
    for name, a, b, old in zip(("netmon", "dqn", "target"), out, (g, q, qt), before):
        assert not torch.equal(b, old), name  # the update changed the weights
        assert torch.equal(a, b), name


# ---- 7. learning ---------------------------------------------------------------------------------------------------------
# half the gain of the greedy policy over the epsilon = 1 policy that this run measured on one B200 (DESIGN.md section 5)
LEARNING_MARGIN = 0.35


def test_trainer_learns(capsys):
    from graph_marl_b200.trainer import Trainer

    tr = Trainer("cfg2", 256, math="bf16x3", batch_size=256, sequence_length=1, train_every=1, updates_per_train=2,
                 step_before_train=20, epsilon=1.0, epsilon_decay=0.95, epsilon_update_freq=20, lr=1e-3, gamma=0.98,
                 tau=0.01, capacity_steps=64, seed=11, graph_steps=0)
    random_reward = tr.evaluate(1, epsilon=1.0)
    losses = tr.train(1200)
    greedy = tr.evaluate(1, epsilon=0.0)
    assert len(losses) == 2 * (1200 - 20 + 1) and all(np.isfinite(losses))
    ckpt = tr.state_dict()
    assert ckpt["type"] == "DQN" and "netmon_state_dict" in ckpt
    with capsys.disabled():
        print(f"\n[trainer cfg2, 256 envs, 1200 steps / {len(losses)} updates] reward greedy {greedy:.4f} vs epsilon=1 "
              f"{random_reward:.4f} (gain {greedy - random_reward:.4f}); loss first {losses[0]:.4g} last {losses[-1]:.4g}")
    assert greedy > random_reward + LEARNING_MARGIN
