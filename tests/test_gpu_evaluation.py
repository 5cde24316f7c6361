"""Batched evaluation on held-out topologies (graph_marl_b200.evaluation, csrc/eval_metrics.cu):

  - gm_eval_accumulate against an fp64 torch restatement that sums in the kernel's order (B in {1, 7, 1000, 4096}, A in
    {1, 20, 100}; random, no done packets, all packets done, large delays), two runs and a captured launch bit-identical;
  - env b's pool slot holds the topology of EVAL_SEEDS[b], for all 1000; an invalid provided seed raises;
  - evaluate_topologies against a batched Routing stepped on the same pool with the same module copies, every metric
    restated in torch fp64 (cfg2- and cfg3-shaped modules, fp32 and bf16x3), per topology and pooled;
  - the same reward_mean as Trainer.evaluate on the training topology;
  - an evaluation in the middle of a captured training run changes nothing of that run (cfg2, cfg3);
  - a short cfg3 training run beats the epsilon = 1 policy on 256 evaluation graphs;
  - the refusals.
"""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _rel(a, b):
    """Largest relative difference, NaN where both are NaN counting as equal."""
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    assert torch.equal(torch.isnan(a), torch.isnan(b)), (a, b)
    ok = ~torch.isnan(b)
    if not ok.any():
        return 0.0
    return float(((a[ok] - b[ok]).abs() / b[ok].abs().clamp_min(1e-300)).max())


# ---- 1. the kernel ---------------------------------------------------------------------------------------------------
def _step_outputs(B, A, mode, gen):
    dev = "cuda"
    reward = (torch.randn((B, A), generator=gen, device=dev) * 3).float()
    if mode == "none_done":
        done = torch.zeros((B, A), dtype=torch.uint8, device=dev)
    elif mode == "all_done":
        done = torch.ones((B, A), dtype=torch.uint8, device=dev)
    else:
        done = (torch.rand((B, A), generator=gen, device=dev) < 0.3).to(torch.uint8)
    arrived = done * (torch.rand((B, A), generator=gen, device=dev) < 0.7).to(torch.uint8)
    hi = 2**30 if mode == "large" else 300
    delays = torch.randint(0, hi, (B, A), generator=gen, device=dev, dtype=torch.int32)
    spr = 1.0 + torch.rand((B, A), generator=gen, device=dev, dtype=torch.float64) * 4
    spr = torch.where(arrived.bool(), spr, torch.full_like(spr, float("nan")))  # never read for packets that did not arrive
    info = torch.randint(0, hi, (B, 4), generator=gen, device=dev, dtype=torch.int32)
    return dict(reward=reward, done=done, arrived=arrived, delays=delays, spr=spr, info=info)


def _lane_sum(v):
    """[B, A] f64 summed in gm_eval_accumulate's order: lane l adds agents l, l + 32, ... in turn, then the shuffle tree
    lane i += lane i + o for o = 16, 8, 4, 2, 1."""
    B, A = v.shape
    L = -(-A // 32) * 32
    p = torch.zeros((B, L), dtype=torch.float64, device=v.device)
    p[:, :A] = v
    p = p.view(B, L // 32, 32)
    s = torch.zeros((B, 32), dtype=torch.float64, device=v.device)
    for j in range(L // 32):
        s = s + p[:, j]
    for o in (16, 8, 4, 2, 1):
        s = s[:, :o] + s[:, o:2 * o]
    return s[:, 0]


def _restate(acc, out):
    A = out["reward"].shape[1]
    done, arrived = out["done"].bool(), out["arrived"].bool()
    d = out["delays"].double()
    zero = torch.zeros_like(d)
    add = [_lane_sum(out["reward"].double()), torch.full_like(acc[:, 0], float(A)), _lane_sum(torch.where(done, d, zero)),
           _lane_sum(done.double()), _lane_sum(torch.where(arrived, d, zero)), _lane_sum(arrived.double()),
           _lane_sum(torch.where(arrived, out["spr"], zero))] + [out["info"][:, k].double() for k in range(4)] + \
          [torch.ones_like(acc[:, 0])]
    acc += torch.stack(add, 1)


@pytest.mark.parametrize("mode", ["random", "none_done", "all_done", "large"])
@pytest.mark.parametrize("A", [1, 20, 100])
@pytest.mark.parametrize("B", [1, 7, 1000, 4096])
def test_accumulate_against_fp64(B, A, mode):
    from graph_marl_b200 import _lib
    from graph_marl_b200.evaluation import accumulate

    gen = torch.Generator(device="cuda").manual_seed(B * 1000 + A)
    steps = [_step_outputs(B, A, mode, gen) for _ in range(3)]
    F_ = len(_lib.EVAL_FIELDS)
    ref = torch.zeros((B, F_), dtype=torch.float64, device="cuda")
    for out in steps:
        _restate(ref, out)
    runs = []
    for _ in range(2):
        acc = torch.zeros((B, F_), dtype=torch.float64, device="cuda")
        for out in steps:
            accumulate(acc, out)
        runs.append(acc)
    torch.cuda.synchronize()
    assert torch.equal(runs[0], runs[1]), "two runs differ"
    acc = runs[0]
    exact = [i for i, k in enumerate(_lib.EVAL_FIELDS) if k not in ("reward_sum", "spr_sum")]
    assert torch.equal(acc[:, exact], ref[:, exact])
    for k in ("reward_sum", "spr_sum"):
        i = _lib.EVAL_FIELDS.index(k)
        assert _rel(acc[:, i].cpu(), ref[:, i].cpu()) <= 1e-12, k
    if mode == "none_done":
        assert not acc[:, 2:7].any()
    # a captured launch sequence computes the same bits
    cap = torch.zeros_like(acc)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for out in steps:
            accumulate(cap, out)
    cap.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(cap, acc), "captured != eager"


# ---- 2. placement ----------------------------------------------------------------------------------------------------
def test_eval_pool_holds_every_evaluation_graph_in_its_slot():
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.env.network import generate_tables
    from graph_marl_b200.evaluation import topology_pool

    pool, slot = topology_pool(EVAL_SEEDS, 20, "cuda")
    assert torch.equal(slot.cpu(), torch.arange(len(EVAL_SEEDS), dtype=torch.int32))
    edges, apsp = pool.edges.cpu().numpy(), pool.apsp.cpu().numpy()
    ne, nn_ = pool.node_edges.cpu().numpy(), pool.node_nbrs.cpu().numpy()
    for b, s in enumerate(EVAL_SEEDS):
        t = generate_tables(20, s)
        assert np.array_equal(edges[b], t["edges"]) and np.array_equal(apsp[b], t["apsp"]), (b, s)
        assert np.array_equal(ne[b], t["node_edges"]) and np.array_equal(nn_[b], t["node_nbrs"]), (b, s)
    assert pool.seeds == list(EVAL_SEEDS)


def test_invalid_provided_seed_raises():
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.evaluation import evaluate_topologies, topology_pool

    with pytest.raises(AssertionError, match="Provided seed 4 is invalid."):
        topology_pool([EVAL_SEEDS[0], 4, EVAL_SEEDS[1]], 20, "cuda")
    nm, dqn = _modules("cfg2", "fp32")
    with pytest.raises(AssertionError, match="Provided seed 4 is invalid."):
        evaluate_topologies(nm, dqn, [4], 20, 5)


# ---- 3. end to end against a restatement -----------------------------------------------------------------------------
SHAPES = {"cfg2": dict(K=3, congestion=True), "cfg3": dict(K=1, congestion=False)}


def _modules(cfg, math, N=20, seed=0):
    from graph_marl_b200.model import DQN, NetMon

    torch.manual_seed(seed)
    H = 128
    nm = NetMon(4 * N + 8, H, (512, 256), SHAPES[cfg]["K"], F.leaky_relu, rnn_type="lstm", agg_type="sum",
                output_neighbor_hidden=True, math=math).cuda().eval()
    dqn = DQN(6 * N + 10 + nm.get_out_features(), (512, 256), 4, F.leaky_relu, math=math).cuda().eval()
    return nm, dqn


def _restated_metrics(nm, dqn, seeds, A, steps, congestion, epsilon, env_seed, episodes):
    """The evaluation restated: a plain batched Routing reset onto the pool by hand, NetMonWrapper, model.act; every
    metric in torch fp64 from the per-step tensors, as eval.py defines them."""
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from graph_marl_b200.env.wrapper import NetMonWrapper
    from graph_marl_b200.evaluation import _private_copy, topology_pool

    B = len(seeds)
    pool, slot = topology_pool(seeds, 20, "cuda")
    be = Routing(Network(20), A, 1, enable_congestion=congestion, num_envs=B, device="cuda", seed=env_seed, batched=True)
    env = NetMonWrapper(be, _private_copy(nm), 1, split_obs=True, graph_obs_fp32=True)
    model = _private_copy(dqn)
    z = lambda: torch.zeros((B,), dtype=torch.float64, device="cuda")
    s = {k: z() for k in ("reward", "agent_steps", "d", "dn", "da", "an", "spr", "looped", "throughput", "dropped",
                          "blocked", "steps")}
    lists = {"delays": [], "delays_arrived": [], "spr": []}
    k = 0
    with torch.no_grad():
        for _ in range(episodes):
            env.last_netmon_state = env.current_netmon_state = None
            obs, _ = be.reset_on_pool(pool, slot)
            obs_a, obs_g = env._with_graph_obs(obs)
            for _ in range(steps):
                k += 1
                _, act = model.act(obs_a, obs_g, epsilon=epsilon, seed=12345, step=k, want_q=False)
                (obs_a, obs_g), _, reward, done, info = env.step(act)
                d = info["delays"].double()
                arr = info["arrived"].bool()
                s["reward"] += reward.double().sum(1)
                s["agent_steps"] += A
                s["d"] += torch.where(done, d, 0.0).sum(1)
                s["dn"] += done.double().sum(1)
                s["da"] += torch.where(arr, d, 0.0).sum(1)
                s["an"] += arr.double().sum(1)
                s["spr"] += torch.where(arr, info["spr"], 0.0).sum(1)
                for key in ("looped", "throughput", "dropped", "blocked"):
                    s[key] += info[key].double()
                s["steps"] += 1
                lists["delays"].append(d[done])
                lists["delays_arrived"].append(d[arr])
                lists["spr"].append(info["spr"][arr])
    per = dict(reward_mean=s["reward"] / s["agent_steps"], delays=s["d"] / s["dn"], delays_arrived=s["da"] / s["an"],
               spr=s["spr"] / s["an"])
    per.update({key: s[key] / s["steps"] for key in ("looped", "throughput", "dropped", "blocked")})
    pooled = {key: float(torch.cat(v).mean()) if sum(x.numel() for x in v) else float("nan") for key, v in lists.items()}
    pooled["reward_mean"] = float(s["reward"].sum() / s["agent_steps"].sum())
    for key in ("looped", "throughput", "dropped", "blocked"):
        pooled[key] = float(s[key].sum() / s["steps"].sum())
    return {k: v.cpu() for k, v in per.items()}, pooled


@pytest.mark.parametrize("math", ["fp32", "bf16x3"])
@pytest.mark.parametrize("cfg,steps,episodes,epsilon", [("cfg2", 40, 2, 0.0), ("cfg3", 50, 1, 0.1)])
def test_evaluate_topologies_against_restatement(cfg, steps, episodes, epsilon, math):
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.evaluation import METRICS, evaluate_topologies

    seeds = list(EVAL_SEEDS[:64])
    nm, dqn = _modules(cfg, math)
    cong = SHAPES[cfg]["congestion"]
    got = evaluate_topologies(nm, dqn, seeds, 20, steps, congestion=cong, epsilon=epsilon, env_seed=17, episodes=episodes)
    per, pooled = _restated_metrics(nm, dqn, seeds, 20, steps, cong, epsilon, 17, episodes)
    for k in METRICS:
        assert got["per_topology"][k].dtype == torch.float64 and got["per_topology"][k].shape == (64,)
        assert _rel(got["per_topology"][k], per[k]) <= 1e-12, k
        assert _rel(got[k], pooled[k]) <= 1e-12, (k, got[k], pooled[k])
    assert np.isfinite(got["reward_mean"]) and got["throughput"] > 0


# ---- 4. consistency with Trainer.evaluate -----------------------------------------------------------------------------
def test_same_reward_mean_as_trainer_evaluate():
    """fp32: there NetMon's encoder reads the dense rows on both sides.  (In the tensor-core modes Trainer.evaluate's
    one-topology pool has static rows that the weight pack folds into layer 1, a different rounding of the same sum.)"""
    from graph_marl_b200.trainer import Trainer

    tr = Trainer("cfg2", 256, math="fp32", seed=5, graph_learner=False)
    want = tr.evaluate(1)
    c = tr.rollout.cfg
    got = tr.evaluate_topologies([c["topo_seed"]] * 256)
    assert _rel(got["reward_mean"], want) <= 1e-12, (got["reward_mean"], want)


# ---- 5. non-interference ---------------------------------------------------------------------------------------------
def _run(cfg, evaluate, k=20):
    """k captured rollout steps with captured learner updates, optionally an evaluation on 128 graphs, k more.  lr = 0:
    the device backward accumulates some gradients with float atomics, so two runs with a step size differ in their last
    bits whatever happens between them; with lr = 0 the weights stay put bit for bit (the Polyak target update, the
    moments, the losses and the whole rollout still run), and any difference is the evaluation's doing."""
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.trainer import Trainer

    tr = Trainer(cfg, 256, math="bf16x3", batch_size=32, sequence_length=2, train_every=5, capacity_steps=20, graph_steps=5,
                 lr=0.0, seed=6, graph_learner=True)
    r = tr.rollout
    np.random.seed(123)
    losses = tr.train(k)
    res = None
    if evaluate:
        before = _trainer_state(tr, same_run=True)
        rng = np.random.get_state()
        res = tr.evaluate_topologies(EVAL_SEEDS[:128], episode_steps=10)
        after = _trainer_state(tr, same_run=True)
        rng2 = np.random.get_state()
        assert rng[0] == rng2[0] and np.array_equal(rng[1], rng2[1]) and rng[2:] == rng2[2:], "numpy stream moved"
        for name in before:
            assert _same(before[name], after[name]), name
    assert r._graphs and tr.learner._graphs, "the run did not replay captured units"
    losses += tr.train(k)
    return losses, _trainer_state(tr), res


def _same(a, b):
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    if torch.is_tensor(a):
        return torch.equal(a, b)
    return a == b


def _trainer_state(tr, same_run=False):
    """Everything the rest of a run reads; same_run: also what holds addresses of this run's tensors (pack keys, captured
    graphs, the weight packs the captured rollout units read) and the Adam moments."""
    r, ln, buff = tr.rollout, tr.learner, tr.rollout.buff
    obs_a, obs_g = r.obs
    g = obs_g.buf if hasattr(obs_g, "buf") else obs_g
    st = dict(
        weights=[p.detach().clone() for p in ln.params] + [p.detach().clone() for p in ln.target.parameters()],
        steps=ln.opt.step_count.clone(),
        state=r.netmon.state.clone(), ring=[t.clone() for t in (buff.rec, buff.next_rec, buff.topo, buff.action, buff.reward,
                                                               buff.done, buff.episode_done, buff.node_state)],
        obs=[obs_a.clone(), g.clone()], node_obs=r.base_env._out["node_obs"].clone(), env_state=r.base_env._state.clone(),
        counters=[r._counters(), r.policy._epsilon, r.base_env._episode, buff.steps_total],
        unit_keys=sorted(r._graphs), seeds=list(r.base_env._pool.seeds))
    if same_run:
        mods = (r.netmon, r.model, ln.target)
        # the Adam moments follow the gradients, whose atomics differ between runs: compared within the run only
        st.update(moments=[t.clone() for t in ln.opt.exp_avg + ln.opt.exp_avg_sq], packs=[m._pack.buf.clone() for m in mods], pack_keys=[m._pack.key for m in mods],
                  graphs=[dict(r._graphs), dict(ln._graphs)], pool=r.base_env._pool)
    return st


@pytest.mark.parametrize("cfg", ["cfg2", "cfg3"])
def test_evaluation_leaves_a_captured_training_run_unchanged(cfg):
    la, sa, res = _run(cfg, True)
    lb, sb, _ = _run(cfg, False)
    assert len(la) > 0 and la == lb, "losses differ"
    for name in sa:
        assert _same(sa[name], sb[name]), name
    assert np.isfinite(res["reward_mean"])


# ---- 6. signal -------------------------------------------------------------------------------------------------------
# half the gain of the greedy policy over the epsilon = 1 policy on the 256 evaluation graphs that this recipe measured on
# one B200 (1000 W power limit): 0.451-0.491 after 2400 steps over seeds 11-14 (0.680-0.805 after 3600, 0.081-0.136 after
# 1200; at lr = 1e-3 the 1200-step gains were -0.011 to 0.030)
LEARNING_MARGIN = 0.22


def test_cfg3_training_beats_random_on_evaluation_graphs(capsys):
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.trainer import Trainer

    tr = Trainer("cfg3", 256, math="bf16x3", batch_size=256, sequence_length=1, train_every=1, updates_per_train=2,
                 step_before_train=20, epsilon=1.0, epsilon_decay=0.95, epsilon_update_freq=20, lr=3e-4, gamma=0.98,
                 tau=0.01, capacity_steps=64, seed=11, graph_steps=0)
    seeds = EVAL_SEEDS[:256]
    random_reward = tr.evaluate_topologies(seeds, epsilon=1.0)["reward_mean"]
    losses = tr.train(2400)
    greedy = tr.evaluate_topologies(seeds, epsilon=0.0)
    assert all(np.isfinite(losses))
    gain = greedy["reward_mean"] - random_reward
    with capsys.disabled():
        print(f"\n[trainer cfg3, 256 envs, 2400 steps / {len(losses)} updates] on 256 evaluation graphs: reward greedy "
              f"{greedy['reward_mean']:.4f} vs epsilon=1 {random_reward:.4f} (gain {gain:.4f}); "
              + ", ".join(f"{k} {greedy[k]:.4g}" for k in ("delays", "delays_arrived", "spr", "throughput", "dropped")))
    assert greedy["reward_mean"] > random_reward + LEARNING_MARGIN


# ---- 7. refusals -----------------------------------------------------------------------------------------------------
def test_refusals():
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.evaluation import evaluate_topologies

    nm, dqn = _modules("cfg3", "fp32")
    with pytest.raises(ValueError, match="at least one"):
        evaluate_topologies(nm, dqn, [], 20, 5)
    with pytest.raises(ValueError, match="episode_steps >= 1"):
        evaluate_topologies(nm, dqn, EVAL_SEEDS[:2], 20, 0)
    from graph_marl_b200.model import NetMon

    for width in (4 * 20 + 9, 4 * 2 + 8):  # not 4N + 8 for an integer N; N = 2 has no 3-regular graph
        odd = NetMon(width, 128, (512, 256), 1, F.leaky_relu, rnn_type="lstm", output_neighbor_hidden=True).cuda().eval()
        with pytest.raises(ValueError, match="node rows"):
            evaluate_topologies(odd, dqn, EVAL_SEEDS[:2], 20, 5)
    nm10, _ = _modules("cfg3", "fp32", N=10)  # 10-node NetMon, 20-node DQN
    with pytest.raises(ValueError, match="the DQN takes"):
        evaluate_topologies(nm10, dqn, EVAL_SEEDS[:2], 20, 5)
