"""The device topology generator (csrc/topology.cu, gm_topology_generate_device) and the fresh-topology mode of the batched
Routing env built on it (a pool of B * S slots at fixed addresses, Routing.set_topology_episodes), up the stack:

  - generator parity: every table, the seed used and the repetitions bit-equal to the host generator (generate_tables
    with reseeding), at N = 20 for 100 000+ seeds (reseeding seeds, the 1000 EVAL_SEEDS, the recorded reference draws,
    an exclusion list that a reseed actually hits), at N = 200 and at the smallest N; a cap on attempts is an error;
  - reset parity: after k batched resets the slots, the global numpy stream and the Network match B * k network.reset();
  - the env on fresh graphs against the C oracle built from each env's seed;
  - the compact replay ring returns the observations of an earlier episode on that episode's graphs;
  - captured rollout units and captured learner updates survive resets.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _host(N, seeds, exclude=None):
    from graph_marl_b200.env.network import generate_tables

    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:  # the native generator releases the GIL
        return list(ex.map(lambda s: generate_tables(N, int(s), allow_reseed=True, exclude=exclude), seeds))


def _device(N, seeds, exclude=None, max_attempts=10000):
    from graph_marl_b200.env.routing import TopologyPool

    pool = TopologyPool.slots(len(seeds), N, "cuda")
    slot = torch.arange(len(seeds), dtype=torch.int32, device="cuda")
    exd = torch.tensor(sorted(exclude), dtype=torch.int64, device="cuda") if exclude else None
    used, reps = pool.generate(np.asarray(seeds, np.int64), slot, exd, max_attempts)
    return pool, used, reps


def _assert_parity(N, seeds, exclude=None, chunk=25000):
    """Device tables of `seeds` bit-equal to the host generator's; returns (seed_used, repetitions)."""
    from graph_marl_b200.env.network import lists_from_tables

    all_used, all_reps = [], []
    for lo in range(0, len(seeds), chunk):
        part = seeds[lo:lo + chunk]
        pool, used, reps = _device(N, part, exclude)
        host = _host(N, part, exclude)
        np.testing.assert_array_equal(used, [t["seed"] for t in host])
        np.testing.assert_array_equal(reps, [t["repetitions"] for t in host])
        for key in ("edges", "node_edges", "node_nbrs", "apsp"):
            got, want = getattr(pool, key).cpu().numpy(), np.stack([t[key] for t in host])
            bad = np.nonzero((got != want).reshape(len(part), -1).any(1))[0]
            assert bad.size == 0, f"{key} differs for seeds {[int(part[i]) for i in bad[:8]]}"
        lists = [lists_from_tables(t) for t in host]
        np.testing.assert_array_equal(pool.nbr_all.cpu().numpy(), np.stack([l[0] for l in lists]))
        np.testing.assert_array_equal(pool.deg.cpu().numpy(), np.stack([l[1] for l in lists]))
        all_used.append(used)
        all_reps.append(reps)
    return np.concatenate(all_used), np.concatenate(all_reps)


# ---- 1. generator parity -------------------------------------------------------------------------------------------------
def test_device_generator_matches_host_at_20_nodes(capsys):
    from graph_marl_b200.env.constants import EVAL_SEEDS

    g = np.load(os.path.join(GOLDEN, "topology.npz"))
    recorded = np.concatenate([g["chain_seed"], g["pool_seeds"], g["fixed_seeds"]]).astype(np.int64)
    drawn = np.random.default_rng(2024).integers(0, 2**31 - 1, 100_000)
    seeds = np.concatenate([drawn, np.asarray(EVAL_SEEDS, np.int64), recorded])
    _, reps = _assert_parity(20, seeds)
    assert (reps > 1).sum() > 10_000 and reps.max() > 5  # plenty of seeds that needed reseeding
    with capsys.disabled():
        print(f"\n[device generator, N=20] {len(seeds)} seeds bit-equal to the host; {(reps > 1).sum()} reseeded, "
              f"up to {reps.max()} attempts")


def test_device_generator_skips_excluded_seeds_like_host():
    """An exclusion list that the reseed loop hits: EVAL_SEEDS plus the first reseed candidate of seeds that needed one
    reseed (the host then skips it and draws the next)."""
    from graph_marl_b200.env.constants import EVAL_SEEDS

    seeds = np.random.default_rng(99).integers(0, 2**31 - 1, 4000)
    plain = _host(20, seeds)
    first_reseed = {int(t["seed"]) for t in plain if t["repetitions"] == 2}
    assert len(first_reseed) > 100
    exclude = set(EVAL_SEEDS) | first_reseed
    used, _ = _assert_parity(20, seeds, exclude)
    assert not set(used.tolist()) & exclude
    assert sum(int(u) != t["seed"] for u, t in zip(used, plain)) >= len(first_reseed)


@pytest.mark.parametrize("N,n", [(200, 300), (4, 300), (6, 300)])
def test_device_generator_matches_host_at_other_sizes(N, n):
    seeds = np.random.default_rng(N).integers(0, 2**31 - 1, n)
    _, reps = _assert_parity(N, seeds)
    if N != 4:  # 4 nodes always give K4 at the first attempt
        assert (reps > 1).any()


def test_device_generator_attempt_cap_is_an_error():
    from graph_marl_b200 import _lib

    seeds = np.random.default_rng(5).integers(0, 2**31 - 1, 64)
    reps = np.array([t["repetitions"] for t in _host(20, seeds)])
    needs = int(seeds[np.argmax(reps > 1)])
    with pytest.raises(_lib.GraphMarlError, match=str(needs)):
        _device(20, [needs], max_attempts=1)
    _device(20, [needs], max_attempts=int(reps.max()))  # the same seed with enough attempts is fine
    with pytest.raises(_lib.GraphMarlError, match="even"):
        _device(_lib.GM_TOPOLOGY_MAX_NODES + 2, [1])


# ---- 2. reset parity -----------------------------------------------------------------------------------------------------
def test_batched_fresh_reset_equals_host_resets():
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing

    B, k, S = 96, 3, 2
    env = Routing(Network(20, random_topology=True, excluded_seeds=EVAL_SEEDS), 20, 1, enable_congestion=False,
                  num_envs=B, device="cuda", batched=True)
    env.set_topology_episodes(S)
    np.random.seed(77)
    slots, ptrs = [], None
    for e in range(k):
        env.reset()
        p = env._pool
        assert p.T == B * S and p.static_rows is None
        idx = env._topo_index.cpu().numpy()
        np.testing.assert_array_equal(idx, (e % S) * B + np.arange(B))
        slots.append({key: getattr(p, key)[idx].cpu().numpy() for key in ("edges", "node_edges", "node_nbrs", "apsp")})
        now = [t.data_ptr() for t in (p.edges, p.node_edges, p.node_nbrs, p.apsp, p.nbr_all, p.deg, env._topo_index)]
        assert ptrs is None or now == ptrs
        ptrs = now
    dev_state = np.random.get_state()
    ref = Network(20, random_topology=True, excluded_seeds=EVAL_SEEDS)
    np.random.seed(77)
    for e in range(k):
        for b in range(B):
            ref.reset()
            for key, arr in slots[e].items():
                np.testing.assert_array_equal(arr[b], ref.tables[key], err_msg=f"episode {e} env {b} {key}")
    host_state = np.random.get_state()
    assert host_state[0] == dev_state[0] and np.array_equal(host_state[1], dev_state[1]) and host_state[2:] == dev_state[2:]
    assert env.network.sampled_topology_seeds == ref.sampled_topology_seeds
    assert env.network.current_topology_seed == ref.current_topology_seed
    np.testing.assert_array_equal(env.network.tables["apsp"], ref.tables["apsp"])
    np.testing.assert_array_equal(env.network.adj_matrix, ref.adj_matrix)


# ---- 3. the env on fresh graphs against the C oracle ---------------------------------------------------------------------
def test_fresh_topology_env_matches_oracle():
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from graph_marl_b200.rollout import CONFIGS
    from oracle import oracle as O

    c = CONFIGS["cfg3fresh"]
    N, A, B = c["n_nodes"], c["n_data"], 48
    env = Routing(Network(N, random_topology=True), A, 1, enable_congestion=c["congestion"], num_envs=B, device="cuda",
                  batched=True)
    env.set_topology_episodes(2)
    rng = np.random.default_rng(3)
    draws = lambda: (rng.integers(0, N, (B, A)).astype(np.int32), rng.integers(0, N, (B, A)).astype(np.int32),
                     rng.random((B, A)))
    np.random.seed(8)
    sample = [0, 17, 47]
    for episode in range(3):
        d = draws()
        env.set_draws(*d)
        env.reset()
        seeds = env.network.sampled_topology_seeds[-B:]
        orcs = {b: O.RoutingOracle(O.generate_topology(N, seed=seeds[b]), A, enable_congestion=c["congestion"]) for b in sample}
        for b, o in orcs.items():
            o.reset(d[0][b], d[1][b], d[2][b])
        for t in range(12):
            act = rng.integers(0, 4, (B, A)).astype(np.int32)
            d = draws()
            env.set_draws(*d)
            _, _, reward, _, _ = env.step(torch.from_numpy(act).cuda())
            s = env.get_state()
            rw = reward.cpu().numpy()
            for b, o in orcs.items():
                r = o.step(act[b], d[0][b], d[1][b], d[2][b])
                np.testing.assert_array_equal(rw[b], r["reward"][0], err_msg=f"episode {episode} step {t} env {b}")
                for key in ("now", "target", "edge", "time", "spw", "start", "agent_steps", "size", "load"):
                    np.testing.assert_array_equal(s[key][b], getattr(o, key)[0], err_msg=f"{key} episode {episode} step {t} env {b}")


# ---- 4. the compact ring keeps each transition's graph -------------------------------------------------------------------
def test_compact_ring_returns_earlier_episodes_on_their_own_graphs():
    from graph_marl_b200.rollout import CONFIGS, Rollout

    E, B, cap_steps = 5, 64, 12
    cfg = dict(CONFIGS["cfg3fresh"], episode_steps=E, H=64, enc=(64,), dqn=(64,))
    ro = Rollout(cfg, num_envs=B, math="fp32", seed=3, replay_capacity=B * cap_steps, replay="compact", device_sampler=True)
    be = ro.base_env
    assert be._topo_episodes == -(-cap_steps // E) + 1
    records = []
    for t in range(cap_steps):  # three episodes, all of them still in the ring at the end
        if ro.episode_step is None or ro.episode_step >= E:
            ro.reset()
        i0 = ro.buff.index
        rec = dict(obs=ro.obs[0].clone(), node_obs=be._out["node_obs"].clone(), node_adj=be.get_nodes_adjacency().clone(),
                   node_aux=be.get_node_aux().clone())
        ro.step()
        rec.update(next_obs=ro.obs[0].clone(), next_node_obs=be._out["node_obs"].clone())
        records.append((i0, rec))
    torch.cuda.synchronize()
    first, last = records[0][1], records[-1][1]
    assert not torch.equal(first["node_aux"], last["node_aux"])  # the episodes really ran on different graphs
    for t in (0, 3, 4):  # transitions of the first episode
        i0, rec = records[t]
        slots = np.arange(i0, i0 + B)
        v = ro.buff.learner_views(torch.from_numpy(slots).cuda())
        batch = ro.buff._get_transition_batch(slots, "cuda")
        for key in ("obs", "node_obs", "next_obs", "next_node_obs"):
            assert torch.equal(v[key], rec[key]), (t, key)
        assert torch.equal(batch.node_obs, rec["node_obs"]) and torch.equal(batch.next_node_obs, rec["next_node_obs"]), t
        assert torch.equal(batch.node_adj, rec["node_adj"].float()), t
        assert torch.equal(batch.node_aux, rec["node_aux"]), t
        assert torch.equal(batch.obs[..., :rec["obs"].shape[-1]], rec["obs"]), t


# ---- 5. captured rollout units across resets -----------------------------------------------------------------------------
def test_fresh_topology_rollout_graph_equals_eager_across_resets():
    from graph_marl_b200.rollout import CONFIGS, Rollout

    cfg = dict(CONFIGS["cfg3fresh"], H=64, enc=(64,), dqn=(64,), episode_steps=9)
    mk = lambda g: Rollout(cfg, num_envs=40, math="bf16x3", seed=11, replay_capacity=40 * 8, graph_steps=g, replay="dense")
    a, b = mk(0), mk(3)
    for ro in (a, b):
        np.random.seed(5)
        ro.reset()
    p = b.base_env._pool
    ptrs = [t.data_ptr() for t in (p.edges, p.node_edges, p.node_nbrs, p.apsp, p.nbr_all, p.deg, b.base_env._topo_index)]
    for ro in (a, b):
        np.random.seed(6)
        ro.run(6)
    units = dict(b._graphs)
    assert units, "no CUDA graph unit was captured"
    for ro in (a, b):
        np.random.seed(7)  # the resets draw their seeds from the global stream: the same one for both runs
        ro.run(25)  # three more resets
    torch.cuda.synchronize()
    assert b.base_env._pool is p and b.base_env._episode == 4
    assert [t.data_ptr() for t in (p.edges, p.node_edges, p.node_nbrs, p.apsp, p.nbr_all, p.deg, b.base_env._topo_index)] == ptrs
    assert all(b._graphs.get(k) is g for k, g in units.items()), "units captured before a reset were dropped"
    assert a.base_env.network.sampled_topology_seeds == b.base_env.network.sampled_topology_seeds
    sa, sb = a.base_env.get_state(), b.base_env.get_state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    assert torch.equal(a.obs[0], b.obs[0]) and torch.equal(a.obs[1], b.obs[1])
    for name in ("obs", "next_obs", "node_adj", "node_aux", "reward", "node_state", "node_obs", "action"):
        assert torch.equal(getattr(a.buff, name), getattr(b.buff, name)), name


# ---- 6. training ---------------------------------------------------------------------------------------------------------
def _snapshot(ln, buff):
    ts = [p.data for p in ln.params] + list(ln.target.parameters()) + ln.opt.exp_avg + ln.opt.exp_avg_sq
    ts += [ln.opt.step_count, buff._pcg_dev]
    return ts, [t.clone() for t in ts]


def _restore(snap, ln):
    with torch.no_grad():
        for t, c in zip(*snap):
            t.copy_(c)
    ln.refresh_packs()


def test_trainer_on_fresh_topologies_captures_each_update_once():
    from graph_marl_b200.learner import Learner
    from graph_marl_b200.trainer import Trainer

    tr = Trainer("cfg3fresh", 256, math="bf16x3", batch_size=32, sequence_length=2, train_every=5, capacity_steps=16,
                 graph_steps=5, seed=4)
    be = tr.rollout.base_env
    losses = tr.train(60)
    key = next(iter(tr.learner._graphs))
    g = tr.learner._graphs[key]
    pool = be._pool
    losses += tr.train(90)  # 150 steps: three episode resets
    torch.cuda.synchronize()
    assert be._episode == 3 and be._pool is pool and be._topo_episodes == 2
    assert len(tr.learner._graphs) == 1 and tr.learner._graphs[key] is g, "the captured update was re-captured"
    assert len(losses) >= 25 and np.isfinite(losses).all()
    # the replayed update against an eager one from the same start, after the resets
    buff, r = tr.rollout.buff, tr.rollout
    snap = _snapshot(tr.learner, buff)
    lg = float(tr.learner.update(buff, 32, 2))
    gg = [p.grad.clone() for p in tr.learner.params]
    _restore(snap, tr.learner)
    eager = Learner(r.netmon, r.model, 1e-3, 0.98, 0.01, graph=False)
    eager.target.load_state_dict(tr.learner.target.state_dict())
    le = float(eager.update(buff, 32, 2))
    ge = [p.grad.clone() for p in eager.params]
    assert lg == le
    worst = max(float((a - b).abs().max() / b.abs().max().clamp_min(1e-12)) for a, b in zip(gg, ge))
    assert worst < 1e-5
