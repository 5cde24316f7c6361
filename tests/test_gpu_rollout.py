"""GPU checks of the batched rollout loop (graph_marl_b200/rollout.py): CUDA-graph replay of captured
step units must reproduce the eager (kernel-by-kernel) rollout exactly -- same env state, observations,
NetMon state, replay ring contents -- with device Philox draws and with host-supplied draw tables."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _mk(graph_steps, host_draws=False, replay="dense", B=96, **kw):
    from graph_marl_b200.rollout import Rollout

    ro = Rollout("cfg2", num_envs=B, math="bf16x3", seed=7, replay_capacity=B * 16, graph_steps=graph_steps,
                 host_draws=host_draws, host_draw_steps=40, replay=replay, **kw)
    ro.reset()
    return ro


def _graph_obs(ro):
    g = ro.obs[1]
    return g.buf if hasattr(g, "buf") else g


DENSE_FIELDS = ("obs", "next_obs", "action", "reward", "done", "node_state", "node_obs", "next_node_agent_matrix")
COMPACT_FIELDS = ("rec", "next_rec", "topo", "action", "reward", "done", "episode_done", "node_state")


@pytest.mark.parametrize("replay", ["dense", "compact"])
@pytest.mark.parametrize("host_draws", [False, True])
def test_graph_replay_equals_eager(host_draws, replay):
    a, b = _mk(0, host_draws, replay), _mk(5, host_draws, replay)
    if host_draws:
        # graph units consume aligned blocks of the host draw table (skipping to the next block when needed):
        # record which table rows the graph run used and feed the eager run the same rows
        b._h_trace = []
        b.run(23)
        assert len(b._h_trace) == 23
        for i in b._h_trace:
            a._h_cursor = i
            a.run(1)
    else:
        a.run(23)
        b.run(23)
    torch.cuda.synchronize()
    assert b._graphs, "no CUDA graph unit was captured"
    sa, sb = a.base_env.get_state(), b.base_env.get_state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    assert torch.equal(a.obs[0], b.obs[0]) and torch.equal(_graph_obs(a), _graph_obs(b)) and torch.equal(a.adj, b.adj)
    assert torch.equal(a.env.current_netmon_state, b.env.current_netmon_state)
    assert torch.equal(a.env.last_netmon_state, b.env.last_netmon_state)
    assert (a.buff.index, a.buff.count) == (b.buff.index, b.buff.count)
    for name in (DENSE_FIELDS if replay == "dense" else COMPACT_FIELDS):
        if name == "node_state" and replay == "compact":
            # state-ring mode: the field is the NetMon state history with its own modulus (a multiple of the unit length),
            # so the two runs lay it out differently: compare the blocks of the transitions the ring still holds
            assert a.buff.state_ring and b.buff.state_ring and a.buff.steps_total == b.buff.steps_total
            T = a.buff.steps_total
            for t in range(max(0, T - a.buff.cap_steps), T + 2):
                assert torch.equal(a.buff.state_block(t), b.buff.state_block(t)), t
            continue
        assert torch.equal(getattr(a.buff, name), getattr(b.buff, name)), name
    assert (a.episode_step, a.base_env._calls, a.policy._step) == (b.episode_step, b.base_env._calls, b.policy._step)
    if host_draws:  # the per-step reward read-back (side stream inside a captured unit) delivered the last step's rewards
        assert torch.equal(a._h_reward, b._h_reward)
        last = b.buff.reward[(b.buff.index - b.B) % b.buff.buffer_size:][:b.B] if b.buff.index >= b.B else None
        if last is not None:
            assert torch.equal(last.reshape(b._h_reward.shape).cpu(), b._h_reward)
    if replay == "compact":  # and the learner's view of both rings is the same
        for x, y in zip(a.buff.get_batch(24, "cuda", sequence_length=4), b.buff.get_batch(24, "cuda", sequence_length=4)):
            assert np.array_equal(x.idx, y.idx)
            for f in ("obs", "next_obs", "node_state", "reward", "node_obs"):
                assert torch.equal(getattr(x, f), getattr(y, f)), f


@pytest.mark.parametrize("graph_steps,B", [(0, 40), (5, 40), (5, 2100)])  # 2100 envs: the one-warp-per-env instance of the step kernel
def test_fused_insert_equals_stage_and_commit(graph_steps, B):
    """The step kernel writing the compact transition itself (gm_routing_io.ring_*: records before / after, actions,
    reward, done, topology index, episode_done) must leave the ring exactly as the two insert launches (stage + commit)
    do, ring wrap and episode ends included."""
    from graph_marl_b200.rollout import Rollout

    cfg = dict(n_nodes=20, n_data=20, topo_seed=476, random_topology=True, n_topologies=5, congestion=True, K=1, rnn="lstm",
               H=64, enc=(64,), dqn=(64,), episode_steps=9)
    mk = lambda fused: Rollout(cfg, num_envs=B, math="bf16x3", seed=5, replay_capacity=B * 10, replay="compact",
                               graph_steps=graph_steps, fused_insert=fused)
    a, b = mk(False), mk(True)
    assert not a.fused_insert and b.fused_insert
    for ro in (a, b):
        np.random.seed(3)
        ro.reset()
        ro.run(27)  # wraps the 10-step ring twice and crosses three episode ends
    torch.cuda.synchronize()
    assert (a.buff.index, a.buff.count, a.buff.steps_total) == (b.buff.index, b.buff.count, b.buff.steps_total)
    for name in COMPACT_FIELDS:
        assert torch.equal(getattr(a.buff, name), getattr(b.buff, name)), name
    assert b.buff.episode_done.any() and b.buff.reward.abs().sum() > 0 and b.buff.action.to(torch.int32).sum() > 0


@pytest.mark.parametrize("math", ["bf16x3", "fp32"])
def test_compact_ring_rebuilds_the_dense_transition(math):
    """SURVEY 8f-3: the compact ring (env records + NetMon state, 23 kB instead of 141 kB per transition at config 2)
    must hand the learner the SAME TransitionBatch as the reference's dense ring: two runs from one seed, one per
    format, sampled with the same index streams (single transitions, then 6-step sequences) -- all 17 fields
    bit-identical, including the graph-observation tails the compact ring recomputes with NetMon."""
    from graph_marl_b200.replaybuffer import TransitionBatch
    from graph_marl_b200.rollout import Rollout

    cfg = dict(n_nodes=20, n_data=20, topo_seed=476, random_topology=True, n_topologies=5, congestion=True, K=2, rnn="lstm",
               H=64, enc=(96, 64), dqn=(64, 32), episode_steps=9)
    mk = lambda fmt, **kw: Rollout(cfg, num_envs=24, math=math, seed=13, replay_capacity=24 * 12, replay=fmt, **kw)
    runs = []
    for fmt, kw in (("dense", {}), ("compact", dict(state_ring=False)), ("compact", dict(device_sampler=True))):
        ro = mk(fmt, **kw)
        np.random.seed(2)
        ro.reset()
        ro.run(22)  # crosses two episode ends: first steps (zero NetMon state), episode_done flags, new topologies
        runs.append(ro)
    d, c, cd = runs
    assert c.buff.bytes_per_transition() * 5 < sum(getattr(d.buff, f)[0].numel() * getattr(d.buff, f).element_size()
                                                  for f in TransitionBatch._fields if f != "idx")
    assert (d.buff.index, d.buff.count) == (c.buff.index, c.buff.count) == (cd.buff.index, cd.buff.count)
    for seq in (0, 6):
        bd = list(d.buff.get_batch(16, "cuda", sequence_length=seq))
        bc = list(c.buff.get_batch(16, "cuda", sequence_length=seq))
        bx = list(cd.buff.get_batch(16, "cuda", sequence_length=seq))
        assert len(bd) == len(bc) == len(bx) == max(seq, 1)
        for x, y, z in zip(bd, bc, bx):
            assert np.array_equal(x.idx, y.idx) and np.array_equal(x.idx, z.idx.cpu().numpy())  # device PCG64 == numpy
            for f in TransitionBatch._fields[1:]:
                u, v, w = getattr(x, f), getattr(y, f), getattr(z, f)
                assert u.dtype == v.dtype and u.shape == v.shape, f
                assert torch.equal(u, v) and torch.equal(u, w), (f, seq)
    assert bd[0].obs.shape == (16, 20, 130 + 4 * 64)


def test_eager_tail_then_graph_unit_keeps_the_ring_consistent():
    """ADVICE r1: run(k) with k % graph_steps != 0 interleaves eager steps (insert on the side stream, reading the ring
    index counter and the static tensors) with graph units that rewrite both: at a batch where the insert takes real
    time the ring must still equal the eager run's."""
    a, b = _mk(0, B=2048), _mk(5, B=2048)
    for _ in range(4):
        a.run(7)
        b.run(7)
    torch.cuda.synchronize()
    assert b._graphs
    assert (a.buff.index, a.buff.count) == (b.buff.index, b.buff.count)
    for name in DENSE_FIELDS + ("adj", "node_agent_matrix"):
        assert torch.equal(getattr(a.buff, name), getattr(b.buff, name)), name


def test_graph_units_respect_episode_boundaries():
    from graph_marl_b200.rollout import Rollout

    cfg = dict(n_nodes=20, n_data=20, topo_seed=923430603, congestion=True, K=1, rnn="lstm", H=64, enc=(64,), dqn=(64,),
               episode_steps=12)
    mk = lambda g: Rollout(cfg, num_envs=33, math="bf16x3", seed=3, replay_capacity=33 * 8, graph_steps=g, replay="dense")
    a, b = mk(0), mk(4)
    a.reset(), b.reset()
    a.run(31)
    b.run(31)  # crosses two episode ends (reset + first/last steps run eagerly)
    torch.cuda.synchronize()
    sa, sb = a.base_env.get_state(), b.base_env.get_state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    assert torch.equal(a.env.current_netmon_state, b.env.current_netmon_state)
    assert a.episode_step == b.episode_step
    for name in ("obs", "node_aux", "node_adj", "reward", "node_state"):  # units captured before a reset stay valid after it
        assert torch.equal(getattr(a.buff, name), getattr(b.buff, name)), name


@pytest.mark.parametrize("rnn,H,enc", [("lstm", 64, (64,)), ("lnlstm", 128, (64, 128))])
def test_random_topology_pool_rollout_graph_equals_eager(rnn, H, enc):
    """BASELINE config 3 shape: every env draws a topology from a pool at each episode start (the pool and the
    per-env index tensor keep their device addresses, so captured units stay valid across resets)."""
    from graph_marl_b200.rollout import Rollout

    cfg = dict(n_nodes=20, n_data=20, topo_seed=476, random_topology=True, n_topologies=7, congestion=False, K=1, rnn=rnn,
               H=H, enc=enc, dqn=(64,), episode_steps=9)
    mk = lambda g: Rollout(cfg, num_envs=40, math="bf16x3", seed=11, replay_capacity=40 * 8, graph_steps=g, replay="dense")
    a, b = mk(0), mk(3)
    # the topology draws come from the global numpy stream (network.py:229-238): give both runs the same one
    for ro in (a, b):
        np.random.seed(5)
        ro.reset()
    assert a.base_env._pool.T == 7 and len(set(a.base_env._topo_index.cpu().tolist())) > 1
    assert torch.equal(a.base_env._topo_index, b.base_env._topo_index)
    for ro in (a, b):
        np.random.seed(6)
        ro.run(25)
    torch.cuda.synchronize()
    assert b._graphs, "no CUDA graph unit was captured"
    assert torch.equal(a.base_env._topo_index, b.base_env._topo_index)
    sa, sb = a.base_env.get_state(), b.base_env.get_state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    assert torch.equal(a.obs[0], b.obs[0]) and torch.equal(a.obs[1], b.obs[1])
    assert torch.equal(a.env.current_netmon_state, b.env.current_netmon_state)
    bad = []
    for name in ("obs", "next_obs", "node_adj", "node_aux", "reward", "node_state", "node_obs", "action"):
        x, y = getattr(a.buff, name), getattr(b.buff, name)
        if not torch.equal(x, y):
            d = (x.float() - y.float()).abs().reshape(x.shape[0], -1).max(dim=1)[0]
            bad.append((name, int((d > 0).sum()), float(d.max()), (d > 0).nonzero().flatten()[:8].tolist()))
    assert not bad, bad


def test_bench_dump_outputs_are_the_last_step(tmp_path):
    """bench.py --dump-outputs: after eager steps the arrays are what the last step handed its caller (the graph
    observation, kept only tile-packed, unpacks to the rows the ring's rebuild of the transition computes in fp32, up to
    the bf16 hi/lo split; the Q-values are the DQN's on the next observations).  After the same steps run as replayed
    CUDA-graph units -- the path bench.py times, where the ring index and the carried tensors come from the replay
    bookkeeping -- the dump is the same, array for array."""
    import bench
    from graph_marl_b200.model import PackedRows
    from oracle import netmon_oracle as NO

    a = _mk(0, replay="compact", B=40)
    a.run(9)
    reward, done, _ = a.step()
    b = _mk(5, replay="compact", B=40)
    b.run(10)
    assert b._graphs and not a._graphs
    dumps = []
    for ro, sub in ((a, "eager"), (b, "graph")):
        bench.dump_outputs(ro, str(tmp_path / sub))
        dumps.append({p.stem: np.load(p) for p in (tmp_path / sub).iterdir()})
    d, dg = dumps
    assert sorted(d) == sorted(dg) == sorted(("obs_agent", "obs_graph", "adj", "netmon_state", "action", "reward", "done", "q_values"))
    assert all(v.dtype == np.float32 and v.shape[0] == a.B for v in d.values())  # 40 envs fit: no sampling
    assert np.array_equal(d["reward"], reward.cpu().numpy()) and np.array_equal(d["done"], done.float().cpu().numpy())
    assert np.array_equal(d["obs_agent"], a.obs[0].cpu().numpy()) and np.array_equal(d["adj"], a.adj.float().cpu().numpy())
    assert np.array_equal(d["netmon_state"], a.env.current_netmon_state.cpu().numpy())
    assert isinstance(a.obs[1], PackedRows)
    tb = a.buff._get_transition_batch((a.buff.index - a.B + np.arange(a.B)) % a.buff.buffer_size, "cuda")
    assert np.array_equal(d["action"], tb.action.float().cpu().numpy())
    tail = tb.next_obs[..., a.sizes["Da"]:].cpu().numpy()
    assert d["obs_graph"].shape == tail.shape and np.abs(tail).max() > 0
    assert np.abs(d["obs_graph"] - tail).max() <= 2.0 ** -14 * np.abs(tail).max()
    w_dq = {k: v.detach().cpu().numpy() for k, v in a.model.state_dict().items()}
    q_ref = NO.dqn_forward(w_dq, np.concatenate([d["obs_agent"], tail], -1))
    assert d["q_values"].shape == (a.B, 20, 4) and np.abs(d["q_values"] - q_ref).max() < 1e-3
    for name in d:
        assert np.array_equal(d[name], dg[name]), name
