"""GPU parity of the batched Routing kernel (through the C ABI) against (1) trajectories
recorded from the reference and (2) the C oracle on seeded random batches.  Integer state,
fp64 loads/sizes and every observation field must be BIT-EXACT."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from helpers import cfg_from_golden, draws_for_step, topo_from_golden

pytestmark = pytest.mark.gpu

CASES = ["routing_A_seed923430603_cong", "routing_B_nocong", "routing_C_mask", "routing_D_ttl",
         "routing_E_a35_nocong_mask_ttl", "routing_F_n200", "routing_G_var2", "routing_H_var3", "routing_I_evalinfo"]


def _make_env(g, c, num_envs=1, batched=None):
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing

    net = Network(c["n_nodes"], random_topology=False, topology_init_seed=c["topo_seed"])
    return Routing(net, c["n_data"], c["env_var"], k=c["k"], enable_congestion=c["congestion"],
                   enable_action_mask=c["mask"], ttl=c["ttl"], num_envs=num_envs, batched=batched)


def _check_state(env, g, t):
    s = env.get_state()
    for k in ("now", "target", "edge", "time", "ttl", "spw", "start", "size", "load", "agent_steps", "visited"):
        assert np.array_equal(s[k][0], g["s_" + k][t]), (k, t)


@pytest.mark.parametrize("case", CASES)
def test_golden_trajectory(case):
    g = load_golden(case)
    c = cfg_from_golden(g)
    A = c["n_data"]
    env = _make_env(g, c)
    env.set_eval_info(c["eval_info"])
    ds, dt, dz, n = draws_for_step(g, -1, A)
    env.set_draws(ds, dt, dz)
    obs, adj = env.reset()
    assert np.array_equal(obs, g["obs"][0]) and obs.dtype == np.float32
    assert np.array_equal(adj, g["adj"][0]) and adj.dtype == np.int8
    assert np.array_equal(env.get_node_observation(), g["node_obs"][0])
    assert np.array_equal(env.get_node_agent_matrix(), g["node_agent"][0])
    assert np.array_equal(env.get_nodes_adjacency().shape, (c["n_nodes"], c["n_nodes"]))
    _check_state(env, g, 0)
    n_dense = g["obs"].shape[0]
    for t in range(c["steps"]):
        ds, dt, dz, n = draws_for_step(g, t, A)
        env.set_draws(ds, dt, dz)
        obs, adj, reward, done, info = env.step(g["actions"][t])
        assert np.array_equal(reward, g["reward"][t]) and reward.dtype == np.float32, t
        assert np.array_equal(done, g["done"][t].astype(bool)), t
        assert [float(info["looped"]), int(info["throughput"]), int(info["dropped"]), int(info["blocked"])] == \
            g["info"][t].tolist(), t
        assert info["delays"] == [float(x) for x in g["delays"][t][g["done"][t] == 1]]
        assert info["spr"] == [float(x) for x in g["spr"][t][g["arrived"][t] == 1]]
        assert int(env._out["n_resets"][0]) == n
        if c["eval_info"]:  # routing.py:414-441
            extra = [info["total_edge_load"], info["occupied_edges"], info["packets_on_edges"], info["total_packet_size"]]
            assert np.array_equal(np.array(extra, dtype=np.float64), g["eval_extra"][t]), t
            assert info["packet_sizes"] == g["s_size"][t].tolist()  # sizes before this step's respawns
        _check_state(env, g, t + 1)
        if c["mask"]:
            assert np.array_equal(env.action_mask, g["s_mask"][t + 1].astype(bool))
        if t + 1 < n_dense:
            assert np.array_equal(obs, g["obs"][t + 1]), t
            assert np.array_equal(adj, g["adj"][t + 1]), t
            assert np.array_equal(env.get_node_observation(), g["node_obs"][t + 1]), t
            assert np.array_equal(env.get_node_agent_matrix(), g["node_agent"][t + 1]), t
    if c["eval_info"]:
        assert np.array_equal(env.sum_packets_per_node, g["sum_packets_per_node"])
        assert np.array_equal(env.sum_packets_per_edge, g["sum_packets_per_edge"])
        assert sum(len(v) for v in env.distance_map.values()) == int(g["arrived"].sum())
    fi = env.get_final_info({"delays": []})
    assert fi["delays"] == g["final_delays"].tolist()
    assert np.array_equal(env.get_node_aux(), g["node_aux"])


def test_compat_mode_consumes_global_numpy_stream_like_the_reference():
    """No set_draws: reset()/step() must pull their draws from np.random in the reference's
    order and leave the stream where the reference leaves it."""
    from oracle import oracle as O

    g = load_golden("routing_A_seed923430603_cong")
    c = cfg_from_golden(g)
    env = _make_env(g, c)
    np.random.seed(0)
    obs, adj = env.reset()
    assert np.array_equal(obs, g["obs"][0])
    for t in range(60):
        obs, adj, reward, done, info = env.step(g["actions"][t])
        assert np.array_equal(obs, g["obs"][t + 1]), t
        assert np.array_equal(reward, g["reward"][t]), t
    n_triples = int((g["draw_t"] < 60).sum())
    ref = O.MT19937(0)
    for _ in range(n_triples):
        ref.randint(20), ref.randint(20), ref.random()
    assert np.random.random() == ref.random()


def _random_batch(B, A, N, steps, seed):
    rng = np.random.default_rng(seed)
    return dict(
        reset=(rng.integers(0, N, (B, A)).astype(np.int32), rng.integers(0, N, (B, A)).astype(np.int32),
               rng.random((B, A))),
        steps=[(rng.integers(0, 4, (B, A)).astype(np.int32), rng.integers(0, N, (B, A)).astype(np.int32),
                rng.integers(0, N, (B, A)).astype(np.int32), rng.random((B, A))) for _ in range(steps)])


@pytest.mark.parametrize("cfg", [
    dict(N=20, A=20, B=257, steps=40, cong=True, mask=False, ttl=0, seed=923430603),
    dict(N=20, A=45, B=64, steps=40, cong=True, mask=True, ttl=15, seed=923430603),
    dict(N=200, A=100, B=9, steps=25, cong=True, mask=False, ttl=0, seed=476),
])
def test_batched_against_oracle(cfg):
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from oracle import oracle as O

    N, A, B = cfg["N"], cfg["A"], cfg["B"]
    net = Network(N, random_topology=False, topology_init_seed=cfg["seed"])
    env = Routing(net, A, 1, enable_congestion=cfg["cong"], enable_action_mask=cfg["mask"], ttl=cfg["ttl"],
                  num_envs=B)
    topo = O.generate_topology(N, seed=cfg["seed"])
    orc = O.RoutingOracle(topo, A, enable_congestion=cfg["cong"], enable_action_mask=cfg["mask"], ttl=cfg["ttl"],
                          num_envs=B, threads=4)
    data = _random_batch(B, A, N, cfg["steps"], 5)
    env.set_draws(*data["reset"])
    obs, adj = env.reset()
    orc.reset(*data["reset"])

    def compare(t):
        o = orc.observe()
        assert np.array_equal(env._out["obs"].cpu().numpy(), o["obs"]), t
        assert np.array_equal(env._out["adj"].cpu().numpy(), o["adj"]), t
        assert np.array_equal(env._out["node_obs"].cpu().numpy(), o["node_obs"]), t
        assert np.array_equal(env._out["node_agent"].cpu().numpy(), o["node_agent"]), t
        assert np.array_equal(env._out["agent_node"].cpu().numpy(), orc.now), t
        # the sparse form of the node rows scatters back to exactly the dense rows: 12 fixed slots of (column, value), or
        # (small pools) six indices into the dictionary env.node_static_rows -- one row per (topology, node) for the
        # constant part, five unit rows for the dynamic fields
        sp = env._out["node_sparse"].cpu().numpy()
        dense = np.zeros_like(o["node_obs"])
        bi, ji = np.meshgrid(np.arange(B), np.arange(N), indexing="ij")
        stat = None if env.node_static_rows is None else env.node_static_rows.cpu().numpy()
        assert env.node_obs_nnz == (12 if stat is None else 6)
        for k in range(12):
            col, val = sp[..., k], sp[..., 12 + k].view(np.float32)
            if stat is not None:
                assert (col < stat.shape[0]).all() and (k < 6 or (val == 0).all())
                assert k != 0 or ((val == 1).all() and (col < stat.shape[0] - 5).all())
                dense += stat[col] * val[..., None]
            else:
                np.add.at(dense, (bi, ji, col), val)
        assert np.array_equal(dense, o["node_obs"]), t
        s = env.get_state()
        for k, ref in (("now", orc.now), ("target", orc.target), ("edge", orc.edge), ("time", orc.time),
                       ("ttl", orc.ttl_left), ("spw", orc.spw), ("size", orc.size), ("load", orc.load),
                       ("agent_steps", orc.agent_steps), ("visited", orc.visited)):
            assert np.array_equal(s[k], ref), (k, t)
        if cfg["mask"]:
            assert np.array_equal(s["mask"], orc.mask), t

    compare(-1)
    for t, (act, ds, dt, dz) in enumerate(data["steps"]):
        env.set_draws(ds, dt, dz)
        obs, adj, reward, done, info = env.step(torch.from_numpy(act).cuda())
        r = orc.step(act, ds, dt, dz)
        assert np.array_equal(reward.cpu().numpy(), r["reward"]), t
        assert np.array_equal(done.cpu().numpy(), r["done"].astype(bool)), t
        assert np.array_equal(info["delays"].cpu().numpy(), r["delays"]), t
        assert np.array_equal(info["arrived"].cpu().numpy(), r["arrived"]), t
        assert np.array_equal(info["spr"].cpu().numpy(), r["spr"]), t
        got = torch.stack([info["looped"], info["throughput"], info["dropped"], info["blocked"]], 1).cpu().numpy()
        assert np.array_equal(got, r["info"]), t
        assert np.array_equal(env._out["n_resets"].cpu().numpy(), r["n_resets"]), t
        compare(t)


def test_full_size_properties_and_philox_draws():
    """BASELINE config 2 size (4096 envs): size-independent invariants of the device-side
    Philox run + observe() idempotence (the oracle comparison at this size is the next test)."""
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from oracle import oracle as O

    N = A = 20
    B = 4096
    net = Network(N, random_topology=False, topology_init_seed=923430603)
    env = Routing(net, A, 1, num_envs=B, seed=11)
    obs, adj = env.reset()
    g = torch.Generator(device="cuda").manual_seed(3)
    s0 = env.get_state()
    assert (s0["size"] >= 0).all() and (s0["size"] < 1).all() and len(np.unique(s0["size"])) > B * A * 0.99
    assert np.bincount(s0["now"].ravel(), minlength=N).min() > 0.8 * B * A / N  # uniform spawn
    for t in range(30):
        act = torch.randint(0, 4, (B, A), device="cuda", generator=g, dtype=torch.int32)
        obs, adj, reward, done, info = env.step(act)
    s = env.get_state()
    # every agent row: exactly one 'now' and one 'target' hot, 3 neighbour one-hots
    o = obs.cpu().numpy()
    assert (o[:, :, :N].sum(-1) == 1).all() and (o[:, :, N:2 * N].sum(-1) == 1).all()
    assert np.array_equal(o[:, :, :N].argmax(-1), s["now"])
    assert np.array_equal(o[:, :, 3 * N + 3], np.broadcast_to(np.arange(A, dtype=np.float32), (B, A)))
    # loads = sum of in-flight packet sizes per edge (fp64, up to rounding) and never above capacity
    load = np.zeros_like(s["load"])
    for b in range(0, B, 97):
        for i in range(A):
            if s["edge"][b, i] >= 0:
                load[b, s["edge"][b, i]] += s["size"][b, i]
        assert np.allclose(load[b], s["load"][b], atol=1e-12)
    assert s["load"].max() <= 1.0 + 1e-12 and s["load"].min() > -1e-12
    # observe() rebuilds identical observations from the stored state
    o2 = env.observe()
    assert torch.equal(o2["obs"], obs) and torch.equal(o2["adj"], adj)
    nam = env._out["node_agent"].cpu().numpy()
    assert (nam.sum(1) == 1).all()
    assert np.array_equal(nam.argmax(1), s["now"])


def test_full_size_spot_check_against_oracle():
    """BASELINE config 2 size (4096 envs in ONE launch) with host-supplied draws: 16 envs spread over the batch
    (first / last warp of a CTA, first / last CTA) are replayed on the C oracle with the same draws and actions;
    every output and every state field of those envs must be bit-identical on all 40 steps."""
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from oracle import oracle as O

    N = A = 20
    B, steps = 4096, 40
    pick = np.array([0, 1, 3, 4, 127, 128, 1023, 1024, 2047, 2048, 2049, 3000, 3583, 4092, 4094, 4095])
    net = Network(N, random_topology=False, topology_init_seed=923430603)
    env = Routing(net, A, 1, num_envs=B, seed=3)
    orc = O.RoutingOracle(O.generate_topology(N, seed=923430603), A, num_envs=len(pick), threads=2)
    data = _random_batch(B, A, N, steps, 19)
    env.set_draws(*data["reset"])
    env.reset()
    orc.reset(*(d[pick] for d in data["reset"]))
    sel = torch.from_numpy(pick).cuda()

    def compare(t):
        o = orc.observe()
        for k in ("obs", "adj", "node_obs", "node_agent"):
            assert np.array_equal(env._out[k][sel].cpu().numpy(), o[k]), (k, t)
        s = env.get_state()
        for k, ref in (("now", orc.now), ("target", orc.target), ("edge", orc.edge), ("time", orc.time),
                       ("spw", orc.spw), ("size", orc.size), ("load", orc.load), ("agent_steps", orc.agent_steps),
                       ("visited", orc.visited)):
            assert np.array_equal(s[k][pick], ref), (k, t)

    compare(-1)
    for t, (act, ds, dt, dz) in enumerate(data["steps"]):
        env.set_draws(ds, dt, dz)
        obs, adj, reward, done, info = env.step(torch.from_numpy(act).cuda())
        r = orc.step(act[pick], ds[pick], dt[pick], dz[pick])
        assert np.array_equal(reward[sel].cpu().numpy(), r["reward"]), t
        assert np.array_equal(done[sel].cpu().numpy(), r["done"].astype(bool)), t
        assert np.array_equal(info["delays"][sel].cpu().numpy(), r["delays"]), t
        assert np.array_equal(env._out["n_resets"][sel].cpu().numpy(), r["n_resets"]), t
        compare(t)


def test_simple_environment_golden():
    """SimpleEnvironment (BASELINE config 1) through gm_simple_step: observations, node tables and
    rewards of 12 recorded episodes per (env_var, random_topology), compat mode; then a batched run
    whose rewards are the scores of the chosen neighbours."""
    from graph_marl_b200.env.simple_environment import SimpleEnvironment

    g = load_golden("simple_env")
    for var in (1, 3):
        for rt in (0, 1):
            tag = f"v{var}_rt{rt}_"
            np.random.seed(10 + var + rt)
            env = SimpleEnvironment(env_var=var, random_topology=rt)
            for ep in range(len(g[tag + "act"])):
                obs, adj = env.reset()
                assert np.array_equal(obs, g[tag + "obs"][ep]) and obs.dtype == np.float32
                assert np.array_equal(adj, np.eye(1, dtype=np.int8))
                assert np.array_equal(env.get_node_observation(), g[tag + "node_obs"][ep])
                assert np.array_equal(env.get_node_agent_matrix(), g[tag + "node_agent"][ep])
                assert np.array_equal(env.get_nodes_adjacency(), g[tag + "node_adj"][ep])
                obs2, adj2, rew, done, info = env.step([int(g[tag + "act"][ep])])
                assert done == [True] and np.array_equal(obs2, obs) and info == {}
                assert np.array_equal(rew.astype(np.float64), g[tag + "reward"][ep])
            assert np.random.random() == g[tag + "after"][0]
    np.random.seed(5)
    env = SimpleEnvironment(env_var=1, random_topology=1, num_envs=257)
    obs, adj = env.reset()
    act = torch.randint(0, 2, (257,), device="cuda", dtype=torch.int32)
    obs2, adj2, rew, done, info = env.step(act)
    assert obs2.shape == (257, 1, 1) and done.all() and rew.shape == (257, 1)
    a = act.cpu().numpy()
    for b, net in enumerate(env._host):
        t = net["start_edges"][a[b]]
        e = net["edges"][t]
        dst = e[1] if e[0] == net["start_node"] else e[0]
        assert rew[b, 0].item() == net["scores"][dst]
