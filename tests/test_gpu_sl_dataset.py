"""The device-built supervised shortest-path dataset (graph_marl_b200.sl_dataset, BASELINE config 5) and the pool's
next-hop tables (gm_topology_next_hops) behind its labels.

* build_sl_dataset reproduces tests/golden/sl_netmon.npz (the unmodified reference's sl.py dataset) bit for bit;
* next_hop equals the first hops of networkx's shortest paths on the 1000 evaluation graphs, on fresh N = 20, 200, 4
  and 6 topologies, with pairs whose equal-weight first hops make networkx's tie-breaking decide counted;
* for each way Network.reset() picks a seed, the builder gives what S compat resets + get_sl_sample labels give, and
  leaves the global numpy stream and the Network as those resets do;
* an invalid provided seed raises as the host path does; the pool refreshes its next-hop cache only once built.
"""
import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu


def _sample_ref(net):
    """get_sl_sample's labels and targets (sl.py:174-219) from the Network API, plus the full next-hop table."""
    N = net.n_nodes
    nh = np.zeros((N, N), np.int8)
    for v in range(N):
        hops = [net.edges[e].get_other_node(v) for e in net.nodes[v].edges]
        for t in range(N):
            if t != v:
                nh[v, t] = hops.index(net.shortest_paths[v][t][1]) + 1
    return nh, np.asarray(net.shortest_paths_weights)


def _ties(net):
    """(v, t) pairs with two or more first hops on a shortest path: networkx's tie-breaking picks between them."""
    d, N, n = np.asarray(net.shortest_paths_weights), net.n_nodes, 0
    for v in range(N):
        via = [(net.edges[e].length, net.edges[e].get_other_node(v)) for e in net.nodes[v].edges]
        for t in range(N):
            n += t != v and sum(w + d[u, t] == d[v, t] for w, u in via) > 1
    return n


def _host_net(N, seed, reseed):
    from graph_marl_b200.env.network import Network, generate_tables

    net = Network(N)
    net._install(generate_tables(N, seed, allow_reseed=reseed))
    return net


def _check_next_hops(N, seeds, reseed):
    """Generate `seeds` into a pool, compare next_hop with networkx on the host; returns the tie count."""
    import torch
    from graph_marl_b200.env.routing import TopologyPool

    seeds = np.asarray(seeds, np.int64)
    pool = TopologyPool.slots(len(seeds), N, "cuda")
    used, _ = pool.generate(seeds, torch.arange(len(seeds), dtype=torch.int32, device="cuda"))
    if not reseed:
        assert np.array_equal(used, seeds)
    nh = pool.next_hop.cpu().numpy()
    assert nh.shape == (len(seeds), N, N) and nh.dtype == np.int8
    ties = 0
    for i, s in enumerate(seeds):
        net = _host_net(N, int(s), reseed)
        assert net.current_topology_seed == int(used[i])
        ref, _ = _sample_ref(net)
        assert np.array_equal(nh[i], ref), (N, int(s))
        ties += _ties(net)
    return ties


def test_fixture_dataset_bit_for_bit():
    """sl.py's test split: Network(20, sequential EVAL_SEEDS) after np.random.seed(5), 32 samples."""
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.sl_dataset import FIELDS, build_sl_dataset

    G = load_golden("sl_netmon")
    np.random.seed(5)
    net = Network(20, random_topology=True, sequential_topology_seeds=True, provided_seeds=EVAL_SEEDS)
    ds = build_sl_dataset(net, 32)
    for k in FIELDS:
        got = ds[k].cpu().numpy()
        assert got.dtype == G[k].dtype and got.shape == G[k].shape, k
        assert np.array_equal(got, G[k]), k


def test_next_hops_on_the_evaluation_graphs():
    from graph_marl_b200.env.constants import EVAL_SEEDS

    assert _check_next_hops(20, EVAL_SEEDS, reseed=False) > 0


def test_next_hops_on_fresh_topologies():
    rng = np.random.RandomState(17)
    ties = _check_next_hops(20, rng.randint(2**31 - 1, size=2000), reseed=True)
    assert ties > 0
    assert _check_next_hops(200, rng.randint(2**31 - 1, size=100), reseed=True) > 0
    for N in (4, 6):
        _check_next_hops(N, rng.randint(2**31 - 1, size=200), reseed=True)


# ---- against the compat loop ---------------------------------------------------------------------
def _compat(net, S, A):
    """S compat resets of Routing(net, A, INDEPENDENT) and get_sl_sample's outputs, as sl.py builds its dataset."""
    from graph_marl_b200.env.routing import Routing

    env = Routing(net, A, 1)
    out = {k: [] for k in ("node_obs", "node_adj", "labels", "targets", "targets_all", "seeds")}
    for _ in range(S):
        env.reset()
        nh, apsp = _sample_ref(net)
        out["node_obs"].append(env.get_node_observation())
        out["node_adj"].append(np.asarray(env.get_nodes_adjacency(), np.int8))
        out["labels"].append(nh[:, 0])
        out["targets"].append(apsp[:, 0].astype(np.int32))
        out["targets_all"].append(apsp.astype(np.int32))
        out["seeds"].append(net.current_topology_seed)
    return {k: np.asarray(np.stack(v) if k != "seeds" else np.array(v, np.int64)) for k, v in out.items()}


def _net_attrs(net):
    return dict(current=net.current_topology_seed, sampled=list(net.sampled_topology_seeds),
                index=net.sequential_topology_index, reps=net.repetitions, adj=net.adj_matrix.tolist(),
                nodes=[(n.x, n.y, n.neighbors, n.edges) for n in net.nodes],
                edges=[(e.start, e.end, e.length) for e in net.edges], apsp=np.asarray(net.shortest_paths_weights).tolist())


def _against_compat(make_net, S, A, chunk, seed=23):
    from graph_marl_b200.sl_dataset import FIELDS, build_sl_dataset

    np.random.seed(seed)
    ref_net = make_net()
    ref = _compat(ref_net, S, A)
    ref_state = np.random.get_state()
    np.random.seed(seed)
    net = make_net()
    ds = build_sl_dataset(net, S, n_data=A, chunk=chunk)
    for k in FIELDS:
        got = ds[k].cpu().numpy()
        assert got.dtype == ref[k].dtype and got.shape == ref[k].shape, k
        assert np.array_equal(got, ref[k]), k
    st = np.random.get_state()
    assert st[0] == ref_state[0] and np.array_equal(st[1], ref_state[1]) and st[2:] == ref_state[2:]
    assert _net_attrs(net) == _net_attrs(ref_net)
    return ref["seeds"]


def test_against_compat_sequential_provided_seeds():
    from graph_marl_b200.env.constants import EVAL_SEEDS
    from graph_marl_b200.env.network import Network

    seeds = _against_compat(lambda: Network(20, random_topology=True, sequential_topology_seeds=True,
                                            provided_seeds=EVAL_SEEDS[:250]), 300, 20, 128)
    assert list(seeds[250:]) == list(EVAL_SEEDS[:50])  # wrapped around the list


def test_against_compat_seed_list():
    from graph_marl_b200.env.network import Network

    _against_compat(lambda: Network(20, random_topology=True, n_random_seeds=40), 300, 20, 128)


def test_against_compat_fresh_seeds_with_exclusions():
    from graph_marl_b200.env.network import Network

    np.random.seed(23)  # the seeds the stream draws next without exclusions
    probe = _compat(Network(20, random_topology=True), 300, 20)["seeds"]
    excluded = [int(probe[0]), int(probe[129]), int(probe[299])]
    seeds = _against_compat(lambda: Network(20, random_topology=True, excluded_seeds=excluded), 300, 20, 128)
    assert not set(seeds.tolist()) & set(excluded) and not np.array_equal(seeds, probe)  # the exclusions were hit


def test_against_compat_n200_a100_uneven_chunks():
    from graph_marl_b200.env.network import Network

    _against_compat(lambda: Network(200, random_topology=True), 7, 100, 3)


def test_invalid_provided_seed_raises_like_the_host_path():
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.sl_dataset import build_sl_dataset

    valid = [476, 923430603]
    host = Network(20, random_topology=True, sequential_topology_seeds=True, provided_seeds=valid + [4])
    host.reset(), host.reset()
    with pytest.raises(AssertionError, match="Provided seed 4 is invalid."):
        host.reset()
    net = Network(20, random_topology=True, sequential_topology_seeds=True, provided_seeds=valid + [4])
    with pytest.raises(AssertionError, match="Provided seed 4 is invalid."):
        build_sl_dataset(net, 5, chunk=2)


def test_pool_next_hop_cache():
    """generate() refreshes a built next_hop cache for the regenerated slots and launches nothing extra without one."""
    import torch
    import graph_marl_b200._lib as L
    from graph_marl_b200.env.routing import TopologyPool

    lib = L.lib()
    slot = torch.arange(8, dtype=torch.int32, device="cuda")
    pool = TopologyPool.slots(8, 20, "cuda")
    n0 = lib.gm_kernel_launch_count()
    pool.generate(np.arange(100, 108), slot)
    plain = lib.gm_kernel_launch_count() - n0
    assert getattr(pool, "_next_hop", None) is None
    before = pool.next_hop.clone()
    n0 = lib.gm_kernel_launch_count()
    pool.generate(np.arange(200, 204), slot[4:])
    assert lib.gm_kernel_launch_count() - n0 == plain + 1
    now = pool.next_hop
    assert torch.equal(now[:4], before[:4]) and not torch.equal(now[4:], before[4:])
    assert torch.equal(now, pool.next_hops(slot))
