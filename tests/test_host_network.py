"""Host-side product code (native topology generator + legacy RNG stream behind the
reference's Network API) against reference outputs in tests/golden.  No GPU needed."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from conftest import load_golden
from graph_marl_b200 import _lib
from graph_marl_b200.env.network import Network, generate_tables


def _mt(seed):
    st = np.zeros(_lib.GM_MT_STATE_WORDS, np.uint32)
    _lib.lib().gm_mt_seed(_lib.ptr(st), seed)
    return st


def test_library_exports_every_declared_symbol():
    import re, os
    hdr = open(os.path.join(os.path.dirname(_lib._HERE), "include", "graphmarl_b200.h")).read()
    declared = sorted(set(re.findall(r"GM_API [\w\s\*]+?(gm_\w+)\(", hdr)))
    assert declared == _lib.EXPORTS
    L = _lib.lib()
    for name in declared:
        assert hasattr(L, name), name
    assert L.gm_abi_version() == 6


def test_native_mt19937_matches_numpy_legacy_stream():
    g = load_golden("rng")
    L = _lib.lib()
    for i, s in enumerate(g["seeds"]):
        st = _mt(int(s))
        assert np.array_equal([L.gm_mt_random(_lib.ptr(st)) for _ in range(10)], g["random10"][i])
        assert np.array_equal([L.gm_mt_randint(_lib.ptr(st), 20) for _ in range(16)], g["randint20"][i])
        assert np.array_equal([L.gm_mt_randint(_lib.ptr(st), 200) for _ in range(16)], g["randint200"][i])
        ra = np.zeros(9, np.int32)
        ru = np.zeros(9, np.float64)
        L.gm_mt_policy_draws(_lib.ptr(st), 4, 9, _lib.ptr(ra), _lib.ptr(ru))  # randint(4,size) then rand(size)
        assert np.array_equal(ra, g["randint4_vec"][i]) and np.array_equal(ru, g["rand_vec"][i])
        assert np.array_equal([L.gm_mt_randint(_lib.ptr(st), 2**31 - 1) for _ in range(6)], g["randint_big"][i])
        assert [L.gm_mt_randint(_lib.ptr(st), 1) for _ in range(3)] == [0, 0, 0]
    # packet draws = (randint(N), randint(N), random()) triples, checked against live numpy
    st = _mt(77)
    np.random.seed(77)
    s_, t_, z_ = np.zeros(50, np.int32), np.zeros(50, np.int32), np.zeros(50, np.float64)
    L.gm_mt_packet_draws(_lib.ptr(st), 20, 50, _lib.ptr(s_), _lib.ptr(t_), _lib.ptr(z_))
    for i in range(50):
        assert (s_[i], t_[i], z_[i]) == (np.random.randint(20), np.random.randint(20), np.random.random())


def _check_net(net, edges, node_edges, apsp):
    assert [[e.start, e.end, e.length] for e in net.edges] == edges.tolist()
    assert [n.edges for n in net.nodes] == node_edges.tolist()
    assert np.array_equal(np.asarray(net.shortest_paths_weights), apsp)
    for i, nd in enumerate(net.nodes):
        assert [net.edges[e].get_other_node(i) for e in nd.edges] == sorted(nd.neighbors)


def test_native_pcg64_matches_numpy_generator_choice():
    """gm_pcg64_seed / gm_pcg64_choice (csrc/replay_sampler.cu) == np.random.default_rng(seed).choice(n, size): the
    index stream of ReplayBuffer.get_batch (replaybuffer.py:101, 111-130), incl. the buffered 32-bit halves, the
    Lemire rejection loop and n == 1 (consumes nothing); then the reference's own recorded index streams."""
    L = _lib.lib()
    for seed in (0, 1, 3, 12345, 2**32 + 5, 2**63 + 11, 923430603):
        st = np.zeros(_lib.GM_PCG64_STATE_WORDS, np.uint64)
        L.gm_pcg64_seed(_lib.ptr(st), seed)
        g = np.random.default_rng(seed)
        for n, size in ((10, 4), (1, 3), (4096 * 8, 32), (7, 5), (100000, 64), (3, 33), (2**32 - 1, 9), (2**31 + 7, 40)):
            out = np.zeros(size, np.int64)
            L.gm_pcg64_choice(_lib.ptr(st), n, size, _lib.ptr(out))
            assert np.array_equal(out, g.choice(n, size, replace=True)), (seed, n, size)
    from conftest import load_golden

    g = load_golden("replay")
    seed, cap = int(g["cfg"][0]), int(g["cfg"][1])
    st = np.zeros(_lib.GM_PCG64_STATE_WORDS, np.uint64)
    L.gm_pcg64_seed(_lib.ptr(st), seed)

    def batch(count, index, size, seq):
        out = np.zeros(size, np.int64)
        if seq <= 1:
            L.gm_pcg64_choice(_lib.ptr(st), count, size, _lib.ptr(out))
            return out[None]
        L.gm_pcg64_choice(_lib.ptr(st), count - seq, size, _lib.ptr(out))
        start = (index % count + out) % count
        return np.stack([(start + o) % count for o in range(seq)])

    assert np.array_equal(batch(10, 10, 4, 0)[0], g["idx_partial"])
    assert np.array_equal(batch(10, 10, 4, 3), g["idx_seq_partial"])
    index, count = [int(x) for x in g["final_index_count"]]
    assert np.array_equal(batch(count, index, 6, 0)[0], g["idx_full"])
    assert np.array_equal(batch(count, index, 5, 4), g["idx_seq_full"])


def test_fixed_seed_networks():
    g = load_golden("topology")
    for i, s in enumerate(g["fixed_seeds"]):
        np.random.seed(12345)
        before = np.random.get_state()[2]
        net = Network(20, random_topology=False, topology_init_seed=int(s))
        net.reset()
        assert net.repetitions == 1 and net.current_topology_seed == s
        _check_net(net, g["fixed_edges"][i], g["fixed_node_edges"][i], g["fixed_apsp"][i])
        assert [n.neighbors for n in net.nodes] == g["fixed_node_nbrs_creation"][i].tolist()
        assert np.random.get_state()[2] == before  # a 1-element seed list consumes nothing
    assert np.array_equal(net.adj_matrix, g["fixed_adj"]) and net.adj_matrix.dtype == np.int8


def test_all_eval_seeds_and_n200():
    g = load_golden("topology")
    for s, d in zip(g["eval_seeds"], g["eval_digest64"]):
        t = generate_tables(20, int(s))
        h = hashlib.sha256()
        h.update(np.ascontiguousarray(t["edges"][:, :3]).tobytes()), h.update(t["node_edges"].tobytes())
        h.update(t["apsp"].tobytes())
        assert np.frombuffer(h.digest()[:8], dtype=np.uint64)[0] == d, s
    net = Network(200, random_topology=False, topology_init_seed=476)
    net.reset()
    _check_net(net, g["n200_edges"], g["n200_node_edges"], g["n200_apsp"])
    with pytest.raises(AssertionError):
        Network(50, random_topology=False, topology_init_seed=476).reset()


def test_eval_seeds_constant_is_the_reference_list():
    """env/constants.py derives EVAL_SEEDS with the native generator instead of hard-coding it."""
    from graph_marl_b200.env.constants import EVAL_SEEDS

    g = load_golden("topology")
    state = np.random.get_state()[1].copy()
    assert EVAL_SEEDS == [int(x) for x in g["eval_seeds"]] and EVAL_SEEDS[350] == 923430603
    assert np.array_equal(np.random.get_state()[1], state)  # the caller's global stream is untouched


def test_random_topology_chain_pool_and_sequential():
    g = load_golden("topology")
    ex = [int(x) for x in g["eval_seeds"]]
    np.random.seed(7)
    net = Network(20, random_topology=True, excluded_seeds=ex)
    for i in range(len(g["chain_seed"])):
        net.reset()
        assert net.current_topology_seed == g["chain_seed"][i]
        assert net.repetitions == g["chain_rep"][i]
        assert [[e.start, e.end, e.length] for e in net.edges] == g["chain_edges"][i].tolist()
        assert np.random.get_state()[2] == g["chain_pos"][i]
    assert np.random.random() == g["chain_next_u"][0]
    np.random.seed(99)
    net = Network(20, random_topology=True, n_random_seeds=10, topology_init_seed=476, excluded_seeds=ex)
    assert net.seeds == g["pool_seeds"].tolist()
    picks = []
    for _ in range(len(g["pool_picks"])):
        net.reset()
        picks.append(net.current_topology_seed)
    assert picks == g["pool_picks"].tolist()
    net.seeds = ex
    net.sequential_topology_seeds = True
    seq = []
    for _ in range(4):
        net.reset()
        seq.append(net.current_topology_seed)
    assert seq == g["seq_picks"].tolist()


def test_networkx_views_and_weight_randomisation():
    net = Network(20, random_topology=False, topology_init_seed=923430603)
    net.reset()
    sp = net.shortest_paths
    assert sp[0][3] == [0, 3] and net.G.number_of_edges() == 30
    w0 = np.array(net.shortest_paths_weights).copy()
    np.random.seed(3)
    res = net.randomize_edge_weights("shuffle")
    assert len(res) == 3 and 0 <= res[2] <= 1
    import networkx as nx
    d = dict(nx.all_pairs_dijkstra_path_length(net.G))
    for a in range(20):
        for b in range(20):
            assert net.shortest_paths_weights[a][b] == d[a][b]
    assert not np.array_equal(w0, net.shortest_paths_weights)


def test_simple_environment_topology_draws_match_reference():
    """SimpleEnvironment._draw_network consumes the global legacy stream like the reference's
    _build_network (simple_environment.py:106-187): scores, edges, start node / edge order and the
    stream position after 12 episodes are those recorded from the reference."""
    from conftest import load_golden
    from graph_marl_b200.env.simple_environment import SimpleEnvironment

    g = load_golden("simple_env")
    for var in (1, 3):
        for rt in (0, 1):
            tag = f"v{var}_rt{rt}_"
            np.random.seed(10 + var + rt)
            env = SimpleEnvironment(env_var=var, random_topology=rt)
            for ep in range(len(g[tag + "act"])):
                net = env._draw_network()
                assert np.array_equal(net["scores"], g[tag + "scores"][ep])
                assert np.array_equal(net["edges"], g[tag + "edges"][ep])
                assert [net["start_node"]] + net["start_edges"].tolist() == g[tag + "start_edges"][ep].tolist()
            assert np.random.random() == g[tag + "after"][0]
