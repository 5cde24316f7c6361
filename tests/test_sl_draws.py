"""The native replay of sl.py's dataset draws (gm_mt_reset_draws behind sl_dataset.reset_draws) against the same calls
on numpy's legacy global stream: Network.pick_seed's seed choice, then A packet triples per compat Routing.reset(),
for each way Network.reset() picks a seed.  The produced seeds and tables and the final stream state must match.
No GPU needed."""
import numpy as np
import pytest

from graph_marl_b200.env.network import Network
from graph_marl_b200.sl_dataset import reset_draws


def _numpy_draws(net, n, A):
    """n Network.reset() seed choices + routing.py:130-135 packet triples on the global stream, as the host does."""
    N = net.n_nodes
    seeds, st, tg, sz = [], np.zeros((n, A), np.int32), np.zeros((n, A), np.int32), np.zeros((n, A))
    for s in range(n):
        idx = net.next_topology_seed_index(advance_index=not net.sequential_topology_seeds_frozen)
        seeds.append(net.pick_seed(net.seeds, idx, net.exclude_seeds)[0])
        for i in range(A):
            st[s, i] = np.random.randint(N)
            tg[s, i] = np.random.randint(N)
            sz[s, i] = np.random.random()
    return np.array(seeds, np.int64), st, tg, sz


def _state_equal(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


def _check(make_net, n, A, seed=11, chunks=(1,)):
    np.random.seed(seed)
    ref_net = make_net()
    ref = _numpy_draws(ref_net, n, A)
    ref_state = np.random.get_state()
    np.random.seed(seed)
    net = make_net()
    parts, lo = [], 0
    for c in chunks:
        parts.append(reset_draws(net, c, A))
        lo += c
    assert lo == n
    got = [np.concatenate([p[k] for p in parts]) for k in range(4)]
    for r, g in zip(ref, got):
        assert r.dtype == g.dtype and np.array_equal(r, g)
    assert _state_equal(np.random.get_state(), ref_state)
    assert net.sequential_topology_index == ref_net.sequential_topology_index
    return ref[0]


SEED_LIST = [101, 202, 303, 404, 505, 606, 707]


@pytest.mark.parametrize("chunks", [(40,), (16, 16, 7, 1)])
def test_sequential_provided_seeds_draw_only_packets(chunks):
    mk = lambda: Network(20, random_topology=True, sequential_topology_seeds=True, provided_seeds=SEED_LIST)
    seeds = _check(mk, 40, 20, chunks=chunks)
    assert list(seeds[:9]) == SEED_LIST + SEED_LIST[:2]


def test_frozen_sequential_seeds_repeat_one_seed():
    def mk():
        net = Network(20, random_topology=True, sequential_topology_seeds=True, provided_seeds=SEED_LIST)
        net.sequential_topology_index = 3
        net.freeze_sequential_topology_seeds()
        return net
    assert set(_check(mk, 12, 5, chunks=(5, 7)).tolist()) == {SEED_LIST[3]}


@pytest.mark.parametrize("seeds", [SEED_LIST, [4242]])
def test_seed_list_draws_np_random_choice(seeds):
    mk = lambda: Network(20, random_topology=True, provided_seeds=seeds)
    got = _check(mk, 50, 20, chunks=(25, 24, 1))
    assert set(got.tolist()) <= set(seeds)


@pytest.mark.parametrize("N,A", [(20, 20), (200, 100), (6, 3)])
def test_fresh_seeds(N, A):
    _check(lambda: Network(N, random_topology=True), 30, A, chunks=(10, 20))


def test_fresh_seeds_skip_excluded_ones():
    """The exclusion list holds seeds the stream is known to draw next (a random one is practically never drawn), so
    the redraw runs; the native replay must redraw exactly as pick_seed does."""
    N, A, n = 20, 20, 60
    np.random.seed(11)
    probe = Network(N, random_topology=True)
    drawn = _numpy_draws(probe, n, A)[0]
    excluded = [int(drawn[3]), int(drawn[17]), int(drawn[40]), 12345]
    mk = lambda: Network(N, random_topology=True, excluded_seeds=excluded)
    got = _check(mk, n, A, chunks=(7, 33, 20))
    assert not set(got.tolist()) & set(excluded)
    assert not np.array_equal(got, drawn)  # the exclusions were hit
