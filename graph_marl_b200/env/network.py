"""Topology management, mirrors the public surface of src/env/network.py of the reference.

Graph construction (network.py:122-213), the reseed loop (:215-272) and the shortest-path
weights (:274-290) run natively in libgraphmarl_b200 (csrc/host_topology.cpp); this class
keeps the reference's attribute names (`nodes[i].edges`, `edges[e].start/end/length`,
`shortest_paths_weights[i][j]`, `adj_matrix`, `seeds`, `current_topology_seed`, ...) and its
consumption of the global legacy `np.random` stream (:229-238), so a seeded run draws the
same topologies as the reference.
"""
import ctypes as C
from typing import List, Optional

import numpy as np

from .. import _lib


class Node:
    """Router: position, neighbour ids in creation order and incident edge ids (network.py:9-18)."""

    __slots__ = ("x", "y", "neighbors", "edges")

    def __init__(self, x, y):
        self.x, self.y = x, y
        self.neighbors, self.edges = [], []


class Edge:
    """Undirected link start-end with an integer length in steps (network.py:21-39)."""

    __slots__ = ("start", "end", "length")

    def __init__(self, start, end, length):
        self.start, self.end, self.length = start, end, length

    def get_other_node(self, node):
        ends = (self.start, self.end)
        if node not in ends:
            raise ValueError(f"Is neither start nor end of edge {self.start}-{self.end}: {node}")
        return ends[1] if node == ends[0] else ends[0]


def generate_tables(n_nodes, seed, allow_reseed=False, exclude=None):
    """One topology as flat int32 tables (host numpy). `seed` was chosen by the caller."""
    L = _lib.lib()
    N, E = n_nodes, 3 * n_nodes // 2
    t = dict(
        edges=np.zeros((E + 8, 4), np.int32), node_edges=np.zeros((N, 3), np.int32),
        node_nbrs=np.zeros((N, 3), np.int32), nbr_creation=np.zeros((N, 3), np.int32),
        apsp=np.zeros((N, N), np.int32), xy=np.zeros((N, 2), np.float64))
    rep = C.c_int32(0)
    used = C.c_int64(0)
    ex = None
    if exclude is not None and len(exclude):
        ex = np.ascontiguousarray(np.fromiter(exclude, dtype=np.int64))
    rc = L.gm_topology_generate(None, N, 2 if allow_reseed else 1, int(seed), _lib.ptr(ex),
                                0 if ex is None else ex.size, _lib.ptr(t["edges"]),
                                _lib.ptr(t["node_edges"]), _lib.ptr(t["node_nbrs"]),
                                _lib.ptr(t["nbr_creation"]), _lib.ptr(t["apsp"]), _lib.ptr(t["xy"]),
                                C.byref(rep), C.byref(used))
    if rc == -4:
        raise AssertionError(f"Provided seed {seed} is invalid.")
    _lib.check(rc)
    t["edges"] = np.ascontiguousarray(t["edges"][:E])
    t["seed"] = int(used.value)
    t["repetitions"] = int(rep.value)
    return t


def lists_from_tables(t):
    """NetMon adjacency lists of one topology: ascending ids incl. self, degree 4."""
    N = t["node_nbrs"].shape[0]
    full = np.concatenate([np.arange(N, dtype=np.int32)[:, None], t["node_nbrs"]], axis=1)
    full.sort(axis=1)
    return np.ascontiguousarray(full), np.full((N,), 4, np.int32)


class Network:
    """Network class that manages the creation of graphs (network.py:42-389)."""

    def __init__(
        self,
        n_nodes=20,
        random_topology=False,
        n_random_seeds=None,
        sequential_topology_seeds=False,
        topology_init_seed=476,
        excluded_seeds: Optional[List[int]] = None,
        provided_seeds: Optional[List[int]] = None,
    ):
        self.n_nodes = n_nodes
        self.nodes = []
        self.edges = []
        self.G_weight_key = "weight"
        self._G = None
        self._shortest_paths = None
        self.shortest_paths_weights = None
        self.adj_matrix = None
        self.tables = None
        self.repetitions = 0
        self.random_topology = random_topology
        self.current_topology_seed = None
        self.sampled_topology_seeds = []
        self.sequential_topology_seeds = sequential_topology_seeds
        self.sequential_topology_seeds_frozen = False
        self.sequential_topology_index = 0
        self.topology_init_seed = topology_init_seed
        self.exclude_seeds = None if excluded_seeds is None else set(excluded_seeds)
        self.provide_seeds = provided_seeds
        if provided_seeds is not None and len(provided_seeds) > 0:
            self.seeds = provided_seeds
        else:
            self.seeds = self.build_seed_list(random_topology, n_random_seeds, self.exclude_seeds)
        if self.exclude_seeds is not None:
            assert all([s not in self.exclude_seeds for s in self.seeds])

    # ---- seed management (network.py:100-120, 353-371) --------------------------------------
    def build_seed_list(self, random_topology, n_random_seeds, exclude_seeds=None):
        """Fixed topology: [init seed].  Random topologies: `n_random_seeds` distinct valid seeds drawn from
        a stream seeded with the init seed, leaving the caller's global stream untouched; [] = unrestricted."""
        if not random_topology:
            return [self.topology_init_seed]
        wanted = n_random_seeds or 0
        found = []
        if wanted > 0:
            saved = np.random.get_state()
            try:
                np.random.seed(self.topology_init_seed)
                while len(found) < wanted:
                    candidate = self._create_valid_network(seeds_exclude=exclude_seeds)
                    if candidate not in found:
                        found.append(candidate)
            finally:
                np.random.set_state(saved)
        return found

    def freeze_sequential_topology_seeds(self):
        self.sequential_topology_seeds_frozen = True

    def next_topology_seed_index(self, advance_index=True):
        seed_index = (self.sequential_topology_index
                      if len(self.seeds) > 1 and self.sequential_topology_seeds else None)
        if seed_index is not None and advance_index:
            self.sequential_topology_index = (seed_index + 1) % len(self.seeds)
        return seed_index

    def pick_seed(self, seed_list=None, seed_index=None, seeds_exclude=None):
        """Seed choice of _create_valid_network (network.py:228-238) on the global stream.
        Returns (seed, no_seed_provided)."""
        no_seed_provided = seed_list is None or len(seed_list) == 0
        if no_seed_provided:
            topology_seed = np.random.randint(2**31 - 1)
            while seeds_exclude is not None and topology_seed in seeds_exclude:
                topology_seed = np.random.randint(2**31 - 1)
        elif seed_index is not None:
            topology_seed = seed_list[seed_index]
        else:
            topology_seed = np.random.choice(seed_list)
        return int(topology_seed), no_seed_provided

    def pick_fresh_seeds(self, n):
        """n fresh topology seeds (int64 [n]) drawn from the global stream exactly as n calls of pick_seed() without a
        seed list draw them, this network's exclusion list included: one vectorised draw, replayed call by call from the
        same stream state when it hit an excluded seed (which pick_seed redraws at once)."""
        state = np.random.get_state()
        seeds = np.random.randint(2**31 - 1, size=n).astype(np.int64)
        ex = self.exclude_seeds
        if ex and np.isin(seeds, np.fromiter(ex, np.int64, len(ex))).any():
            np.random.set_state(state)
            seeds = np.array([self.pick_seed(None, None, ex)[0] for _ in range(n)], np.int64)
        return seeds

    def _create_valid_network(self, seed_list=None, seed_index=None, seeds_exclude=None):
        seed, fresh = self.pick_seed(seed_list, seed_index, seeds_exclude)
        t = generate_tables(self.n_nodes, seed, allow_reseed=fresh, exclude=seeds_exclude)
        self._install(t)
        return t["seed"]

    def _install(self, t):
        self.tables = t
        self.repetitions = t["repetitions"]
        self.current_topology_seed = t["seed"]
        N = self.n_nodes
        self.nodes = []
        for i in range(N):
            nd = Node(float(t["xy"][i, 0]), float(t["xy"][i, 1]))
            nd.neighbors = [int(v) for v in t["nbr_creation"][i]]
            nd.edges = [int(v) for v in t["node_edges"][i]]
            self.nodes.append(nd)
        self.edges = [Edge(int(a), int(b), int(l)) for a, b, l, _ in t["edges"]]
        self.shortest_paths_weights = t["apsp"]
        self._G = None
        self._shortest_paths = None
        self._update_nodes_adjacency()

    def reset(self):
        seed_index = self.next_topology_seed_index(advance_index=not self.sequential_topology_seeds_frozen)
        self._create_valid_network(self.seeds, seed_index, self.exclude_seeds)
        self.sampled_topology_seeds.append(self.current_topology_seed)

    # ---- lazily built networkx views (only the drivers / heuristics need them) --------------
    @property
    def G(self):
        if self._G is None:
            import networkx as nx

            g = nx.Graph()
            for i, nd in enumerate(self.nodes):
                g.add_node(i, pos=(nd.x, nd.y))
            for e in self.edges:
                g.add_edge(e.start, e.end, weight=e.length)
            self._G = g
        return self._G

    @property
    def shortest_paths(self):
        if self._shortest_paths is None:
            import networkx as nx

            self._shortest_paths = dict(nx.shortest_path(self.G, weight=self.G_weight_key))
        return self._shortest_paths

    def _update_shortest_paths(self):
        """network.py:274-290 after edge lengths changed."""
        t = self.tables
        for i, e in enumerate(self.edges):
            t["edges"][i, 2] = e.length
        _lib.check(_lib.lib().gm_topology_apsp(self.n_nodes, len(self.edges), _lib.ptr(t["edges"]),
                                               _lib.ptr(t["apsp"])))
        self.shortest_paths_weights = t["apsp"]
        self._G = None
        self._shortest_paths = None

    def randomize_edge_weights(self, mode: str, **kwargs):
        """network.py:292-351."""
        if mode == "shuffle":
            edge_lengths = np.array([e.length for e in self.edges])
            np.random.shuffle(edge_lengths)
            for i, e in enumerate(self.edges):
                e.length = int(edge_lengths[i])
        elif mode == "randint":
            for e in self.edges:
                e.length = int(np.random.randint(kwargs["low"], kwargs["high"]))
        elif mode == "bottleneck-971182936":
            for e in self.edges:
                if e.start == 2 and e.end == 7:
                    e.length = 10
            if self.current_topology_seed != 971182936:
                print("Warning: mode only meant to be used in graph 971182936.")
        else:
            raise ValueError(f"Unknown mode {mode}")
        old_paths = self.shortest_paths.copy()
        old_weights = self.shortest_paths_weights.copy()
        self._update_shortest_paths()
        n_paths = self.n_nodes * (self.n_nodes - 1)
        first = changed = wchanged = 0
        for a in range(self.n_nodes):
            for b in range(self.n_nodes):
                if a == b:
                    continue
                first += self.shortest_paths[a][b][1] != old_paths[a][b][1]
                changed += self.shortest_paths[a][b] != old_paths[a][b]
                wchanged += self.shortest_paths_weights[a][b] != old_weights[a][b]
        return (first / n_paths, changed / n_paths, wchanged / n_paths)

    def render(self):
        import matplotlib.pyplot as plt
        import networkx as nx

        nx.draw_networkx(self.G, with_labels=True, node_color="pink")
        plt.show()

    def get_nodes_adjacency(self):
        return self.adj_matrix

    def _update_nodes_adjacency(self):
        self.adj_matrix = np.eye(self.n_nodes, self.n_nodes, dtype=np.int8)
        for i in range(self.n_nodes):
            for neighbor in self.nodes[i].neighbors:
                self.adj_matrix[i][neighbor] = 1
