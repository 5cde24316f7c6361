"""sl.py's supervised dataset built on the device (build_sl_dataset) against the compat loop it replaces.  Prints one
JSON line:

  * the card and its power limit;
  * per case (N, S): samples/s of build_sl_dataset over S samples, host clock around the call and a device synchronise,
    after one warm-up build of one chunk (module loads, allocator); the whole build, seed and packet replay included;
  * samples/s of the compat loop from the same seed -- one `Routing(num_envs=1).reset()` per sample and get_sl_sample's
    networkx labels (sl.py:174-219) -- over its first `compat` samples, with the first `compat` samples of both checked
    equal (labels, targets, node observations, seeds).

Both start from np.random.seed(seed) on Network(N, random_topology=True): fresh seeds, as sl.py's training split draws.

    python tools/sl_dataset_bench.py [--cases 20:10000:2000,20:100000:2000,200:300:100] [--chunk 4096]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from graph_marl_b200.env.network import Network  # noqa: E402
from graph_marl_b200.env.routing import Routing  # noqa: E402
from graph_marl_b200.sl_dataset import build_sl_dataset  # noqa: E402
from topology_gen_bench import card  # noqa: E402


def compat(N, S, A, seed):
    """The reference's loop: a compat reset and networkx's first hops towards node 0 per sample."""
    np.random.seed(seed)
    net = Network(N, random_topology=True)
    env = Routing(net, A, 1)
    labels, targets, obs, seeds = [], [], [], []
    t0 = time.perf_counter()
    for _ in range(S):
        env.reset()
        lab = np.zeros(N, np.int8)
        for v in range(N):
            path = net.shortest_paths[v][0]
            if len(path) > 1:
                hops = [net.edges[e].get_other_node(v) for e in net.nodes[v].edges]
                lab[v] = hops.index(path[1]) + 1
        labels.append(lab)
        targets.append(np.asarray(net.shortest_paths_weights)[:, 0])
        obs.append(env.get_node_observation())
        seeds.append(net.current_topology_seed)
    s = time.perf_counter() - t0
    return s, dict(labels=np.stack(labels), targets=np.stack(targets), node_obs=np.stack(obs), seeds=np.array(seeds))


def device(N, S, A, seed, chunk):
    np.random.seed(seed)
    build_sl_dataset(Network(N, random_topology=True), min(S, chunk), n_data=A, chunk=chunk)  # warm-up
    torch.cuda.synchronize()
    np.random.seed(seed)
    net = Network(N, random_topology=True)
    t0 = time.perf_counter()
    ds = build_sl_dataset(net, S, n_data=A, chunk=chunk)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, ds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="20:10000:2000,20:100000:2000,200:300:100",
                    help="N:S:compat samples, comma-separated")
    ap.add_argument("--n-data", type=int, default=20)
    ap.add_argument("--chunk", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=5)
    a = ap.parse_args()
    name, power = card()
    rows = []
    for case in a.cases.split(","):
        N, S, Sc = (int(x) for x in case.split(":"))
        dev_s, ds = device(N, S, a.n_data, a.seed, a.chunk)
        host_s, ref = compat(N, Sc, a.n_data, a.seed)
        same = all(np.array_equal(ds[k][:Sc].cpu().numpy(), ref[k]) for k in ref)
        rows.append(dict(N=N, samples=S, device_s=dev_s, device_samples_per_s=S / dev_s, compat_samples=Sc,
                         compat_s=host_s, compat_samples_per_s=Sc / host_s, equal_on_compat_samples=bool(same)))
    print(json.dumps(dict(card=name, power_limit=power, chunk=a.chunk, n_data=a.n_data, cases=rows)))


if __name__ == "__main__":
    main()
