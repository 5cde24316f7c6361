"""Evaluation on the 1000 EVAL_SEEDS graphs: evaluate_topologies (all graphs as the envs of one batched run, metrics
accumulated on the device) against the loop of the reference's eval.py, one graph at a time through the compat
`Routing` (num_envs = 1) + `NetMonWrapper` on the same modules.  Prints one JSON line:

  * the card and its power limit, read in the same run;
  * per (config, math): seconds per evaluate_topologies call over all 1000 graphs (host clock around the call, which
    ends in its host read; median of 3 after a warm-up call) and env-steps/s;
  * the compat loop's env-steps/s, host clock around `--compat-graphs` whole episodes after a warm-up episode (the loop
    is the same for every graph, so its rate does not depend on how many are timed), and the ratio of the two rates.

Workload: cfg2- and cfg3-shaped NetMon + DQN (H = 128, encoder and DQN (512, 256), lstm, sum, neighbour readout; K = 3
with congestion, K = 1 without), N = A = 20, 50-step episodes, greedy policy, untrained weights.

    python tools/eval_bench.py [--steps 50] [--maths bf16x3,fp32] [--compat-graphs 10]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from graph_marl_b200.env.constants import EVAL_SEEDS  # noqa: E402
from graph_marl_b200.env.network import Network  # noqa: E402
from graph_marl_b200.env.routing import Routing  # noqa: E402
from graph_marl_b200.env.wrapper import NetMonWrapper  # noqa: E402
from graph_marl_b200.evaluation import evaluate_topologies  # noqa: E402
from graph_marl_b200.model import DQN, NetMon  # noqa: E402
from topology_gen_bench import card  # noqa: E402

N = A = 20
SHAPES = {"cfg2": dict(K=3, congestion=True), "cfg3": dict(K=1, congestion=False)}


def modules(cfg, math, seed=0):
    torch.manual_seed(seed)
    nm = NetMon(4 * N + 8, 128, (512, 256), SHAPES[cfg]["K"], F.leaky_relu, rnn_type="lstm", agg_type="sum",
                output_neighbor_hidden=True, math=math).cuda().eval()
    dqn = DQN(6 * N + 10 + nm.get_out_features(), (512, 256), 4, F.leaky_relu, math=math).cuda().eval()
    return nm, dqn


def batched(nm, dqn, cfg, steps):
    run = lambda: evaluate_topologies(nm, dqn, EVAL_SEEDS, A, steps, congestion=SHAPES[cfg]["congestion"])
    run()
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        run()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def compat(nm, dqn, cfg, steps, graphs):
    """eval.py's loop: env.reset() on the next evaluation graph, then greedy actions from the wrapped observations."""
    np.random.seed(0)
    net = Network(N, random_topology=True, sequential_topology_seeds=True, provided_seeds=list(EVAL_SEEDS))
    env = NetMonWrapper(Routing(net, A, 1, enable_congestion=SHAPES[cfg]["congestion"]), nm, 1)

    def episode():
        nm.state = None
        obs, _ = env.reset()
        for _ in range(steps):
            _, act = dqn.act(torch.from_numpy(obs).cuda(), epsilon=0.0, want_q=False)
            obs, _, _, _, _ = env.step(act.cpu().numpy())

    with torch.no_grad():
        episode()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(graphs):
            episode()
        torch.cuda.synchronize()
        return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--maths", default="bf16x3,fp32")
    ap.add_argument("--configs", default="cfg2,cfg3")
    ap.add_argument("--compat-graphs", type=int, default=10)
    a = ap.parse_args()
    name, power = card()
    rows = []
    for cfg in a.configs.split(","):
        for math in a.maths.split(","):
            nm, dqn = modules(cfg, math)
            s = batched(nm, dqn, cfg, a.steps)
            sc = compat(nm, dqn, cfg, a.steps, a.compat_graphs)
            rate, rate_c = len(EVAL_SEEDS) * a.steps / s, a.compat_graphs * a.steps / sc
            rows.append(dict(config=cfg, math=math, graphs=len(EVAL_SEEDS), steps=a.steps, batched_s=s,
                             batched_env_steps_per_s=rate, compat_env_steps_per_s=rate_c,
                             compat_s_for_all_graphs=len(EVAL_SEEDS) * a.steps / rate_c, speedup=rate / rate_c))
    print(json.dumps(dict(card=name, power_limit=power, N=N, A=A, rows=rows)))


if __name__ == "__main__":
    main()
