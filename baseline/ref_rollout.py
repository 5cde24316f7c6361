"""Timing of the UNMODIFIED reference rollout loop (src/main.py:673-737) on host cores.

Used only by bench.py (`cpu_baseline_reference`, kind "reference") next to the oracle port.  The reference's own
classes are imported from an unedited copy of its src/ placed at baseline/_ref/src (git-ignored, not part of this
repository; without it the reference arm is skipped); gymnasium / matplotlib / torch_geometric, which the reference
imports for features this timing does not use, are stubbed by tools/ref_stubs.py.  P worker processes (SURVEY 8d: one
per host core, torch threads = 1) each run

    policy(obs, adj) -> NetMonWrapper.step(actions) -> buff.add(...)            [one env instance per process]

for BASELINE config 2 (Routing N=20, A=20, seed 923430603, NetMon H=128 (512,256) K=3 lstm + DQN (512,256)),
epsilon 1.0 like the GPU arm, and report env-steps/s summed over the workers.
"""
import multiprocessing as mp
import os
import sys
import time
from types import SimpleNamespace

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_SRC = os.path.join(HERE, "_ref", "src")


def available():
    return os.path.exists(os.path.join(REF_SRC, "main.py"))


def _worker(rank, cfg, seconds, warmup_steps, q):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import ref_stubs

    ref_stubs.REFERENCE_SRC = REF_SRC
    ref_stubs.install()
    sys.path.insert(0, REF_SRC)
    import numpy as np
    import torch
    import torch.nn.functional as F

    torch.set_num_threads(1)
    from env.environment import reset_and_get_sizes
    from env.network import Network
    from env.routing import Routing
    from env.wrapper import NetMonWrapper
    from model import DQN, NetMon
    from policy import EpsilonGreedy
    from replaybuffer import ReplayBuffer

    np.random.seed(1000 + rank)
    torch.manual_seed(0)
    net = Network(n_nodes=cfg["n_nodes"], random_topology=False, topology_init_seed=cfg["topo_seed"])
    env = Routing(net, cfg["n_data"], 1, enable_congestion=cfg["congestion"])
    n_agents, agent_obs_size, n_nodes, node_obs_size = reset_and_get_sizes(env)
    netmon = NetMon(node_obs_size, cfg["H"], list(cfg["enc"]), cfg["K"], activation_fn=F.leaky_relu, rnn_type=cfg["rnn"],
                    rnn_carryover=True, agg_type="sum", output_neighbor_hidden=True, output_global_hidden=False)
    node_state_size = netmon.get_state_size()
    node_aux_size = len(env.get_node_aux()[0])
    env = NetMonWrapper(env, netmon, 1)
    _, agent_obs_size, _, _ = reset_and_get_sizes(env)
    model = DQN(agent_obs_size, list(cfg["dqn"]), env.action_space.n, F.leaky_relu)
    args = SimpleNamespace(epsilon=1.0, step_before_train=10**9, epsilon_update_freq=100, epsilon_decay=0.996)
    policy = EpsilonGreedy(env, model, env.action_space.n, args)
    buff = ReplayBuffer(0, 512, n_agents, agent_obs_size, 0, n_nodes, node_obs_size, node_state_size, node_aux_size)
    model.eval(), netmon.eval()

    episode_step, episode_done = None, False
    steps, t_start = 0, None
    while True:
        # ---- src/main.py:676-737 ----
        if episode_step is None or episode_done:
            episode_step = 0
            obs, adj = env.reset()
        buffer_node_state = env.last_netmon_state.cpu().detach().numpy() if env.last_netmon_state is not None else 0
        netmon_info = env.get_netmon_info()
        buffer_node_aux = env.get_node_aux()
        joint_actions = policy(obs, adj)
        next_obs, next_adj, reward, done, info = env.step(joint_actions)
        next_netmon_info = env.get_netmon_info()
        episode_step += 1
        episode_done = episode_step >= cfg["episode_steps"]
        buff.add(obs, joint_actions, reward, next_obs, adj, next_adj, done, episode_done, 0, buffer_node_state,
                 buffer_node_aux, *netmon_info, *next_netmon_info)
        obs, adj = next_obs, next_adj
        # ----
        steps += 1
        if t_start is None and steps >= warmup_steps:
            t_start, steps = time.perf_counter(), 0
        elif t_start is not None and time.perf_counter() - t_start >= seconds:
            break
    q.put((steps, time.perf_counter() - t_start))


def time_reference(cfg, seconds=10.0, warmup_steps=20, procs=None):
    """env-steps/s of the unmodified reference loop over `procs` single-threaded processes."""
    procs = procs or len(os.sched_getaffinity(0))
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ws = [ctx.Process(target=_worker, args=(r, dict(cfg), seconds, warmup_steps, q)) for r in range(procs)]
    for w in ws:
        w.start()
    res = [q.get(timeout=seconds * 6 + 300) for _ in ws]
    for w in ws:
        w.join(timeout=60)
    value = sum(s / t for s, t in res)
    return dict(value=value, unit="env-steps/s", cores=procs, kind="reference",
                sample=f"unmodified src/main.py:673-737 loop, {procs} processes x 1 env (torch threads = 1), "
                       f"{sum(s for s, _ in res)} env-steps in {max(t for _, t in res):.1f} s after {warmup_steps} warm-up steps each",
                per_process=value / procs)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    from graph_marl_b200.rollout import CONFIGS

    print(time_reference(CONFIGS["cfg2"], seconds=float(sys.argv[1]) if len(sys.argv) > 1 else 5.0))
