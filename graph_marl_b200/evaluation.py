"""Evaluation of a policy on held-out topologies in one batched run: the reference's eval.py loop (a greedy policy, one
episode per graph, the mean of the reward and of every info key, SURVEY §3.6) with B graphs as the B envs of one
batched Routing, and the metrics summed per env on the device (gm_eval_accumulate, csrc/eval_metrics.cu).

The packet draws are the env's device Philox stream, not the reference's global numpy stream (whose consumption depends
on the actions of every earlier episode): the numbers are eval.py's metrics by definition, not bit for bit.
"""
import copy

import numpy as np
import torch

from . import _lib
from .env.environment import EnvironmentVariant
from .env.network import Network
from .env.routing import Routing, TopologyPool
from .env.wrapper import NetMonWrapper

# the metrics, in the order of per_topology and of the pooled means
METRICS = ("reward_mean", "delays", "delays_arrived", "spr", "looped", "throughput", "dropped", "blocked")


def run_episodes(env, model, episodes, episode_steps, epsilon):
    """The evaluation loop: `episodes` rounds of env.reset() followed by `episode_steps` steps of model.act -> env.step on
    a batched NetMonWrapper(split_obs=True); yields each step's (reward, done, info).  Actions are epsilon-greedy with the
    device Philox draws of seed 12345 at steps 1, 2, ... counted across rounds.  Run it under torch.no_grad()."""
    step = 0
    for _ in range(int(episodes)):
        (obs_a, obs_g), _ = env.reset()
        for _ in range(int(episode_steps)):
            step += 1
            _, act = model.act(obs_a, obs_g, epsilon=float(epsilon), seed=12345, step=step, want_q=False)
            (obs_a, obs_g), _, reward, done, info = env.step(act)
            yield reward, done, info


def accumulate(acc, out):
    """gm_eval_accumulate: add one batched step's outputs `out` (Routing's output dict: reward, done, arrived, delays,
    spr, info) into acc f64 [B, len(_lib.EVAL_FIELDS)]."""
    B, A = out["reward"].shape
    assert acc.dtype == torch.float64 and acc.shape == (B, len(_lib.EVAL_FIELDS)) and acc.is_contiguous()
    t = [out[k].contiguous() for k in ("reward", "done", "arrived", "delays", "spr", "info")]
    with torch.cuda.device(acc.device):
        _lib.check(_lib.lib().gm_eval_accumulate(*(x.data_ptr() for x in t), B, A, acc.data_ptr(), _lib.current_stream()))


def summarize(acc):
    """The metrics of accumulated rows acc f64 [B, F], read to the host once.  Returns per_topology (a dict of f64 [B]
    CPU tensors, one per metric: each env's own means) and the pooled means over all envs:

      reward_mean              sum of rewards / agent-steps
      delays                   sum of the delays of done packets / their number
      delays_arrived           sum of the delays of arrived packets / their number
      spr                      sum of the spr of arrived packets / their number
      looped, throughput,      sum of the info counter / env-steps
      dropped, blocked

    A list key (delays, delays_arrived, spr: eval.py extends a list with the step's values and takes np.mean) is the sum
    of its values over all envs and steps over their count; an empty set gives NaN, as np.mean([]) does.  A scalar key is
    its mean per env-step."""
    h = acc.cpu()
    f = {k: h[:, i] for i, k in enumerate(_lib.EVAL_FIELDS)}
    tot = {k: v.sum() for k, v in f.items()}
    res = {}
    for src in (f, tot):
        m = dict(reward_mean=src["reward_sum"] / src["agent_steps"], delays=src["delay_sum"] / src["delay_count"],
                 delays_arrived=src["arrived_delay_sum"] / src["arrived_count"], spr=src["spr_sum"] / src["arrived_count"])
        for k in ("looped", "throughput", "dropped", "blocked"):
            m[k] = src[k] / src["steps"]
        if src is f:
            res["per_topology"] = m
        else:
            res.update({k: float(v) for k, v in m.items()})
    return res


def topology_pool(seeds, n_nodes, device):
    """The topologies of `seeds` generated on the device into a pool of their own: returns (pool, slot), seeds[b] in
    slot[b] = b.  A seed that is not a valid topology raises AssertionError (the device generator would reseed)."""
    seeds = np.asarray(seeds, dtype=np.int64).reshape(-1)
    pool = TopologyPool.slots(seeds.size, n_nodes, device)
    slot = torch.arange(seeds.size, dtype=torch.int32, device=device)
    used, _ = pool.generate(seeds, slot)
    if not np.array_equal(used, seeds):
        bad = int(np.flatnonzero(used != seeds)[0])
        raise AssertionError(f"Provided seed {int(seeds[bad])} is invalid.")
    return pool, slot


class _PoolRouting(Routing):
    """A batched Routing that stays on the topologies of its pool: reset() puts env b back on slot topo_index[b] and
    never reads or resets the Network."""

    def reset(self):
        return self.reset_on_pool(self._pool, self._topo_index)


def _private_copy(module):
    """`module` with copies of its parameters and its own weight pack and workspace, and without NetMon's carried state.
    NetMon folds the pool's static rows into its weight pack, and the pack is repacked into the same buffer that captured
    rollout units read: evaluation must not run on the training modules."""
    memo = {id(module._ws): type(module._ws)(), id(module._pack): type(module._pack)()}
    if getattr(module, "state", None) is not None:
        memo[id(module.state)] = None
    return copy.deepcopy(module, memo)


def evaluate_topologies(netmon, model, seeds, n_data, episode_steps, congestion=True, epsilon=0.0, env_seed=0, episodes=1):
    """Evaluate the NetMon + DQN policy on the topologies of `seeds`, of the node count N that NetMon's input width
    4N + 8 gives: env b runs on the topology of
    seeds[b], generated on the device into a pool of its own (slot b).  Each of `episodes` rounds resets every env
    (packets from the env's device Philox stream of seed `env_seed`) and runs `episode_steps` steps; NetMon starts each
    round from no state, and actions come from model.act with `epsilon` (device Philox draws, run_episodes).
    gm_eval_accumulate sums the metrics of every step per env, and the host reads them once at the end.

    A provided seed that is not a valid topology raises AssertionError, as Network.reset() and build_sl_dataset do (no
    reseed).  The run uses copies of the modules, so nothing of a live training run is touched: not NetMon's state or
    weight pack, not the global numpy stream.  Returns summarize()'s dict: per_topology and the pooled means of METRICS."""
    _lib.require_device()
    seeds = np.asarray(seeds, dtype=np.int64).reshape(-1)
    B, N = seeds.size, (netmon.in_features - 8) // 4
    if B < 1:
        raise ValueError("evaluate_topologies needs at least one topology seed")
    if int(episode_steps) < 1 or int(episodes) < 1:
        raise ValueError(f"evaluate_topologies needs episode_steps >= 1 and episodes >= 1, got {episode_steps}, {episodes}")
    if netmon.in_features != 4 * N + 8 or N < 4:
        raise ValueError(f"NetMon takes {netmon.in_features}-wide node rows, which are no N-node topology's 4N + 8")
    if model.in_features != 6 * N + 10 + netmon.get_out_features():
        raise ValueError(f"the DQN takes {model.in_features} inputs, {N}-node topologies and this NetMon give "
                         f"{6 * N + 10 + netmon.get_out_features()}")
    dev = next(netmon.parameters()).device
    pool, slot = topology_pool(seeds, N, dev)
    be = _PoolRouting(Network(N), n_data, EnvironmentVariant.INDEPENDENT, enable_congestion=congestion, num_envs=B,
                      device=dev, seed=env_seed, batched=True)
    be.set_topology_pool(pool, slot)
    env = NetMonWrapper(be, _private_copy(netmon), 1, split_obs=True, graph_obs_fp32=True)
    dqn = _private_copy(model)
    acc = torch.zeros((B, len(_lib.EVAL_FIELDS)), dtype=torch.float64, device=dev)
    with torch.no_grad():
        for _ in run_episodes(env, dqn, episodes, episode_steps, epsilon):
            accumulate(acc, be._out)
    return summarize(acc)
