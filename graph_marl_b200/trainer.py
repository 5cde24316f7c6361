"""Training loop at batched throughput: the rollout of rollout.Rollout (B envs per step, the env kernel writing every
transition into the compact state ring) interleaved with learner.Learner updates -- src/main.py:667-1026 for B envs.
"""
import torch

from .env.routing import Routing
from .env.wrapper import NetMonWrapper
from .evaluation import evaluate_topologies, run_episodes
from .learner import Learner
from .rollout import Rollout
from .util import get_state_dict


class Trainer:
    def __init__(self, cfg="cfg2", num_envs=4096, math="bf16x3", batch_size=32, sequence_length=1, train_every=1,
                 updates_per_train=1, step_before_train=0, epsilon=1.0, epsilon_decay=0.996, epsilon_update_freq=100,
                 lr=1e-3, gamma=0.98, tau=0.01, capacity_steps=64, seed=0, graph_steps=0, graph_learner=True):
        """Counts are in batched steps (one step advances all num_envs envs): step_before_train, train_every,
        epsilon_update_freq, capacity_steps.  Every `train_every` rollout steps the learner runs `updates_per_train`
        updates on `batch_size` per-env sequences of `sequence_length` transitions.  epsilon decays like
        EpsilonGreedy (policy.py): times `epsilon_decay` every `epsilon_update_freq` steps after step_before_train,
        floored at 0.01."""
        self.rollout = r = Rollout(cfg, num_envs, math=math, replay_capacity=int(capacity_steps) * num_envs, epsilon=epsilon,
                                   seed=seed, graph_steps=graph_steps, device_sampler=True, state_ring=True,
                                   fused_insert=True)
        assert r.state_ring, "the trainer samples per-env sequences from the compact state ring"
        a = r.policy._args
        a.step_before_train, a.epsilon_decay, a.epsilon_update_freq = int(step_before_train), float(epsilon_decay), int(epsilon_update_freq)
        self.args = dict(cfg=cfg, num_envs=num_envs, math=math, batch_size=batch_size, sequence_length=sequence_length,
                         train_every=train_every, updates_per_train=updates_per_train, step_before_train=step_before_train,
                         epsilon=epsilon, epsilon_decay=epsilon_decay, epsilon_update_freq=epsilon_update_freq, lr=lr,
                         gamma=gamma, tau=tau, capacity_steps=capacity_steps, seed=seed, graph_steps=graph_steps)
        self.batch_size, self.sequence_length = int(batch_size), int(sequence_length)
        self.train_every, self.updates_per_train = int(train_every), int(updates_per_train)
        self.step_before_train = int(step_before_train)
        self.learner = Learner(r.netmon, r.model, lr, gamma, tau, graph=graph_learner)
        self.steps = 0
        self.losses = []  # device scalars, one per update
        self._eval = None

    @property
    def epsilon(self):
        return self.rollout.policy._epsilon

    def _evict_stale_units(self):
        """Captured rollout units bake epsilon in as a launch argument: drop those of superseded values."""
        r, eps = self.rollout, float(self.epsilon)
        for k in [k for k in r._graphs if k[2] != eps]:
            del r._graphs[k]
        if not r._graphs:
            r._graph_pool = None  # the memory pool lives only as long as a graph captured into it

    def train(self, steps):
        """Advance `steps` batched rollout steps, with learner updates every train_every steps once step_before_train
        steps are done and the ring holds more steps than a sequence needs.  Returns the losses of these updates (host
        floats, read once at the end)."""
        r, buff = self.rollout, self.rollout.buff
        first = len(self.losses)
        done = 0
        while done < steps:
            n = min(self.train_every, steps - done)
            r.run(n)
            done += n
            self.steps += n
            self._evict_stale_units()
            if self.steps >= self.step_before_train and buff.count // r.B > self.sequence_length:
                for _ in range(self.updates_per_train):
                    self.losses.append(self.learner.update(buff, self.batch_size, self.sequence_length))
        new = self.losses[first:]
        return torch.cat(new).tolist() if new else []

    def evaluate(self, episodes=1, epsilon=0.0, seed=None):
        """Mean reward per agent and step of `episodes` fresh episodes of all B envs, acting with `epsilon` (0: the greedy
        policy) on an env of its own (same topology and sizes; the training env, its episode and the replay ring are not
        touched).  Actions come from the DQN's fused Q head with the device Philox draws."""
        r = self.rollout
        c = r.cfg
        if self._eval is None:
            if c.get("random_topology"):
                raise NotImplementedError("evaluate() shares the training env's fixed topology")
            be = Routing(r.base_env.network, c["n_data"], 1, enable_congestion=c["congestion"], num_envs=r.B,
                         device=r.device, seed=(self.args["seed"] if seed is None else seed) + 7919, batched=True)
            # the same device topology tables: NetMon's weight pack (which folds in the pool's static rows) stays the one
            # the captured rollout units read
            be._pool = r.base_env._pool
            self._eval = NetMonWrapper(be, r.netmon, 1, split_obs=True, graph_obs_fp32=True)
        saved = r.netmon.state
        total = torch.zeros((), dtype=torch.float64, device=r.device)
        steps = 0
        with torch.no_grad():
            for reward, _, _ in run_episodes(self._eval, r.model, episodes, c["episode_steps"], epsilon):
                steps += 1
                total += reward.double().mean()
        r.netmon.state = saved
        return float(total) / steps

    def evaluate_topologies(self, seeds, episode_steps=None, epsilon=0.0):
        """evaluation.evaluate_topologies of the current policy on the topologies of `seeds` (e.g. env.constants.EVAL_SEEDS),
        with the rollout's n_data, congestion and (by default) episode length.  Works for every config: it runs on copies
        of the modules and on a topology pool of its own, so the training run is not touched."""
        r = self.rollout
        c = r.cfg
        return evaluate_topologies(r.netmon, r.model, seeds, c["n_data"],
                                   c["episode_steps"] if episode_steps is None else episode_steps,
                                   congestion=c["congestion"], epsilon=epsilon, env_seed=self.args["seed"] + 7919)

    def state_dict(self):
        """Checkpoint in the reference's layout (util.get_state_dict): loads with the reference's util.load_state_dict."""
        return get_state_dict(self.rollout.model, self.rollout.netmon, self.args)
