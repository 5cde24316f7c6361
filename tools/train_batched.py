"""Measures the batched trainer (graph_marl_b200.trainer.Trainer) at BASELINE config 2 and prints one JSON line:

  - the card's name and power limit;
  - env-steps/s while training (4096 envs, captured rollout units of 4 steps, one captured learner update of 32
    sequences after each unit, epsilon at its floor) and of the same rollout alone;
  - learner update ms, eager and captured, at two batch sizes;
  - gm_optimizer_step us against the torch tail (clip_grad_value_ + clip_grad_norm_ + AdamW(foreach=False) +
    util.interpolate_model) on the same cfg2 parameters (~0.94 M);
  - the greedy policy's mean reward every --curve-every updates.

    python tools/train_batched.py [--envs 4096] [--steps 256] [--curve-updates 1200] [--curve-every 300]

Times come from CUDA events around work on the current stream (ended by a synchronise).  Nothing is written to disk.
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from graph_marl_b200.learner import FusedOptimizer, Learner  # noqa: E402
from graph_marl_b200.trainer import Trainer  # noqa: E402
from graph_marl_b200.util import interpolate_model  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"name": out[0], "power_limit": out[1]}
    except Exception as e:  # the measurement still names the device torch sees
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def timed(fn, n):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--graph-steps", type=int, default=4)
    ap.add_argument("--batches", default="32,256")
    ap.add_argument("--seq-len", type=int, default=1)
    ap.add_argument("--curve-batch", type=int, default=256)
    ap.add_argument("--curve-updates", type=int, default=1200)
    ap.add_argument("--curve-every", type=int, default=300)
    a = ap.parse_args(argv)
    res = {"card": card(), "config": "cfg2", "math": "bf16x3", "envs": a.envs}
    n = a.graph_steps
    tr = Trainer("cfg2", a.envs, math="bf16x3", batch_size=32, sequence_length=a.seq_len, train_every=n, updates_per_train=1,
                 step_before_train=4 * n, epsilon=1.0, epsilon_decay=0.9, epsilon_update_freq=20, capacity_steps=32, seed=0,
                 graph_steps=n)
    r = tr.rollout
    while tr.epsilon > 0.01:  # epsilon at its floor: no captured rollout unit is superseded inside the timed region
        tr.train(n)
    tr.train(4 * n)
    ms = timed(lambda: tr.train(n), a.steps // n) / n
    res["train_env_steps_per_s"] = a.envs / (ms * 1e-3)
    res["train_ms_per_step"] = ms
    res["rollout_only_env_steps_per_s"] = a.envs / (timed(lambda: r.run(n), a.steps // n) / n * 1e-3)

    upd = {}
    for batch in [int(b) for b in a.batches.split(",")]:
        for graph in (False, True):
            ln = Learner(r.netmon, r.model, 1e-3, 0.98, 0.01, graph=graph)
            for _ in range(3):
                ln.update(r.buff, batch, a.seq_len)
            upd[f"batch{batch}_{'captured' if graph else 'eager'}_ms"] = timed(lambda: ln.update(r.buff, batch, a.seq_len), 20)
    res["learner_update"] = dict(upd, seq_len=a.seq_len, agents=r.sizes["A"])

    # optimizer tail on the cfg2 parameter set: device kernels vs the torch calls of the reference's learner
    model, nm = copy.deepcopy(r.model), copy.deepcopy(r.netmon)
    target = copy.deepcopy(model)
    params = list(model.parameters()) + list(nm.parameters())
    for p in params:
        p.grad = torch.randn_like(p) * 1e-3
    opt = FusedOptimizer(params, list(zip(model.parameters(), target.parameters())), 1e-3, 0.01)
    t_dev = timed(opt.step, 200)
    torch_opt = torch.optim.AdamW(params, lr=1e-3, foreach=False)

    def torch_tail():
        torch.nn.utils.clip_grad_value_(params, 0.5)
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        torch_opt.step()
        interpolate_model(model, target, 0.01, target)

    for _ in range(3):
        torch_tail()
    t_torch = timed(torch_tail, 50)
    res["optimizer"] = {"parameters": sum(p.numel() for p in params), "gm_optimizer_step_us": t_dev * 1e3,
                        "torch_tail_us": t_torch * 1e3}

    # greedy reward curve on a fresh trainer (one update of --curve-batch sequences after every rollout unit)
    tc = Trainer("cfg2", a.envs, math="bf16x3", batch_size=a.curve_batch, sequence_length=a.seq_len, train_every=n, updates_per_train=1,
                 step_before_train=4 * n, epsilon=1.0, epsilon_decay=0.9, epsilon_update_freq=20, capacity_steps=32, seed=1,
                 graph_steps=n)
    curve = [{"updates": 0, "greedy_reward": tc.evaluate(1), "epsilon1_reward": tc.evaluate(1, epsilon=1.0)}]
    while tc.learner.updates < a.curve_updates:
        goal = tc.learner.updates + a.curve_every
        losses = []
        while tc.learner.updates < goal:
            losses += tc.train(n)
        curve.append({"updates": tc.learner.updates, "greedy_reward": tc.evaluate(1), "last_loss": losses[-1] if losses else None,
                      "epsilon": tc.epsilon})
    res["greedy_reward_curve"] = curve
    print(json.dumps(res))
    return res


if __name__ == "__main__":
    main()
