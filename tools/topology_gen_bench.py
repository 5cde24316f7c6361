"""Fresh-topology generation on the device against the host generator, and what it costs the rollout.  Prints one JSON line:

  * the card and its power limit;
  * device generation of B topologies into a pool (TopologyPool.generate: seed upload, gm_topology_generate_device, the
    status / seed read-back), CUDA events, warmed, at N = 20 for B = 2048 / 4096 / 16384 and at N = 200 for B = 4096;
  * the host generator (generate_tables, one thread) on the same seeds -- all of them at N = 20, the first 256 at N = 200,
    reported per topology;
  * cfg3fresh env-steps/s with its episode resets (B device-generated topologies each) inside the timed window, against
    cfg3's finite pool of 4096 topologies, same env count, graph units and steps.

    python tools/topology_gen_bench.py [--envs 2048] [--episodes 4]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from graph_marl_b200.env.network import generate_tables  # noqa: E402
from graph_marl_b200.env.routing import TopologyPool  # noqa: E402
from graph_marl_b200.rollout import Rollout  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else (torch.cuda.get_device_name(0), "?")
    return name, power


def device_generation(N, B, reps=5):
    seeds = np.random.default_rng(N * 100003 + B).integers(0, 2**31 - 1, B)
    pool = TopologyPool.slots(B, N, "cuda")
    slot = torch.arange(B, dtype=torch.int32, device="cuda")
    pool.generate(seeds, slot)  # warm-up
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        pool.generate(seeds, slot)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    n_host = B if N <= 20 else 256
    t0 = time.perf_counter()
    for s in seeds[:n_host]:
        generate_tables(N, int(s), allow_reseed=True)
    host_ms = (time.perf_counter() - t0) * 1e3
    return dict(N=N, B=B, device_ms_median=float(np.median(ms)), device_ms_min=float(min(ms)),
                host_ms_per_topology=host_ms / n_host, host_topologies_timed=n_host)


def rollout_rate(cfg, B, episodes, graph_steps=10):
    ro = Rollout(cfg, num_envs=B, math="bf16x3", seed=1000, graph_steps=graph_steps)
    E = ro.cfg["episode_steps"]
    ro.precapture()
    ro.run(E)  # warm: a whole episode, its reset included
    steps = episodes * E
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    ro.run(steps)  # `episodes` resets inside the window
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    return dict(workload=cfg, envs=B, steps=steps, resets=episodes, ms=ms, env_steps_per_s=B * steps / (ms * 1e-3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=2048)
    ap.add_argument("--episodes", type=int, default=4)
    a = ap.parse_args()
    name, power = card()
    gen = [device_generation(20, B) for B in (2048, 4096, 16384)] + [device_generation(200, 4096)]
    roll = [rollout_rate(c, a.envs, a.episodes) for c in ("cfg3fresh", "cfg3")]
    print(json.dumps(dict(card=name, power_limit=power, generation=gen, rollout=roll)))


if __name__ == "__main__":
    main()
