#!/usr/bin/env python
"""Benchmark of the rollout hot path (BASELINE.json metric: batched env-steps/sec incl. NetMon
forward; % of HBM roofline for the env-step kernel).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg2ln|cfg3|cfg4]
                    [--dump-outputs DIR]

One "step" = one batched rollout step over B environment instances per GPU
(src/main.py:673-737): DQN epsilon-greedy action selection -> Routing env step with agent and
node observations -> NetMon forward -> replay insert.  1 env-step = one env instance advanced
one tick.  Environment instances shard across GPUs with no collective on the path (weak
scaling: B per GPU is fixed).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput; `e2e` = the same step
driven through the public classes with the step's random draws supplied from pinned HOST memory
(a pre-generated pinned table, each step copies its own slice) and the reward read back every step; `roofline` = dominant kernel of the step;
`roofline_env_step` = the HBM-bound env-step kernel named by the metric; `cpu_baseline` = the
oracle (CPU port of the reference path) on this box's host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "batched_env_steps_per_sec_incl_netmon_fwd"
UNIT = "env-steps/s"


def peaks():
    p = dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")
    f = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(f):
        try:
            j = json.load(open(f))
            p.update(hbm_gbs=float(j["hbm_gbs"]), bf16_tflops=float(j["bf16_tflops"]),
                     bf16_tflops_sustained=float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), source="measured")
        except Exception:
            pass
    return p


def env_step_bytes(N, A, sparse_rows=False):
    """SURVEY.md 8(d): algorithmic bytes of one env-step with dense outputs materialised.  sparse_rows: the launch also
    writes the node rows in sparse form for NetMon's fused encoder (96 bytes per node, `gm_routing_io.node_sparse`)."""
    E = 3 * N // 2
    state = A * (40 + 4 * ((N + 31) // 32)) + 8 * E
    return (2 * state + 4 * A + 4 * A * (6 * N + 10) + 4 * N * (4 * N + 8) + A * A + N * A + 4 * A + A + 32 + 4 * A
            + (96 * N if sparse_rows else 0))


def gemm_flops(N, A, H, K, enc, dqn, n_act=4):
    """SURVEY.md 8(d): dense GEMM FLOPs per env-step (NetMon + DQN)."""
    Dn, Dj = 4 * N + 8, 6 * N + 10 + 4 * H
    nm, prev = 0, Dn
    for u in list(enc) + [H]:
        nm += 2 * prev * u
        prev = u
    nm += (1 + K) * 16 * H * H
    dq, prev = 0, Dj
    for u in dqn:
        dq += 2 * prev * u
        prev = u
    dq += 2 * prev * n_act
    return N * nm + A * dq


class ClockSampler:
    """SM clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  Sampled in-process
    through NVML every 10 ms (an external `nvidia-smi -lms` loop was seen to stall kernel launches of the
    timed process on some boxes); falls back to one nvidia-smi query if NVML is unavailable."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.rows, self.stop_flag, self.h, self.nv = [], False, None, None
        self.index = index
        try:
            import pynvml as nv

            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].strip().isdigit() else index
            self.h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.nv = nv
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.time(), sm, rs))
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self, t0, t1):
        if self.nv is None:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout
                f = [float(x) for x in out.strip().split(",")]
                return {"sm_mhz": f[0], "sm_max_mhz": f[1], "reasons": [], "samples": 1, "note": "after the timed region (NVML unavailable)"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"]}
        self.stop_flag = True
        self.t.join(timeout=1.0)
        nv = self.nv
        rows = [r for r in self.rows if t0 <= r[0] <= t1] or self.rows[-3:]
        sm = sorted(r[1] for r in rows)
        reasons = set()
        for r in rows:
            for bit, name in self.REASONS.items():
                if r[2] & bit:
                    reasons.add(name)
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def _init_weights(c):
    """Default-initialised NetMon / DQN parameters under the reference's state_dict names (model.py:256-401, 187-203),
    built from plain torch.nn layers: the CPU arm shares no code with the package it is compared with."""
    import torch
    import torch.nn as nn

    torch.manual_seed(0)
    N, H = c["n_nodes"], c["H"]
    w_nm, w_dq = {}, {}
    prev = 4 * N + 8
    for i, u in enumerate(list(c["enc"]) + [H]):
        l = nn.Linear(prev, u)
        w_nm[f"encode.linear_layers.{i}.weight"], w_nm[f"encode.linear_layers.{i}.bias"] = l.weight, l.bias
        prev = u
    for cell in ("rnn_obs", "rnn_update"):
        m = nn.LSTMCell(H, H)
        w_nm[f"{cell}.weight_ih"], w_nm[f"{cell}.weight_hh"], w_nm[f"{cell}.bias_ih"] = m.weight_ih, m.weight_hh, m.bias_ih
        if c["rnn"] == "lnlstm":
            for ln, width in (("ln_input", 4 * H), ("ln_hidden", 4 * H), ("ln_cell", H)):
                w_nm[f"{cell}.{ln}.weight"], w_nm[f"{cell}.{ln}.bias"] = torch.ones(width), torch.zeros(width)
        else:
            w_nm[f"{cell}.bias_hh"] = m.bias_hh
    prev = 6 * N + 10 + 4 * H
    for i, u in enumerate(c["dqn"]):
        l = nn.Linear(prev, u)
        w_dq[f"encoder.linear_layers.{i}.weight"], w_dq[f"encoder.linear_layers.{i}.bias"] = l.weight, l.bias
        prev = u
    q = nn.Linear(prev, 4)
    w_dq["q_net.fc.weight"], w_dq["q_net.fc.bias"] = q.weight, q.bias
    f = lambda d: {k: v.detach().numpy().copy() for k, v in d.items()}
    return f(w_nm), f(w_dq)


def cpu_arm(cfg_name, steps, warmup, envs=None, budget_s=20.0):
    """The oracle's rollout step on the host cores, bounded sample of the same workload."""
    from graph_marl_b200.rollout import CONFIGS  # the workload table only (sizes, seeds): no kernels, no classes
    from oracle.cpu_rollout import CpuRollout

    c = CONFIGS[cfg_name]
    cores = len(os.sched_getaffinity(0))
    N, A = c["n_nodes"], c["n_data"]
    w_nm, w_dq = _init_weights(c)
    B = envs or (64 * cores if N <= 50 else 2 * cores)
    ro = CpuRollout(N, A, c["topo_seed"], c["congestion"], c["K"], c["rnn"], c["H"], c["enc"], c["dqn"], B, cores,
                    w_nm, w_dq, replay_capacity=4 * B)
    ro.reset()
    for _ in range(max(1, min(warmup, 2))):
        ro.step()
    t0 = time.perf_counter()
    n = 0
    while n < steps and (time.perf_counter() - t0 < budget_s or n < 1):
        ro.step()
        n += 1
    dt = time.perf_counter() - t0
    return dict(value=B * n / dt, unit=UNIT, cores=cores, kind="port",
                sample=f"{B} envs x {n} rollout steps of {cfg_name}{' (CPU arm: one shared topology instead of the pool)' if c.get('random_topology') else ''} (C env oracle on {cores} threads + torch CPU NetMon+DQN on {cores} threads, "
                       f"replay insert incl.), {dt:.1f} s"), dt / max(n, 1), B


def reference_arm(cfg_name, seconds=8.0):
    """The UNMODIFIED Python reference (a copy of its src/ placed at baseline/_ref/src) running its own rollout loop, one
    process per host core (baseline/ref_rollout.py).  None when that copy is absent or the workload is not config 2's."""
    try:
        from baseline import ref_rollout
        from graph_marl_b200.rollout import CONFIGS

        c = CONFIGS[cfg_name]
        if not ref_rollout.available() or c.get("random_topology"):
            return None
        return ref_rollout.time_reference(c, seconds=seconds, warmup_steps=5 if c["n_nodes"] <= 50 else 1)
    except Exception as ex:  # never hide the GPU number behind the baseline
        return dict(value=None, unit=UNIT, kind="reference", sample=f"failed: {ex}")


def dump_outputs(ro, out_dir, budget_bytes=60_000_000):
    """Writes what the rollout's last step handed its caller to out_dir/<name>.npy (float32): the next agent and graph
    observations, agent adjacency and NetMon state, and the actions, rewards and done flags the step wrote into the
    replay ring.  The rollout acts with epsilon 1 (random actions), so `q_values` adds the DQN's Q-values on the next
    observations (a greedy act(): no random draws) to cover its GEMMs.  Files hold the same fixed, seeded sample of env
    instances, as many as fit `budget_bytes`."""
    import math

    import numpy as np
    import torch

    ro.join_streams()  # a dense-ring insert may still run on its side stream
    B, buff = ro.B, ro.buff
    slots = (buff.index - B + torch.arange(B, device=buff.reward.device)) % buff.buffer_size  # env e -> its ring slot
    obs_a, obs_g = ro.obs  # obs_g may exist only tile-packed (model.PackedRows): .float() unpacks it
    with torch.no_grad():
        q, _ = ro.model.act(obs_a, obs_g, epsilon=0.0, want_q=True)
    full = dict(obs_agent=obs_a, obs_graph=obs_g, adj=ro.adj, netmon_state=ro.env.current_netmon_state,
                action=buff.action[slots], reward=buff.reward[slots], done=buff.done[slots], q_values=q)
    per_env = 4 * sum(math.prod(t.shape[1:]) for t in full.values())
    k = min(B, budget_bytes // per_env)
    env = np.sort(np.random.default_rng(0).choice(B, k, replace=False))
    sel = torch.from_numpy(env).to(obs_a.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in full.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().index_select(0, sel).cpu().numpy())
    print(f"dump: outputs of the last timed step, {k} of {B} env instances -> {out_dir}", file=sys.stderr)


_REAL_STDOUT = None


def _claim_stdout():
    """Rank 0 must print exactly ONE JSON line on stdout, but C libraries (NCCL's version banner, the CUDA runtime)
    write to file descriptor 1 as they please: keep a private copy of the real stdout for the JSON line and point
    fd 1 (and sys.stdout) at stderr for everything else."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        sys.stdout = sys.stderr


def _emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg2ln", "cfg3", "cfg4"])
    ap.add_argument("--envs", type=int, default=0, help="env instances per GPU (default: BASELINE config size)")
    ap.add_argument("--math", default=os.environ.get("GM_BENCH_MATH", "bf16x3"), choices=["fp32", "bf16x3", "bf16"],
                    help="GEMM arithmetic: bf16x3 = tcgen05 with the fp32-accurate hi/lo split (default, parity mode), "
                         "bf16 = single tensor-core pass (reduced precision, reported only on request), fp32 = CUDA-core FFMA")
    ap.add_argument("--graph-steps", type=int, default=int(os.environ.get("GM_BENCH_GRAPH_STEPS", "10")),
                    help="rollout steps per captured CUDA graph unit (0 = launch every kernel from Python)")
    ap.add_argument("--no-replay", action="store_true")
    ap.add_argument("--replay", default="compact", choices=["compact", "dense"],
                    help="replay ring format: compact (env records + NetMon state, dense fields rebuilt when sampled; default) "
                         "or dense (the reference's 17 dense fields per transition)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --envs (default: the config's size) per GPU; strong: the config's TOTAL env count "
                         "(cfg2 4096, cfg3 16384) sharded over the ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--per-kernel", action="store_true", help="also print a per-stage CUDA-event breakdown to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one and the DQN's Q-values on its next "
                         "observations to DIR/<name>.npy (float32, rank 0's env instances, a fixed seeded sample of them "
                         "under 64 MB): same arguments, same inputs, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "ours" or a.no_replay):
        ap.error("--dump-outputs reads the last step's actions, rewards and done flags from the replay ring of the GPU "
                 "rollout: it needs --impl ours without --no-replay")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    from graph_marl_b200.rollout import CONFIGS

    c = CONFIGS[a.workload]
    N, A = c["n_nodes"], c["n_data"]
    B = a.envs or {"cfg2": 4096, "cfg2ln": 4096, "cfg3": 2048}.get(a.workload, 1024)
    B_weak = B
    if a.scaling == "strong":
        from graph_marl_b200.rollout import shard_envs

        total = a.envs or {"cfg2": 4096, "cfg2ln": 4096, "cfg3": 16384, "cfg4": 8192}[a.workload]
        lo, hi = shard_envs(total, world, rank)
        B = hi - lo
    # every step of a captured unit keeps its own observation / state tensors alive in the graph's pool:
    # bound the unit so that those stay under ~24 GB (cfg4 at 8192 envs holds ~15 GB per step)
    step_bytes = 4 * B * (1.5 * A * (6 * N + 10 + 4 * c["H"]) + N * (4 * N + 8) + 2 * N * c["H"])
    a.graph_steps = int(max(1, min(a.graph_steps, 24e9 // step_bytes))) if a.graph_steps > 0 else a.graph_steps
    if a.graph_steps > 2 and c["episode_steps"] % a.graph_steps != 0:
        # units that tile the episode exactly leave only the reset outside the captured graphs: prefer the largest
        # divisor of the episode length in [graph_steps / 2, graph_steps]
        divs = [g for g in range(max(2, a.graph_steps // 2), a.graph_steps + 1) if c["episode_steps"] % g == 0]
        if divs:
            a.graph_steps = divs[-1]
    config = dict(workload=f"{a.workload}: routing N={N} A={A} topo_seed={c['topo_seed']} congestion={c['congestion']} "
                           f"episode={c['episode_steps']} NetMon H={c['H']} enc={list(c['enc'])} K={c['K']} {c['rnn']} sum "
                           f"+ DQN {list(c['dqn'])}", envs_per_gpu=B, envs_total=(B * world if a.scaling == "weak" else total), math=a.math,
                  replay_insert=not a.no_replay,
                  replay_format=("compact: env records before/after + actions/reward/done + NetMon state per transition, dense fields rebuilt by get_batch"
                                 if a.replay == "compact" else "dense: the reference's 17 fields per transition"),
                  replay_overlap=("written by the env step kernel itself (gm_routing_io.ring_*), no insert launch" if a.replay == "compact" else "side stream, joined before the end event"),
                  cuda_graph_steps=a.graph_steps, sharding=f"env instances, {world} rank(s), no collective",
                  l2="per-step working set (obs + node_obs + NetMon activations + replay slots) exceeds the 126 MB L2")

    if a.impl == "reference":
        if rank != 0:
            return
        # The reference's own CPU implementation of the path: the UNMODIFIED Python rollout loop (src/main.py:673-737,
        # a copy placed at baseline/_ref/src) with one process per host core -- the reference has no batching, every process
        # advances one env instance.  The oracle port (C env + torch CPU tensors, all cores, the GPU arm's env count) is
        # timed beside it and becomes the line's value only where that copy is absent.
        cbr = reference_arm(a.workload, seconds=max(6.0, min(20.0, 0.4 * (a.steps + a.warmup))))
        cb, sec_per_step, Bc = cpu_arm(a.workload, a.steps, a.warmup, envs=(B_weak if N <= 50 else None), budget_s=45.0)
        use_ref = cbr is not None and cbr.get("value")
        main = cbr if use_ref else cb
        envs = main["cores"] if use_ref else Bc
        line = dict(metric=METRIC, value=main["value"], unit=UNIT, n_gpus=a.gpus, steps=a.steps, warmup=a.warmup,
                    ms_per_step=(envs / main["value"] * 1e3) if use_ref else sec_per_step * 1e3, higher_is_better=True,
                    scaling=a.scaling, vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                    config=dict(config, envs_per_gpu=envs, envs_total=envs,
                                math="fp32 (torch CPU)" if use_ref else "fp32 (oracle port: C env + torch CPU tensors)",
                                replay_format="dense: the reference's 17 fields per transition (numpy ring)", replay_overlap="none (host)",
                                cuda_graph_steps=0,
                                sharding=(f"{envs} single-env processes (the reference is not batched), one per host core" if use_ref
                                          else f"{Bc} envs batched over {cb['cores']} host threads")),
                    cpu_baseline=main, gpu_launches=0,
                    e2e=dict(value=main["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        line["cpu_baseline_port" if use_ref else "cpu_baseline_reference"] = cb if use_ref else cbr
        _emit(line)
        return

    import torch
    import torch.distributed as dist

    from graph_marl_b200 import _lib
    from graph_marl_b200.rollout import Rollout, aggregate_throughput

    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    _lib.require_device()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = [0.0]

    def timed(ro, steps, warmup, host):
        # untimed warm-up: at least the requested steps and one full wrap of the replay ring (8 x B slots), so
        # first-touch effects of the ring are outside the timed region
        ro.precapture()  # CUDA-graph units are captured before anything is timed
        g = max(ro.graph_steps, 1)
        ro.run(-(-(max(warmup, 10) + 2 * g) // g) * g)  # whole units: the timed region starts on a unit boundary (same ring phase)
        if g > 1 and steps % g != 0:
            # K is not a whole number of units: its last K % g steps run kernel by kernel.  Warm that path up too (one
            # unit's worth of eager steps keeps the unit boundary), or the caching allocator's first eager allocations
            # would fall into the timed region
            for _ in range(g):
                ro.step()
        ro.join_streams()
        n0 = _lib.lib().gm_kernel_launch_count() + ro.graph_launches
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        e0.record()
        ro.run(steps)
        ro.join_streams()  # the side-stream replay inserts of these steps finish inside the timed region
        e1.record()
        host_ms[0] = (time.time() - w0) * 1e3 / steps  # host-side issue time per step (before the final sync)
        barrier()
        w1 = time.time()
        ms = e0.elapsed_time(e1)
        # whole-job units / MAX device time over ranks
        value, ms_max = aggregate_throughput(B * steps, ms, world)
        return value, ms_max, _lib.lib().gm_kernel_launch_count() + ro.graph_launches - n0, w0, w1

    # ---- device-resident arm ---------------------------------------------------------------
    G = a.graph_steps
    ro = Rollout(a.workload, num_envs=B, device=dev, math=a.math, with_replay=not a.no_replay, seed=1000 + rank, graph_steps=G,
                 replay=a.replay)
    ro.reset()
    sampler = ClockSampler(local) if rank == 0 else None
    value, ms, launches, w0, w1 = timed(ro, a.steps, max(a.warmup, 3), host=False)
    clocks = sampler.stop(w0, w1) if sampler else None
    host_issue_ms = host_ms[0]
    if a.dump_outputs and rank == 0:
        dump_outputs(ro, a.dump_outputs)

    # ---- per-kernel timing for the roofline (CUDA events on the launching stream) -------------
    stage = ro.profile_stages(iters=max(5, min(a.steps, 20)))
    stage["note"] = ("dqn_act / env_step / netmon / replay_insert: CUDA events around the stages of an EAGER step (kernel-by-kernel issue; "
                     "they include GPU idle time whenever the host issues slower than the GPU runs, so they can exceed ms_per_step, "
                     "which is timed on captured CUDA-graph units); *_kernel_ms and gemm_ms: per-launch events inside the library")
    sparse_out = getattr(ro.base_env, "_out", {}).get("node_sparse") is not None
    # fused insert: the step launch also writes the transition's compact replay record (records before / after, int8
    # actions, f32 reward, done, topology index, episode_done) -- bytes of that launch, no separate insert kernel
    ring_bytes = (2 * ro.base_env._layout["stride"] + 6 * A + 5) if getattr(ro, "fused_insert", False) else 0
    del ro
    torch.cuda.empty_cache()

    # ---- end-to-end arm: host-supplied draws in, reward out, every step --------------------------
    ro = Rollout(a.workload, num_envs=B, device=dev, math=a.math, with_replay=not a.no_replay, seed=1000 + rank,
                 host_draws=True, graph_steps=G, replay=a.replay,
                 host_draw_steps=((a.steps + 2 * max(a.warmup, 10) + 4 * max(G, 1)) // max(G, 1) + 1) * max(G, 1))
    ro.reset()
    value_e, ms_e, _, _, _ = timed(ro, a.steps, max(a.warmup, 3), host=True)
    e2e = dict(value=value_e, unit=UNIT, h2d_bytes_per_step=ro.h2d_bytes_per_step() * world,
               d2h_bytes_per_step=ro.d2h_bytes_per_step() * world, ms_per_step=ms_e / a.steps,
               host_issue_ms_per_step=host_ms[0])
    del ro
    torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    traffic = {}
    try:  # DRAM bytes from the committed ncu --set full capture of this workload (cfg2, B=4096 only)
        if a.workload == "cfg2" and B == 4096:
            if a.replay == "compact":
                traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        traffic = {}
    H, K = c["H"], c["K"]
    flops_step = gemm_flops(N, A, H, K, c["enc"], c["dqn"]) * B
    gemm_ms = stage["gemm_ms"]
    env_ms = stage["env_kernel_ms"] if stage.get("env_kernel_ms", 0) > 0 else stage["env_step_ms"]
    agg_ms = stage.get("aggregate_kernel_ms", 0.0) / max(stage.get("aggregate_kernel_launches_per_step", 1.0), 1.0)
    # the step launch also writes the node rows in sparse form (the fused encoder's input): real output bytes of the
    # kernel, counted next to SURVEY 8(d)'s dense outputs (tools/env_only.py times the kernel against the same figure)
    per_env = env_step_bytes(N, A, sparse_rows=sparse_out) + ring_bytes
    env_bytes = per_env * B
    roof_env = dict(bound="hbm", kernel="routing_kernel<STEP>", achieved=env_bytes / (env_ms * 1e-3) / 1e9,
                    peak=pk["hbm_gbs"], unit="GB/s", frac=env_bytes / (env_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
                    traffic=traffic.get("routing_step_bytes_per_launch"), algorithmic_bytes_per_launch=env_bytes,
                    peak_source=pk["source"], bytes_per_env_step=per_env, ms_per_launch=env_ms,
                    note="SURVEY 8(d) dense outputs" + (" + 96 B per node of sparse node rows (gm_routing_io.node_sparse)" if sparse_out else "")
                         + (f" + {ring_bytes} B of compact replay transition (gm_routing_io.ring_*)" if ring_bytes else ""))
    tf = flops_step / (gemm_ms * 1e-3) / 1e12
    passes = {"fp32": 1, "bf16x3": 3, "bf16": 1}[a.math]
    roof_gemm = dict(bound="tensor", kernel=stage["gemm_kernel"], achieved=tf, peak=pk["bf16_tflops_sustained"], unit="TFLOP/s",
                     frac=tf / pk["bf16_tflops_sustained"], traffic=traffic.get("linear_tc_bytes_per_step"),
                     traffic_note="DRAM read+write bytes of the step's 9 launches (ncu, cold caches)" if traffic else None,
                     peak_source=pk["source"] + " (sustained bf16)",
                     flops_per_env_step=flops_step // B, ms_per_step_in_gemms=gemm_ms,
                     launches_per_step=stage.get("gemm_launches_per_step"),
                     note=f"achieved = algorithmic dense-GEMM flops of one step (2mnk, fp32 semantics) / summed CUDA-event time of the "
                          f"step's GEMM launches; the tensor pipe executes {passes}x that in bf16 MMAs",
                     tensor_pipe_tflops_executed=tf * passes)
    agg_bytes = 8 * N * H * B  # SURVEY 8(d): read h + write M per iteration
    roof_agg = dict(bound="hbm", kernel="aggregate_pk_pipe_kernel", achieved=(agg_bytes / (agg_ms * 1e-3) / 1e9) if agg_ms > 0 else None,
                    peak=pk["hbm_gbs"], unit="GB/s", frac=(agg_bytes / (agg_ms * 1e-3) / 1e9 / pk["hbm_gbs"]) if agg_ms > 0 else None,
                    traffic=traffic.get("aggregate_pk_bytes_per_launch"), algorithmic_bytes_per_launch=agg_bytes, ms_per_launch=agg_ms)
    dominant = roof_gemm if gemm_ms >= env_ms else roof_env
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=max(a.warmup, 3),
                ms_per_step=ms / a.steps, higher_is_better=True, scaling=a.scaling, vs_baseline=None,
                dtype={"fp32": "f32", "bf16x3": "f32 (tcgen05 bf16 hi/lo split x3, fp32 accumulate; env state int32/f64)",
                       "bf16": "bf16 (single pass, fp32 accumulate) -- reduced precision"}[a.math],
                data="synthetic", config=config, agent_steps_per_sec=value * A, host_issue_ms_per_step=host_issue_ms, gpu_launches=int(launches), clocks=clocks, e2e=e2e,
                roofline=dominant, roofline_env_step=roof_env, roofline_aggregate=roof_agg, roofline_gemm=roof_gemm, stage_ms=stage)
    if not a.no_cpu_baseline and world == 1:
        try:
            cb, _, _ = cpu_arm(a.workload, steps=10**6, warmup=1, budget_s=12.0)
            cbr = reference_arm(a.workload, seconds=8.0)
            if cbr is not None and cbr.get("value"):
                line["cpu_baseline"] = cbr       # the unmodified Python reference, one process per host core
                line["cpu_baseline_port"] = cb   # the oracle port (C env + torch CPU tensors) on the same cores
            else:
                line["cpu_baseline"] = cb
        except Exception as ex:  # the baseline must never hide the GPU number
            line["cpu_baseline"] = dict(value=None, unit=UNIT, cores=len(os.sched_getaffinity(0)), kind="port", sample=f"failed: {ex}")
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
