"""sl.py's supervised training (BASELINE config 5) on the device dataset: the captured SLTrainer update against the path
the unmodified sl.py takes today, and SLTrainer.evaluate.  Prints one JSON line:

  * the card and its power limit, read in the same run;
  * per (batch, math) at T = 8 steps: ms per update and samples x steps / s of
      - the captured update (SLTrainer, graph=True), CUDA events around `--updates` updates after 3 warm-up updates;
      - sl.py's path in the same process on the same data, timed the same way: np.random.choice indices copied to the
        device, the batch gathered there, the NetMon module in grad mode on the dense mask (identity node-agent
        matrix), an nn.Linear head, F.mse_loss per step, loss.backward() and torch.optim.AdamW;
  * evaluation samples/s over the 1000-sample EVAL_SEEDS split at T = 1 and 4, host clock around evaluate() (which ends
    in its host read), median of 5 after a warm-up call.

Workload: paper dims (H = 128, encoder (512, 256), K = 2, lstm, sum, neighbour readout: O = 4H), N = 20, 10 000 fresh
training samples from build_sl_dataset.

    python tools/sl_train_bench.py [--updates 200] [--batches 32,512] [--maths fp32,bf16x3] [--seq-len 8]
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
from graph_marl_b200.model import MLP, NetMon  # noqa: E402
from graph_marl_b200.sl_dataset import build_sl_dataset  # noqa: E402
from graph_marl_b200.sl_trainer import SLTrainer  # noqa: E402
from topology_gen_bench import card  # noqa: E402

N = 20


def modules(math, seed=0):
    torch.manual_seed(seed)
    nm = NetMon(4 * N + 8, 128, (512, 256), 2, F.leaky_relu, rnn_type="lstm", agg_type="sum",
                output_neighbor_hidden=True, math=math).cuda()
    return nm


def timed(fn, n):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(n):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / n


def captured(data, math, B, T, n):
    nm = modules(math)
    head = MLP(nm.out_width(3), N, F.leaky_relu, activation_on_output=False).cuda()
    tr = SLTrainer(nm, head, data, lr=1e-3, seed=0, graph=True)
    for _ in range(3):
        tr.update(B, T)
    return timed(lambda: tr.update(B, T), n), tr


def sl_py_path(data, math, B, T, n):
    nm = modules(math)
    head = torch.nn.Linear(nm.get_out_features(), N).cuda()
    opt = torch.optim.AdamW(list(nm.parameters()) + list(head.parameters()), lr=1e-3)
    S = data["node_obs"].shape[0]
    eye = torch.eye(N, device="cuda").expand(B, N, N)

    def step():
        idx = torch.from_numpy(np.random.choice(S, B)).cuda()
        x, mask = data["node_obs"][idx], data["node_adj"][idx].float()
        y = data["targets_all"][idx].float()
        nm.state = None
        opt.zero_grad()
        loss = 0.0
        for _ in range(T):
            loss = loss + F.mse_loss(head(nm(x, mask, eye)), y)
        loss.backward()
        opt.step()

    for _ in range(3):
        step()
    return timed(step, n)


def evaluation(tr, data, T, reps=5):
    tr.evaluate(data, [T])
    s = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tr.evaluate(data, [T])
        s.append(time.perf_counter() - t0)
    return data["node_obs"].shape[0] / statistics.median(s)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--updates", type=int, default=200)
    ap.add_argument("--batches", default="32,512")
    ap.add_argument("--maths", default="fp32,bf16x3")
    ap.add_argument("--seq-len", type=int, default=8)
    ap.add_argument("--samples", type=int, default=10000)
    a = ap.parse_args()
    name, power = card()
    np.random.seed(0)
    train = build_sl_dataset(Network(N, random_topology=True), a.samples)
    np.random.seed(5)
    test = build_sl_dataset(Network(N, random_topology=True, sequential_topology_seeds=True, provided_seeds=EVAL_SEEDS),
                            1000)
    T, rows = a.seq_len, []
    for math in a.maths.split(","):
        for B in (int(b) for b in a.batches.split(",")):
            ms, tr = captured(train, math, B, T, a.updates)
            ref_ms = sl_py_path(train, math, B, T, a.updates)
            row = dict(math=math, batch=B, seq_len=T, updates=a.updates, captured_ms=ms,
                       captured_sample_steps_per_s=B * T / ms * 1e3, sl_py_path_ms=ref_ms,
                       sl_py_path_sample_steps_per_s=B * T / ref_ms * 1e3, speedup=ref_ms / ms)
            row.update({f"eval_T{t}_samples_per_s": evaluation(tr, test, t) for t in (1, 4)})
            rows.append(row)
    print(json.dumps(dict(card=name, power_limit=power, N=N, train_samples=a.samples, test_samples=1000, rows=rows)))


if __name__ == "__main__":
    main()
