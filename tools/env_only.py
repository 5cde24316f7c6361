"""Env-step kernel alone (profiling / A-B timing): B envs of config 2, device Philox draws, random actions.
usage: python tools/env_only.py [B] [iters] -- prints the CUDA-event time per launch and the HBM-roofline fraction."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from bench import env_step_bytes, peaks
from graph_marl_b200.env.network import Network
from graph_marl_b200.env.routing import Routing

B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 50
N = A = 20
env = Routing(Network(N, random_topology=False, topology_init_seed=923430603), A, 1, num_envs=B, seed=1, batched=True)
env.reset()
acts = [torch.randint(0, 4, (B, A), device="cuda", dtype=torch.int32) for _ in range(8)]
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for i in range(10):
    env.step(acts[i % 8])
torch.cuda.synchronize()
# kernel time from the library's own CUDA events around the launch (gm_profile_*): Python's issue time stays outside
import ctypes as C  # noqa: E402

from graph_marl_b200 import _lib  # noqa: E402

ts = []
for i in range(iters):
    flush.zero_()  # outputs of the previous launch leave L2, like in the rollout where GEMMs run in between
    _lib.lib().gm_profile_enable(1)
    env.step(acts[i % 8])
    _lib.lib().gm_profile_enable(0)
    ms, cnt = (C.c_double * 8)(), (C.c_int32 * 8)()
    _lib.check(_lib.lib().gm_profile_collect(ms, cnt))
    ts.append(ms[1] * 1e3)
ts.sort()
med = ts[len(ts) // 2]
by = env_step_bytes(N, A, sparse_rows=env._out.get("node_sparse") is not None) * B
print(f"B={B} median {med:.2f} us  min {ts[0]:.2f} us  "
      f"roofline frac (median) {by / (med * 1e-6) / 1e9 / peaks()['hbm_gbs']:.3f}")

try:  # probe build (-DGM_ROUTING_PROBES=1): mean SM clocks between the phase boundaries of the last launch
    import ctypes as C

    import numpy as np

    from graph_marl_b200 import _lib

    fn = _lib.lib().gm_routing_probe_read
    n = min(B, 16384)
    out = np.zeros((n, 10), np.int64)
    fn.argtypes, fn.restype = [C.c_void_p, C.c_int], C.c_int
    assert fn(out.ctypes.data, n) == 0
    t = out - out[:, :1]
    print("phase ends (mean SM clocks since the warp started):")
    for k, nm in zip(range(1, 8), ["record loaded", "loop 1 done", "loop 2 done", "agent obs emitted", "record written back",
                                   "waiting sums done", "node obs emitted"]):
        print(f"  {nm:24s} {t[:, k].mean():9.0f}   (+{(t[:, k] - t[:, k - 1]).mean():8.0f})")
    print(f"  {'adj / node-agent done':24s} {max(t[:, 8].mean(), t[:, 9].mean()):9.0f}")
    print(f"  warp start spread: {(out[:, 0].max() - out[:, 0].min())} clocks; last end - first start: {out[:, 8:].max() - out[:, 0].min()} clocks")
except AttributeError:
    pass
