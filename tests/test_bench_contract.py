"""CPU checks of bench.py: the one-line JSON contract of the reference arm, and the --dump-outputs writer on a stand-in
rollout.  The device arm needs a B200 (tests/test_gpu_rollout.py)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--envs", "32"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout  # exactly one line on stdout, whatever libraries print
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "e2e", "cpu_baseline"):
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["unit"] == "env-steps/s" and d["value"] > 0 and d["steps"] == 1
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]


def _pack_rows(x):
    """[R, K] fp32 -> tile-packed bf16 hi/lo bytes, element by element as csrc/gemm_sm100.cuh states the layout."""
    import torch

    R, K = x.shape
    kb = K // 32
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    r, k = np.arange(R)[:, None], np.arange(K)[None, :]
    byte = ((r // 128) * kb + k // 32) * 16384 + (r % 128 >> 3) * 512 + ((k & 31) >> 3) * 128 + (r % 128 & 7) * 16 + (k & 7) * 2
    buf = np.zeros(-(-R // 128) * kb * 8192, np.int16)
    buf[byte // 2] = hi.view(torch.int16).numpy()
    buf[byte // 2 + 4096] = lo.view(torch.int16).numpy()
    return torch.from_numpy(buf.view(np.uint8)), hi.float(), lo.float()


def test_packed_rows_float_unpacks_the_tile_layout():
    import torch

    from graph_marl_b200.model import PackedRows

    B, A, K = 3, 50, 96  # 150 rows: the second 128-row tile is partial
    x = torch.randn(B * A, K, generator=torch.Generator().manual_seed(0))
    buf, hi, lo = _pack_rows(x)
    y = PackedRows(buf, (B, A, K), "bf16x3").float()
    assert y.dtype == torch.float32 and y.shape == (B, A, K)
    assert torch.equal(y.reshape(B * A, K), hi + lo)
    assert torch.equal(PackedRows(buf, (B, A, K), "bf16").float().reshape(B * A, K), hi)  # single pass: no lo part


def test_dump_outputs_writes_the_last_step_of_a_seeded_env_sample(tmp_path):
    """bench.py --dump-outputs: env e's transition of the last step sits at ring slot (index - B + e) % capacity (here
    across the end of the ring), the sample is the same seeded one for every array, and it stays inside the byte budget."""
    from types import SimpleNamespace

    import torch

    import bench
    from graph_marl_b200.model import PackedRows

    B, A, N, S, D, cap, index = 12, 3, 4, 6, 5, 40, 7
    g = torch.Generator().manual_seed(1)
    obs_g = torch.randn(B * A, 32, generator=g)
    buff = SimpleNamespace(index=index, buffer_size=cap, reward=torch.randn(cap, A, generator=g),
                           action=torch.randint(0, 4, (cap, A), generator=g).to(torch.int8),
                           done=torch.rand(cap, A, generator=g) < 0.5)
    ro = SimpleNamespace(B=B, buff=buff, join_streams=lambda: None, obs=(torch.randn(B, A, D, generator=g),
                         PackedRows(_pack_rows(obs_g)[0], (B, A, 32), "bf16x3")),
                         adj=torch.randint(0, 2, (B, A, A), generator=g).to(torch.int8),
                         env=SimpleNamespace(current_netmon_state=torch.randn(B, N, S, generator=g)))
    q = torch.randn(B, A, 4, generator=g)
    calls = []

    def act(obs_a, obs_g, **kw):
        calls.append((obs_a, obs_g, kw))
        return q, None

    ro.model = SimpleNamespace(act=act)
    per_env = 4 * (A * D + A * 32 + A * A + N * S + 3 * A + 4 * A)
    bench.dump_outputs(ro, str(tmp_path), budget_bytes=5 * per_env + 7)
    env = np.sort(np.random.default_rng(0).choice(B, 5, replace=False))
    slots = (index - B + env) % cap
    want = dict(obs_agent=ro.obs[0][env], obs_graph=ro.obs[1].float()[env], adj=ro.adj[env], netmon_state=ro.env.current_netmon_state[env],
                action=buff.action[slots], reward=buff.reward[slots], done=buff.done[slots], q_values=q[env])
    # Q-values: one greedy act() (no random draws) on the observations the step left
    assert len(calls) == 1 and calls[0][0] is ro.obs[0] and calls[0][1] is ro.obs[1]
    assert calls[0][2]["epsilon"] == 0 and calls[0][2]["want_q"]
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(n + ".npy" for n in want)
    for name, t in want.items():
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, t.float().numpy()), name
