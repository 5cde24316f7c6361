"""The DQN's action selection and the device Philox draws against exact references.

Every batched rollout step picks its actions in one place: the Q head, action mask, argmax and epsilon mix that run either
in the epilogue of the tensor-core kernel (linear_tc_kernel with EPI_QHEAD) or in dqn_head_kernel after the hidden layers.
These tests run each dispatch branch at row counts around the 128-row tile and at a count that gives every CTA at least
two M tiles, and compare

- Q-values with the fp64 numpy oracle within the stated bars (bf16x3 1e-4, bf16 5e-2, fp32 2e-5);
- random rows (u < epsilon) with the draws exactly: host tables, or the numpy Philox restatement (oracle/philox.py);
- greedy rows with the masked argmax of the reference Q-values exactly wherever the reference's masked top-2 gap exceeds
  twice the Q tolerance, and elsewhere with an action within twice the tolerance of the maximum.  At least 99 % of the
  greedy rows of a case must fall in the exact class, so that a case cannot pass on ambiguous rows alone.

Single-pass bf16 rounds every operand to 8 bits, so its Q-values sit up to 5e-4 from the fp64 values of the unrounded
operands (bar 5e-2).  Its actions are therefore checked against an fp64 reference of the same rounded operands (hi part
of the split, as the kernel forms it) at 2e-4.

The env's device packet draws are checked the same way: a batched Routing run without host draws is replayed on the C
oracle with the draw tables of oracle/philox.env_draws, and every state field and output must be bit-identical.
"""
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden
from helpers import det_weights, dqn_shapes

pytestmark = pytest.mark.gpu

DA = 130
BIG = 2 * 148 * 128 + 77  # every CTA of a 148-SM grid gets at least two M tiles
ROWS = [1, 127, 128, 129, BIG]
TOL = {"bf16x3": 1e-4, "bf16": 5e-2, "fp32": 2e-5}
BF16_ACT_TOL = 2e-4  # bf16: Q against the fp64 reference of the bf16-rounded operands

# name: (hidden, Dg, n_act, math, Q-head instance (BN, PASSES, EPI, NCG) of linear_tc_kernel, or None: dqn_head_kernel)
CASES = {
    "cfg2": ((512, 256), 512, 4, "bf16x3", (256, 3, 2, 4)),
    "n48": ((64, 48), 128, 4, "bf16x3", (256, 3, 2, 4)),
    "one_action": ((64, 32), 128, 1, "bf16x3", (256, 3, 2, 4)),
    "fp32_input_n36": ((100, 36), 128, 5, "bf16x3", (256, 3, 2, 2)),
    "one_layer_8_actions": ((252,), 128, 8, "bf16x3", (256, 3, 2, 2)),
    "bf16": ((128, 64), 128, 7, "bf16", (256, 1, 2, 2)),
    "head_after_wide_layer": ((256, 512), 128, 4, "bf16x3", None),
    "head_n_not_multiple_of_4": ((64, 130), 128, 3, "bf16x3", None),
    "fp32": ((512, 256), 512, 4, "fp32", None),
}
TC_CASES = [c for c in CASES if CASES[c][3] != "fp32"]

_TC_NAME = re.compile(r"linear_tc_kernel(?:<(\d+), (\d+), (\d+), (\d+)>|ILi(\d+)ELi(\d+)ELi(\d+)ELi(\d+)E)")


def _bf16(x):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16).float().numpy()


def _bf16_forward(w, x):
    """fp64 DQN forward on bf16-rounded layer inputs and weights (single-pass tensor-core layers); the Q head is fp32."""
    h = np.asarray(x, np.float32)
    i = 0
    while f"encoder.linear_layers.{i}.weight" in w:
        h = _bf16(h).astype(np.float64) @ _bf16(w[f"encoder.linear_layers.{i}.weight"]).astype(np.float64).T
        h = h + w[f"encoder.linear_layers.{i}.bias"]
        h = np.where(h >= 0, h, 0.01 * h)
        i += 1
    return h @ w["q_net.fc.weight"].astype(np.float64).T + w["q_net.fc.bias"]


class Case:
    """One dispatch branch: the DQN, inputs for BIG rows (row counts below use a prefix), and the reference Q-values of a
    sample of rows that holds the first 130 rows, 1500 random ones and the last 8 of BIG."""

    def __init__(self, name):
        from oracle import netmon_oracle as NO

        self.name = name
        self.hidden, self.Dg, self.n_act, self.math, self.qhead = CASES[name]
        seed = 100 + list(CASES).index(name)
        self.w = det_weights(dqn_shapes(DA + self.Dg, self.hidden, self.n_act), seed)
        self.dqn = self.make_dqn(self.w)
        rng = np.random.default_rng(seed)
        self.xa = (rng.random((BIG, DA)) < 0.1).astype(np.float32)
        self.xg = (rng.standard_normal((BIG, self.Dg)) * 0.3).astype(np.float32)
        self.obs_a, self.obs_g = torch.from_numpy(self.xa).cuda(), torch.from_numpy(self.xg).cuda()
        self.sample = np.unique(np.concatenate([np.arange(130), rng.choice(BIG, 1500, replace=False), np.arange(BIG - 8, BIG)]))
        x = np.concatenate([self.xa[self.sample], self.xg[self.sample]], 1)
        self.q_ref = NO.dqn_forward(self.w, x, dtype=np.float64)
        self.tol = TOL[self.math]
        # the reference the actions are held to, and its tolerance
        self.q_act, self.act_tol = (_bf16_forward(self.w, x), BF16_ACT_TOL) if self.math == "bf16" else (self.q_ref, self.tol)
        self.greedy = self.exact = 0

    def make_dqn(self, w):
        from graph_marl_b200.model import DQN

        dqn = DQN(DA + self.Dg, self.hidden, self.n_act, F.leaky_relu, math=self.math)
        dqn.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
        return dqn.cuda().eval()

    def act(self, R, dqn=None, obs_g=None, **kw):
        with torch.no_grad():
            q, a = (dqn or self.dqn).act(self.obs_a[:R], self.obs_g[:R] if obs_g is None else obs_g, **kw)
        return (None if q is None else q.cpu().numpy()), a.cpu().numpy()

    def rows(self, R):
        """Positions in the sample, and row indices, of the sampled rows below R."""
        pos = np.nonzero(self.sample < R)[0]
        return pos, self.sample[pos]

    def check_q(self, q, R):
        pos, rows = self.rows(R)
        err = np.abs(q[rows] - self.q_ref[pos]).max()
        assert err < self.tol, (self.name, R, err)
        if self.math == "bf16":
            err = np.abs(q[rows] - self.q_act[pos]).max()
            assert err < self.act_tol, (self.name, R, err)

    def check_actions(self, act, R, eps, ra, ru, mask, greedy_ref=None):
        """ra / ru: the draws of all R rows; mask [R, n_act] or None.  Random rows are checked on every row, greedy rows on
        the sampled rows against the reference (and on every row against `greedy_ref`, the actions at epsilon 0)."""
        assert act.shape == (R,) and act.min() >= 0 and act.max() < self.n_act, (self.name, R)
        rand = ru < eps
        assert np.array_equal(act[rand], ra[rand]), (self.name, R, eps, np.nonzero(act[rand] != ra[rand])[0][:8])
        if greedy_ref is not None:
            assert np.array_equal(act[~rand], greedy_ref[~rand]), (self.name, R, eps)
        pos, rows = self.rows(R)
        qm = self.q_act[pos].copy()
        if mask is not None:
            qm[mask[rows].astype(bool)] = -np.inf
        best = np.argmax(qm, axis=-1)
        srt = np.sort(qm, axis=-1)
        with np.errstate(invalid="ignore"):
            gap = srt[:, -1] - srt[:, -2] if self.n_act > 1 else np.full(len(rows), np.inf)
        exact = ~(gap <= 2 * self.act_tol)  # nan (every action masked: argmax 0) counts as exact
        g = ~rand[rows]
        got = act[rows]
        bad = g & exact & (got != best)
        assert not bad.any(), (self.name, R, eps, rows[bad][:8], got[bad][:8], best[bad][:8], qm[bad][:4])
        amb = g & ~exact
        near = qm[np.arange(len(rows)), got] >= qm.max(-1) - 2 * self.act_tol
        assert near[amb].all(), (self.name, R, eps, rows[amb & ~near][:8])
        self.greedy += int(g.sum())
        self.exact += int((g & exact).sum())

    def check_exact_share(self):
        assert self.greedy > 0 and self.exact >= 0.99 * self.greedy, (self.name, self.exact, self.greedy)


_cases = {}


def _case(name):
    if name not in _cases:
        _cases[name] = Case(name)
    c = _cases[name]
    c.greedy = c.exact = 0
    return c


def _masks(R, n_act, rng):
    out = {"none": None, "random30": (rng.random((R, n_act)) < 0.3).astype(np.uint8)}
    half = rng.random(R) < 0.5
    m = np.zeros((R, n_act), np.uint8)
    m[half, 0] = 1
    out["first"] = m
    m = np.zeros((R, n_act), np.uint8)
    m[half, :n_act - 1] = 1
    out["all_but_last"] = m
    m = np.zeros((R, n_act), np.uint8)
    m[rng.random(R) < 0.3] = 1
    out["all"] = m
    return out


def _kernels(fn):
    """Runs fn() under torch.profiler; returns its result and the CUDA kernel names."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def _tc_instances(names):
    """Template arguments (BN, PASSES, EPI, NCG) of the linear_tc_kernel instances among kernel names (demangled or not)."""
    inst = set()
    for n in names:
        m = _TC_NAME.search(n)
        if m:
            inst.add(tuple(int(x) for x in (m.groups()[:4] if m.group(1) else m.groups()[4:])))
    return inst


def _check_kernels(c, names):
    inst = _tc_instances(names)
    qheads = {i for i in inst if i[2] == 2}
    head = any("dqn_head_kernel" in n for n in names)
    if c.qhead is not None:
        assert qheads == {c.qhead} and not head, (c.name, inst, names)
    else:
        assert not qheads and head, (c.name, inst, names)
        if c.math == "fp32":
            assert not inst, (c.name, inst)
        else:
            assert inst, (c.name, names)


# ---- A. Q head, mask and epsilon mix with host draws ---------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_q_head_and_epsilon_greedy_host_draws(name):
    c = _case(name)
    rng = np.random.default_rng(7)
    for R in ROWS:
        ra = rng.integers(0, c.n_act, R).astype(np.int32)
        ru = rng.random(R)
        ra_t, ru_t = torch.from_numpy(ra).cuda(), torch.from_numpy(ru).cuda()
        if R == BIG:
            (q, _), names = _kernels(lambda: c.act(R))
            _check_kernels(c, names)
        else:
            q, _ = c.act(R)
        c.check_q(q, R)
        for kind, mask in _masks(R, c.n_act, rng).items():
            mask_t = None if mask is None else torch.from_numpy(mask).cuda()
            for eps in (0.0, 0.4, 1.0):
                q2, a = c.act(R, action_mask=mask_t, epsilon=eps, rand_action=ra_t, rand_u=ru_t)
                assert np.array_equal(q2, q), (name, R, kind, eps)  # Q-values before masking, every call the same
                c.check_actions(a, R, eps, ra, ru, mask)
                if eps == 0.4:
                    _, a2 = c.act(R, action_mask=mask_t, epsilon=eps, rand_action=ra_t, rand_u=ru_t, want_q=False)
                    assert np.array_equal(a2, a), (name, R, kind)
    c.check_exact_share()


@pytest.mark.parametrize("name", [n for n in CASES if CASES[n][2] > 1])
def test_exact_ties_pick_the_lower_action(name):
    """Two actions with identical Q-head weights and bias, lifted above the others: their Q-values are bit-identical, the
    lower index wins, and the higher one wherever the lower one is masked (numpy argmax: first maximum)."""
    c = _case(name)
    lo, hi = 0, c.n_act - 1
    w = dict(c.w)
    qw, qb = w["q_net.fc.weight"].copy(), w["q_net.fc.bias"].copy()
    qw[lo] = qw[hi]
    qb[lo] = qb[hi] = qb[hi] + 10.0
    w["q_net.fc.weight"], w["q_net.fc.bias"] = qw, qb
    dqn = c.make_dqn(w)
    rng = np.random.default_rng(3)
    for R in ROWS:
        mask = np.zeros((R, c.n_act), np.uint8)
        sel = rng.random(R) < 0.5
        mask[sel, lo] = 1
        q, a = c.act(R, dqn=dqn)
        assert np.array_equal(q[:, lo].view(np.uint32), q[:, hi].view(np.uint32)), (name, R)
        assert (q[:, lo] > np.delete(q, [lo, hi], axis=1).max(axis=1, initial=-np.inf)).all()
        assert (a == lo).all(), (name, R, np.nonzero(a != lo)[0][:8])
        _, a = c.act(R, dqn=dqn, action_mask=torch.from_numpy(mask).cuda(), want_q=False)
        assert np.array_equal(a, np.where(sel, hi, lo)), (name, R)


# ---- B. device Philox draws of the policy --------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_policy_device_draws_match_philox_restatement(name):
    """Without host draws the kernel draws (rand_action, u) from Philox4x32-10 at counter (row lo, row hi, step lo,
    step hi ^ 0x5bd1e995) and key seed ^ 0xA5A5A5A5DEADBEEF.  Every branch must give exactly the draws of the numpy
    restatement; u does not depend on n_act, so for a seed, step and row count every branch takes the random action on
    the same rows.  The steps cross 2^32 and the seeds 2^32, so the high words are used."""
    from graph_marl_b200 import _lib
    from oracle import philox as P

    c = _case(name)
    rng = np.random.default_rng(11)
    for R in ROWS:
        mask = (rng.random((R, c.n_act)) < 0.3).astype(np.uint8)
        mask_t = torch.from_numpy(mask).cuda()
        _, greedy = c.act(R, action_mask=mask_t, want_q=False)
        c.check_actions(greedy, R, 0.0, np.zeros(R, np.int64), np.ones(R), mask)
        for seed in (0, 3, 2**40 + 7):
            for step in (0, 9, 2**32 + 5):
                ra, ru = P.policy_draws(R, c.n_act, seed, step)
                for eps in (1.0, 0.5):
                    _, a = c.act(R, action_mask=mask_t, epsilon=eps, seed=seed, step=step, want_q=False)
                    c.check_actions(a, R, eps, ra, ru, mask, greedy_ref=greedy)
    # step_dev: the captured rollout passes step = s - base and a device counter holding base
    cnt = _lib.DeviceCounter("cuda")
    for k, s in ((5, 4), (2**32 - 3, 7)):
        cnt.set(k)
        _, a = c.act(BIG, epsilon=0.5, seed=3, step=s, step_dev=cnt.ptr(), want_q=False)
        _, b = c.act(BIG, epsilon=0.5, seed=3, step=s + k, want_q=False)
        assert np.array_equal(a, b), (name, k, s)
        ra, ru = P.policy_draws(BIG, c.n_act, 3, s + k)
        rand = ru < 0.5
        assert np.array_equal(a[rand], ra[rand])
    c.check_exact_share()


# ---- C. tile-packed graph observation ------------------------------------------------------------------------------------
def _pack_rows(x, math):
    """fp32 rows [R, K] (K % 32 == 0) -> PackedRows in the layout of csrc/gemm_sm100.cuh: per (128-row tile mt, 32-column
    block kb) 16 KiB, hi = bf16(x) at +0 and lo = bf16(x - hi) at +8 KiB, element (r, k) at
    (r>>3)*512 + ((k&31)>>3)*128 + (r&7)*16 + (k&7)*2; rows padded to 128 with zeros."""
    from graph_marl_b200.model import PackedRows

    R, K = x.shape
    mt, kb = -(-R // 128), K // 32
    xp = torch.zeros((mt * 128, K), dtype=torch.float32, device=x.device)
    xp[:R] = x
    hi = xp.to(torch.bfloat16)
    lo = (xp - hi.float()).to(torch.bfloat16)
    # [mt][r>>3][r&7][kb][(k&31)>>3][k&7] -> [mt][kb][r>>3][(k&31)>>3][r&7][k&7]
    planes = [p.reshape(mt, 16, 8, kb, 4, 8).permute(0, 3, 1, 4, 2, 5) for p in (hi, lo)]
    buf = torch.stack(planes, 2).contiguous().view(torch.uint8).reshape(-1)
    assert buf.numel() == mt * kb * 16384
    return PackedRows(buf, (R, K), math), hi[:R].float(), lo[:R].float()


@pytest.mark.parametrize("name", TC_CASES)
def test_tile_packed_graph_observation(name):
    c = _case(name)
    for R in ROWS:
        pk, hi, lo = _pack_rows(c.obs_g[:R], c.math)
        back = pk.float()
        assert torch.equal(back, hi if c.math == "bf16" else hi + lo), (name, R)
        q_ref, a_ref = c.act(R, epsilon=0.0)
        q, a = c.act(R, obs_g=pk, epsilon=0.0)
        err = np.abs(q - q_ref).max()
        assert err < c.tol, (name, R, err)
        c.check_q(q, R)
        for x in (a, a_ref):
            c.check_actions(x, R, 0.0, np.zeros(R, np.int64), np.ones(R), None)
    c.check_exact_share()


# ---- D. the recorded policy through the fused Q head ---------------------------------------------------------------------
def test_recorded_policy_through_fused_q_head():
    """dqn_policy.npz (the unmodified reference's EpsilonGreedy on one env: recorded masks, legacy np.random draws) replayed
    through the compat EpsilonGreedy over a bf16x3 DQN, i.e. the fused Q head with host draws.  The actions equal the
    recording, except on greedy rows whose recorded masked top-2 gap is below 2e-4: there either near-max action passes."""
    from types import SimpleNamespace

    from graph_marl_b200.model import DQN
    from graph_marl_b200.policy import EpsilonGreedy

    g = load_golden("dqn_policy")
    D, h1, h2, n_act, wseed = [int(x) for x in g["cfg"]]
    dqn = DQN(D, (h1, h2), n_act, F.leaky_relu, math="bf16x3")
    dqn.load_state_dict({k: torch.from_numpy(v) for k, v in det_weights(dqn_shapes(D, [h1, h2], n_act), wseed).items()})
    dqn = dqn.cuda().eval()
    env = SimpleNamespace(enable_action_mask=True, action_mask=None)
    args = SimpleNamespace(epsilon=0.5, step_before_train=3, epsilon_update_freq=2, epsilon_decay=0.5)
    pol = EpsilonGreedy(env, dqn, 4, args)
    np.random.seed(5)
    draws = np.random.RandomState(5)  # the same legacy stream, read alongside: randint(n_act, size=A), then rand(A)
    A = g["obs"].shape[1]
    n_near = 0
    (_, _), names = _kernels(lambda: dqn.act(torch.from_numpy(g["obs"][0]).cuda()))
    assert (256, 3, 2, 4) in _tc_instances(names), names
    for t in range(g["obs"].shape[0]):
        mask = g["masks"][t].astype(bool)
        env.action_mask = mask
        eps = pol._epsilon
        ra, ru = draws.randint(n_act, size=A), draws.rand(A)
        a = pol(g["obs"][t], np.ones((A, A), np.int8))
        rec = g["actions"][t]
        qm = np.where(mask, -np.inf, g["q"][t].astype(np.float64))
        srt = np.sort(qm, -1)
        near = (srt[:, -1] - srt[:, -2] < 2e-4) & (ru >= eps)
        assert np.array_equal(a[~near], rec[~near]), t
        assert (qm[np.arange(A), a] >= qm.max(-1) - 2e-4)[near].all(), t
        assert np.array_equal(a[ru < eps], ra[ru < eps]), t
        assert pol._epsilon == g["eps_after"][t]
        n_near += int(near.sum())
    assert n_near < 0.01 * g["actions"].size


# ---- E. env device draws and the mask hand-off ---------------------------------------------------------------------------
ENV_CFGS = {
    "n20_congestion": dict(N=20, A=20, B=4096, cong=True, mask=False, ttl=0, topo=923430603, seed=11,
                           pick=[0, 3, 4, 7, 1020, 1023, 2048, 2051, 4092, 4095]),
    "a45_mask_ttl": dict(N=20, A=45, B=64, cong=True, mask=True, ttl=15, topo=923430603, seed=2**33 + 5, pick=None),
    "n200_a100": dict(N=200, A=100, B=9, cong=True, mask=False, ttl=0, topo=476, seed=7, pick=None),
}


@pytest.mark.parametrize("cfg", list(ENV_CFGS))
def test_env_device_draws_against_oracle(cfg):
    """A batched Routing run with no host draws: the env draws packets from Philox4x32-10 at counter (slot, env, call lo,
    call hi) and key seed.  Picked envs (first and last warp of a CTA, the last env) are replayed on the C oracle with the
    tables of oracle.philox.env_draws and must match bit for bit on reset and every step.  In the masked config a bf16x3 DQN
    acts through the batched EpsilonGreedy on the env's observations and its own action mask; its actions must equal the
    oracle's epsilon-greedy of fp64 Q-values, that mask and the policy's Philox draws."""
    from types import SimpleNamespace

    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from graph_marl_b200.model import DQN
    from graph_marl_b200.policy import EpsilonGreedy
    from oracle import netmon_oracle as NO
    from oracle import oracle as O
    from oracle import philox as P

    k = ENV_CFGS[cfg]
    N, A, B = k["N"], k["A"], k["B"]
    pick = np.arange(B) if k["pick"] is None else np.array(k["pick"])
    env = Routing(Network(N, random_topology=False, topology_init_seed=k["topo"]), A, 1, enable_congestion=k["cong"],
                  enable_action_mask=k["mask"], ttl=k["ttl"], num_envs=B, seed=k["seed"], batched=True)
    orc = O.RoutingOracle(O.generate_topology(N, seed=k["topo"]), A, enable_congestion=k["cong"],
                          enable_action_mask=k["mask"], ttl=k["ttl"], num_envs=len(pick), threads=2)
    sel = torch.from_numpy(pick).cuda()

    def draws():
        return tuple(d[pick] for d in P.env_draws(B, A, N, k["seed"], env._calls))

    def compare(t):
        o = orc.observe()
        for key in ("obs", "adj", "node_obs", "node_agent"):
            assert np.array_equal(env._out[key][sel].cpu().numpy(), o[key]), (key, t)
        s = env.get_state()
        for key, ref in (("now", orc.now), ("target", orc.target), ("edge", orc.edge), ("time", orc.time),
                         ("ttl", orc.ttl_left), ("spw", orc.spw), ("start", orc.start), ("size", orc.size),
                         ("load", orc.load), ("agent_steps", orc.agent_steps), ("visited", orc.visited)):
            assert np.array_equal(s[key][pick], ref), (key, t)
        if k["mask"]:
            assert np.array_equal(s["mask"][pick], orc.mask), t
            assert np.array_equal(env._out["action_mask_out"][sel].cpu().numpy(), orc.mask), t

    d = draws()
    env.reset()
    orc.reset(*d)
    compare(-1)
    pol = None
    if k["mask"]:
        Da = env.obs_width()
        dqn = DQN(Da, (512, 256), 4, F.leaky_relu, math="bf16x3")
        w = det_weights(dqn_shapes(Da, [512, 256], 4), 21)
        dqn.load_state_dict({n: torch.from_numpy(v) for n, v in w.items()})
        dqn = dqn.cuda().eval()
        args = SimpleNamespace(epsilon=0.5, step_before_train=10**9, epsilon_update_freq=1, epsilon_decay=0.5)
        pol = EpsilonGreedy(env, dqn, 4, args, seed=2**35 + 9)
    gen = torch.Generator(device="cuda").manual_seed(3)
    n_greedy = n_exact = respawned = 0
    for t in range(30):
        if pol is None:
            act = torch.randint(0, 4, (B, A), device="cuda", generator=gen, dtype=torch.int32)
        else:
            obs = env._out["obs"]
            mask = env._out["action_mask_out"].cpu().numpy().reshape(B * A, 4).astype(bool)
            act = pol(obs, env._out["adj"])
            q = NO.dqn_forward(w, obs.cpu().numpy().reshape(B * A, -1), dtype=np.float64)
            ra, ru = P.policy_draws(B * A, 4, pol._seed, pol._step)
            got = act.cpu().numpy().reshape(-1)
            rand = ru < pol._epsilon
            assert np.array_equal(got[rand], ra[rand]), t
            qm = np.where(mask, -np.inf, q)
            srt = np.sort(qm, -1)
            with np.errstate(invalid="ignore"):
                exact = ~(srt[:, -1] - srt[:, -2] <= 2e-4)
            g = ~rand
            assert np.array_equal(got[g & exact], np.argmax(qm, -1)[g & exact]), t
            assert (qm[np.arange(B * A), got] >= qm.max(-1) - 2e-4)[g & ~exact].all(), t
            n_greedy, n_exact = n_greedy + int(g.sum()), n_exact + int((g & exact).sum())
        d = draws()
        _, _, reward, done, info = env.step(act)
        r = orc.step(act.cpu().numpy()[pick], *d)
        assert np.array_equal(reward[sel].cpu().numpy(), r["reward"]), t
        assert np.array_equal(done[sel].cpu().numpy(), r["done"].astype(bool)), t
        for key in ("delays", "arrived", "spr"):
            assert np.array_equal(info[key][sel].cpu().numpy(), r[key]), (key, t)
        got = torch.stack([info["looped"], info["throughput"], info["dropped"], info["blocked"]], 1)[sel].cpu().numpy()
        assert np.array_equal(got, r["info"]), t
        assert np.array_equal(env._out["n_resets"][sel].cpu().numpy(), r["n_resets"]), t
        respawned += int(r["n_resets"].sum())
        compare(t)
    assert respawned > 0  # the steps drew packets, not only the reset
    if pol is not None:
        assert n_exact >= 0.99 * n_greedy > 0, (n_exact, n_greedy)
