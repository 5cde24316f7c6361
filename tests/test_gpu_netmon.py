"""GPU parity of NetMon / DQN / epsilon-greedy / replay (through the C ABI) against outputs of
the reference recorded in tests/golden and against the numpy oracle on larger random batches.

Stated fp32 tolerances (max abs error, identical weights + inputs, GM_MATH_FP32 arithmetic):
  lstm / gru / none : 2e-5 single step from identical state, 1e-4 over a 4-step recurrent rollout
  lnlstm            : 2e-3 (ill-conditioned LayerNorm over gate vectors, SURVEY 7.4)
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden
from helpers import det_weights, dqn_shapes, netmon_case, netmon_shapes

pytestmark = pytest.mark.gpu

G = load_golden("netmon")
TOL_ROLLOUT = {"lstm": 1e-4, "gru": 1e-4, "none": 1e-4, "lnlstm": 2e-3}
SKIP = set()  # gru_nocarry_k2: the reference's scrambled state layout (model.py:571, :449) is reproduced


def _netmon(cfg, in_features, math="fp32"):
    from graph_marl_b200.model import NetMon

    nm = NetMon(in_features, cfg["hidden"], cfg["enc"], cfg["iterations"], F.leaky_relu, rnn_type=cfg["rnn_type"],
                rnn_carryover=cfg["rnn_carryover"], agg_type=cfg["agg_type"],
                output_neighbor_hidden=cfg["output_neighbor_hidden"],
                output_global_hidden=cfg["output_global_hidden"], math=math)
    w = det_weights(netmon_shapes(in_features, cfg["hidden"], cfg["enc"], cfg["rnn_type"]), cfg["wseed"])
    assert list(nm.state_dict().keys()) == list(w.keys())  # same parameter names/order as the reference
    nm.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    return nm.cuda().eval(), w


@pytest.mark.parametrize("entry", [str(x) for x in G["case_names"] if str(x).split("|")[0] not in SKIP])
def test_netmon_golden_rollout(entry):
    import graph_marl_b200._lib as L

    name, cfg = netmon_case(G, entry)
    X, ADJ, NAM = G["node_obs"], G["node_adj"], G["node_agent"]
    nm, _ = _netmon(cfg, X.shape[-1])
    tol = TOL_ROLLOUT[cfg["rnn_type"]]
    n0 = L.lib().gm_kernel_launch_count()
    with torch.no_grad():
        nm.state = None
        for t in range(X.shape[0]):
            out = nm(torch.from_numpy(X[t]).cuda(), torch.from_numpy(ADJ[t]).float().cuda(),
                     torch.from_numpy(NAM[t]).float().cuda())
            assert out.shape == G[name + "_agent_out"][t].shape
            err = np.abs(out.cpu().numpy() - G[name + "_agent_out"][t]).max()
            serr = np.abs(nm.state.cpu().numpy() - G[name + "_state"][t]).max()
            assert err < tol and serr < tol, (t, err, serr)
    assert L.lib().gm_kernel_launch_count() > n0  # the CUDA path ran, not a fallback


def test_netmon_lists_path_and_single_step_tolerance():
    """forward_lists (no dense mask, gather readout) from the reference's recorded state."""
    name, cfg = netmon_case(G, [x for x in G["case_names"] if str(x).startswith("lstm_sum_k3_paper")][0])
    X, ADJ, NAM = G["node_obs"], G["node_adj"], G["node_agent"]
    nm, _ = _netmon(cfg, X.shape[-1])
    from graph_marl_b200.model import NetMon

    with torch.no_grad():
        for t in range(1, X.shape[0]):
            nbr, deg, dm = NetMon.lists_from_mask(torch.from_numpy(ADJ[t]).float().cuda())
            assert dm == 4 and int(deg.min()) == 4
            nm.state = torch.from_numpy(G[name + "_state"][t - 1]).cuda()
            agent_node = torch.from_numpy(NAM[t].argmax(axis=1).astype(np.int32)).cuda()
            _, ao = nm.forward_lists(torch.from_numpy(X[t]).cuda(), nbr, deg, None, 3, agent_node=agent_node)
            assert np.abs(ao.cpu().numpy() - G[name + "_agent_out"][t]).max() < 2e-5
            assert np.abs(nm.state.cpu().numpy() - G[name + "_state"][t]).max() < 2e-5


def test_netmon_simple_env_degree2():
    cfg = dict(hidden=8, iterations=2, rnn_type="lstm", rnn_carryover=True, agg_type="sum",
               output_neighbor_hidden=True, output_global_hidden=False, enc=[6], wseed=4242)
    nm, _ = _netmon(cfg, 1)
    with torch.no_grad():
        out = nm(torch.from_numpy(G["simple_node_obs"][None]).cuda(),
                 torch.from_numpy(G["simple_node_adj"][None]).float().cuda(), None, no_agent_mapping=True)
    assert out.shape == (1, 3, 24)
    assert np.abs(out.cpu().numpy() - G["simple_node_out"]).max() < 2e-5


@pytest.mark.parametrize("rnn,K,H,enc,B,N", [("lstm", 3, 128, (512, 256), 96, 20), ("lnlstm", 4, 128, (512, 256), 8, 200),
                                             ("gru", 2, 64, (96,), 33, 20)])
def test_netmon_against_oracle_random_batch(rnn, K, H, enc, B, N):
    """Larger seeded batch vs the numpy oracle in fp64 (truth) -- both GPU and fp32 oracle
    must sit within the stated tolerance of it."""
    from oracle import netmon_oracle as NO
    from oracle import oracle as O

    Dn = 4 * N + 8
    cfg = dict(hidden=H, iterations=K, rnn_type=rnn, rnn_carryover=True, agg_type="sum",
               output_neighbor_hidden=True, output_global_hidden=False, enc=list(enc), wseed=77)
    nm, w = _netmon(cfg, Dn)
    topo = O.generate_topology(N, seed=923430603 if N == 20 else 476)
    rng = np.random.default_rng(1)
    x = (rng.random((B, N, Dn)) < 0.05).astype(np.float32) + rng.random((B, N, Dn)).astype(np.float32) * (rng.random((B, N, Dn)) < 0.02)
    mask = np.broadcast_to(topo["adj"], (B, N, N)).astype(np.float32)
    st = (rng.standard_normal((B, N, nm.state_size)) * 0.3).astype(np.float32)
    ref_out, ref_state, _ = NO.netmon_forward(w, cfg, x, mask, st, dtype=np.float64)
    with torch.no_grad():
        nm.state = torch.from_numpy(st).cuda()
        out = nm(torch.from_numpy(x).cuda(), torch.from_numpy(mask.copy()).cuda(), None, no_agent_mapping=True)
    tol = 2e-3 if rnn == "lnlstm" else 2e-5
    assert np.abs(out.cpu().numpy() - ref_out).max() < tol
    assert np.abs(nm.state.cpu().numpy() - ref_state).max() < tol


def test_dqn_q_values_and_epsilon_greedy_golden():
    from types import SimpleNamespace

    from graph_marl_b200.model import DQN
    from graph_marl_b200.policy import EpsilonGreedy

    g = load_golden("dqn_policy")
    D, h1, h2, n_act, wseed = [int(x) for x in g["cfg"]]
    dqn = DQN(D, (h1, h2), n_act, F.leaky_relu)
    w = det_weights(dqn_shapes(D, [h1, h2], n_act), wseed)
    assert list(dqn.state_dict().keys()) == list(w.keys())
    dqn.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    dqn = dqn.cuda().eval()
    with torch.no_grad():
        q = dqn(torch.from_numpy(g["obs"]).cuda(), None)
        # two-segment input == concatenated input
        q2, _ = dqn.act(torch.from_numpy(g["obs"][..., :130].copy()).cuda(), torch.from_numpy(g["obs"][..., 130:].copy()).cuda())
    assert np.abs(q.cpu().numpy() - g["q"]).max() < 2e-5
    assert np.abs(q2.cpu().numpy() - g["q"]).max() < 2e-5
    env = SimpleNamespace(enable_action_mask=True, action_mask=None)
    args = SimpleNamespace(epsilon=0.5, step_before_train=3, epsilon_update_freq=2, epsilon_decay=0.5)
    pol = EpsilonGreedy(env, dqn, 4, args)
    np.random.seed(5)
    A = g["obs"].shape[1]
    for t in range(g["obs"].shape[0]):
        env.action_mask = g["masks"][t].astype(bool)
        a = pol(g["obs"][t], np.ones((A, A), np.int8))
        assert np.array_equal(a, g["actions"][t]), t
        assert pol._epsilon == g["eps_after"][t]
    pol.eval()
    assert pol._epsilon == 0
    pol.train()
    assert pol._epsilon == 0  # reference quirk (App. D.1)
    # batched Philox path: epsilon=1 -> uniform random actions, epsilon=0 -> argmax of masked q
    obs = torch.from_numpy(g["obs"]).cuda()
    _, a0 = dqn.act(obs, None, epsilon=0.0)
    assert np.array_equal(a0.cpu().numpy(), g["q"].argmax(-1))
    _, a1 = dqn.act(obs.repeat(200, 1, 1), None, epsilon=1.0, seed=3, step=9)
    cnt = np.bincount(a1.cpu().numpy().ravel(), minlength=4) / a1.numel()
    assert np.abs(cnt - 0.25).max() < 0.02


def test_replay_ring_golden():
    from graph_marl_b200.replaybuffer import ReplayBuffer

    g = load_golden("replay")
    seed, cap, A, D, S, N, Dn, Sn, Ax, n_add = [int(x) for x in g["cfg"]]
    rb = ReplayBuffer(seed, cap, A, D, S, N, Dn, Sn, Ax)
    T = lambda k, i: g["tr_" + k][i]
    for i in range(n_add):
        rb.add(T("obs", i), T("action", i), T("reward", i), T("next_obs", i), T("adj", i), T("next_adj", i),
               T("done", i), bool(T("episode_done", i)), 0, T("node_state", i), T("node_aux", i), T("node_obs", i),
               T("node_adj", i), T("node_agent", i), T("next_node_obs", i), T("next_node_adj", i),
               T("next_node_agent", i))
        if i == 9:
            b = next(rb.get_batch(4, "cuda"))
            assert np.array_equal(b.idx, g["idx_partial"])
            assert np.array_equal(b.obs.cpu().numpy(), g["obs_partial"])
            seq = list(rb.get_batch(4, "cuda", sequence_length=3))
            assert np.array_equal(np.stack([s.idx for s in seq]), g["idx_seq_partial"])
    b = next(rb.get_batch(6, "cuda"))
    assert np.array_equal(b.idx, g["idx_full"])
    for f in b._fields:
        if f == "idx":
            continue
        got = getattr(b, f)
        ref = g["full_" + f]
        assert got.cpu().numpy().dtype == ref.dtype, f
        assert np.array_equal(got.cpu().numpy(), ref), f
    seq = list(rb.get_batch(5, "cuda", sequence_length=4))
    assert np.array_equal(np.stack([s.idx for s in seq]), g["idx_seq_full"])
    assert np.array_equal(np.stack([s.node_state.cpu().numpy() for s in seq]), g["seq_full_node_state"])
    assert [rb.index, rb.count] == g["final_index_count"].tolist()
    # batched insert == n single inserts
    rb2 = ReplayBuffer(seed, cap, A, D, S, N, Dn, Sn, Ax)
    for lo in (0, 7, 14, 21):
        hi = min(n_add, lo + 7)
        sl = slice(lo, hi)
        rb2.add(*[torch.from_numpy(np.ascontiguousarray(g["tr_" + k][sl])).cuda() for k in
                  ("obs", "action", "reward", "next_obs", "adj", "next_adj", "done", "episode_done")], 0,
                *[torch.from_numpy(np.ascontiguousarray(g["tr_" + k][sl])).cuda() for k in
                  ("node_state", "node_aux", "node_obs", "node_adj", "node_agent", "next_node_obs", "next_node_adj",
                   "next_node_agent")], num=hi - lo)
    for name in ("obs", "action", "done", "node_state", "next_node_agent_matrix", "episode_done"):
        assert torch.equal(getattr(rb, name), getattr(rb2, name)), name
    assert (rb2.index, rb2.count) == (rb.index, rb.count)


def test_wrapper_closed_loop_golden():
    """NetMonWrapper over the CUDA env in compat mode reproduces the reference's joint
    observations, last/current NetMon state bookkeeping and startup iterations."""
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from graph_marl_b200.env.wrapper import NetMonWrapper
    from graph_marl_b200.model import NetMon

    g = load_golden("wrapper")
    Dn, H, e1, K, wseed, startup = [int(x) for x in g["cfg"]]
    nm = NetMon(Dn, H, (e1,), K, F.leaky_relu, rnn_type="lstm", output_neighbor_hidden=True)
    w = det_weights(netmon_shapes(Dn, H, [e1], "lstm"), wseed)
    nm.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    nm = nm.cuda().eval()
    np.random.seed(31)
    net = Network(20, random_topology=False, topology_init_seed=923430603)
    env = NetMonWrapper(Routing(net, 20, 1), nm, startup)
    obs, adj = env.reset()
    assert obs.shape == g["joint_obs"][0].shape
    assert np.array_equal(obs[:, :130], g["joint_obs"][0][:, :130])
    assert np.abs(obs - g["joint_obs"][0]).max() < 1e-4
    for t in range(g["actions"].shape[0]):
        assert np.abs(env.last_netmon_state.cpu().numpy()[0] - g["last_state"][t][0]).max() < 1e-4
        obs, adj, rew, done, info = env.step(g["actions"][t])
        assert np.array_equal(obs[:, :130], g["joint_obs"][t + 1][:, :130]), t
        assert np.abs(obs - g["joint_obs"][t + 1]).max() < 1e-4, t
        assert np.abs(env.current_netmon_state.cpu().numpy()[0] - g["cur_state"][t][0]).max() < 1e-4
        node_obs, node_adj, nam = env.get_netmon_info()
        assert node_obs.shape == (20, 88) and node_adj.shape == (20, 20) and nam.shape == (20, 20)


def test_replay_half_precision_golden():
    """ReplayBuffer(half_precision=True) (replaybuffer.py:52-54): float fields are stored as fp16 (round to nearest
    even, like numpy's assignment) and sampled back as fp32 (gm_replay_sample convert 3); flags / actions as usual."""
    from graph_marl_b200.replaybuffer import ReplayBuffer

    g = load_golden("replay_half")
    seed, cap, A, D, S, N, Dn, Sn, Ax, n_add = [int(x) for x in g["cfg"]]
    rb = ReplayBuffer(seed, cap, A, D, S, N, Dn, Sn, Ax, half_precision=True)
    assert rb.obs.dtype == torch.float16 and rb.node_state.dtype == torch.float16 and rb.reward.dtype == torch.float16
    T = lambda k, i: g["tr_" + k][i]
    for i in range(n_add):
        rb.add(T("obs", i), T("action", i), T("reward", i), T("next_obs", i), T("adj", i), T("next_adj", i),
               T("done", i), bool(T("episode_done", i)), 0, T("node_state", i), T("node_aux", i), T("node_obs", i),
               T("node_adj", i), T("node_agent", i), T("next_node_obs", i), T("next_node_adj", i),
               T("next_node_agent", i))
    b = next(rb.get_batch(6, "cuda"))
    assert np.array_equal(b.idx, g["idx_full"])
    for f in b._fields:
        if f == "idx":
            continue
        got, ref = getattr(b, f).cpu().numpy(), g["full_" + f]
        assert got.dtype == ref.dtype, f
        assert np.array_equal(got, ref), f


def test_wrapper_freeze_golden():
    """NetMonWrapper.freeze() (wrapper.py:53-75) in compat mode against the reference: after the freeze the NetMon
    state stops advancing and the agents read the frozen node readout at their new nodes; `env.data` exposes the
    packets with the reference's attribute names (routing.py:12-40) for the heuristic policies (policy.py:90-139)."""
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from graph_marl_b200.env.wrapper import NetMonWrapper
    from graph_marl_b200.model import NetMon

    g = load_golden("wrapper_freeze")
    Dn, H, e1, K, wseed, startup = [int(x) for x in g["cfg"]]
    nm = NetMon(Dn, H, (e1,), K, F.leaky_relu, rnn_type="lstm", output_neighbor_hidden=True)
    nm.load_state_dict({k: torch.from_numpy(v) for k, v in det_weights(netmon_shapes(Dn, H, [e1], "lstm"), wseed).items()})
    nm = nm.cuda().eval()
    np.random.seed(77)
    net = Network(20, random_topology=False, topology_init_seed=923430603)
    env0 = Routing(net, 20, 1)
    env = NetMonWrapper(env0, nm, startup)
    obs, adj = env.reset()
    assert np.abs(obs - g["joint_obs"][0]).max() < 1e-4
    fz = int(g["freeze_at"][0])
    for t in range(g["actions"].shape[0]):
        if t == fz:
            env.freeze()
        obs, adj, rew, done, info = env.step(g["actions"][t])
        assert np.array_equal(obs[:, :130], g["joint_obs"][t + 1][:, :130]), t
        assert np.abs(obs - g["joint_obs"][t + 1]).max() < 1e-4, t
        assert np.abs(env.current_netmon_state.cpu().numpy()[0] - g["cur_state"][t][0]).max() < 1e-4, t
        assert np.array_equal(env.get_netmon_info()[2], g["node_agent"][t]), t
        got = np.array([[p.now, p.target, p.edge, p.time, p.ttl, p.shortest_path_weight, p.start] for p in env0.data], dtype=np.int32)
        assert np.array_equal(got, g["data"][t]), t
    assert np.array_equal(g["cur_state"][fz - 1], g["cur_state"][-1])  # the recording itself: no step after the freeze
    assert np.array_equal(np.array([p.size for p in env0.data]), g["sizes"])
    assert [p.id for p in env0.data] == list(range(20))


@pytest.mark.parametrize("math", ["fp32", "bf16x3"])
def test_wrapper_freeze_batched_lean_mode(math):
    """freeze() in the batched split mode the rollout uses (only the agents' rows are read out, tile-packed on the
    tensor-core path): the node readout of the latest NetMon step is rebuilt when freeze() is called, and the frozen
    graph observations equal those of a wrapper that kept the full node readout all along."""
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from graph_marl_b200.env.wrapper import NetMonWrapper
    from graph_marl_b200.model import NetMon

    B, N, A, H = 37, 20, 20, 64
    torch.manual_seed(3)
    nm = NetMon(4 * N + 8, H, (96,), 2, F.leaky_relu, rnn_type="lstm", output_neighbor_hidden=True, math=math).cuda().eval()
    mk = lambda split, fp32: NetMonWrapper(Routing(Network(N, random_topology=False, topology_init_seed=923430603), A, 1,
                                                   num_envs=B, seed=5, batched=True), nm, 1, split_obs=split, graph_obs_fp32=fp32)
    full, lean = mk(False, True), mk(True, False)
    jo, _ = full.reset()
    (la, lg), _ = lean.reset()
    g = torch.Generator(device="cuda").manual_seed(1)
    for t in range(7):
        if t == 3:
            full.freeze(), lean.freeze()
        act = torch.randint(0, 4, (B, A), device="cuda", generator=g, dtype=torch.int32)
        jo, _, r0, _, _ = full.step(act)
        (la, lg), _, r1, _, _ = lean.step(act)
        assert torch.equal(r0, r1) and torch.equal(jo[..., :6 * N + 10], la)
        if t >= 3:
            assert torch.is_tensor(lg) and torch.equal(jo[..., 6 * N + 10:], lg), t
            assert torch.equal(full.current_netmon_state, lean.current_netmon_state)


def test_ci_known_answer_simple_env_training_reaches_reward_mean_1():
    """The reference's only known-answer test (.github/workflows/train-example.yml:26-27, BASELINE
    config 1): DQN + NetMon on SimpleEnvironment, 5000 steps, final evaluation reward_mean == 1.0 --
    with the classes of this package dropped into the reference's rollout/learner/eval loop."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import train_simple

    metrics = train_simple.main(["--total-steps", "5000", "--step-before-train", "1000", "--eval-episodes", "100"])
    assert metrics["reward_mean"] == 1.0


def test_unmodified_reference_main_py_runs_on_the_package(tmp_path):
    """The drop-in claim, demonstrated: the reference's own src/main.py (staged, unedited, at baseline/_ref/src) runs its
    CI command (.github/workflows/train-example.yml:26-27, BASELINE config 1; --device=cuda because this package has no
    CPU path) with env.* / model.NetMon,DQN,MLP / policy.EpsilonGreedy / replaybuffer / buffer aliased to graph_marl_b200
    (tools/run_reference_driver.py) and prints the known answer `"reward_mean": 1.0`."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.exists(os.path.join(root, "baseline", "_ref", "src", "main.py")):
        pytest.skip("runs the original project's own driver: needs a copy of its src/ at baseline/_ref/src")
    cmd = [sys.executable, os.path.join(root, "tools", "run_reference_driver.py"), "main.py"] + (
        "--model=dqn --hidden-dim=8 --random-topology=1 --mini-batch-size=32 --device=cuda --episode-steps=1 "
        "--eval-episode-steps=1 --lr=0.001 --tau=0.01 --netmon --netmon-encoder-dim=4 --hidden-dim=4 --netmon-dim=2 "
        "--netmon-iterations=1 --sequence-length=1 --step-before-train=1_000 --capacity=10_000 --eval-episodes=100 "
        "--total-steps=5_000 --env-type=simple --epsilon=0.1 --epsilon-decay=1.0 --seed=0 --disable-progress").split()
    r = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert '"reward_mean": 1.0' in r.stdout, r.stdout[-3000:]


def test_unmodified_reference_sl_py_runs_on_the_package(tmp_path):
    """BASELINE config 5 through the reference's own, unedited src/sl.py (tools/run_reference_driver.py): dataset generation
    with the native topology generator behind `Network` / `Routing`, 40 training iterations of NetMonSL (8-... step
    sequences unrolled through the device-side backward: no torch-composed fallback may be reported), validation and the
    test evaluations on the EVAL_SEEDS graphs."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.exists(os.path.join(root, "baseline", "_ref", "src", "sl.py")):
        pytest.skip("runs the original project's own driver: needs a copy of its src/ at baseline/_ref/src")
    cmd = [sys.executable, os.path.join(root, "tools", "run_reference_driver.py"), "sl.py", "--iterations", "40",
           "--num-samples-train", "200", "--validate-after", "20", "--test-sequence-lengths", "1,4", "--disable-progressbar"]
    r = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "NetMon Module (libgraphmarl_b200)" in r.stdout and "Extended test data eval (seq_len=4)" in r.stdout
    assert "torch-composed" not in r.stderr and "torch-composed" not in r.stdout
    losses = [float(l.split()[-1]) for l in r.stdout.splitlines() if l.startswith("Pred_all loss")]
    assert len(losses) >= 3 and all(np.isfinite(losses))
