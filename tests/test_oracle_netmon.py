"""The numpy oracle for NetMon / DQN / epsilon-greedy / replay against reference outputs."""
import numpy as np
import pytest

from conftest import load_golden
from helpers import det_weights, dqn_shapes, netmon_case, netmon_shapes
from oracle import netmon_oracle as NO

G = load_golden("netmon")
# fp32 tolerance of the oracle restatement vs torch CPU fp32 (different summation order).
# lnlstm is ill-conditioned (SURVEY 7.4): LayerNorm over near-constant gate vectors.
TOL = {"lstm": 2e-6, "gru": 2e-6, "none": 2e-5, "lnlstm": 2e-4}


@pytest.mark.parametrize("entry", [str(x) for x in G["case_names"]])
def test_netmon_recurrent_rollout(entry):
    name, cfg = netmon_case(G, entry)
    X, ADJ, NAM = G["node_obs"], G["node_adj"], G["node_agent"]
    w = det_weights(netmon_shapes(X.shape[-1], cfg["hidden"], cfg["enc"], cfg["rnn_type"]), cfg["wseed"])
    state = None
    tol = TOL[cfg["rnn_type"]]
    for t in range(X.shape[0]):
        out, state, agent_out = NO.netmon_forward(w, cfg, X[t], ADJ[t], state, node_agent=NAM[t])
        assert agent_out.shape == G[name + "_agent_out"][t].shape
        assert np.abs(agent_out - G[name + "_agent_out"][t]).max() < tol, t
        assert np.abs(state - G[name + "_state"][t]).max() < tol, t
        # gather == bmm with the one-hot node-agent matrix
        agent_node = NAM[t].argmax(axis=1)
        _, _, ao2 = NO.netmon_forward(w, cfg, X[t], ADJ[t], G[name + "_state"][t - 1] if t else None,
                                      agent_node=agent_node)
        assert np.abs(ao2 - G[name + "_agent_out"][t]).max() < tol


@pytest.mark.parametrize("entry", [str(x) for x in G["case_names"] if str(x).split("|")[1] in ("lstm", "lnlstm")
                                   and netmon_case(G, x)[1]["rnn_carryover"]])
def test_fp64_autograd_reference_reproduces_recording(entry):
    """`NetMon._forward_autograd` of a `.double()` module, the fp64 reference that tests/test_gpu_train_kernels.py
    differentiates, reproduces the reference's recorded agent outputs and carried states."""
    import torch
    import torch.nn.functional as F

    from graph_marl_b200.model import NetMon

    name, cfg = netmon_case(G, entry)
    X, ADJ, NAM = G["node_obs"], G["node_adj"], G["node_agent"]
    T, B, N, Dn = X.shape
    nm = NetMon(Dn, cfg["hidden"], cfg["enc"], cfg["iterations"], F.leaky_relu, rnn_type=cfg["rnn_type"],
                agg_type=cfg["agg_type"], output_neighbor_hidden=cfg["output_neighbor_hidden"],
                output_global_hidden=cfg["output_global_hidden"])
    w = det_weights(netmon_shapes(Dn, cfg["hidden"], cfg["enc"], cfg["rnn_type"]), cfg["wseed"])
    nm.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    nm.double()
    nm.state = torch.zeros((B, N, nm.state_size), dtype=torch.float64)
    tol = TOL[cfg["rnn_type"]]
    with torch.no_grad():
        for t in range(T):
            out = nm._forward_autograd(torch.from_numpy(X[t]).double(), torch.from_numpy(ADJ[t]).double(),
                                       torch.from_numpy(NAM[t]).double(), None, False)
            assert out.dtype == torch.float64 and out.shape == G[name + "_agent_out"][t].shape
            assert np.abs(out.numpy() - G[name + "_agent_out"][t]).max() < tol, t
            assert np.abs(nm.state.numpy() - G[name + "_state"][t]).max() < tol, t


def test_netmon_simple_env_degree2_readout():
    cfg = dict(hidden=8, iterations=2, rnn_type="lstm", rnn_carryover=True, agg_type="sum",
               output_neighbor_hidden=True, output_global_hidden=False)
    w = det_weights(netmon_shapes(1, 8, [6], "lstm"), 4242)
    out, _, _ = NO.netmon_forward(w, cfg, G["simple_node_obs"][None], G["simple_node_adj"][None])
    assert out.shape == G["simple_node_out"].shape == (1, 3, 8 * 3)  # max degree 2 (App. D.3)
    assert np.abs(out - G["simple_node_out"]).max() < 2e-6


def test_dqn_and_epsilon_greedy():
    g = load_golden("dqn_policy")
    D, h1, h2, n_act, wseed = [int(x) for x in g["cfg"]]
    w = det_weights(dqn_shapes(D, [h1, h2], n_act), wseed)
    q = NO.dqn_forward(w, g["obs"])
    assert np.abs(q - g["q"]).max() < 5e-6
    eps = 0.5
    for t in range(g["obs"].shape[0]):
        a = NO.epsilon_greedy(g["q"][t], eps, g["rand_action"][t], g["rand_u"][t], g["masks"][t])
        assert np.array_equal(a, g["actions"][t]), t
        eps = NO.epsilon_decay(eps, t + 1, 3, 2, 0.5)
        assert eps == g["eps_after"][t]
    assert g["eps_eval"][0] == 0 and g["eps_train"][0] == 0  # train() never restores (App. D.1)


def test_replay_index_sampling():
    g = load_golden("replay")
    seed, cap = int(g["cfg"][0]), int(g["cfg"][1])
    n_add = int(g["cfg"][-1])
    r = NO.ReplayIndexOracle(seed, cap)
    slots = []
    for i in range(n_add):
        slots.append(r.add())
        if i == 9:
            assert np.array_equal(r.sample(4)[0], g["idx_partial"])
            assert np.array_equal(g["obs_partial"], g["tr_obs"][g["idx_partial"]])
            assert np.array_equal(np.stack(r.sample(4, 3)), g["idx_seq_partial"])
    assert np.array_equal(r.sample(6)[0], g["idx_full"])
    assert np.array_equal(np.stack(r.sample(5, 4)), g["idx_seq_full"])
    assert [r.index, r.count] == g["final_index_count"].tolist()
    # ring content: slot s holds the last transition written to it
    last_writer = {s: i for i, s in enumerate(slots)}
    src = np.array([last_writer[int(s)] for s in g["idx_full"]])
    assert np.array_equal(g["full_obs"], g["tr_obs"][src])
    assert np.array_equal(g["full_action"], g["tr_action"][src].astype(np.int64))
    assert g["full_adj"].dtype == np.float32 and np.array_equal(g["full_adj"], g["tr_adj"][src].astype(np.float32))
    assert np.array_equal(g["full_done"], g["tr_done"][src])


def test_cpu_rollout_torch_backend_matches_numpy_backend():
    """oracle/cpu_rollout.py (the timed CPU baseline): the multi-threaded torch backend computes the same
    rollout as the numpy restatement (same seeds -> same draws; fp32 summation-order noise only)."""
    import torch
    from oracle.cpu_rollout import CpuRollout
    from helpers import det_weights, dqn_shapes, netmon_shapes

    N = A = 20
    H, K, enc, dq = 32, 2, (48, 40), (36, 28)
    w_nm = det_weights(netmon_shapes(4 * N + 8, H, list(enc), "lstm"), 3)
    w_dq = det_weights(dqn_shapes(6 * N + 10 + 4 * H, list(dq), 4), 5)
    mk = lambda be: CpuRollout(N, A, 923430603, True, K, "lstm", H, enc, dq, 6, 2, w_nm, w_dq, replay_capacity=12, seed=1, backend=be)
    a, b = mk("numpy"), mk("torch")
    a.reset(), b.reset()
    for t in range(4):
        ra, rb = a.step(epsilon=1.0), b.step(epsilon=1.0)  # epsilon 1: actions come from the shared draw stream
        assert np.array_equal(ra, rb), t
        assert np.array_equal(a.env.now, b.env.now) and np.array_equal(a.env.load, b.env.load)
        assert np.abs(np.asarray(a.joint) - b.joint.numpy()).max() < 1e-5
        assert np.abs(np.asarray(a.state) - b.state.numpy()).max() < 1e-5
