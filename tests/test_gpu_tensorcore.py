"""GPU parity of the tcgen05 paths of NetMon / DQN (fused aggregate + gate GEMM + LSTM-cell kernel,
packed-weight cache, two-segment DQN input) against the reference's recorded outputs and the fp64
numpy oracle.

Stated tolerances (max abs error on outputs of magnitude O(1), identical weights + inputs):
  bf16x3 (fp32-accurate split): 1e-4 single step, 3e-4 over the recorded recurrent rollouts
  bf16   (single pass)        : 3e-2 -- reported as a speed/accuracy option, not the parity mode
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden
from helpers import det_weights, dqn_shapes, netmon_case, netmon_shapes

pytestmark = pytest.mark.gpu

G = load_golden("netmon")
LSTM_CASES = [str(x) for x in G["case_names"] if str(x).split("|")[1] in ("lstm", "gru", "none")]


def _netmon(cfg, in_features, math):
    from graph_marl_b200.model import NetMon

    nm = NetMon(in_features, cfg["hidden"], cfg["enc"], cfg["iterations"], F.leaky_relu, rnn_type=cfg["rnn_type"],
                rnn_carryover=cfg["rnn_carryover"], agg_type=cfg["agg_type"],
                output_neighbor_hidden=cfg["output_neighbor_hidden"],
                output_global_hidden=cfg["output_global_hidden"], math=math)
    w = det_weights(netmon_shapes(in_features, cfg["hidden"], cfg["enc"], cfg["rnn_type"]), cfg["wseed"])
    nm.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    return nm.cuda().eval(), w


@pytest.mark.parametrize("entry", LSTM_CASES)
def test_netmon_golden_rollout_bf16x3(entry):
    name, cfg = netmon_case(G, entry)
    X, ADJ, NAM = G["node_obs"], G["node_adj"], G["node_agent"]
    nm, _ = _netmon(cfg, X.shape[-1], "bf16x3")
    with torch.no_grad():
        nm.state = None
        for t in range(X.shape[0]):
            out = nm(torch.from_numpy(X[t]).cuda(), torch.from_numpy(ADJ[t]).float().cuda(),
                     torch.from_numpy(NAM[t]).float().cuda())
            err = np.abs(out.cpu().numpy() - G[name + "_agent_out"][t]).max()
            serr = np.abs(nm.state.cpu().numpy() - G[name + "_state"][t]).max()
            assert err < 3e-4 and serr < 3e-4, (t, err, serr)


@pytest.mark.parametrize("math,tol", [("bf16x3", 1e-4), ("bf16", 3e-2)])
@pytest.mark.parametrize("K,agg,B,N", [(3, "sum", 96, 20), (1, "mean", 7, 20), (2, "sum", 5, 200)])
def test_netmon_fused_cells_against_fp64_oracle(K, agg, B, N, math, tol):
    from oracle import netmon_oracle as NO
    from oracle import oracle as O

    Dn, H = 4 * N + 8, 128
    cfg = dict(hidden=H, iterations=K, rnn_type="lstm", rnn_carryover=True, agg_type=agg, output_neighbor_hidden=True,
               output_global_hidden=False, enc=[512, 256], wseed=31)
    nm, w = _netmon(cfg, Dn, math)
    topo = O.generate_topology(N, seed=923430603 if N == 20 else 476)
    rng = np.random.default_rng(2)
    x = ((rng.random((B, N, Dn)) < 0.05).astype(np.float32) + rng.random((B, N, Dn)).astype(np.float32) * (rng.random((B, N, Dn)) < 0.02))
    mask = np.broadcast_to(topo["adj"], (B, N, N)).astype(np.float32)
    st = (rng.standard_normal((B, N, 2 * H)) * 0.3).astype(np.float32)
    agent_node = rng.integers(0, N, (B, 11)).astype(np.int32)
    ref_out, ref_state, ref_agent = NO.netmon_forward(w, cfg, x, mask, st, agent_node=agent_node, dtype=np.float64)
    from graph_marl_b200.model import NetMon

    with torch.no_grad():
        # dense-mask API
        nm.state = torch.from_numpy(st).cuda()
        out = nm(torch.from_numpy(x).cuda(), torch.from_numpy(mask.copy()).cuda(), None, no_agent_mapping=True)
        assert np.abs(out.cpu().numpy() - ref_out).max() < tol
        assert np.abs(nm.state.cpu().numpy() - ref_state).max() < tol
        # list API with a shared list table + agent gather, state None on a second module call chain
        nbr, deg, dm = NetMon.lists_from_mask(torch.from_numpy(mask[:1].copy()).cuda())
        nm.state = torch.from_numpy(st).cuda()
        _, ao = nm.forward_lists(torch.from_numpy(x).cuda(), nbr, deg, None, 3, agent_node=torch.from_numpy(agent_node).cuda())
        assert np.abs(ao.cpu().numpy() - ref_agent).max() < tol
        # zero initial state
        ref0, ref_state0, _ = NO.netmon_forward(w, cfg, x, mask, None, dtype=np.float64)
        nm.state = None
        out0 = nm(torch.from_numpy(x).cuda(), torch.from_numpy(mask.copy()).cuda(), None, no_agent_mapping=True)
        assert np.abs(out0.cpu().numpy() - ref0).max() < tol
        assert np.abs(nm.state.cpu().numpy() - ref_state0).max() < tol


# the last case gives every CTA 2-3 M tiles (320 tiles over 148 SMs): both epilogue groups and the reuse of the
# resident activation blocks are exercised
@pytest.mark.parametrize("K,agg,B,N,A", [(3, "sum", 96, 20, 20), (1, "mean", 7, 20, 11), (4, "sum", 5, 200, 100),
                                         (2, "sum", 2048, 20, 20)])
def test_netmon_fused_layernorm_cell_against_fp64_oracle(K, agg, B, N, A):
    """LayerNormLSTM cell on the tensor cores (EPI_LNLSTM: Gram-matrix row statistics + two accumulators per tile).
    Stated tolerance: 1e-3 max abs on the new state and the readout, single step from an identical state
    (SURVEY Appendix B: 'lnlstm atol 1e-3'; the fp32 reference itself sits 5e-6 from fp64 here)."""
    from oracle import netmon_oracle as NO
    from oracle import oracle as O
    from graph_marl_b200.model import NetMon

    Dn, H, tol = 4 * N + 8, 128, 1e-3
    cfg = dict(hidden=H, iterations=K, rnn_type="lnlstm", rnn_carryover=True, agg_type=agg, output_neighbor_hidden=True,
               output_global_hidden=False, enc=[512, 256], wseed=41)
    nm, w = _netmon(cfg, Dn, "bf16x3")
    topo = O.generate_topology(N, seed=923430603 if N == 20 else 476)
    rng = np.random.default_rng(5)
    x = ((rng.random((B, N, Dn)) < 0.05).astype(np.float32) + rng.random((B, N, Dn)).astype(np.float32) * (rng.random((B, N, Dn)) < 0.02))
    mask = np.broadcast_to(topo["adj"], (B, N, N)).astype(np.float32)
    st = (rng.standard_normal((B, N, 2 * H)) * 0.3).astype(np.float32)
    agent_node = rng.integers(0, N, (B, A)).astype(np.int32)
    ref_out, ref_state, ref_agent = NO.netmon_forward(w, cfg, x, mask, st, agent_node=agent_node, dtype=np.float64)
    with torch.no_grad():
        nbr, deg, dm = NetMon.lists_from_mask(torch.from_numpy(mask[:1].copy()).cuda())
        nm.state = torch.from_numpy(st).cuda()
        no, ao = nm.forward_lists(torch.from_numpy(x).cuda(), nbr, deg, None, 3, agent_node=torch.from_numpy(agent_node).cuda(),
                                  want_node_out=True, want_agent_pk=True)
        got_state = nm.state.cpu().numpy()
        eh = np.abs(got_state[..., :H] - ref_state[..., :H]).max()
        ec = np.abs(got_state[..., H:] - ref_state[..., H:]).max()
        assert eh < tol and ec < tol, (eh, ec)
        assert np.abs(no.cpu().numpy() - ref_out).max() < tol
        assert np.abs(ao.cpu().numpy() - ref_agent).max() < tol
        # zero initial state (h = 0: the hidden-side gate vector is constant, LayerNorm divides by sqrt(eps))
        ref0, ref_state0, _ = NO.netmon_forward(w, cfg, x, mask, None, dtype=np.float64)
        nm.state = None
        out0 = nm(torch.from_numpy(x).cuda(), torch.from_numpy(mask.copy()).cuda(), None, no_agent_mapping=True)
        assert np.abs(out0.cpu().numpy() - ref0).max() < tol
        assert np.abs(nm.state.cpu().numpy() - ref_state0).max() < tol
        # same inputs through the fp32 SIMT path of the library: both implementations agree
        nm32, _ = _netmon(cfg, Dn, "fp32")
        nm32.state = torch.from_numpy(st).cuda()
        no32, _ = nm32.forward_lists(torch.from_numpy(x).cuda(), nbr, deg, None, 3, want_node_out=True)
        assert np.abs(no32.cpu().numpy() - no.cpu().numpy()).max() < tol


@pytest.mark.parametrize("math,tol", [("bf16x3", 1e-3), ("fp32", 1e-3)])
def test_netmon_layernorm_cell_single_step_from_reference_recording(math, tol):
    """The LayerNormLSTM cell (tcgen05 EPI_LNLSTM for bf16x3, the FFMA path for fp32) against the UNMODIFIED reference:
    every step of the `lnlstm_sum_k4_paper` recording restarted from the reference's own recorded state (single step
    from identical state; SURVEY Appendix B tolerance 1e-3)."""
    from graph_marl_b200.model import NetMon

    name, cfg = netmon_case(G, [x for x in G["case_names"] if str(x).startswith("lnlstm_sum_k4_paper")][0])
    X, ADJ, NAM = G["node_obs"], G["node_adj"], G["node_agent"]
    nm, _ = _netmon(cfg, X.shape[-1], math)
    with torch.no_grad():
        for t in range(X.shape[0]):
            nbr, deg, dm = NetMon.lists_from_mask(torch.from_numpy(ADJ[t]).float().cuda())
            nm.state = torch.from_numpy(G[name + "_state"][t - 1]).cuda() if t else None
            agent_node = torch.from_numpy(NAM[t].argmax(axis=1).astype(np.int32)).cuda()
            _, ao = nm.forward_lists(torch.from_numpy(X[t]).cuda(), nbr, deg, None, 3, agent_node=agent_node,
                                     want_agent_pk=(math != "fp32"))
            err = np.abs(ao.cpu().numpy() - G[name + "_agent_out"][t]).max()
            serr = np.abs(nm.state.cpu().numpy() - G[name + "_state"][t]).max()
            assert err < tol and serr < tol, (t, err, serr)


def _tc_launches(fn):
    """Tensor-core launches (library profile category 0) that fn() makes."""
    import ctypes as C
    from graph_marl_b200 import _lib
    L = _lib.lib()
    L.gm_profile_enable(1)
    try:
        out = fn()
    finally:
        L.gm_profile_enable(0)
    ms, cnt = (C.c_double * 8)(), (C.c_int32 * 8)()
    _lib.check(L.gm_profile_collect(ms, cnt))
    return out, int(cnt[0])


@pytest.mark.parametrize("B", [37, 512, 2048])  # 2048 envs = 320 M tiles: up to three tiles per CTA, rings wrap
def test_netmon_fused_encoder_with_static_rows_from_the_env(B):
    """The 6-term form: the Routing env hands NetMon its node rows as sparse entries whose constant part (one-hots,
    edge lengths) is ONE entry naming a static row that the weight pack folded into layer 1 (single-topology pool).
    Same state and observations through the dense tensor-core path: 2e-5; the pack follows a topology change."""
    from graph_marl_b200.env.network import Network
    from graph_marl_b200.env.routing import Routing
    from graph_marl_b200.model import NetMon

    N = A = 20
    env = Routing(Network(N, random_topology=False, topology_init_seed=923430603), A, 1, num_envs=B, seed=2, batched=True)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(5):
        env.step(torch.randint(0, 4, (B, A), device="cuda", generator=g, dtype=torch.int32))
    assert env.node_obs_nnz == 6 and env.node_static_rows.shape == (N + 5, 4 * N + 8)
    torch.manual_seed(1)
    nm = NetMon(4 * N + 8, 128, (512, 256), 2, F.leaky_relu, output_neighbor_hidden=True, math="bf16x3").cuda().eval()
    nbr_all, deg, list_index = env.get_adjacency_lists()
    st = torch.randn(B, N, 256, device="cuda") * 0.3
    outs, n_tc = [], []
    with torch.no_grad():
        # the same rows once more in the mixed form (static_only=False): entry 0 names static row s as column Dn + s, the
        # dynamic entries are ordinary input columns
        Dn = 4 * N + 8
        dyn_cols = torch.tensor([N, N + 1] + [N + 2 + q * (N + 2) + N + 1 for q in range(3)], device="cuda", dtype=torch.int32)
        mixed = env._out["node_sparse"].clone()
        mixed[..., 0] += Dn
        mixed[..., 1:6] = dyn_cols
        for kw in (dict(), dict(sparse_nnz=12), dict(sparse_nnz=env.node_obs_nnz, sparse_rows=env._out["node_sparse"], static_rows=env.node_static_rows),
                   dict(sparse_nnz=6, sparse_rows=mixed, static_rows=env.node_static_rows[:N].contiguous(), static_only=False)):
            nm.state = st.clone()
            (no, _), n = _tc_launches(lambda: nm.forward_lists(env._out["node_obs"], nbr_all, deg, list_index, 3, want_node_out=True, **kw))
            outs.append((no, nm.state))
            n_tc.append(n)
    # the 6-term forms run layers 1 + 2 as ONE tensor-core launch; derived 12-term rows take the two-layer path by default
    assert n_tc[1] == n_tc[0] and n_tc[2] == n_tc[0] - 1 and n_tc[3] == n_tc[0] - 1, n_tc
    for no, s2 in outs[1:]:
        assert float((no - outs[0][0]).abs().max()) < 2e-5 and float((s2 - outs[0][1]).abs().max()) < 2e-5
    # another topology: new static rows -> the cached pack must be rebuilt (same module, same weights)
    env2 = Routing(Network(N, random_topology=False, topology_init_seed=476 if False else 923430603 + 0), A, 1, num_envs=B, seed=3, batched=True)
    env2.network = Network(N, random_topology=True, n_random_seeds=1, topology_init_seed=5)
    env2.reset()
    assert env2.node_static_rows is not None and not torch.equal(env2.node_static_rows, env.node_static_rows)
    nbr2, deg2, li2 = env2.get_adjacency_lists()
    with torch.no_grad():
        nm.state = st.clone()
        a, _ = nm.forward_lists(env2._out["node_obs"], nbr2, deg2, li2, 3, want_node_out=True)
        nm.state = st.clone()
        b, _ = nm.forward_lists(env2._out["node_obs"], nbr2, deg2, li2, 3, want_node_out=True, sparse_nnz=env2.node_obs_nnz,
                                sparse_rows=env2._out["node_sparse"], static_rows=env2.node_static_rows)
    assert float((a - b).abs().max()) < 2e-5
    # a pool of three topologies: the dictionary holds 3N + 5 rows and an env's rows index its own topology's block
    env3 = Routing(Network(N, random_topology=True, n_random_seeds=3, topology_init_seed=11), A, 1, num_envs=B, seed=4, batched=True)
    env3.reset()
    for _ in range(3):
        env3.step(torch.randint(0, 4, (B, A), device="cuda", generator=g, dtype=torch.int32))
    assert env3.node_obs_nnz == 6 and env3.node_static_rows.shape == (3 * N + 5, 4 * N + 8)
    nbr3, deg3, li3 = env3.get_adjacency_lists()
    assert int(li3.max()) > 0  # more than one topology in use
    with torch.no_grad():
        nm.state = st.clone()
        a, _ = nm.forward_lists(env3._out["node_obs"], nbr3, deg3, li3, 3, want_node_out=True)
        nm.state = st.clone()
        (b, _), n = _tc_launches(lambda: nm.forward_lists(env3._out["node_obs"], nbr3, deg3, li3, 3, want_node_out=True,
                                                          sparse_nnz=env3.node_obs_nnz, sparse_rows=env3._out["node_sparse"],
                                                          static_rows=env3.node_static_rows))
    assert n == n_tc[0] - 1 and float((a - b).abs().max()) < 2e-5


def test_packed_weight_cache_follows_parameter_updates():
    cfg = dict(hidden=64, iterations=1, rnn_type="lstm", rnn_carryover=True, agg_type="sum", output_neighbor_hidden=True,
               output_global_hidden=False, enc=[32], wseed=3)
    from oracle import netmon_oracle as NO
    from oracle import oracle as O

    N = 20
    nm, w = _netmon(cfg, 4 * N + 8, "bf16x3")
    topo = O.generate_topology(N, seed=923430603)
    rng = np.random.default_rng(0)
    x = rng.random((3, N, 4 * N + 8)).astype(np.float32)
    mask = np.broadcast_to(topo["adj"], (3, N, N)).astype(np.float32)
    with torch.no_grad():
        for scale in (1.0, 0.5):
            for q in nm.parameters():
                q.mul_(scale)  # in-place update bumps the version counter -> repack
            w2 = {k: v.detach().cpu().numpy() for k, v in nm.state_dict().items()}
            ref, _, _ = NO.netmon_forward(w2, cfg, x, mask, None, dtype=np.float64)
            nm.state = None
            out = nm(torch.from_numpy(x).cuda(), torch.from_numpy(mask.copy()).cuda(), None, no_agent_mapping=True)
            assert np.abs(out.cpu().numpy() - ref).max() < 1e-4, scale


@pytest.mark.parametrize("math,tol", [("bf16x3", 1e-4), ("bf16", 5e-2)])
def test_dqn_tensorcore_q_values(math, tol):
    from graph_marl_b200.model import DQN

    g = load_golden("dqn_policy")
    D, h1, h2, n_act, wseed = [int(x) for x in g["cfg"]]
    dqn = DQN(D, (h1, h2), n_act, F.leaky_relu, math=math)
    w = det_weights(dqn_shapes(D, [h1, h2], n_act), wseed)
    dqn.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    dqn = dqn.cuda().eval()
    obs = torch.from_numpy(g["obs"]).cuda()
    with torch.no_grad():
        q, a = dqn.act(obs)
        q2, a2 = dqn.act(obs[..., :130].contiguous(), obs[..., 130:].contiguous())
        q3, a3 = dqn.act(obs[..., :130], obs[..., 130:])  # strided views of the joint tensor
    for qq in (q, q2, q3):
        assert np.abs(qq.cpu().numpy() - g["q"]).max() < tol
    if math == "bf16x3":
        assert np.array_equal(a.cpu().numpy(), g["q"].argmax(-1))
        assert np.array_equal(a2.cpu().numpy(), g["q"].argmax(-1))


def test_dqn_q_head_with_several_tiles_per_cta():
    """The config-2 DQN over 4096 envs x 20 agents (640 M tiles, several per CTA): the Q head's epilogue sums the partial
    Q-values of its four column groups through shared memory behind a barrier of all epilogue warps.  Every row must match
    the fp64 oracle, in every call (greedy actions = argmax)."""
    from graph_marl_b200.model import DQN
    from oracle import netmon_oracle as NO

    torch.manual_seed(4)
    dqn = DQN(130 + 512, (512, 256), 4, F.leaky_relu, math="bf16x3").cuda().eval()
    w = {k: v.detach().cpu().numpy() for k, v in dqn.state_dict().items()}
    rng = np.random.default_rng(4)
    obs_a = torch.from_numpy((rng.random((4096, 20, 130)) < 0.1).astype(np.float32)).cuda()
    obs_g = torch.from_numpy(rng.standard_normal((4096, 20, 512)).astype(np.float32) * 0.3).cuda()
    rows = rng.choice(4096 * 20, 4096, replace=False)
    x = torch.cat((obs_a, obs_g), -1).reshape(-1, 642).cpu().numpy()[rows]
    ref = NO.dqn_forward(w, x, dtype=np.float64)
    for _ in range(3):
        with torch.no_grad():
            q, a = dqn.act(obs_a, obs_g)
        q = q.reshape(-1, 4).cpu().numpy()
        assert np.abs(q[rows] - ref).max() < 1e-4
        assert np.array_equal(a.reshape(-1).cpu().numpy(), q.argmax(-1))


# (N, H, agg_type, batch, kernel that must run): the pipelined kernel's <H = 128, DM = 4> instance and its run-time
# instance, and the L2 gather kernel for graphs too large for the pipeline's stages.  "wrap" takes a batch from the SM
# count: 3 CTAs per SM of 2 graphs per row block, so every CTA goes round its 3-stage ring at least twice (both mbarrier
# phases in use), and an odd last graph leaves the last block, 8-row group and M tile partial.
AGG_CASES = {
    "pipe_sum": (20, 128, "sum", 301, ("aggregate_pk_pipe_kernel<128, 4>", "aggregate_pk_pipe_kernelILi128ELi4E")),
    "pipe_mean": (20, 128, "mean", 301, ("aggregate_pk_pipe_kernel<128, 4>", "aggregate_pk_pipe_kernelILi128ELi4E")),
    "pipe_wrap": (20, 128, "sum", "wrap", ("aggregate_pk_pipe_kernel<128, 4>", "aggregate_pk_pipe_kernelILi128ELi4E")),
    "pipe_generic": (20, 64, "sum", 301, ("aggregate_pk_pipe_kernel<0, 0>", "aggregate_pk_pipe_kernelILi0ELi0E")),
    "gather": (200, 128, "sum", 5, ("aggregate_pk_kernel(", "aggregate_pk_kernelEPKf")),
}


@pytest.mark.parametrize("case", list(AGG_CASES))
def test_netmon_aggregation_kernels(case):
    """Each aggregation kernel of the fused tensor-core path, chosen by the shapes alone: NetMon output and state against
    the fp64 oracle (graphs are independent, so a large batch is checked on a sample of graphs that includes the last
    ones), and the torch.profiler kernel names show which aggregation kernel ran."""
    from torch.profiler import ProfilerActivity, profile

    from graph_marl_b200.model import NetMon
    from oracle import netmon_oracle as NO
    from oracle import oracle as O

    N, H, agg, B, names = AGG_CASES[case]
    if B == "wrap":
        B = 36 * torch.cuda.get_device_properties(0).multi_processor_count + 1
    K, Dn = 3, 4 * N + 8
    cfg = dict(hidden=H, iterations=K, rnn_type="lstm", rnn_carryover=True, agg_type=agg, output_neighbor_hidden=True,
               output_global_hidden=False, enc=[512, 256], wseed=5)
    nm = NetMon(Dn, H, cfg["enc"], K, F.leaky_relu, output_neighbor_hidden=True, math="bf16x3", agg_type=agg)
    w = det_weights(netmon_shapes(Dn, H, cfg["enc"], "lstm"), 5)
    nm.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
    nm = nm.cuda().eval()
    topo = O.generate_topology(N, seed=923430603 if N == 20 else 476)
    rng = np.random.default_rng(0)
    x = (rng.random((B, N, Dn)) < 0.05).astype(np.float32)
    mask = np.broadcast_to(topo["adj"], (B, N, N)).astype(np.float32)
    st = (rng.standard_normal((B, N, 2 * H)) * 0.3).astype(np.float32)
    with torch.no_grad(), profile(activities=[ProfilerActivity.CUDA]) as prof:
        nm.state = torch.from_numpy(st).cuda()
        out = nm(torch.from_numpy(x).cuda(), torch.from_numpy(mask.copy()).cuda(), None, no_agent_mapping=True)
        torch.cuda.synchronize()
    ran = {e.name for e in prof.events() if "aggregate" in e.name}
    assert ran and all(any(n in r for n in names) for r in ran), ran
    g = np.arange(B) if B <= 512 else np.unique(np.concatenate([rng.choice(B, 504, replace=False), np.arange(B - 8, B)]))
    ref, ref_state, _ = NO.netmon_forward(w, cfg, x[g], mask[g], st[g], dtype=np.float64)
    e1, e2 = np.abs(out.cpu().numpy()[g] - ref).max(), np.abs(nm.state.cpu().numpy()[g] - ref_state).max()
    assert e1 < 1e-4 and e2 < 1e-4, (e1, e2)
