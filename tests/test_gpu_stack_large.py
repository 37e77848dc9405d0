"""Stacked GAT Q-networks on large swarms (swarm_gatstack_forward_large / swarm_rollout_stack above 128 agents): one launch
with one CTA per env for every SwarmStackSpec, the attention in input space per layer, the graph built once per forward
(uniform grid for the radius graph, sorted-prefix factorisation for the complete graph, the caller's topk table for kNN).

Bar, per env: |Q - Q64| <= 1e-5 * max|Q64| against the float64 oracle (oracle/swarm_oracle.gat_conv stacked layer by
layer on the explicit graph), and greedy actions equal to the oracle's wherever the float64 top-2 gap exceeds
4e-5 * max|Q64|.  The rollout equals the composed per-tick calls bit for bit."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from helpers import load_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q_RTOL = 1e-5
GAP = 4e-5


def _dev():
    return torch.device("cuda:0")


def _flocking_sd(seed):
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    pre = f"{seed}/"
    return {k[len(pre):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(pre)}


def _random_sd(layers, hidden, in_features, seed, att_scale=1.0):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for l in range(1, layers + 1):
        cin = in_features if l == 1 else hidden
        sd[f"conv{l}.lin.weight"] = (0.5 if l > 1 else 0.3) * torch.randn(hidden, cin, generator=g)
        sd[f"conv{l}.att_src"] = att_scale * torch.randn(1, 1, hidden, generator=g)
        sd[f"conv{l}.att_dst"] = att_scale * torch.randn(1, 1, hidden, generator=g)
        sd[f"conv{l}.bias"] = 0.1 * torch.randn(hidden, generator=g)
    sd["lin1.weight"] = 0.4 * torch.randn(hidden, hidden, generator=g)
    sd["lin1.bias"] = 0.1 * torch.randn(hidden, generator=g)
    sd["lin2.weight"] = 0.4 * torch.randn(9, hidden, generator=g)
    sd["lin2.bias"] = 0.1 * torch.randn(9, generator=g)
    return sd


def _states(B, N, seed, scenario="go_to"):
    from oracle import swarm_oracle as so, batched_oracle as bo
    g = torch.Generator().manual_seed(seed)
    centers = torch.stack([so.draw_center(scenario, True, g) for _ in range(B)])
    pos, vel = bo.reset_grid(scenario, centers, N)
    pos = pos + 0.03 * torch.randn(B, N, 2, generator=g)
    vel = 0.3 * torch.randn(B, N, 2, generator=g)
    return pos.contiguous(), vel.contiguous()


def _cfg(graph, B, N, k, scenario=None):
    import swarm_b200 as sb
    L = sb._lib
    gm = {"complete": L.GRAPH_COMPLETE, "knn": L.GRAPH_KNN, "radius": L.GRAPH_RADIUS}[graph]
    return sb.ops.make_config(L.SCENARIO_GOTO if scenario is None else scenario, B, N, gm,
                              int(k) if graph == "knn" else 10, graph_radius=float(k) if graph == "radius" else 0.35)


def _edges(graph, pos, k, nbr=None):
    """Explicit per-env edge list int64[B,2,E] of the reference's builders; kNN from the library's topk table."""
    from oracle import batched_oracle as bo
    if graph == "knn":
        return bo.edges_from_knn(nbr.cpu().long())
    return bo.graph_edges(pos, graph, k)


def _oracle_q64(sd, acts, pos, vel, edges, in_features=7, device=None, dtype=torch.float64):
    """float64 oracle: swarm_oracle.gat_conv stacked layer by layer, run on `device` (the GPU: the complete graph of 4 096
    agents has 16.8 M edges)."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    dev = device or torch.device("cpu")
    B, N, _ = pos.shape
    x = bo.node_features(pos.to(dtype), vel.to(dtype))
    if in_features == 5:
        x = torch.cat([x[..., :4], x[..., 6:7]], dim=-1)
    h = x.reshape(B * N, -1).to(dev)
    ei = bo.batch_edge_index(edges, N).to(dev)
    sdd = {k: v.to(dtype).to(dev) for k, v in sd.items()}
    l = 1
    while f"conv{l}.lin.weight" in sdd:
        h = so.gat_conv(h, ei, sdd[f"conv{l}.lin.weight"], sdd[f"conv{l}.att_src"], sdd[f"conv{l}.att_dst"],
                        sdd[f"conv{l}.bias"])
        h = torch.tanh(h) if acts[l - 1] == "tanh" else torch.relu(h)
        l += 1
    h = torch.relu(h @ sdd["lin1.weight"].T + sdd["lin1.bias"])
    return (h @ sdd["lin2.weight"].T + sdd["lin2.bias"]).reshape(B, N, 9).cpu().double()


def _check(q, act, q64, what="", bar=Q_RTOL):
    """The bar per env; returns the worst relative error."""
    q = q.cpu().double()
    scale = q64.abs().flatten(1).amax(dim=1).clamp_min(1e-30).view(-1, 1, 1)
    err = ((q - q64).abs() / scale).amax().item()
    assert torch.isfinite(q).all(), f"{what}: non-finite Q"
    assert err <= bar, f"{what}: Q relative error {err:.3e}"
    if act is not None:
        top2 = torch.topk(q64, 2, dim=-1).values
        clear = (top2[..., 0] - top2[..., 1]) > GAP * scale.view(-1, 1)
        ref = torch.argmax(q64, dim=-1)
        assert torch.equal(act.cpu().long()[clear], ref[clear]), f"{what}: greedy actions differ outside the near-tie band"
    return err


def _forward_large(cfg, spec, w, state):
    import swarm_b200 as sb
    B, N = cfg.num_envs, cfg.n_agents
    q = torch.empty(B, N, 9, dtype=torch.float32, device=state.device)
    act = torch.empty(B, N, dtype=torch.int32, device=state.device)
    nbr = None
    if cfg.graph_mode == sb._lib.GRAPH_KNN:
        _, nbr = sb.ops.graph_build(cfg, state, want_neighbours=True)
    sb.ops.gatstack_forward_large(cfg, spec, w, state, neighbours=nbr, q=q, actions=act)
    return q, act, nbr


FLOCK_CASES = [("complete", 129, 3, 0), ("radius", 300, 2, 0.35), ("knn", 129, 3, 2), ("knn", 640, 2, 10),
               ("complete", 1024, 2, 0), ("radius", 1024, 2, 0.25), ("knn", 1024, 2, 10), ("complete", 4096, 1, 0),
               ("radius", 4096, 1, 0.35)]


@pytest.mark.gpu
@pytest.mark.parametrize("graph,N,B,k", FLOCK_CASES)
def test_flocking_checkpoint_matches_float64_oracle(graph, N, B, k):
    """The three-layer Flocking checkpoint (conv1 7 -> 8, conv2 / conv3 8 -> 8).  Worst measured relative Q error on a
    B200: 2.6e-7 (radius, N = 300)."""
    import swarm_b200 as sb
    ops = sb.ops
    sd = _flocking_sd(0)
    acts = ["tanh", "relu", "relu"]
    pos, vel = _states(B, N, seed=N + B)
    cfg = _cfg(graph, B, N, k)
    spec = ops.stack_spec(3, 8, 7, acts)
    w = ops.pack_stack_weights(sd, spec, _dev())
    state = torch.cat([pos, vel], 2).contiguous().to(_dev())
    q, act, nbr = _forward_large(cfg, spec, w, state)
    q64 = _oracle_q64(sd, acts, pos, vel, _edges(graph, pos, k, nbr), device=_dev())
    _check(q, act, q64, f"{graph} N={N}")
    # ops.gatstack_forward routes N > 128 to the same entry point
    q2, a2 = ops.gatstack_forward(cfg, spec, w, state, want_actions=True)
    assert torch.equal(q2, q) and torch.equal(a2, act)


RANDOM_SPECS = [(1, 32, 7), (2, 16, 5), (4, 5, 7), (4, 32, 5), (2, 32, 7)]


@pytest.mark.gpu
@pytest.mark.parametrize("layers,hidden,inf", RANDOM_SPECS)
@pytest.mark.parametrize("graph,N,B,k", [("complete", 300, 2, 0), ("radius", 1024, 2, 0.35), ("knn", 1024, 2, 10)])
def test_random_specs_match_float64_oracle(layers, hidden, inf, graph, N, B, k):
    """Every width class (8 / 16 / 32 padded), 1 to 4 layers, both input widths, mixed activations.  Worst measured
    relative Q error on a B200: 8.7e-7 (kNN)."""
    import swarm_b200 as sb
    ops = sb.ops
    sd = _random_sd(layers, hidden, inf, seed=layers * 100 + hidden)
    acts = (["tanh", "relu"] * 2)[:layers]
    pos, vel = _states(B, N, seed=layers + hidden)
    cfg = _cfg(graph, B, N, k)
    spec = ops.stack_spec(layers, hidden, inf, acts)
    w = ops.pack_stack_weights(sd, spec, _dev())
    q, act, nbr = _forward_large(cfg, spec, w, torch.cat([pos, vel], 2).contiguous().to(_dev()))
    _check(q, act, _oracle_q64(sd, acts, pos, vel, _edges(graph, pos, k, nbr), inf, device=_dev()), f"{graph} {spec}")


@pytest.mark.gpu
@pytest.mark.parametrize("graph,k", [("complete", 0), ("radius", 0.35), ("knn", 10)])
def test_matches_generic_layer_path_at_size(graph, k):
    """StackedGCN.forward through the generic layer kernels on the library's own graph (swarm_graph_build edges /
    graph_build_radius_csr), 16 envs x 1 024 agents.  Worst measured relative Q difference on a B200: 5.3e-6 (complete
    graph: sums over 1 023 sources in two different float32 orders)."""
    import swarm_b200 as sb
    ops = sb.ops
    B, N = 16, 1024
    sd = _flocking_sd(0)
    model = sb.StackedGCN.from_state_dict(sd).to(_dev()).eval()
    pos, vel = _states(B, N, seed=5)
    state = torch.cat([pos, vel], 2).contiguous().to(_dev())
    cfg = _cfg(graph, B, N, k)
    spec = model.stack_spec()
    w = model.packed_stack_weights(_dev())
    q, act, _ = _forward_large(cfg, spec, w, state)
    if graph == "radius":
        row_ptr, src = ops.graph_build_radius_csr(cfg, state)
        dst = torch.repeat_interleave(torch.arange(B * N, device=_dev()), (row_ptr[1:] - row_ptr[:-1]).long())
        ei = torch.stack([src.long(), dst])
    else:
        edges, _ = ops.graph_build(cfg, state)
        offs = (torch.arange(B, device=_dev(), dtype=torch.int64) * N).view(B, 1, 1)
        ei = (edges.long() + offs).permute(1, 0, 2).reshape(2, -1)
    ids = torch.arange(N, device=_dev(), dtype=torch.float32).view(1, N, 1).expand(B, N, 1)
    goal = torch.tensor([cfg.goal_x, cfg.goal_y], device=_dev()).view(1, 1, 2).expand(B, N, 2)
    x = torch.cat([state, goal, ids], 2).reshape(B * N, 7)
    with torch.no_grad():
        q_gen = model(sb.Data(x=x, edge_index=ei)).view(B, N, 9)
    _check(q, act, q_gen.double().cpu(), graph)


@pytest.mark.gpu
@pytest.mark.parametrize("graph,N,k", [("complete", 2, 0), ("complete", 12, 0), ("complete", 128, 0), ("radius", 12, 0.25),
                                       ("radius", 128, 0.35), ("knn", 12, 5), ("knn", 16, 6), ("knn", 2, 2)])
def test_small_swarms_match_the_env_tile_kernel(graph, N, k):
    """Any N >= 1 is accepted; at N <= 128 the large entry point agrees with swarm_gatstack_forward within the bar.
    Worst measured relative Q difference on a B200: 6.5e-7 (complete, N = 128)."""
    import swarm_b200 as sb
    ops = sb.ops
    B = 20
    sd = _flocking_sd(2)
    pos, vel = _states(B, N, seed=N)
    cfg = _cfg(graph, B, N, k)
    spec = ops.stack_spec(3, 8, 7)
    w = ops.pack_stack_weights(sd, spec, _dev())
    state = torch.cat([pos, vel], 2).contiguous().to(_dev())
    q, act, _ = _forward_large(cfg, spec, w, state)
    q_tile = ops.gatstack_forward(cfg, spec, w, state)
    _check(q, act, q_tile.double().cpu(), f"{graph} N={N}")


@pytest.mark.gpu
@pytest.mark.parametrize("exp,graph,k", [("GoTo", "complete", 0), ("ObstacleAvoidance", "radius", 0.35),
                                         ("ObstacleAvoidance", "knn", 10)])
def test_one_layer_stack_is_the_shipped_gcn(exp, graph, k):
    """L = 1, width 32, tanh on the shipped weights: the one-layer large kernels (gatq_forward_large /
    gatq_forward_knn_large) within the bar (separate layer code: float32-level different rounding).  Worst measured
    relative Q difference on a B200: 1.4e-6 (kNN)."""
    import swarm_b200 as sb
    ops = sb.ops
    B, N = 4, 1024
    params = load_params(exp, 0)
    pos, vel = _states(B, N, seed=9)
    state = torch.cat([pos, vel], 2).contiguous().to(_dev())
    cfg = _cfg(graph, B, N, k)
    spec = ops.stack_spec(1, 32, 7)
    w = ops.pack_stack_weights(params, spec, _dev())
    q, act, nbr = _forward_large(cfg, spec, w, state)
    w1 = sb.pack_weights(params, _dev())
    q1 = ops.gatq_forward_knn_large(cfg, w1, state, nbr) if graph == "knn" else ops.gatq_forward_large(cfg, w1, state)
    _check(q, act, q1.double().cpu(), graph)


@pytest.mark.gpu
@pytest.mark.parametrize("graph,k", [("complete", 0), ("radius", 0.35)])
def test_stretched_attention_logits(graph, k):
    """Attention vectors scaled until the logits of an env spread over more than 100: only the softmax shift keeps the
    exponentials finite (and, on the complete graph, the factorisation against the env's largest alpha_src).  Worst
    measured relative Q error on a B200: 5.0e-7 (complete)."""
    import swarm_b200 as sb
    ops = sb.ops
    B, N = 2, 1024
    sd = _random_sd(2, 8, 7, seed=17, att_scale=6.0)
    acts = ["tanh", "relu"]
    pos, vel = _states(B, N, seed=4)
    from oracle import batched_oracle as bo
    x = bo.node_features(pos.double(), vel.double())
    a = (x @ sd["conv1.lin.weight"].double().T) @ sd["conv1.att_src"].double().reshape(-1)
    assert (a.amax(dim=1) - a.amin(dim=1)).min().item() > 100.0
    cfg = _cfg(graph, B, N, k)
    spec = ops.stack_spec(2, 8, 7, acts)
    w = ops.pack_stack_weights(sd, spec, _dev())
    q, act, nbr = _forward_large(cfg, spec, w, torch.cat([pos, vel], 2).contiguous().to(_dev()))
    _check(q, act, _oracle_q64(sd, acts, pos, vel, _edges(graph, pos, k, nbr), device=_dev()), graph)


@pytest.mark.gpu
@pytest.mark.parametrize("graph,k", [("complete", 0), ("radius", 0.35), ("knn", 10)])
def test_collapsed_swarm(graph, k):
    """Every agent at one point: every pair is a radius edge, the topk table is all ties, every alpha_src of a layer
    differs only through the agent id.  Worst measured relative Q error on a B200: 1.2e-5 on the kNN graph (inside twice
    the float32 oracle's own error there), 1.8e-6 on the others."""
    import swarm_b200 as sb
    ops = sb.ops
    B, N = 2, 1024
    sd = _flocking_sd(4)
    acts = ["tanh", "relu", "relu"]
    pos = torch.tensor([[0.3, -0.2], [-0.5, 0.1]]).view(B, 1, 2).expand(B, N, 2).contiguous()
    vel = torch.zeros(B, N, 2)
    cfg = _cfg(graph, B, N, k)
    spec = ops.stack_spec(3, 8, 7, acts)
    w = ops.pack_stack_weights(sd, spec, _dev())
    q, act, nbr = _forward_large(cfg, spec, w, torch.cat([pos, vel], 2).contiguous().to(_dev()))
    edges = _edges(graph, pos, k, nbr)
    q64 = _oracle_q64(sd, acts, pos, vel, edges, device=_dev())
    # the all-tie kNN table gives nodes 0 .. k-1 an in-degree of N: float32 sums of ~1 000 rows that carry the agent ids
    # (up to 1 023).  The bar there is the float32 oracle's own error on the same graph, doubled, if that is larger.
    q32 = _oracle_q64(sd, acts, pos, vel, edges, device=_dev(), dtype=torch.float32)
    err32 = ((q32 - q64).abs() / q64.abs().flatten(1).amax(dim=1).view(-1, 1, 1)).amax().item()
    _check(q, act, q64, graph, bar=max(Q_RTOL, 2 * err32))


def _composed(cfg, spec, w, state, ticks):
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    B, N = cfg.num_envs, cfg.n_agents
    returns = torch.zeros(B, N, dtype=torch.float32, device=state.device)
    hits = torch.zeros(B, dtype=torch.int32, device=state.device)
    for _ in range(ticks):
        _, act, _ = _forward_large(cfg, spec, w, state)
        out = ops.sim_step(cfg, state, act, state_out=state, want_obs=False)
        returns += out["rewards"]
        hits += ((out["flags"] & L.FLAG_HIT) != 0).sum(dim=1, dtype=torch.int32)
    return state, returns, hits


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", ["GoTo", "ObstacleAvoidance"])
@pytest.mark.parametrize("graph,N,k", [("complete", 1024, 0), ("radius", 1024, 0.35), ("knn", 1024, 10), ("radius", 300, 0.35)])
def test_rollout_equals_composed_calls(scenario, graph, N, k):
    """ops.rollout_stack above 128 agents == [topk table ->] gatstack_forward_large -> sim_step in place -> returns / hits,
    bit for bit (final state, returns, hits)."""
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    B, T = 3, 5
    sid = L.SCENARIO_GOTO if scenario == "GoTo" else L.SCENARIO_OBSTACLE_AVOIDANCE
    pos, vel = _states(B, N, seed=N + 1, scenario="go_to" if scenario == "GoTo" else "obstacle_avoidance")
    cfg = _cfg(graph, B, N, k, sid)
    spec = ops.stack_spec(3, 8, 7)
    w = ops.pack_stack_weights(_flocking_sd(0), spec, _dev())
    s0 = torch.cat([pos, vel], 2).contiguous().to(_dev())
    out = ops.rollout_stack(cfg, spec, w, s0.clone(), T)
    st, ret, hits = _composed(cfg, spec, w, s0.clone(), T)
    assert torch.equal(out["state"], st)
    assert torch.equal(out["returns"], ret)
    assert torch.equal(out["hits"], hits)
    assert not torch.equal(st, s0)


@pytest.mark.gpu
def test_rollout_cuda_graph_replay_equals_eager():
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    B, N, T = 2, 1024, 3
    pos, vel = _states(B, N, seed=3, scenario="obstacle_avoidance")
    cfg = _cfg("knn", B, N, 10, L.SCENARIO_OBSTACLE_AVOIDANCE)
    spec = ops.stack_spec(3, 8, 7)
    w = ops.pack_stack_weights(_flocking_sd(1), spec, _dev())
    s0 = torch.cat([pos, vel], 2).contiguous().to(_dev())
    eager = ops.rollout_stack(cfg, spec, w, s0.clone(), T)
    state = s0.clone()
    returns = torch.zeros(B, N, device=_dev())
    hits = torch.zeros(B, dtype=torch.int32, device=_dev())
    ops.rollout_stack(cfg, spec, w, state, T, returns=returns, hits=hits)          # warm-up (kernel attributes)
    state.copy_(s0); returns.zero_(); hits.zero_()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            ops.rollout_stack(cfg, spec, w, state, T, returns=returns, hits=hits)
    torch.cuda.current_stream().wait_stream(s)
    state.copy_(s0); returns.zero_(); hits.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(state, eager["state"]) and torch.equal(returns, eager["returns"]) and torch.equal(hits, eager["hits"])


@pytest.mark.gpu
def test_simulator_runs_a_flocking_checkpoint_on_a_large_swarm(tmp_path):
    """Simulator with a shipped three-layer Flocking checkpoint on a 1 024-agent ObstacleAvoidance env (kNN, k = 10):
    the large stacked forward + world step per tick writes the reference's CSV tree, and the trajectory equals the
    script-level loop (create_graph_from_observations -> StackedGCN.forward through the generic layer kernels -> argmax
    -> env.step) wherever that loop has no near-tie."""
    import csv
    import swarm_b200 as sb
    n, T, k = 1024, 4, 10
    model = sb.StackedGCN.from_state_dict(_flocking_sd(0)).to(_dev()).eval()

    def make():
        return sb.make_env(scenario=sb.ObstacleAvoidanceScenario(), num_envs=1, device=_dev(), continuous_actions=False,
                           max_steps=T, dict_spaces=True, seed=3, n_agents=n)

    env = make()
    sim = sb.Simulator(env, model, 1, "obstacle", 3, output_dir=str(tmp_path / "stats"), k=k)
    torch.manual_seed(11)
    sim.run_simulation()
    with open(tmp_path / "stats" / "positions" / "positions_episode_0_x.csv") as f:
        rows = list(csv.reader(f))
    assert rows[0] == ["Tick"] + [f"X{a}" for a in range(n)] and len(rows) == T + 1
    xs = torch.tensor([[float(v) for v in r[1:]] for r in rows[1:]])
    env2 = make()
    torch.manual_seed(11)
    obs = env2.reset()
    safe = True
    for t in range(T):
        data = sb.create_graph_from_observations(obs, n, mode="knn", k=k)
        with torch.no_grad():
            q = model(data)
        top2 = torch.topk(q, 2, dim=1).values
        if ((top2[:, 0] - top2[:, 1]) <= GAP * q.abs().amax()).any():
            safe = False
        act = torch.argmax(q, dim=1)
        obs, rew, done, info = env2.step({f"agent{i}": act[i:i + 1] for i in range(n)})
        if safe:
            got = torch.stack([obs[f"agent{i}"][0, 0] for i in range(n)]).cpu()
            assert torch.equal(got, xs[t]), f"tick {t}"
    assert safe or t > 0


# ---- argument errors (no device needed: rejected before any launch) ------------------------------------------------
def test_stack_large_argument_errors():
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    lib = L.lib()
    spec = ops.stack_spec(3, 8, 7)
    ws = lambda c, s=spec: int(lib.swarm_gatstack_large_workspace_bytes(C.byref(c), C.byref(s)))   # noqa: E731

    def fwd(c, s=spec, nbr=8, wb=1 << 40):
        return lib.swarm_gatstack_forward_large(C.byref(c), C.byref(s), 8, 8, nbr, 8, 8, 8, wb, None)

    big = ops.make_config(L.SCENARIO_GOTO, 2, 4097, L.GRAPH_RADIUS)
    assert fwd(big) == -2 and ws(big) == 0
    knn = ops.make_config(L.SCENARIO_GOTO, 2, 1024, L.GRAPH_KNN, 10)
    assert fwd(knn, nbr=None) == -1 and b"neighbours" in lib.swarm_last_error()
    assert ws(knn) > 2 * 2 * 1024 * 8 * 4
    assert fwd(knn, wb=ws(knn) - 1) == -1 and b"workspace too small" in lib.swarm_last_error()
    knn20 = ops.make_config(L.SCENARIO_GOTO, 2, 1024, L.GRAPH_KNN, 20)                  # 64 k > N: no partial_sort table
    assert fwd(knn20) == -2 and ws(knn20) == 0
    bad = ops.stack_spec(3, 8, 7)
    bad.n_layers = 5
    rad = ops.make_config(L.SCENARIO_GOTO, 2, 1024, L.GRAPH_RADIUS)
    assert fwd(rad, s=bad) == -1 and b"n_layers" in lib.swarm_last_error() and ws(rad, bad) == 0
    assert lib.swarm_gatstack_forward_large(C.byref(rad), C.byref(spec), 8, 8, None, None, None, 8, 1 << 40, None) == -1
    assert b"no output" in lib.swarm_last_error()
    # rollout above 128 agents: the world's reward only
    rs = L.SwarmRewardSpec()
    lib.swarm_default_reward_spec(C.byref(rs), L.REWARD_FLOCKING, 2, 1024)
    wb = int(lib.swarm_rollout_stack_workspace_bytes(C.byref(rad)))
    assert lib.swarm_rollout_stack(C.byref(rad), C.byref(spec), 8, 8, 1, C.byref(rs), 8, None, None, 8, wb, None) == -2
    assert b"n_agents <= 128" in lib.swarm_last_error()
    assert lib.swarm_rollout_stack(C.byref(rad), C.byref(spec), 8, 8, 1, None, None, None, None, 8, wb - 1, None) == -1
    assert b"workspace too small" in lib.swarm_last_error()
    # the env-tile entry point and the stacked DQN update keep their limits
    assert lib.swarm_gatstack_forward(C.byref(rad), C.byref(spec), 8, 8, 8, None, None) == -2
    assert int(lib.swarm_dqn_stack_workspace_bytes(C.byref(rad), C.byref(spec), 4)) == 0
    assert b"n_agents <= 128" in lib.swarm_last_error()
