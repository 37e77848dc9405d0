"""Multi-layer GAT Q-networks in one launch (swarm_gatstack_forward / swarm_rollout_stack; SURVEY 8f rank 4): the
three-layer form the reference ships as data/models/experiment_Flocking-seed_*.pth (conv2 / conv3 are comments in
train_gcn_dqn.py:54-55, 64-67) against the oracle's GATConv restatement (oracle/swarm_oracle.py gat_conv) stacked the same
way, the one-layer GCN as the special case L = 1, the 5-feature input of scenarios that observe cat[pos, vel], and the
library tick loop against the composed calls.  Tolerance: Q within 1e-5 of the row's largest magnitude (float32 kernels
against the float32 oracle)."""
import os

import numpy as np
import pytest
import torch

from helpers import load_params

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q_RTOL = 1e-5


def _dev():
    return torch.device("cuda:0")


def _flocking_sd(seed):
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    pre = f"{seed}/"
    return {k[len(pre):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(pre)}


def _states(B, N, seed):
    from oracle import swarm_oracle as so, batched_oracle as bo
    g = torch.Generator().manual_seed(seed)
    centers = torch.stack([so.draw_center("go_to", True, g) for _ in range(B)])
    pos, vel = bo.reset_grid("go_to", centers, N)
    pos[1:] += 0.03 * torch.randn(B - 1, N, 2, generator=g)
    vel = 0.3 * torch.randn(B, N, 2, generator=g)
    return pos.contiguous(), vel.contiguous()


def _oracle_q(sd, acts, pos, vel, edges, in_features=7):
    from oracle import swarm_oracle as so, batched_oracle as bo
    B, N, _ = pos.shape
    x = bo.node_features(pos, vel)
    if in_features == 5:
        x = torch.cat([x[..., :4], x[..., 6:7]], dim=-1)
    h = x.reshape(B * N, -1)
    ei = bo.batch_edge_index(edges, N)
    l = 1
    while f"conv{l}.lin.weight" in sd:
        h = so.gat_conv(h, ei, sd[f"conv{l}.lin.weight"], sd[f"conv{l}.att_src"], sd[f"conv{l}.att_dst"], sd[f"conv{l}.bias"])
        h = torch.tanh(h) if acts[l - 1] == "tanh" else torch.relu(h)
        l += 1
    h = torch.relu(h @ sd["lin1.weight"].T + sd["lin1.bias"])
    return (h @ sd["lin2.weight"].T + sd["lin2.bias"]).reshape(B, N, 9)


def _check_q(q, q_ref):
    scale = q_ref.abs().amax(dim=-1, keepdim=True).clamp_min(1e-3)
    err = ((q.cpu().double() - q_ref.double()).abs() / scale.double()).max().item()
    assert err <= Q_RTOL, f"Q relative error {err:.3e}"


@pytest.mark.parametrize("graph,N,B,k", [("complete", 12, 40, 0), ("knn", 12, 40, 5), ("knn", 5, 30, 5), ("radius", 20, 12, 0.25),
                                         ("complete", 100, 3, 0), ("knn", 16, 20, 6), ("complete", 2, 64, 0)])
@pytest.mark.parametrize("acts", [("tanh", "relu", "relu"), ("tanh", "tanh", "tanh")])
def test_three_layer_flocking_checkpoints_match_oracle(graph, N, B, k, acts):
    import swarm_b200 as sb
    from oracle import batched_oracle as bo
    ops, L = sb.ops, sb._lib
    sd = _flocking_sd(3)
    assert sd["conv1.lin.weight"].shape == (8, 7) and sd["conv3.lin.weight"].shape == (8, 8)
    pos, vel = _states(B, N, seed=N + B)
    edges = bo.graph_edges(pos, graph, k)
    with torch.no_grad():
        q_ref = _oracle_q(sd, acts, pos, vel, edges)
    gm = {"complete": L.GRAPH_COMPLETE, "knn": L.GRAPH_KNN, "radius": L.GRAPH_RADIUS}[graph]
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N, gm, int(k) if graph == "knn" else 5,
                          graph_radius=float(k) if graph == "radius" else 0.35)
    spec = ops.stack_spec(3, 8, 7, list(acts))
    w = ops.pack_stack_weights(sd, spec, _dev())
    q, a = ops.gatstack_forward(cfg, spec, w, torch.cat([pos, vel], 2).contiguous().to(_dev()), want_actions=True)
    _check_q(q, q_ref)
    assert torch.equal(a.cpu().long(), torch.argmax(q.cpu(), dim=-1)), "argmax of the kernel's own Q (first maximum wins)"


@pytest.mark.parametrize("exp,graph,N", [("GoTo", "complete", 9), ("ObstacleAvoidance", "knn", 12)])
def test_one_layer_stack_is_the_shipped_gcn(exp, graph, N):
    """L = 1, H = 32, tanh: the reference's active GCN (train:50-70) through the stack kernel == oracle == the dedicated
    one-layer kernels (bit-faithful path) within the tolerance."""
    import swarm_b200 as sb
    from oracle import batched_oracle as bo
    ops, L = sb.ops, sb._lib
    B = 50
    params = load_params(exp, 2)
    pos, vel = _states(B, N, seed=7)
    edges = bo.graph_edges(pos, graph, 5)
    with torch.no_grad():
        q_ref = bo.gatq(params, pos, vel, edges)
    gm = L.GRAPH_COMPLETE if graph == "complete" else L.GRAPH_KNN
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N, gm, 5)
    spec = ops.stack_spec(1, 32, 7)
    w = ops.pack_stack_weights(params, spec, _dev())
    q = ops.gatstack_forward(cfg, spec, w, torch.cat([pos, vel], 2).contiguous().to(_dev()))
    _check_q(q, q_ref)


@pytest.mark.parametrize("hidden,layers", [(32, 1), (12, 2), (16, 4)])
def test_five_feature_input_matches_oracle(hidden, layers):
    """[pos, vel, agent id]: the node features of a scenario whose observation() is cat[pos, vel]
    (cohesion_scenario.py:87-94) under train:95-99; random weights of odd widths (zero-padded channels)."""
    import swarm_b200 as sb
    from oracle import batched_oracle as bo
    ops, L = sb.ops, sb._lib
    g = torch.Generator().manual_seed(hidden)
    sd = {}
    for l in range(1, layers + 1):
        cin = 5 if l == 1 else hidden
        sd[f"conv{l}.lin.weight"] = 0.5 * torch.randn(hidden, cin, generator=g)
        sd[f"conv{l}.att_src"] = torch.randn(1, 1, hidden, generator=g)
        sd[f"conv{l}.att_dst"] = torch.randn(1, 1, hidden, generator=g)
        sd[f"conv{l}.bias"] = 0.1 * torch.randn(hidden, generator=g)
    sd["lin1.weight"] = 0.4 * torch.randn(hidden, hidden, generator=g)
    sd["lin1.bias"] = 0.1 * torch.randn(hidden, generator=g)
    sd["lin2.weight"] = 0.4 * torch.randn(9, hidden, generator=g)
    sd["lin2.bias"] = 0.1 * torch.randn(9, generator=g)
    B, N = 30, 9
    pos, vel = _states(B, N, seed=3)
    acts = ["tanh"] + ["relu"] * (layers - 1)
    with torch.no_grad():
        q_ref = _oracle_q(sd, acts, pos, vel, bo.graph_edges(pos, "complete", 0), in_features=5)
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N, L.GRAPH_COMPLETE)
    spec = ops.stack_spec(layers, hidden, 5, acts)
    q = ops.gatstack_forward(cfg, spec, ops.pack_stack_weights(sd, spec, _dev()), torch.cat([pos, vel], 2).contiguous().to(_dev()))
    _check_q(q, q_ref)


@pytest.mark.parametrize("graph", ["knn", "complete", "radius"])
@pytest.mark.parametrize("reward", ["world_oa", "world_goto", "flocking", "cohesion"])
def test_rollout_stack_equals_composed_calls(reward, graph):
    """swarm_rollout_stack (forward -> step -> reward -> totals in one launch) == the same calls composed by hand, bit
    for bit; Flocking carries its shaping memory, Cohesion uses the 5-feature input."""
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    dev = _dev()
    B, N, T = 300, 9, 12
    scen = L.SCENARIO_OBSTACLE_AVOIDANCE if reward == "world_oa" else L.SCENARIO_GOTO
    gm = {"knn": L.GRAPH_KNN, "complete": L.GRAPH_COMPLETE, "radius": L.GRAPH_RADIUS}[graph]
    cfg = ops.make_config(scen, B, N, gm, 5, graph_radius=0.25)
    sd = _flocking_sd(0)
    in_features = 5 if reward == "cohesion" else 7
    if in_features == 5:
        sd = dict(sd)
        sd["conv1.lin.weight"] = sd["conv1.lin.weight"][:, [0, 1, 2, 3, 6]].contiguous()
    spec = ops.stack_spec(3, 8, in_features)
    w = ops.pack_stack_weights(sd, spec, dev)
    g = torch.Generator().manual_seed(1)
    centers = (torch.tensor([0.3, -0.3]) + 0.2 * torch.randn(B, 2, generator=g)).to(dev)
    state0 = ops.reset_grid(cfg, centers)
    rs = shaping0 = None
    if reward == "flocking":
        rs = ops.reward_spec(L.REWARD_FLOCKING, B, N)
        shaping0 = torch.zeros(B, N, 2, device=dev)
        ops.scenario_reward(rs, state0, shaping0, reset=True)
    elif reward == "cohesion":
        rs = ops.reward_spec(L.REWARD_COHESION, B, N)
    # composed
    st = state0.clone()
    sh = shaping0.clone() if shaping0 is not None else None
    ret = torch.zeros(B, N, device=dev)
    hits = torch.zeros(B, dtype=torch.int32, device=dev)
    for _ in range(T):
        act = ops.gatstack_forward(cfg, spec, w, st, want_q=False, want_actions=True)
        out = ops.sim_step(cfg, st, act, state_out=st, want_obs=False)
        if reward == "flocking":
            ret += ops.scenario_reward(rs, st, sh).view(B, 1)
        elif reward == "cohesion":
            ret += ops.scenario_reward(rs, st)
        else:
            ret += out["rewards"]
        hits += ((out["flags"] & L.FLAG_HIT) != 0).sum(dim=1, dtype=torch.int32)
    res = ops.rollout_stack(cfg, spec, w, state0.clone(), T, reward=rs,
                            shaping=shaping0.clone() if shaping0 is not None else None)
    assert torch.equal(res["state"], st), "state"
    assert torch.equal(res["returns"], ret), "returns"
    assert torch.equal(res["hits"], hits), "hits"
    if reward == "flocking":
        assert torch.equal(res["shaping"], sh), "shaping"
    assert (st != state0).any() and torch.isfinite(ret).all()
    # running totals continue
    res2 = ops.rollout_stack(cfg, spec, w, res["state"].clone(), 3, reward=rs, shaping=res.get("shaping"),
                             returns=res["returns"].clone(), hits=res["hits"].clone())
    assert not torch.equal(res2["returns"], res["returns"])


def test_stack_argument_errors():
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    dev = _dev()
    cfg = ops.make_config(L.SCENARIO_GOTO, 4, 20, L.GRAPH_KNN, 5)
    spec = ops.stack_spec(3, 8, 7)
    w = torch.zeros(int(L.lib().swarm_stack_weight_count(__import__("ctypes").byref(spec))), device=dev)
    with pytest.raises(sb.SwarmError, match="n_agents <= 16"):
        ops.gatstack_forward(cfg, spec, w, torch.zeros(4, 20, 4, device=dev))
    bad = ops.stack_spec(3, 8, 7)
    bad.hidden = 40
    with pytest.raises(Exception):
        ops.gatstack_forward(ops.clone_config(cfg, graph_mode=L.GRAPH_COMPLETE), bad, w, torch.zeros(4, 20, 4, device=dev))
    oa = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, 4, 9, L.GRAPH_COMPLETE)
    with pytest.raises(ValueError, match="GoTo world"):
        ops.rollout_stack(oa, spec, w, torch.zeros(4, 9, 4, device=dev), 1, reward=ops.reward_spec(L.REWARD_COHESION, 4, 9))


def test_simulator_runs_the_shipped_flocking_checkpoint(tmp_path):
    """Simulator (simulator.py:28-166) with a StackedGCN built from a shipped three-layer Flocking checkpoint on a
    FlockingScenario env: the one-launch forward + world step per tick writes the reference's CSV tree, and the trajectory
    equals the script-level loop (create_graph_from_observations -> model(data) through the generic layer kernels ->
    argmax -> env.step) wherever that loop's top-2 Q gap is outside the tolerance band."""
    import csv
    import swarm_b200 as sb
    n, T, k = 5, 12, 5
    model = sb.StackedGCN.from_state_dict(_flocking_sd(1)).to(_dev()).eval()
    assert model.n_layers == 3 and model.lin1.in_features == 8

    def make():
        return sb.make_env(scenario=sb.FlockingScenario(), num_envs=1, device=_dev(), continuous_actions=False,
                           max_steps=T, dict_spaces=True, seed=3, n_agents=n)

    env = make()
    sim = sb.Simulator(env, model, 1, "flocking", 3, output_dir=str(tmp_path / "stats"), k=k)
    torch.manual_seed(11)
    sim.run_simulation()
    with open(tmp_path / "stats" / "positions" / "positions_episode_0_x.csv") as f:
        rows = list(csv.reader(f))
    assert rows[0] == ["Tick"] + [f"X{a}" for a in range(n)] and len(rows) == T + 1
    xs = torch.tensor([[float(v) for v in r[1:]] for r in rows[1:]])
    # the script-level loop on a fresh env from the same generator state
    env2 = make()
    torch.manual_seed(11)
    obs = env2.reset()
    safe = True
    for t in range(T):
        data = sb.create_graph_from_observations(obs, n, mode="knn", k=k)
        with torch.no_grad():
            q = model(data)
        top2 = torch.topk(q, 2, dim=1).values
        if ((top2[:, 0] - top2[:, 1]) <= 4 * Q_RTOL * q.abs().amax(dim=1)).any():
            safe = False                                  # a near-tie: the two float32 forwards may pick different actions
        act = torch.argmax(q, dim=1)
        obs, rew, done, info = env2.step({f"agent{i}": act[i:i + 1] for i in range(n)})
        if safe:
            got = torch.stack([obs[f"agent{i}"][0, 0] for i in range(n)]).cpu()
            assert torch.equal(got, xs[t]), f"tick {t}"
    assert safe or t > 0
