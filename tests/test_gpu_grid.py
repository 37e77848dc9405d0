"""Uniform-grid broad phase for large swarms (SURVEY 8(f) rank 4; BASELINE config 4 with the radius / complete graph):
the radius graph as a compact CSR against its oracle definition (oracle/batched_oracle.py::edges_radius, vectorised over
a row), the edge-list-free Q forward against the bit-faithful CSR forward and the oracle, and the library tick loop."""
import pytest
import torch

from helpers import load_params


Q_RTOL = 1e-5


def _dev():
    return torch.device("cuda:0")


def _swarm(B, N, seed, spread=1.0, jitter=0.02):
    """Grid starts (spacing 0.15) squeezed / jittered; env 0 keeps the exact lattice, whose pair distances sit exactly on
    multiples of the spacing (boundary cases of the inclusive radius test)."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    g = torch.Generator().manual_seed(seed)
    centers = torch.stack([so.draw_center("obstacle_avoidance", True, g) for _ in range(B)])
    pos, vel = bo.reset_grid("obstacle_avoidance", centers, N)
    ctr = pos.mean(dim=1, keepdim=True)
    pos = ctr + (pos - ctr) * spread
    if B > 1:
        pos[1:] += jitter * torch.randn(B - 1, N, 2, generator=g)
    vel = 0.2 * torch.randn(B, N, 2, generator=g)
    return pos.contiguous(), vel.contiguous()


def _radius_csr_ref(pos, radius):
    """edges_radius + stable sort by target, vectorised over j: in-edges of t are the sources s != t with
    ||p_s - p_t|| <= r (float32 norm of the row difference, as simulator.py:18 computes it) in ascending s, node 0 also
    (0 -> 0) last.  Global node ids."""
    B, N, _ = pos.shape
    r = torch.tensor(radius, dtype=torch.float32)
    deg = torch.zeros(B * N, dtype=torch.int64)
    srcs = []
    for b in range(B):
        for t in range(N):
            d = torch.linalg.norm(pos[b] - pos[b, t], dim=1)
            m = d <= r
            m[t] = False
            s = torch.nonzero(m).flatten() + b * N
            if t == 0:
                s = torch.cat([s, torch.tensor([b * N])])
            deg[b * N + t] = s.numel()
            srcs.append(s)
    row_ptr = torch.zeros(B * N + 1, dtype=torch.int64)
    row_ptr[1:] = torch.cumsum(deg, 0)
    return row_ptr, torch.cat(srcs)


def test_vectorised_radius_reference_is_the_oracle_edge_list():
    """CPU: the per-target formulation above == oracle edge list -> stable sort by target."""
    from oracle import batched_oracle as bo
    pos, _ = _swarm(3, 14, seed=2, spread=0.9)
    for radius in (0.15, 0.3, 0.2):
        e = bo.edges_radius(pos, radius)
        ei = bo.batch_edge_index(e, 14)
        order = torch.sort(ei[1], stable=True).indices
        row_ptr, src = _radius_csr_ref(pos, radius)
        assert torch.equal(ei[0][order], src)
        assert torch.equal(torch.bincount(ei[1], minlength=3 * 14), row_ptr[1:] - row_ptr[:-1])


@pytest.mark.gpu
@pytest.mark.parametrize("N,B,radius,spread", [(300, 3, 0.3, 1.0), (1024, 2, 0.35, 1.0), (12, 50, 0.2, 1.0),
                                               (4096, 1, 0.15, 1.0), (200, 3, float("inf"), 1.0), (150, 3, 0.0, 1.0),
                                               (640, 2, 0.45, 0.3), (129, 4, 1e-3, 0.0)])
def test_radius_csr_bitexact(N, B, radius, spread):
    import swarm_b200 as sb
    pos, vel = _swarm(B, N, seed=N + B, spread=spread)
    cfg = sb.ops.make_config(sb._lib.SCENARIO_OBSTACLE_AVOIDANCE, B, N, sb._lib.GRAPH_RADIUS, graph_radius=radius)
    row_ptr, src = sb.ops.graph_build_radius_csr(cfg, torch.cat([pos, vel], 2).contiguous().to(_dev()))
    rp_ref, src_ref = _radius_csr_ref(pos, radius)
    assert torch.equal(row_ptr.cpu().long(), rp_ref), "in-degrees differ"
    assert torch.equal(src.cpu().long(), src_ref), "sources differ"
    if 0 < radius < 1 and spread == 1.0:
        assert (rp_ref[1:] - rp_ref[:-1]).max() < N - 1, "the radius must prune"


@pytest.mark.gpu
def test_radius_csr_degenerate_positions():
    """NaN / infinite coordinates never enter an edge (the oracle's `d <= r` is False for them) and do not disturb the
    binning of the others."""
    import swarm_b200 as sb
    B, N, radius = 2, 260, 0.3
    pos, vel = _swarm(B, N, seed=5)
    pos[0, 7, 0] = float("nan")
    pos[1, 100] = float("inf")
    pos[1, 3, 1] = -float("inf")
    cfg = sb.ops.make_config(sb._lib.SCENARIO_OBSTACLE_AVOIDANCE, B, N, sb._lib.GRAPH_RADIUS, graph_radius=radius)
    row_ptr, src = sb.ops.graph_build_radius_csr(cfg, torch.cat([pos, vel], 2).contiguous().to(_dev()))
    rp_ref, src_ref = _radius_csr_ref(pos, radius)
    assert torch.equal(row_ptr.cpu().long(), rp_ref) and torch.equal(src.cpu().long(), src_ref)


def _x(cfg, state):
    B, N = cfg.num_envs, cfg.n_agents
    dev = state.device
    ids = torch.arange(N, device=dev, dtype=torch.float32).view(1, N, 1).expand(B, N, 1)
    goal = torch.tensor([cfg.goal_x, cfg.goal_y], device=dev).view(1, 1, 2).expand(B, N, 2)
    return torch.cat([state, goal, ids], dim=2).reshape(B * N, 7)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,N,B,radius", [("radius", 1024, 3, 0.35), ("radius", 300, 4, 0.2), ("radius", 12, 64, 0.22),
                                             ("radius", 4096, 1, 0.3), ("complete", 200, 3, 0.0), ("complete", 1024, 2, 0.0),
                                             ("complete", 9, 40, 0.0), ("radius", 200, 2, float("inf"))])
def test_forward_large_matches_csr_forward(mode, N, B, radius):
    """swarm_gatq_forward_large (no edge list, attention in input space) against the bit-faithful generic forward on the
    same graph: Q within the float32 tolerance of the tensor-core path, greedy actions equal except at near-ties."""
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    dev = _dev()
    pos, vel = _swarm(B, N, seed=N, spread=0.8)
    state = torch.cat([pos, vel], 2).contiguous().to(dev)
    w = sb.pack_weights(load_params("ObstacleAvoidance", 1), dev)
    if mode == "radius":
        cfg = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B, N, L.GRAPH_RADIUS, graph_radius=radius)
        row_ptr, src = ops.graph_build_radius_csr(cfg, state)
    else:
        cfg = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B, N, L.GRAPH_COMPLETE)
        edges, _ = ops.graph_build(cfg, state)
        offs = (torch.arange(B, device=dev, dtype=torch.int64) * N).view(B, 1, 1)
        ei = (edges.to(torch.int64) + offs).permute(1, 0, 2).reshape(2, -1).contiguous()
        row_ptr, src, _ = ops.csr_from_edges(ei, B * N)
    q_ref, a_ref = ops.gatq_forward_csr(w, _x(cfg, state), row_ptr, src, want_q=True, want_actions=True)
    q, a = ops.gatq_forward_large(cfg, w, state, want_q=True, want_actions=True)
    q, a = q.view(B * N, 9), a.view(-1)
    scale = q_ref.abs().amax(dim=1, keepdim=True)
    err = ((q.double() - q_ref.double()).abs() / scale.double()).max().item()
    assert err <= Q_RTOL, f"Q relative error {err:.3e}"
    flips = a != a_ref
    if flips.any():
        top2 = torch.topk(q_ref[flips], 2, dim=1).values
        gap = ((top2[:, 0] - top2[:, 1]) / scale[flips].squeeze(1)).max().item()
        assert gap <= 4 * Q_RTOL, f"an action flipped at a top-2 gap of {gap:.3e}"
    assert flips.float().mean().item() <= 0.005


@pytest.mark.gpu
def test_forward_large_against_oracle():
    """Directly against the oracle's GCN.forward on the oracle's radius edge list."""
    import swarm_b200 as sb
    from oracle import batched_oracle as bo
    ops, L = sb.ops, sb._lib
    B, N, radius = 2, 150, 0.25
    params = load_params("GoTo", 2)
    pos, vel = _swarm(B, N, seed=3, spread=0.9)
    with torch.no_grad():
        q_ref = bo.gatq(params, pos, vel, bo.edges_radius(pos, radius))
    # the oracle's node features carry GoTo's goal: same constant in both scenarios
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N, L.GRAPH_RADIUS, graph_radius=radius)
    q = ops.gatq_forward_large(cfg, sb.pack_weights(params, _dev()), torch.cat([pos, vel], 2).contiguous().to(_dev()))
    scale = q_ref.abs().amax(dim=-1, keepdim=True)
    err = ((q.cpu().double() - q_ref.double()).abs() / scale.double()).max().item()
    assert err <= Q_RTOL, f"Q relative error {err:.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("mode,N,B,radius", [("radius", 1024, 3, 0.35), ("complete", 300, 3, 0.0), ("radius", 4096, 2, 0.2)])
def test_rollout_large_radius_and_complete(mode, N, B, radius):
    """swarm_rollout_large on the radius / complete graph (forward_large + world step per tick, launched from the
    library) against the generic tick loop (CSR graph -> bit-faithful forward -> world step): same states except where a
    near-tie flips a greedy action; returns / hits accumulate on the device and continue running totals."""
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    dev = _dev()
    pos, vel = _swarm(B, N, seed=N + 1, spread=0.7)
    vel.zero_()
    state = torch.cat([pos, vel], 2).contiguous().to(dev)
    w = sb.pack_weights(load_params("ObstacleAvoidance", 0), dev)
    gm = L.GRAPH_RADIUS if mode == "radius" else L.GRAPH_COMPLETE
    cfg = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B, N, gm, graph_radius=radius if mode == "radius" else 0.35)
    T = 3
    rx = ops.rollout_large(cfg, w, state.clone(), T, fused=True)
    rg = ops.rollout_large(cfg, w, state.clone(), T, fused=False)
    assert torch.isfinite(rx["state"]).all()
    same = (rx["state"] == rg["state"]).all(dim=-1).float().mean().item()
    assert same >= 0.995, f"only {same:.4f} of the agents end in the generic path's state"
    clean = (rx["state"] == rg["state"]).all(dim=-1)
    assert torch.allclose(rx["returns"][clean], rg["returns"][clean], rtol=1e-5, atol=1e-5)
    # a single tick: no action can have been influenced by an earlier flip
    r1 = ops.rollout_large(cfg, w, state.clone(), 1, fused=True)
    g1 = ops.rollout_large(cfg, w, state.clone(), 1, fused=False)
    assert (r1["state"] == g1["state"]).all(dim=-1).float().mean().item() >= 0.998
    # running totals continue; GoTo's collective reward through the same loop
    cg = ops.make_config(L.SCENARIO_GOTO, B, N, gm, graph_radius=radius if mode == "radius" else 0.35)
    r2 = ops.rollout_large(cg, w, rx["state"].clone(), 2, returns=rx["returns"].clone(), hits=rx["hits"].clone())
    assert (r2["returns"] < rx["returns"]).all() and torch.equal(r2["hits"], rx["hits"])


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", ["obstacle_avoidance", "go_to"])
@pytest.mark.parametrize("N,B,spread", [(1024, 6, 0.5), (300, 5, 0.45), (4096, 2, 0.55), (640, 3, 0.02), (129, 4, 0.6)])
def test_grid_world_step_equals_full_sweep(scenario, N, B, spread, monkeypatch):
    """World step of a large env with its contact partners from the uniform grid (visited in ascending agent order) ==
    the full partner sweep (SWARM_STEP_GRID=0; pinned against the oracle in test_gpu_large.py), bit for bit: squeezed
    swarms full of contacts, a collapsed swarm (more candidates than the merge handles: per-agent fallback), in place."""
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    dev = _dev()
    pos, vel = _swarm(B, N, seed=N + 3, spread=spread, jitter=0.01)
    if scenario == "obstacle_avoidance":
        pos[0] += torch.tensor([-0.1, 0.1]) - pos[0].mean(dim=0)        # park one swarm on the obstacle
    state = torch.cat([pos, vel], 2).contiguous().to(dev)
    actions = torch.randint(0, 9, (B, N), generator=torch.Generator().manual_seed(2)).to(torch.int32).to(dev)
    cfg = ops.make_config(L.SCENARIO_GOTO if scenario == "go_to" else L.SCENARIO_OBSTACLE_AVOIDANCE, B, N)
    d = torch.cdist(pos[-1], pos[-1]) + 10 * torch.eye(N)
    assert (d <= 0.1).any(), "the fixture must contain agent-agent contacts"
    monkeypatch.setenv("SWARM_STEP_GRID", "0")
    ref = ops.sim_step(cfg, state, actions)
    monkeypatch.setenv("SWARM_STEP_GRID", "1")                        # forced: the default starts at 512 agents
    out = ops.sim_step(cfg, state, actions)
    for key in ("state", "rewards", "flags", "dist", "obs"):
        assert torch.equal(out[key], ref[key]), key
    work = state.clone()
    inplace = ops.sim_step(cfg, work, actions, state_out=work, want_obs=False)
    assert torch.equal(inplace["state"], ref["state"]) and torch.equal(inplace["rewards"], ref["rewards"])


@pytest.mark.gpu
@pytest.mark.parametrize("N,B,vscale", [(1024, 3, 0.2), (129, 5, 0.2), (1000, 2, 3.0), (2048, 2, 1.0), (300, 4, 30.0),
                                        (640, 2, 0.0), (4096, 2, 0.5), (1022, 2, 1.0), (131, 3, 5.0), (5, 64, 1.0)])
def test_complete_graph_sorted_forward_equals_csr(N, B, vscale):
    """Complete graph of a large env in O(N log N) (sources sorted by alpha_src, prefix / suffix scans of the factorised
    softmax weights, own term removed, the holder of the largest alpha_src summed directly) against the bit-faithful CSR
    forward on the materialised complete graph (about 34 M edges at 2 x 4 096 agents): Q within 1e-5 of the row's
    largest magnitude, also with velocities that stretch the attention logits over hundreds of units."""
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    dev = _dev()
    pos, vel = _swarm(B, N, seed=N + 7, spread=0.8)
    vel = vel * (vscale / 0.2)
    if vscale == 0.0:
        pos[0] = pos[0, :1]                                   # an env whose agents all share one state: every alpha ties
    state = torch.cat([pos, vel], 2).contiguous().to(dev)
    cfg = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B, N, L.GRAPH_COMPLETE)
    edges, _ = ops.graph_build(cfg, state)
    offs = (torch.arange(B, device=dev, dtype=torch.int64) * N).view(B, 1, 1)
    ei = (edges.to(torch.int64) + offs).permute(1, 0, 2).reshape(2, -1).contiguous()
    del edges
    row_ptr, src, _ = ops.csr_from_edges(ei, B * N)
    del ei
    x = _x(cfg, state)
    for model in (0, 3):
        w = sb.pack_weights(load_params("ObstacleAvoidance", model), dev)
        q_sort, a_sort = ops.gatq_forward_large(cfg, w, state, want_q=True, want_actions=True)
        assert torch.isfinite(q_sort).all()
        assert torch.equal(a_sort.long(), torch.argmax(q_sort, dim=-1))
        q_ref = ops.gatq_forward_csr(w, x, row_ptr, src, want_q=True, want_actions=False)
        scale = q_ref.abs().amax(dim=1, keepdim=True).clamp_min(1e-3)
        err = ((q_sort.view(B * N, 9).double() - q_ref.double()).abs() / scale.double()).max().item()
        assert err <= Q_RTOL, f"model {model}: sorted vs CSR forward Q relative error {err:.3e}"
