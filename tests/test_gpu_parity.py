"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star):
  * bit-exact: start grids, kNN / complete edge lists, collision masks, obstacle flags, and -- whenever no
    contact force acts on the agent -- positions, velocities and rewards;
  * float32 tolerance 1e-6 relative for states / rewards of agents under a contact force (logaddexp);
  * Q-values within 1e-5 relative; greedy actions equal except where the oracle's own top-2 Q gap is below
    that tolerance (counted and bounded).
"""
import numpy as np
import pytest
import torch

from helpers import eval_centers, golden_eval, load_params, rel_err

pytestmark = pytest.mark.gpu

Q_RTOL = 1e-5
STATE_RTOL = 1e-6


def _swarm():
    import swarm_b200
    return swarm_b200


def _dev():
    return torch.device("cuda:0")


def _scen_id(sb, scenario):
    from oracle import swarm_oracle as so
    return sb._lib.SCENARIO_GOTO if scenario == so.GOTO else sb._lib.SCENARIO_OBSTACLE_AVOIDANCE


def _pack_state(pos, vel):
    return torch.cat([pos, vel], dim=2).contiguous()


def _random_states(scenario, B, N, seed, crowd=True):
    """Grid starts perturbed so that agent-agent and agent-obstacle contacts occur."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    g = torch.Generator().manual_seed(seed)
    centers = torch.stack([so.draw_center(scenario, True, g) for _ in range(B)])
    if scenario == so.OBSTACLE_AVOIDANCE:
        # move a third of the swarms onto the obstacle
        centers[::3] = torch.tensor(list(so.OBSTACLE_POS)) + 0.1 * torch.randn(len(centers[::3]), 2, generator=g)
    pos, vel = bo.reset_grid(scenario, centers, N)
    if crowd:
        scale = torch.rand(B, 1, 1, generator=g) * 0.6 + 0.4            # squeeze grids: spacing 0.06 .. 0.15
        ctr = pos.mean(dim=1, keepdim=True)
        pos = ctr + (pos - ctr) * scale + 0.01 * torch.randn(B, N, 2, generator=g)
        vel = 0.3 * torch.randn(B, N, 2, generator=g)
    return pos.contiguous(), vel.contiguous()


def _assert_state_close(name, got, ref, touched):
    """bit-exact where no contact force acted; STATE_RTOL (relative, with a 1e-7 absolute floor) elsewhere."""
    free = ~touched
    g, r = got[free], ref[free]
    assert torch.equal(g, r), f"{name}: {int((g != r).any(-1).sum() if g.dim() > 1 else (g != r).sum())} contact-free agents differ"
    g, r = got[touched].double(), ref[touched].double()
    if g.numel():
        err = ((g - r).abs() / r.abs().clamp_min(1e-1)).max().item()
        assert err <= STATE_RTOL, f"{name}: relative error {err:.3e} under contact"


@pytest.mark.parametrize("scenario", ["go_to", "obstacle_avoidance"])
@pytest.mark.parametrize("n", [1, 5, 9, 12, 32])
def test_reset_grid_bitexact(scenario, n):
    from oracle import swarm_oracle as so, batched_oracle as bo
    sb = _swarm()
    g = torch.Generator().manual_seed(n)
    centers = torch.stack([so.draw_center(scenario, True, g) for _ in range(64)])
    ref, _ = bo.reset_grid(scenario, centers, n)
    cfg = sb.ops.make_config(_scen_id(sb, scenario), 64, n)
    state = sb.ops.reset_grid(cfg, centers.to(_dev()))
    assert torch.equal(state[:, :, :2].cpu(), ref)
    assert torch.count_nonzero(state[:, :, 2:]) == 0


@pytest.mark.parametrize("scenario", ["go_to", "obstacle_avoidance"])
@pytest.mark.parametrize("n,B", [(5, 600), (12, 600), (7, 37), (32, 64), (40, 9),
                                 # >= 148 full tiles: the TMA-pipelined streaming kernel (+ ragged tail on the plain one)
                                 (12, 4100), (5, 8000), (32, 1200), (7, 16001),
                                 # 65 .. 128 agents: the one-tile kernel, two envs per CTA
                                 (96, 40), (127, 300), (128, 300)])
def test_sim_step_parity(scenario, n, B):
    from oracle import batched_oracle as bo
    sb = _swarm()
    pos, vel = _random_states(scenario, B, n, seed=100 + n)
    g = torch.Generator().manual_seed(7)
    actions = torch.randint(0, 9, (B, n), generator=g)
    ref = bo.step(scenario, pos, vel, actions)
    cfg = sb.ops.make_config(_scen_id(sb, scenario), B, n)
    out = sb.ops.sim_step(cfg, _pack_state(pos, vel).to(_dev()), actions.to(torch.int32).to(_dev()),
                          want_contact=(n <= 32))
    st = out["state"].cpu()
    flags = out["flags"].cpu()
    assert torch.equal(flags, ref["flags"]), "obstacle contact / hit / penalty flags differ"
    if n <= 32:
        mask = out["contact"].cpu().to(torch.int64) & 0xFFFFFFFF
        assert torch.equal(mask, ref["contact"]), "agent-agent collision masks differ"
    touched = ref["agent_contact"] | ((ref["flags"] & 1) != 0)
    assert touched.any(), "test inputs should exercise contacts"
    _assert_state_close("pos", st[:, :, :2], ref["pos"], touched)
    _assert_state_close("vel", st[:, :, 2:], ref["vel"], touched)
    rew_touched = touched if scenario == "obstacle_avoidance" else touched.any(dim=1, keepdim=True).expand_as(touched)
    _assert_state_close("rewards", out["rewards"].cpu(), ref["rewards"], rew_touched)
    _assert_state_close("d_goal", out["dist"][:, :, 0].cpu(), ref["d_goal"], touched)
    if scenario == "obstacle_avoidance":
        _assert_state_close("d_obs", out["dist"][:, :, 1].cpu(), ref["d_obs"], touched)
    obs = out["obs"].cpu()
    assert torch.equal(obs[:, :, :4], st) and torch.all(obs[:, :, 4] == -0.8) and torch.all(obs[:, :, 5] == 0.8)


def test_contact_force_known_answers():
    """SURVEY.md D.5: f(p_a - p_b) for p_a = (0,0)."""
    sb = _swarm()
    cases = [((0.06, 0.08), (-0.041588831692934036, -0.05545177310705185)),
             ((0.03, 0.04), (-3.0, -4.0)),
             ((0.0600001, 0.08), (0.0, 0.0))]
    for (bx, by), (fx, fy) in cases:
        cfg = sb.ops.make_config(sb._lib.SCENARIO_GOTO, 1, 2)
        state = torch.tensor([[[0.0, 0.0, 0.0, 0.0], [bx, by, 0.0, 0.0]]], device=_dev())
        out = sb.ops.sim_step(cfg, state, torch.zeros(1, 2, dtype=torch.int32, device=_dev()))
        v = out["state"][0, 0, 2:].cpu().double() / 0.1         # v = F * dt from rest, action 0
        assert abs(v[0].item() - fx) <= 2e-6 * max(1.0, abs(fx)) and abs(v[1].item() - fy) <= 2e-6 * max(1.0, abs(fy))


@pytest.mark.parametrize("n", [5, 6, 7, 8, 9, 10, 11, 12, 20, 32])
def test_graph_knn_bitexact(n):
    """Edge lists incl. order, duplicates and torch.topk tie behaviour; regular grids make ties the norm."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    sb = _swarm()
    B = 96
    g = torch.Generator().manual_seed(n)
    centers = torch.stack([so.draw_center(so.GOTO, True, g) for _ in range(B)])
    pos, vel = bo.reset_grid(so.GOTO, centers, n)
    pos[B // 2:] += 0.02 * torch.randn(B - B // 2, n, 2, generator=g)      # half exact grids, half perturbed
    for k in sorted({min(5, n), min(10, n), n, 1}):
        nbr_ref = bo.knn_table(pos, k)
        edges_ref = bo.edges_from_knn(nbr_ref)
        cfg = sb.ops.make_config(sb._lib.SCENARIO_GOTO, B, n, sb._lib.GRAPH_KNN, k)
        edges, nbr = sb.ops.graph_build(cfg, _pack_state(pos, vel).to(_dev()), want_neighbours=True)
        assert torch.equal(nbr.cpu().long(), nbr_ref), f"N={n} k={k}: topk index rows differ"
        assert torch.equal(edges.cpu().long(), edges_ref), f"N={n} k={k}: edge lists differ"


def test_graph_knn_k_out_of_range():
    """simulator.py:19 with n_agents < k raises in the reference (torch.topk); same error class and text."""
    sb = _swarm()
    cfg = sb.ops.make_config(sb._lib.SCENARIO_GOTO, 1, 5, sb._lib.GRAPH_KNN, 10)
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        sb.ops.graph_build(cfg, torch.zeros(1, 5, 4, device=_dev()))


@pytest.mark.parametrize("n", [1, 2, 5, 12, 31])
def test_graph_complete_bitexact(n):
    from oracle import batched_oracle as bo
    sb = _swarm()
    cfg = sb.ops.make_config(sb._lib.SCENARIO_GOTO, 7, n, sb._lib.GRAPH_COMPLETE)
    edges, _ = sb.ops.graph_build(cfg, torch.zeros(7, n, 4, device=_dev()))
    assert torch.equal(edges.cpu().long(), bo.edges_complete(7, n))


def _check_q_and_actions(q, act, q_ref, label):
    """Q within Q_RTOL; actions equal unless the oracle's top-2 gap is inside the tolerance band."""
    scale = q_ref.abs().amax(dim=-1, keepdim=True)
    err = ((q.double() - q_ref.double()).abs() / scale.double()).max().item()
    assert err <= Q_RTOL, f"{label}: Q relative error {err:.3e}"
    a_ref = torch.argmax(q_ref, dim=-1)
    top2 = torch.topk(q_ref, 2, dim=-1).values
    gap = (top2[..., 0] - top2[..., 1])
    flips = act.long() != a_ref
    excused = gap <= 2 * Q_RTOL * scale.squeeze(-1)
    bad = flips & ~excused
    assert not bad.any(), f"{label}: {int(bad.sum())} greedy actions differ outside the Q tolerance band"
    assert flips.float().mean().item() <= 2e-3, f"{label}: too many excused flips ({int(flips.sum())})"
    return int(flips.sum())


@pytest.mark.parametrize("exp,scenario", [("GoTo", "go_to"), ("ObstacleAvoidance", "obstacle_avoidance")])
@pytest.mark.parametrize("n,mode,k", [(5, "knn", 5), (12, "knn", 5), (12, "complete", 0), (5, "complete", 0),
                                      (10, "knn", 10), (32, "complete", 0)])
def test_gatq_forward_parity(exp, scenario, n, mode, k):
    from oracle import batched_oracle as bo
    sb = _swarm()
    B = 200
    pos, vel = _random_states(scenario, B, n, seed=n, crowd=(mode == "knn"))
    total_flips = 0
    for model in (0, 3, 7):
        params = load_params(exp, model)
        edges = bo.graph_edges(pos, mode, k)
        with torch.no_grad():
            q_ref = bo.gatq(params, pos, vel, edges)
        gm = sb._lib.GRAPH_KNN if mode == "knn" else sb._lib.GRAPH_COMPLETE
        cfg = sb.ops.make_config(_scen_id(sb, scenario), B, n, gm, max(k, 1))
        q, act = sb.ops.gatq_forward(cfg, sb.pack_weights(params, _dev()), _pack_state(pos, vel).to(_dev()))
        total_flips += _check_q_and_actions(q.cpu(), act.cpu(), q_ref, f"{exp} m{model} N{n} {mode}")
    print(f"excused flips: {total_flips}")


def test_known_answer_q_values():
    """SURVEY.md D.3 / D.4: GoTo model 0 at the first golden state."""
    sb = _swarm()
    from oracle import batched_oracle as bo
    center = torch.tensor([[1.0912246704101562, -1.1671851873397827]])
    pos, vel = bo.reset_grid("go_to", center, 5)
    cfg = sb.ops.make_config(sb._lib.SCENARIO_GOTO, 1, 5, sb._lib.GRAPH_KNN, 5)
    st = _pack_state(pos, vel).to(_dev())
    edges, _ = sb.ops.graph_build(cfg, st)
    d3 = [[0,0],[0,0],[0,1],[1,0],[0,3],[3,0],[0,4],[4,0],[0,2],[2,0],[1,1],[1,1],[1,2],[2,1],[1,0],[0,1],[1,4],[4,1],[1,3],[3,1],
          [2,2],[2,2],[2,1],[1,2],[2,4],[4,2],[2,0],[0,2],[2,3],[3,2],[3,3],[3,3],[3,4],[4,3],[3,0],[0,3],[3,1],[1,3],[3,2],[2,3],
          [4,4],[4,4],[4,3],[3,4],[4,1],[1,4],[4,2],[2,4],[4,0],[0,4],[0,0]]
    assert edges[0].t().cpu().tolist() == d3
    q, act = sb.ops.gatq_forward(cfg, sb.pack_weights(load_params("GoTo", 0), _dev()), st)
    row0 = torch.tensor([-480.535125732, -479.557739258, -476.046112061, -478.448791504, -481.078460693,
                         -470.474761963, -477.220703125, -478.659271240, -477.309295654])
    assert rel_err(q[0, 0].cpu(), row0) <= Q_RTOL
    assert act.cpu().tolist() == [[5, 5, 5, 5, 5]]


@pytest.mark.parametrize("exp,scenario", [("GoTo", "go_to"), ("ObstacleAvoidance", "obstacle_avoidance")])
def test_gcn_module_generic_graph(exp, scenario):
    """The nn.Module seam: shipped state dict -> GCN.forward(Batch) through the CSR kernels."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    sb = _swarm()
    params = load_params(exp, 2)
    model = sb.GCN(7, 32, 9)
    model.load_state_dict(params)
    model = model.to(_dev()).eval()
    # ragged batch: graphs of different sizes and kinds, plus an isolated node (no in-edges -> bias only)
    xs, eis = [], []
    g = torch.Generator().manual_seed(0)
    for n, kind in ((5, "knn"), (12, "complete"), (7, "knn"), (1, "complete"), (9, "complete")):
        pos, vel = _random_states(scenario, 1, n, seed=n)
        x = bo.node_features(pos, vel)[0]
        ei = so.graph_knn(x, min(5, n)) if kind == "knn" else so.graph_complete(n)
        xs.append(x)
        eis.append(ei)
    xs.append(torch.randn(3, 7, generator=g))
    eis.append(torch.tensor([[0, 1], [1, 0]]))                     # node 2 isolated
    x_all, ei_all = so.batch_graphs(xs, eis)
    with torch.no_grad():
        q_ref = so.gatq_forward(params, x_all, ei_all)
        batch = sb.Batch.from_data_list([sb.Data(x=x.to(_dev()), edge_index=e.to(_dev())) for x, e in zip(xs, eis)])
        q = model(batch)
    scale = q_ref.abs().amax(dim=-1, keepdim=True)
    assert ((q.cpu().double() - q_ref.double()).abs() / scale.double()).max().item() <= Q_RTOL
    # CSR grouping is the stable sort by target
    row_ptr, src, perm = sb.ops.csr_from_edges(ei_all.to(_dev()), x_all.shape[0])
    order = torch.sort(ei_all[1], stable=True).indices
    assert torch.equal(perm.cpu().long(), order)
    assert torch.equal(src.cpu().long(), ei_all[0][order])
    counts = torch.bincount(ei_all[1], minlength=x_all.shape[0])
    assert torch.equal(row_ptr.cpu().long(), torch.cat([torch.zeros(1, dtype=torch.long), counts.cumsum(0)]))


@pytest.mark.parametrize("exp,scenario,mode", [("GoTo", "go_to", "knn"), ("ObstacleAvoidance", "obstacle_avoidance", "knn"),
                                               ("ObstacleAvoidance", "obstacle_avoidance", "complete"),
                                               ("GoTo", "go_to", "complete")])
def test_rollout_teacher_forced(exp, scenario, mode):
    """Fixed-horizon fused rollout with the oracle's actions injected: every tick's edges / Q / greedy action /
    state / reward / masks are compared with the oracle's trace."""
    from oracle import batched_oracle as bo
    sb = _swarm()
    B, N, T, k = 48, 12, 30, 5
    params = load_params(exp, 1)
    pos, vel = _random_states(scenario, B, N, seed=11, crowd=False)
    ref = bo.rollout(scenario, params, pos, vel, T, mode, k)
    gm = sb._lib.GRAPH_KNN if mode == "knn" else sb._lib.GRAPH_COMPLETE
    cfg = sb.ops.make_config(_scen_id(sb, scenario), B, N, gm, k)
    state = _pack_state(pos, vel).to(_dev())
    forced = ref["actions"].to(torch.int32).to(_dev()).contiguous()
    # greedy actions of the kernel itself are observed through a second, un-forced single-tick forward below
    out = sb.ops.rollout(cfg, sb.pack_weights(params, _dev()), state, T, forced_actions=forced,
                         trace=dict(state=True, actions=True, q=True, rewards=True, flags=True, contact=True, edges=True,
                                    dist=True))
    assert torch.equal(out["trace_actions"].cpu().long(), ref["actions"])
    assert torch.equal(out["trace_edges"].cpu().long(), ref["edges"]), "per-tick edge lists differ"
    assert torch.equal(out["trace_flags"].cpu(), ref["flags"])
    assert torch.equal(out["trace_contact"].cpu().long() & 0xFFFFFFFF, ref["contact"])
    # an agent's trajectory is bit-exact until the first contact force anywhere in its env
    touched = ((ref["contact"] != 0) | ((ref["flags"] & 1) != 0)).any(dim=2, keepdim=True)
    ever = (torch.cumsum(touched.long(), dim=0) > 0).expand(T, B, N)
    st = out["trace_state"].cpu()
    assert torch.equal(st[..., :2][~ever], ref["pos"][~ever])
    assert torch.equal(st[..., 2:][~ever], ref["vel"][~ever])
    assert torch.equal(out["trace_rewards"].cpu()[~ever], ref["rewards"][~ever])
    assert ((st[..., :2] - ref["pos"]).abs().max().item()) <= 1e-4
    # Q parity on the ticks whose input state is bit-identical (tick 0 and every untouched prefix)
    q = out["trace_q"].cpu()
    pre = torch.cat([torch.zeros(1, B, N, dtype=torch.bool), ever[:-1]], dim=0)      # state entering tick t touched?
    clean = ~pre
    scale = ref["q"].abs().amax(dim=-1, keepdim=True)
    err = ((q.double() - ref["q"].double()).abs() / scale.double())[clean].max().item()
    assert err <= Q_RTOL, f"Q relative error {err:.3e}"
    greedy = torch.argmax(q, dim=-1)
    top2 = torch.topk(ref["q"], 2, dim=-1).values
    excused = (top2[..., 0] - top2[..., 1]) <= 2 * Q_RTOL * scale.squeeze(-1)
    bad = (greedy != ref["actions"]) & clean & ~excused
    assert not bad.any(), f"{int(bad.sum())} greedy actions differ outside the tolerance band"
    # returns = sum of per-tick rewards in tick order; hits = sum of hit flags
    ret = torch.zeros(B, N)
    for t in range(T):
        ret = ret + out["trace_rewards"][t].cpu()
    assert torch.equal(out["returns"].cpu(), ret)
    assert torch.equal(out["hits"].cpu().long(), ((out["trace_flags"].cpu() & 2) != 0).sum(dim=(0, 2)))


@pytest.mark.parametrize("exp,models,agents", [("go_to", (0, 4, 9), (5, 8, 12)), ("obstacle_avoidance", (0, 3, 8), (5, 9, 12))])
def test_rollout_reproduces_reference_goldens(exp, models, agents):
    """Free-running fused greedy rollout (kNN k=5) against the reference's own shipped trajectories
    (data/test_stats/**/positions_episode_*.csv, full float32 repr).  The 8 episodes of a golden run are 8
    envs of one batch.  Episodes may only deviate after a greedy action whose oracle Q gap is inside the
    float tolerance band; the bit-identical count is asserted at the measured value."""
    sb = _swarm()
    scen = sb._lib.SCENARIO_GOTO if exp == "go_to" else sb._lib.SCENARIO_OBSTACLE_AVOIDANCE
    T = 50 if exp == "go_to" else 100
    exact = total = 0
    for n in agents:
        centers = eval_centers(exp, n)
        for m in models:
            gold = golden_eval(exp, m, n)
            cfg = sb.ops.make_config(scen, 8, n, sb._lib.GRAPH_KNN, 5)
            state = sb.ops.reset_grid(cfg, centers.to(_dev()))
            out = sb.ops.rollout(cfg, sb.pack_weights(load_params(exp, m), _dev()), state, T,
                                 trace=dict(state=True, flags=True, dist=True))
            pos = out["trace_state"][..., :2].cpu().permute(1, 0, 2, 3).numpy()       # [8, T, n, 2]
            eq = (pos == gold["pos"]).all(axis=(1, 2, 3))
            exact += int(eq.sum())
            total += 8
            hits = ((out["trace_flags"].cpu() & 2) != 0).sum(dim=2).t().numpy().astype(np.float32)   # [8, T]
            for e in np.nonzero(eq)[0]:
                assert (hits[e] == gold["hits"][e]).all()
                d = out["trace_dist"][:, e, :, 0].cpu()
                mean_d = torch.stack([torch.mean(torch.stack([d[t, i] for i in range(n)])) for t in range(T)])
                assert np.array_equal(mean_d.numpy(), gold["dist"][e]), "mean goal distance trace differs"
    print(f"{exp}: {exact}/{total} golden episodes reproduced bit-for-bit by the fused CUDA rollout")
    # measured on B200 (the complete sweep with the per-episode near-tie analysis is tests/test_gpu_golden_sweep.py)
    assert exact >= {"go_to": 72, "obstacle_avoidance": 70}[exp], f"{exact}/{total}"


def _ragged_batch(scenario, seed=0):
    """Graphs of different sizes and kinds, duplicate edges, self loops and an isolated node."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    xs, eis = [], []
    g = torch.Generator().manual_seed(seed)
    for n, kind in ((5, "knn"), (12, "complete"), (7, "knn"), (1, "complete"), (9, "complete"), (30, "knn")):
        pos, vel = _random_states(scenario, 1, n, seed=n + seed)
        x = bo.node_features(pos, vel)[0]
        ei = so.graph_knn(x, min(5, n)) if kind == "knn" else so.graph_complete(n)
        xs.append(x)
        eis.append(ei)
    xs.append(torch.randn(4, 7, generator=g))
    eis.append(torch.tensor([[0, 1, 1, 3, 3], [1, 0, 0, 3, 3]]))     # duplicates, double self loop, node 2 isolated
    return so.batch_graphs(xs, eis)


@pytest.mark.parametrize("exp,scenario", [("GoTo", "go_to"), ("ObstacleAvoidance", "obstacle_avoidance")])
def test_gcn_module_backward_generic_graph(exp, scenario):
    """loss.backward() through GCN.forward on an arbitrary Batch: parameter gradients against torch autograd of the
    oracle network (per tensor, relative to that tensor's largest gradient), bit-reproducible across calls."""
    from oracle.dqn_oracle import OracleGCN
    sb = _swarm()
    params = load_params(exp, 3)
    x_all, ei_all = _ragged_batch(scenario)
    cot = torch.randn(x_all.shape[0], 9, generator=torch.Generator().manual_seed(1))
    ref = OracleGCN(7, 32, 9)
    ref.load_state_dict(params)
    (ref(x_all, ei_all) * cot).sum().backward()
    ref64 = OracleGCN(7, 32, 9).double()
    ref64.load_state_dict({k: v.double() for k, v in params.items()})
    (ref64(x_all.double(), ei_all) * cot.double()).sum().backward()

    model = sb.GCN(7, 32, 9)
    model.load_state_dict(params)
    model = model.to(_dev())
    data = sb.Data(x=x_all.to(_dev()), edge_index=ei_all.to(_dev()))
    grads = []
    for _ in range(2):
        model.zero_grad()
        (model(data) * cot.to(_dev())).sum().backward()
        grads.append({k: p.grad.detach().clone() for k, p in model.named_parameters()})
    for k in grads[0]:
        assert torch.equal(grads[0][k], grads[1][k]), f"{k}: gradient differs between two identical calls"
    for (name, p32), (_, p64) in zip(ref.named_parameters(), ref64.named_parameters()):
        g64 = p64.grad.float()
        got = grads[0][name].cpu().reshape(g64.shape)
        scale = g64.abs().max().item()
        err = (got - g64).abs().max().item()
        err32 = (p32.grad - g64).abs().max().item()
        assert err <= max(1e-5 * scale, 20 * err32), f"{name}: abs error {err:.3e} (float32 autograd {err32:.3e}, |g|max {scale:.3e})"


def test_reference_style_train_step_on_the_module():
    """The reference's train_step_dqn (train:116-126) written against the nn.Module API -- values.gather, TD target from
    a target module, MSELoss, backward, clip_grad_norm_, torch.optim.Adam -- runs on swarm_b200.GCN and tracks the same
    steps on the CPU oracle network."""
    import torch.nn as nn
    from oracle.dqn_oracle import OracleGCN
    sb = _swarm()
    params = load_params("ObstacleAvoidance", 5)
    x, ei = _ragged_batch("obstacle_avoidance", seed=2)
    x2, ei2 = _ragged_batch("obstacle_avoidance", seed=3)
    n = x.shape[0]
    g = torch.Generator().manual_seed(0)
    actions = torch.randint(0, 9, (n,), generator=g)
    rewards = torch.randn(n, generator=g)

    def make(cls, dev):
        m, t = cls(7, 32, 9), cls(7, 32, 9)
        m.load_state_dict(params)
        t.load_state_dict(load_params("ObstacleAvoidance", 6))
        return m.to(dev), t.to(dev).eval()

    def run(model, target, fwd, dev):
        opt = torch.optim.Adam(model.parameters(), lr=0.001)
        losses = []
        for _ in range(5):
            values = fwd(model, x.to(dev), ei.to(dev)).gather(1, actions.to(dev).unsqueeze(1))
            with torch.no_grad():
                nxt = fwd(target, x2.to(dev), ei2.to(dev)).max(dim=1)[0]
            tgt = rewards.to(dev) + 0.99 * nxt
            loss = nn.MSELoss()(values, tgt.unsqueeze(1))
            opt.zero_grad()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            opt.step()
            losses.append(loss.item())
        return losses, {k: v.detach().cpu() for k, v in model.state_dict().items()}

    om, ot = make(OracleGCN, "cpu")
    ref_losses, ref_sd = run(om, ot, lambda m, xx, ee: m(xx, ee), "cpu")
    gm, gt = make(sb.GCN, _dev())
    got_losses, got_sd = run(gm, gt, lambda m, xx, ee: m(sb.Data(x=xx, edge_index=ee)), _dev())
    for a, b in zip(got_losses, ref_losses):
        assert abs(a - b) <= 1e-4 * abs(b), (got_losses, ref_losses)
    assert got_losses[-1] < got_losses[0]
    for k in ref_sd:
        assert torch.allclose(got_sd[k].reshape(ref_sd[k].shape), ref_sd[k], rtol=2e-4, atol=2e-5), k


@pytest.mark.parametrize("exp,scenario", [("GoTo", "go_to"), ("ObstacleAvoidance", "obstacle_avoidance")])
def test_gatconv_layer_alone_forward_backward(exp, scenario):
    """The network class as the reference DEFINES it (train:50-70): its own ``forward`` composed of
    ``GATConv(x, edge_index)`` + torch tanh / Linear / relu, with only the GATConv layer from this package.  Loads the
    shipped state dict (same key set), matches the fused swarm_b200.GCN and the oracle network in value and in every
    parameter gradient, and is bit-reproducible across calls."""
    import torch.nn as nn
    from oracle.dqn_oracle import OracleGCN
    sb = _swarm()

    def nerr(a, b):                        # max error relative to the largest reference magnitude
        return float((a.double() - b.double()).abs().max() / b.double().abs().max())

    class ReferenceStyleGCN(nn.Module):
        def __init__(self, input_dim, hidden_dim, output_dim):
            super().__init__()
            self.conv1 = sb.GATConv(input_dim, hidden_dim, add_self_loops=False, bias=True)
            self.lin1 = nn.Linear(hidden_dim, hidden_dim)
            self.lin2 = nn.Linear(hidden_dim, output_dim)

        def forward(self, data):
            x, edge_index = data.x, data.edge_index
            x = torch.tanh(self.conv1(x, edge_index))
            x = torch.relu(self.lin1(x))
            return self.lin2(x)

    params = load_params(exp, 4)
    x_all, ei_all = _ragged_batch(scenario, seed=5)
    cot = torch.randn(x_all.shape[0], 9, generator=torch.Generator().manual_seed(2))
    ref64 = OracleGCN(7, 32, 9).double()
    ref64.load_state_dict({k: v.double() for k, v in params.items()})
    q64 = ref64(x_all.double(), ei_all)
    (q64 * cot.double()).sum().backward()
    ref32 = OracleGCN(7, 32, 9)
    ref32.load_state_dict(params)
    (ref32(x_all, ei_all) * cot).sum().backward()

    model = ReferenceStyleGCN(7, 32, 9)
    model.load_state_dict(params)
    model = model.to(_dev())
    fused = sb.GCN(7, 32, 9)
    fused.load_state_dict(params)
    fused = fused.to(_dev())
    data = sb.Data(x=x_all.to(_dev()), edge_index=ei_all.to(_dev()))

    # the layer's own output against the oracle's conv stage
    with torch.no_grad():
        conv = model.conv1(data.x, data.edge_index).cpu()
        want = ref64.conv1(x_all.double(), ei_all)
    assert nerr(conv, want) < 2e-6
    q = model(data)
    assert nerr(q.detach().cpu(), q64.detach()) < 5e-6
    assert nerr(q.detach().cpu(), fused(data).detach().cpu()) < 5e-6

    grads = []
    for _ in range(2):
        model.zero_grad()
        (model(data) * cot.to(_dev())).sum().backward()
        grads.append({k: p.grad.detach().clone() for k, p in model.named_parameters()})
    for k in grads[0]:
        if k.startswith("conv1."):
            assert torch.equal(grads[0][k], grads[1][k]), f"{k}: gradient differs between two identical calls"
    for (name, p32), (_, p64) in zip(ref32.named_parameters(), ref64.named_parameters()):
        g64 = p64.grad.float()
        got = grads[0][name].cpu().reshape(g64.shape)
        scale = g64.abs().max().item()
        err = (got - g64).abs().max().item()
        err32 = (p32.grad - g64).abs().max().item()
        assert err <= max(1e-5 * scale, 20 * err32), f"{name}: abs error {err:.3e} (float32 autograd {err32:.3e}, |g|max {scale:.3e})"

    # empty graph and isolated nodes: the layer returns the bias for nodes without in-edges
    xe = x_all[:5].to(_dev())
    out = model.conv1(xe, torch.zeros(2, 0, dtype=torch.int64, device=_dev()))
    assert torch.equal(out, model.conv1.bias.detach().expand(5, 32))
    empty = sb.Data(x=xe, edge_index=torch.zeros(2, 0, dtype=torch.int64, device=_dev()))
    q_empty = fused(empty)
    want_empty = ref32(x_all[:5], torch.zeros(2, 0, dtype=torch.int64))
    assert nerr(q_empty.detach().cpu(), want_empty.detach()) < 5e-6
    fused.zero_grad()
    q_empty.sum().backward()                 # edgeless graph: only the bias / head gradients are non-zero
    assert float(fused.conv1.lin.weight.grad.abs().max()) == 0.0
    assert torch.allclose(fused.lin2.bias.grad.cpu(), torch.full((9,), 5.0))
    with pytest.raises(NotImplementedError):              # widths beyond the generic layer kernels (tests/test_gpu_gat_layer.py)
        sb.GATConv(7, 65).to(_dev())(xe, torch.zeros(2, 0, dtype=torch.int64, device=_dev()))
