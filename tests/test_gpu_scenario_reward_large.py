"""Flocking and Cohesion rewards for swarms of up to 4 096 agents (swarm_scenario_reward_large, and the reward of
swarm_rollout_stack_large), bit for bit.

* For N <= 128 the large kernel equals the env-tile kernel (swarm_scenario_reward).
* Above that it equals a vectorised float32 judge: torch on the CPU over [N, N - 1] partner rows, which adds each row in
  the order torch's CPU row sum takes (tests/test_torch_sum_order_cascade.py pins that order up to 4 095 elements), with
  the collective sum in agent order.  The judge is proven equal to the per-pair single-env oracle
  (oracle/scenario_rewards_oracle.FlockingOracle) at 129 and 600 agents; 600 crosses the cascade at 576.
* The stacked rollout with a reward equals the composed public calls, and the environment, Simulator and DQNTrainer run
  Flocking above 128 agents through them."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32


def _sb():
    import swarm_b200 as sb
    return sb


def _dev():
    return torch.device("cuda:0")


def _flocking_sd(seed):
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    pre = f"{seed}/"
    return {k[len(pre):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(pre)}


def _spec(kind, B, N):
    sb = _sb()
    return sb.ops.reward_spec(kind, B, N)


def _grid(B, N, seed, jitter=0.0, collapse=False):
    """state f32[B,N,4] on the device: the start grid around random centres (+ jitter), velocities small and random;
    collapse: every env's agents within 1e-3 of its centre, so every pair is a near-contact."""
    sb = _sb()
    g = torch.Generator().manual_seed(seed)
    centers = torch.tensor([-1.0, 1.0]) + torch.tensor([-0.6, 0.6]) + 0.4 * torch.randn(B, 2, generator=g)
    cfg = sb.ops.make_config(sb._lib.SCENARIO_GOTO, B, N)
    state = sb.ops.reset_grid(cfg, centers.to(_dev())).cpu()
    if collapse:
        state[..., 0:2] = centers.view(B, 1, 2) + 1e-3 * torch.rand(B, N, 2, generator=g)
    elif jitter:
        state[..., 0:2] += jitter * torch.randn(B, N, 2, generator=g)
    state[..., 2:4] = 0.1 * torch.randn(B, N, 2, generator=g)
    return state.contiguous().to(_dev())


# ---- the judge --------------------------------------------------------------------------------------------------------
def _partners(N):
    k = torch.arange(N - 1).view(1, -1)
    return k + (k >= torch.arange(N).view(-1, 1)).long()          # [N, N-1]: the list comprehension's j != i


def flocking_judge(pos, prev, reset):
    """FlockingOracle.reward / reset vectorised over every env's [N, N-1] partner rows in float32 on the CPU.
    pos f32[B,N,2]; prev f32[B,N,2] = (previous_distance_to_goal, previous_distance_to_agents) before the call.
    Returns (collective f32[B] or None, terms f32[B,N,4] or None, shaping f32[B,N,2])."""
    from oracle import scenario_rewards_oracle as sro, swarm_oracle as so
    pos = pos.cpu().float()
    B, N, _ = pos.shape
    J = _partners(N)
    later = (J > torch.arange(N).view(-1, 1)).unsqueeze(-1)
    goal = torch.tensor([list(sro.GOAL_POS)])
    shaping, terms, per_agent = [], [], []
    for b in range(B):
        p = pos[b]
        q = p[J]
        if reset:                                              # agents after i still sit at the origin (flocking:93-121)
            q = torch.where(later, torch.zeros(()), q)
        d = torch.linalg.vector_norm(p.unsqueeze(1) - q, dim=-1)                        # [N, N-1]
        spacing = (d - sro.DESIRED_DISTANCE).pow(2).mean(-1) * 10.0
        d_goal = torch.linalg.vector_norm(p - goal, dim=-1)
        shaped = d_goal * 10.0
        shaping.append(torch.stack([shaped, spacing], -1))
        if reset:
            continue
        close = (((d - so.SPHERE_RADIUS) - so.SPHERE_RADIUS) <= sro.MIN_COLLISION_DISTANCE).sum(-1)
        pos_rew = prev[b, :, 0].cpu() - shaped
        goal_reward = torch.where(d_goal < so.SPHERE_RADIUS, pos_rew + sro.ON_GOAL_BONUS, pos_rew)
        avoid = (close * sro.AGENT_COLLISION_REWARD).float()
        dist_rew = prev[b, :, 1].cpu() - spacing
        per_agent.append((goal_reward + avoid) + dist_rew)
        terms.append(torch.stack([pos_rew, avoid, dist_rew, d_goal], -1))
    if reset:
        return None, None, torch.stack(shaping)
    t = torch.stack(per_agent).numpy()
    c = np.zeros(B, F)
    for j in range(N):                                         # collective += per agent, in agent order (flocking:125-129)
        c = c + t[:, j]
    return torch.from_numpy(c), torch.stack(terms), torch.stack(shaping)


def cohesion_judge(pos):
    """CohesionOracle.reward (cohesion:66-85) restated over [N, N-1] partner rows (its constructor refuses more than nine
    agents).  Returns (reward f32[B,N], terms f32[B,N,4])."""
    from oracle import scenario_rewards_oracle as sro, swarm_oracle as so
    pos = pos.cpu().float()
    B, N, _ = pos.shape
    J = _partners(N)
    rew, terms = [], []
    for b in range(B):
        p = pos[b]
        dist = (torch.linalg.vector_norm(p.unsqueeze(1) - p[J], dim=-1) - so.SPHERE_RADIUS) - so.SPHERE_RADIUS
        mn, mx = dist.min(-1).values, dist.max(-1).values
        collision = torch.from_numpy(np.exp(-(mn / sro.SIGMA).numpy()))               # numpy's float32 exp
        collision = torch.where(mn > sro.SIGMA, torch.zeros(()), collision)
        cohesion = torch.where(mn < sro.SIGMA, torch.zeros(()), -(mx - sro.SIGMA))
        rew.append(collision + cohesion)
        terms.append(torch.stack([collision, cohesion, mn, mx], -1))
    return torch.stack(rew), torch.stack(terms)


def _check_cohesion(rew, terms, pos):
    """mn / mx and the cohesion factor bit for bit; the collision factor exp(-mn / sigma) is CUDA's expf against numpy's
    float32 exp, which may differ in the last bit; the reward is the kernel's own factors added once."""
    want_r, want_t = cohesion_judge(pos)
    t = terms.cpu()
    assert torch.equal(t[..., 1:4], want_t[..., 1:4])
    assert torch.allclose(t[..., 0], want_t[..., 0], rtol=3e-7, atol=0)
    assert torch.equal(rew.cpu(), t[..., 0] + t[..., 1])
    assert torch.allclose(rew.cpu(), want_r, rtol=3e-7, atol=1e-30)


# ---- 1. the large kernel equals the env-tile kernel for small swarms ----------------------------------------------------
@pytest.mark.parametrize("N", [2, 5, 8, 12, 13, 64, 127, 128])
def test_large_kernel_equals_env_tile_kernel(N):
    sb = _sb()
    ops, L = sb.ops, sb._lib
    B = 5
    s0 = _grid(B, N, seed=N)
    s1 = _grid(B, N, seed=N + 100, jitter=0.02)
    fl = _spec(L.REWARD_FLOCKING, B, N)
    sh_a = torch.zeros(B, N, 2, device=_dev())
    sh_b = torch.zeros(B, N, 2, device=_dev())
    ops.scenario_reward(fl, s0, sh_a, reset=True)
    ops.scenario_reward_large(fl, s0, sh_b, reset=True)
    assert torch.equal(sh_a, sh_b)
    for state, env_index in ((s1, None), (s0, 3), (s1, None)):
        ra, ta = ops.scenario_reward(fl, state, sh_a, env_index=env_index, want_terms=True)
        rb, tb = ops.scenario_reward_large(fl, state, sh_b, env_index=env_index, want_terms=True)
        assert torch.equal(ra, rb) and torch.equal(ta, tb) and torch.equal(sh_a, sh_b)
    ops.scenario_reward(fl, s1, sh_a, reset=True, env_index=1)
    ops.scenario_reward_large(fl, s1, sh_b, reset=True, env_index=1)
    assert torch.equal(sh_a, sh_b)
    co = _spec(L.REWARD_COHESION, B, N)
    for state in (s0, s1, _grid(B, N, seed=7, collapse=True)):
        ra, ta = ops.scenario_reward(co, state, want_terms=True)
        rb, tb = ops.scenario_reward_large(co, state, want_terms=True)
        assert torch.equal(ra, rb) and torch.equal(ta, tb)


# ---- 2. the judge equals the per-pair oracle ----------------------------------------------------------------------------
@pytest.mark.parametrize("N", [129, 600])
def test_judge_equals_flocking_oracle(N):
    from oracle import scenario_rewards_oracle as sro
    g = torch.Generator().manual_seed(N)
    center = torch.tensor([-1.6, 1.6]) + 0.4 * torch.randn(2, generator=g)
    orc = sro.FlockingOracle(N)
    orc.reset(center)
    pos = torch.cat(orc.world.pos).unsqueeze(0)
    _, _, sh = flocking_judge(pos, None, reset=True)
    assert torch.equal(sh[0, :, 0], torch.cat(orc.previous_distance_to_goal))
    assert torch.equal(sh[0, :, 1], torch.cat(orc.previous_distance_to_agents))
    for t in range(3):
        act = torch.randint(0, 9, (N,), generator=g)
        orc.world.step(act)
        pos = torch.cat(orc.world.pos).unsqueeze(0)
        c, terms, sh2 = flocking_judge(pos, sh, reset=False)
        want = orc.reward()
        assert torch.equal(c, want.reshape(1)), f"tick {t}"
        assert torch.equal(terms[0, :, 0], torch.cat(orc.pos_rew)) and torch.equal(terms[0, :, 2], torch.cat(orc.dist_rew))
        assert torch.equal(sh2[0, :, 0], torch.cat(orc.previous_distance_to_goal))
        assert torch.equal(sh2[0, :, 1], torch.cat(orc.previous_distance_to_agents))
        sh = sh2


# ---- 3. exact at large sizes --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,B", [(129, 3), (512, 3), (577, 3), (578, 3), (1025, 3), (2048, 2), (4096, 2)])
def test_large_swarm_rewards_equal_the_judge(N, B):
    sb = _sb()
    ops, L = sb.ops, sb._lib
    g = torch.Generator().manual_seed(N)
    fl = _spec(L.REWARD_FLOCKING, B, N)
    co = _spec(L.REWARD_COHESION, B, N)
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N)
    state = _grid(B, N, seed=N)
    shaping = torch.zeros(B, N, 2, device=_dev())
    ops.scenario_reward(fl, state, shaping, reset=True)                 # routed to the large kernel
    _, _, sh = flocking_judge(state[..., :2], None, reset=True)
    assert torch.equal(shaping.cpu(), sh), "grid reset"
    _check_cohesion(*ops.scenario_reward(co, state, want_terms=True), state[..., :2])

    def step_and_check(st, what):
        prev = shaping.clone()
        r, t = ops.scenario_reward(fl, st, shaping, want_terms=True)
        want_c, want_t, want_sh = flocking_judge(st[..., :2], prev, reset=False)
        assert torch.equal(r.cpu(), want_c), f"{what}: collective reward"
        assert torch.equal(t.cpu(), want_t), f"{what}: terms"
        assert torch.equal(shaping.cpu(), want_sh), f"{what}: shaping"
        _check_cohesion(*ops.scenario_reward(co, st, want_terms=True), st[..., :2])
        return t

    for tick in range(3):                                               # stepped ticks under random actions
        act = torch.randint(0, 9, (B, N), generator=g, dtype=torch.int32).to(_dev())
        ops.sim_step(cfg, state, act, state_out=state, want_obs=False)
        step_and_check(state, f"tick {tick}")
    step_and_check(_grid(B, N, seed=N + 1, jitter=0.05), "perturbed")
    t = step_and_check(_grid(B, N, seed=N + 2, collapse=True), "collapsed")
    assert torch.equal(t[..., 1].cpu(), torch.full((B, N), -(N - 1.0))), "every partner is a near-contact"
    # a reset of one env leaves the others' memory alone
    before = shaping.clone()
    s2 = _grid(B, N, seed=N + 3)
    ops.scenario_reward(fl, s2, shaping, reset=True, env_index=1)
    _, _, sh = flocking_judge(s2[1:2, :, :2], None, reset=True)
    assert torch.equal(shaping[1].cpu(), sh[0])
    assert torch.equal(shaping[0], before[0]) and torch.equal(shaping[2:], before[2:])


# ---- 4. the stacked rollout with a reward -------------------------------------------------------------------------------
def _composed(cfg, spec, w, state, ticks, rs, shaping):
    """[topk table ->] gatstack_forward_large -> sim_step in place -> scenario_reward_large -> returns += per tick."""
    sb = _sb()
    ops, L = sb.ops, sb._lib
    B, N = cfg.num_envs, cfg.n_agents
    returns = torch.zeros(B, N, device=state.device)
    hits = torch.zeros(B, dtype=torch.int32, device=state.device)
    act = torch.empty(B, N, dtype=torch.int32, device=state.device)
    for _ in range(ticks):
        nbr = None
        if cfg.graph_mode == L.GRAPH_KNN:
            _, nbr = ops.graph_build(cfg, state, want_neighbours=True)
        ops.gatstack_forward_large(cfg, spec, w, state, neighbours=nbr, actions=act)
        out = ops.sim_step(cfg, state, act, state_out=state, want_obs=False)
        hits += ((out["flags"] & L.FLAG_HIT) != 0).sum(dim=1, dtype=torch.int32)
        if rs.kind == L.REWARD_FLOCKING:
            returns += ops.scenario_reward_large(rs, state, shaping).view(B, 1)
        else:
            returns += ops.scenario_reward_large(rs, state)
    return state, returns, hits


@pytest.mark.parametrize("kind", ["flocking", "cohesion"])
@pytest.mark.parametrize("graph,k", [("knn", 10), ("radius", 0.35), ("complete", 0)])
def test_rollout_stack_large_equals_composed_calls(kind, graph, k):
    sb = _sb()
    ops, L = sb.ops, sb._lib
    B, N, T = 4, 1024, 5
    gm = {"complete": L.GRAPH_COMPLETE, "knn": L.GRAPH_KNN, "radius": L.GRAPH_RADIUS}[graph]
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N, gm, int(k) if graph == "knn" else 10,
                          graph_radius=float(k) if graph == "radius" else 0.35)
    spec = ops.stack_spec(3, 8, 7)
    w = ops.pack_stack_weights(_flocking_sd(0), spec, _dev())
    s0 = _grid(B, N, seed=5, jitter=0.02)
    rs = _spec(L.REWARD_FLOCKING if kind == "flocking" else L.REWARD_COHESION, B, N)
    sh0 = torch.zeros(B, N, 2, device=_dev())
    if kind == "flocking":
        ops.scenario_reward(rs, s0, sh0, reset=True)
    sh_a, sh_b = sh0.clone(), sh0.clone()
    out = ops.rollout_stack(cfg, spec, w, s0.clone(), T, reward=rs, shaping=sh_a if kind == "flocking" else None)
    st, ret, hits = _composed(cfg, spec, w, s0.clone(), T, rs, sh_b)
    assert torch.equal(out["state"], st) and not torch.equal(st, s0)
    assert torch.equal(out["returns"], ret) and torch.equal(out["hits"], hits)
    assert torch.equal(sh_a, sh_b)
    if kind == "flocking":
        assert torch.equal(ret, ret[:, :1].expand(B, N)), "every agent receives its env's collective reward"
    # without a reward: exactly swarm_rollout_stack above 128 agents
    a = ops.rollout_stack_large(cfg, spec, w, s0.clone(), T)
    b = ops.rollout_stack(cfg, spec, w, s0.clone(), T)
    for key in ("state", "returns", "hits"):
        assert torch.equal(a[key], b[key]), key


def test_rollout_stack_large_cuda_graph_replay_equals_eager():
    sb = _sb()
    ops, L = sb.ops, sb._lib
    B, N, T = 2, 1024, 3
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N, L.GRAPH_KNN, 10)
    spec = ops.stack_spec(3, 8, 7)
    w = ops.pack_stack_weights(_flocking_sd(1), spec, _dev())
    s0 = _grid(B, N, seed=9, jitter=0.02)
    rs = _spec(L.REWARD_FLOCKING, B, N)
    sh0 = torch.zeros(B, N, 2, device=_dev())
    ops.scenario_reward(rs, s0, sh0, reset=True)
    eager = ops.rollout_stack(cfg, spec, w, s0.clone(), T, reward=rs, shaping=sh0.clone())
    state, shaping = s0.clone(), sh0.clone()
    returns = torch.zeros(B, N, device=_dev())
    hits = torch.zeros(B, dtype=torch.int32, device=_dev())
    ops.rollout_stack(cfg, spec, w, state, T, reward=rs, shaping=shaping, returns=returns, hits=hits)     # warm-up
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            ops.rollout_stack(cfg, spec, w, state, T, reward=rs, shaping=shaping, returns=returns, hits=hits)
    torch.cuda.current_stream().wait_stream(s)
    state.copy_(s0); shaping.copy_(sh0); returns.zero_(); hits.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(state, eager["state"]) and torch.equal(returns, eager["returns"])
    assert torch.equal(shaping, eager["shaping"]) and torch.equal(hits, eager["hits"])


# ---- 5. environment level -----------------------------------------------------------------------------------------------
def _flocking_env(n, B, T, seed=3):
    sb = _sb()
    return sb.make_env(scenario=sb.FlockingScenario(), num_envs=B, device=_dev(), continuous_actions=False, max_steps=T,
                       dict_spaces=True, seed=seed, n_agents=n)


def test_flocking_env_with_1024_agents_equals_the_judge():
    n, B, T = 1024, 2, 3
    env = _flocking_env(n, B, T)
    torch.manual_seed(4)
    env.reset()
    sc = env.scenario
    _, _, sh = flocking_judge(env.world.state[..., :2], None, reset=True)
    assert torch.equal(sc.shaping.cpu(), sh)
    g = torch.Generator().manual_seed(5)
    for t in range(T):
        prev = sc.shaping.clone()
        act = torch.randint(0, 9, (B, n), generator=g).to(_dev())
        _, rews, _, _ = env.step({f"agent{i}": act[:, i] for i in range(n)})
        c, terms, sh = flocking_judge(env.world.state[..., :2], prev, reset=False)
        assert torch.equal(rews["agent0"].cpu(), c) and torch.equal(rews[f"agent{n - 1}"].cpu(), c), f"tick {t}"
        assert torch.equal(sc.shaping.cpu(), sh)
        assert torch.equal(sc.world.agents[7].dist_rew.cpu(), terms[:, 7, 2])


def test_simulator_and_evaluate_policy_on_a_1024_agent_flocking_env(tmp_path):
    import csv
    sb = _sb()
    ops, L = sb.ops, sb._lib
    n, T = 1024, 4
    model = sb.StackedGCN.from_state_dict(_flocking_sd(0)).to(_dev()).eval()
    spec = model.stack_spec()
    w = model.packed_stack_weights(_dev())
    # Simulator: the large forward, world step and large Flocking reward per tick; its trajectory equals the rollout's
    env = _flocking_env(n, 1, T)
    sim = sb.Simulator(env, model, 1, "flocking", 3, output_dir=str(tmp_path / "stats"), k=10)
    torch.manual_seed(11)
    sim.run_simulation()
    assert np.isfinite(sim.episode_rewards[0])
    with open(tmp_path / "stats" / "positions" / "positions_episode_0_x.csv") as f:
        rows = list(csv.reader(f))
    assert len(rows) == T + 1
    env2 = _flocking_env(n, 1, T)
    torch.manual_seed(11)
    env2.reset()
    cfg = ops.clone_config(env2.world.cfg, graph_mode=L.GRAPH_KNN, knn_k=10)
    out = ops.rollout_stack(cfg, spec, w, env2.world.state, T, reward=env2.scenario._spec(), shaping=env2.scenario.shaping)
    assert torch.equal(torch.tensor([float(v) for v in rows[-1][1:]]), out["state"][0, :, 0].cpu())
    assert torch.isfinite(out["returns"]).all()
    # DQNTrainer.evaluate_policy: agent 0's return of the stacked rollout with the Flocking reward
    env3 = _flocking_env(n, 2, T)
    tr = sb.DQNTrainer(env3, 0, str(tmp_path), str(tmp_path), "t", graph_mode="knn", knn_k=10, replay_capacity=4,
                       model=sb.StackedGCN.from_state_dict(_flocking_sd(0)))
    torch.manual_seed(12)
    got = tr.evaluate_policy(1)
    env4 = _flocking_env(n, 2, T)
    torch.manual_seed(12)
    env4.reset()
    cfg4 = ops.clone_config(env4.world.cfg, graph_mode=L.GRAPH_KNN, knn_k=10)
    rs = env4.scenario._spec()
    _, ret, _ = _composed(cfg4, spec, w, env4.world.state, T, rs, env4.scenario.shaping)
    assert got == ret[0, 0].item()
