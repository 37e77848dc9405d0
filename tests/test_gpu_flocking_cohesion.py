"""FlockingScenario / CohesionScenario (flocking_scenario.py, cohesion_scenario.py; SURVEY.md 8f rank 3) through the
environment seam: world step in swarm_sim_step (GoTo physics, covered bit-exactly by test_gpu_parity.py), rewards in
swarm_scenario_reward.  Every env is compared with its own single-env oracle (oracle/scenario_rewards_oracle.py) on the
SAME device states, tick by tick, so the reward arithmetic and the shaping memory are what is being checked.

Tolerance: rewards are chains of separately rounded float32 ops in the reference's order; the only op whose rounding
the kernel does not reproduce by construction is torch's ``mean`` (and ``exp`` for Cohesion).  torch sums a contiguous
row with SIMD partial sums whose width depends on the host CPU (8 or 16 lanes), so for more than 8 partners the
reference's own last bit is machine dependent; the kernel adds in partner order, which is what torch does below the SIMD
width.  Results must agree to 2e-5 absolute + 1e-5 relative everywhere, and up to 5 agents at least 90 % of the
collective rewards must be bit-identical."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ATOL, RTOL = 2e-5, 1e-5


def _swarm():
    import swarm_b200 as sb
    return sb


def _dev():
    return torch.device("cuda:0")


def _close(got, want):
    return torch.allclose(got, want, rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("n", [2, 5, 12])
def test_flocking_env_matches_oracle(n):
    from oracle import scenario_rewards_oracle as sro
    sb = _swarm()
    B, T = 6, 25
    g = torch.Generator().manual_seed(n)
    centers = torch.tensor([-1.0, 1.0]) + torch.tensor([-0.6, 0.6]) + 0.4 * torch.randn(B, 2, generator=g)
    scenario = sb.FlockingScenario()
    env = sb.Environment(scenario, num_envs=B, device=_dev(), max_steps=T, continuous_actions=False, seed=0,
                         dict_spaces=True, n_agents=n)
    scenario.set_start_centers(centers)
    obs = env.reset()
    assert obs["agent0"].shape == (B, 6)
    oracles = [sro.FlockingOracle(n) for _ in range(B)]
    for b, orc in enumerate(oracles):
        orc.reset(centers[b])
        pos, _ = orc.world.state()
        assert torch.equal(env.world.state[b, :, 0:2].cpu(), pos), "start grid"
        assert _close(scenario.previous_distance_to_goal[b].cpu(), torch.cat(orc.previous_distance_to_goal))
        assert _close(scenario.previous_distance_to_agents[b].cpu(), torch.cat(orc.previous_distance_to_agents))
    exact = total = 0
    for t in range(T):
        # head for the goal most of the time so that agents bunch up, touch and reach the goal
        act = torch.randint(0, 9, (B, n), generator=g)
        act = torch.where(torch.rand(B, n, generator=g) < 0.7, torch.full_like(act, 5), act)     # 5 = (-1, +1)
        obs, rews, dones, infos = env.step({f"agent{i}": act[:, i] for i in range(n)})
        state = env.world.state.cpu()
        for b, orc in enumerate(oracles):
            orc.world.set_state(state[b, :, 0:2], state[b, :, 2:4])
            want = orc.reward()
            got = rews["agent0"][b].cpu()
            assert _close(got, want[0]), (t, b, float(got), float(want))
            exact += int(got == want[0])
            total += 1
            assert _close(infos["agent0"]["pos_rew"][b].cpu(), orc.pos_rew[0][0])
        for i in range(1, n):
            assert torch.equal(rews[f"agent{i}"], rews["agent0"])         # one collective reward for everybody
        assert obs["agent0"].shape == (B, 6) and torch.equal(obs["agent0"][:, 4:6].cpu(), torch.tensor([[-0.8, 0.8]] * B))
    if n <= 5:
        assert exact >= 0.9 * total, f"only {exact} / {total} collective rewards bit-identical"


def test_flocking_contacts_goal_bonus_and_reset_at():
    """Hand-placed states on the decision boundaries: surface gap just inside / outside 0.005, an agent just inside /
    outside the goal radius; then reset_at(1) re-initialises the memory of that env only."""
    from oracle import scenario_rewards_oracle as sro
    sb = _swarm()
    n, B = 4, 3
    scenario = sb.FlockingScenario()
    env = sb.Environment(scenario, num_envs=B, device=_dev(), max_steps=10, continuous_actions=False, seed=3,
                         dict_spaces=True, n_agents=n)
    centers = torch.tensor([[0.1, 0.1], [-0.3, 0.4], [0.5, -0.2]])
    scenario.set_start_centers(centers)
    env.reset()
    oracles = [sro.FlockingOracle(n) for _ in range(B)]
    for b, orc in enumerate(oracles):
        orc.reset(centers[b])
    placed = torch.tensor([
        [[-0.8, 0.8 + 0.0499], [0.0, 0.0], [0.1049, 0.0], [0.5, 0.5]],          # on goal; pair gap 0.0049
        [[-0.8, 0.8 + 0.0501], [0.0, 0.0], [0.1051, 0.0], [0.5, 0.5]],          # just off goal; pair gap 0.0051
        [[-0.8, 0.8], [0.3, 0.3], [0.3, 0.3], [0.3, 0.4]],                      # coincident pair + a touching third
    ])
    env.world.state[:, :, 0:2] = placed.to(_dev())
    got, terms = sb.ops.scenario_reward(scenario._spec(), env.world.state, scenario.shaping, want_terms=True)
    for b, orc in enumerate(oracles):
        orc.world.set_state(placed[b], torch.zeros(n, 2))
        want = orc.reward()
        assert _close(got[b].cpu(), want[0]), (b, float(got[b]), float(want))
    terms = terms.cpu()
    assert terms[0, 0, 3] < 0.05 <= terms[1, 0, 3]                               # distance_to_goal either side of the radius
    assert terms[0, 1, 1] == -1.0 and terms[0, 2, 1] == -1.0 and terms[0, 3, 1] == 0.0
    assert (terms[1, :, 1] == 0.0).all()
    # env 2: agents 1 and 2 coincide and agent 3 touches both (centre distance 0.1 -> gap 0): two penalties each
    assert terms[2, 0, 1] == 0.0 and (terms[2, 1:, 1] == -2.0).all()
    # reset_at(1): env 1 back on its grid with fresh memory, envs 0 and 2 untouched
    before = scenario.shaping.clone()
    env.reset_at(1)
    oracles[1].reset(centers[1])
    assert torch.equal(scenario.shaping[0], before[0]) and torch.equal(scenario.shaping[2], before[2])
    assert _close(scenario.previous_distance_to_goal[1].cpu(), torch.cat(oracles[1].previous_distance_to_goal))
    assert _close(scenario.previous_distance_to_agents[1].cpu(), torch.cat(oracles[1].previous_distance_to_agents))
    assert torch.equal(env.world.state[1, :, 0:2].cpu(), oracles[1].world.state()[0])


def test_flocking_seeded_reset_follows_the_reference_generator_stream():
    """Without explicit centres the reset draws what flocking:94-98 and :70-71 draw, in that order."""
    from oracle import scenario_rewards_oracle as sro
    sb = _swarm()
    n = 5
    env = sb.make_env(scenario=sb.FlockingScenario(), num_envs=1, device=_dev(), continuous_actions=False,
                      max_steps=5, dict_spaces=True, seed=42, n_agents=n)
    after = torch.rand(1)
    torch.manual_seed(42)
    orc = sro.FlockingOracle(n)
    orc.reset()
    assert torch.equal(after, torch.rand(1))
    assert torch.equal(env.world.state[0, :, 0:2].cpu(), orc.world.state()[0])


@pytest.mark.parametrize("n", [2, 9])
def test_cohesion_env_matches_oracle(n):
    from oracle import scenario_rewards_oracle as sro
    sb = _swarm()
    B, T = 5, 20
    g = torch.Generator().manual_seed(7 + n)
    scenario = sb.CohesionScenario()
    env = sb.Environment(scenario, num_envs=B, device=_dev(), max_steps=T, continuous_actions=False, seed=0,
                         dict_spaces=True, n_agents=n)
    assert env.observation_space["agent0"].shape == (4,)
    obs = env.reset()
    assert obs["agent0"].shape == (B, 4)
    oracles = [sro.CohesionOracle(n) for _ in range(B)]
    for b, orc in enumerate(oracles):
        orc.reset()
        assert torch.equal(env.world.state[b].cpu(), torch.cat(orc.world.state(), dim=1))
    start = scenario.all_rewards().cpu()
    for b, orc in enumerate(oracles):
        assert _close(start[b], orc.reward())
    for t in range(T):
        act = torch.randint(0, 9, (B, n), generator=g)
        obs, rews, dones, infos = env.step({f"agent{i}": act[:, i] for i in range(n)})
        state = env.world.state.cpu()
        got = torch.stack([rews[f"agent{i}"] for i in range(n)], dim=1).cpu()
        for b, orc in enumerate(oracles):
            orc.world.set_state(state[b, :, 0:2], state[b, :, 2:4])
            assert _close(got[b], orc.reward()), (t, b)
        assert torch.equal(obs["agent1"].cpu(), state[:, 1])
    # both branches of cohesion:80,83 at sigma, and agents closer than sigma
    placed = torch.zeros(B, n, 2)
    placed[:, 1, 0] = torch.tensor([0.2, 0.25, 0.2500001, 0.3, 1.0])             # gaps 0.1, 0.15, ~0.15, 0.2, 0.9
    if n > 2:
        placed[:, 2:, 1] = 2.0 + torch.arange(n - 2).float().view(1, -1)
    env.world.state.zero_()
    env.world.state[:, :, 0:2] = placed.to(_dev())
    env.world.version += 1
    got = scenario.all_rewards().cpu()
    for b, orc in enumerate(oracles):
        orc.world.set_state(placed[b], torch.zeros(n, 2))
        assert _close(got[b], orc.reward()), b
    assert got[0, 0] > 0.5                                                       # exp(-(0.1 / 0.15)): the reference's sign


def test_scenario_reward_argument_errors():
    sb = _swarm()
    ops = sb.ops
    state = torch.zeros(4, 1, 4, device=_dev())
    with pytest.raises(ValueError):
        ops.scenario_reward(ops.reward_spec(sb._lib.REWARD_COHESION, 4, 1), state)          # one agent
    state = torch.zeros(4, 3, 4, device=_dev())
    with pytest.raises(ValueError):
        ops.scenario_reward(ops.reward_spec(sb._lib.REWARD_FLOCKING, 4, 3), state)          # no shaping buffer
    with pytest.raises(RuntimeError):                                                       # index errors, like torch
        ops.scenario_reward(ops.reward_spec(sb._lib.REWARD_COHESION, 4, 3), state, env_index=4)
    with pytest.raises(IndexError):
        sb.Environment(sb.CohesionScenario(), num_envs=2, device=_dev(), continuous_actions=False, n_agents=10)
    # zero envs is a no-op
    empty = torch.zeros(0, 3, 4, device=_dev())
    assert ops.scenario_reward(ops.reward_spec(sb._lib.REWARD_COHESION, 0, 3), empty).shape == (0, 3)


def test_scenario_reward_full_size_properties():
    """C2-sized batch (4096 envs x 12 agents): replicated envs give replicated rewards, a second call on an unchanged
    state returns only bonuses / penalties (the shaping memory moved), permutation of envs permutes the rewards."""
    sb = _swarm()
    ops = sb.ops
    B, n = 4096, 12
    g = torch.Generator().manual_seed(0)
    base = torch.randn(64, n, 4, generator=g) * 0.3
    state = base.repeat(B // 64, 1, 1).contiguous().to(_dev())
    spec = ops.reward_spec(sb._lib.REWARD_FLOCKING, B, n)
    shaping = torch.zeros(B, n, 2, device=_dev())
    ops.scenario_reward(spec, state, shaping, reset=True)
    moved = (state + 0.01).contiguous()
    r1, t1 = ops.scenario_reward(spec, moved, shaping, want_terms=True)
    assert torch.equal(r1.view(-1, 64), r1[:64].view(1, 64).expand(B // 64, 64))
    r2, t2 = ops.scenario_reward(spec, moved, shaping, want_terms=True)
    assert (t2[:, :, 0] == 0).all() and (t2[:, :, 2] == 0).all()                 # no progress on an unchanged state
    assert torch.equal(t2[:, :, 1], t1[:, :, 1])
    perm = torch.randperm(B, generator=g).to(_dev())
    shaping_p = torch.zeros(B, n, 2, device=_dev())
    ops.scenario_reward(spec, state[perm].contiguous(), shaping_p, reset=True)
    rp = ops.scenario_reward(spec, moved[perm].contiguous(), shaping_p)
    assert torch.equal(rp, r1[perm])
    cspec = ops.reward_spec(sb._lib.REWARD_COHESION, B, n)
    rc = ops.scenario_reward(cspec, state)
    assert torch.equal(rc[perm], ops.scenario_reward(cspec, state[perm].contiguous()))
    assert torch.isfinite(rc).all()


def test_reference_training_loop_runs_on_flocking():
    """DQNTrainer.train_model (the reference's num_envs = 1 loop, train:139-204) on a Flocking env: the transitions it
    stores carry the Flocking collective reward (not the world-step kernel's GoTo reward), the update changes the
    weights, losses are finite; the whole-run device loop refuses scenarios it cannot reset on the device."""
    sb = _swarm()
    sb.set_seed(1)
    n, T = 5, 40
    env = sb.make_env(scenario=sb.FlockingScenario(), num_envs=1, device=_dev(), continuous_actions=False, wrapper=None,
                      max_steps=T, dict_spaces=True, n_agents=n, seed=1)
    trainer = sb.DQNTrainer(env, 1, "/tmp/swarm_models", "/tmp/swarm_stats", "Flocking", replay_capacity=512)
    w0 = trainer.w.clone()
    seen = []
    step = env.step

    def recording_step(actions):
        out = step(actions)
        seen.append(out[1]["agent0"].clone())
        return out

    env.step = recording_step
    trainer.train_model({"epsilon": 0.99, "epsilon_decay": 0.01, "min_epsilon": 0.05, "episodes": 2, "verbose": False,
                         "save": False})
    assert len(seen) == 2 * T and len(trainer.episode_losses) == 2
    assert all(torch.isfinite(torch.as_tensor(l)) for l in trainer.episode_losses) and trainer.episode_losses[1] > 0
    assert not torch.equal(trainer.w, w0)
    ring = trainer.replay_buffer.ring
    stored = sb.ops.replay_gather(ring, torch.arange(2 * T, device=_dev(), dtype=torch.int64))["rewards"]
    want = torch.stack(seen).reshape(2 * T, 1).expand(2 * T, n)
    assert torch.equal(stored.reshape(2 * T, n), want), "the replay ring holds the Flocking collective reward"
    goto_like = -torch.linalg.vector_norm(env.world.state[0, :, 0:2] - torch.tensor([-0.8, 0.8], device=_dev()), dim=-1).sum()
    assert abs(float(seen[-1]) - float(goto_like)) > 1e-3, "and it is not the GoTo reward of the world-step kernel"


def test_device_loop_training_on_flocking():
    """DQNTrainer.train_model_device on a Flocking env: the reset of flocking:93-121 (start centre from the counter RNG,
    grid at the desired distance, the two shaping memories) happens on the device inside the episode graph.  The
    pushed transitions of episode 0 are re-derived by stepping a second env from the same start states, and the
    CUDA-graph run equals the eager run bit for bit."""
    B, n, T, G = 64, 5, 12, 32
    cfgd = {"epsilon": 0.4, "epsilon_decay": 0.05, "min_epsilon": 0.05, "episodes": 3, "graphs_per_update": G,
            "update_target_every": 5}

    def run(use_graph):
        sb, env, env_ref, _ = _flocking_pair(B, n, T, seed=11)
        sb.set_seed(5)
        trainer = sb.DQNTrainer(env, 5, "/tmp/swarm_models", "/tmp/swarm_stats", "Flocking", replay_capacity=B * T * 4)
        stats = trainer.train_model_device(dict(cfgd, cuda_graph=use_graph))
        torch.cuda.synchronize()
        return sb, trainer, env_ref, stats

    sb, trainer, env_ref, stats = run(False)
    ring = trainer.replay_buffer.ring
    assert len(ring) == 3 * T * B and trainer.opt_step == 3 * T and torch.isfinite(stats).all()
    first = sb.ops.replay_gather(ring, torch.arange(T * B, device=_dev(), dtype=torch.int64))     # episode 0
    start = first["state"][:B]
    # the device reset: zero velocities, agents on the 0.15-spaced grid around a centre drawn from (-1, 1) + N((-0.6, 0.6), 0.4)
    assert (start[..., 2:] == 0).all()
    centres = start[..., :2].mean(dim=1).cpu()
    assert abs(centres[:, 0].mean().item() + 1.6) < 0.3 and abs(centres[:, 1].mean().item() - 1.6) < 0.3
    assert 0.2 < centres[:, 0].std().item() < 0.6
    dx = (start[:, 1, 0] - start[:, 0, 0]).cpu()
    assert torch.allclose(dx, torch.full_like(dx, 0.15), atol=1e-6)
    # rewards: the second env starts from the same states with the reset shaping memory and replays the stored actions
    env_ref.world.state.copy_(start)
    sb.ops.scenario_reward(env_ref.scenario._spec(), env_ref.world.state, env_ref.scenario.shaping, reset=True)
    for t in range(T):
        sl = slice(t * B, (t + 1) * B)
        assert torch.equal(first["state"][sl], env_ref.world.state), f"pre-step state of tick {t}"
        _, rews, _, _ = env_ref.step(first["actions"][sl])
        assert torch.equal(first["next_state"][sl], env_ref.world.state)
        assert torch.equal(first["rewards"][sl], rews["agent0"][:, None].expand(B, n)), f"reward of tick {t}"
    _, graphed, _, stats_g = run(True)
    assert torch.equal(graphed.w, trainer.w) and torch.equal(graphed.w_target, trainer.w_target)
    assert torch.equal(stats_g, stats)


@pytest.mark.parametrize("which", ["flocking", "obstacle_avoidance"])
def test_stepwise_batched_training_any_scenario(which):
    """DQNTrainer.train_model_stepwise: B envs per tick through env.step and the scenario's own reward().  The ring
    receives B transitions per tick carrying that reward, updates start once G transitions exist, weights move, the
    target network is synchronised on schedule, and a second run with the same seeds is bit-identical."""
    sb = _swarm()
    B, n, T, G = 48, 5, 12, 32

    def run():
        sb.set_seed(2)
        scenario = sb.FlockingScenario() if which == "flocking" else sb.ObstacleAvoidanceScenario()
        env = sb.make_env(scenario=scenario, num_envs=B, device=_dev(), continuous_actions=False, wrapper=None,
                          max_steps=T, dict_spaces=True, n_agents=n, seed=2, per_env_centers=True)
        trainer = sb.DQNTrainer(env, 2, "/tmp/swarm_models", "/tmp/swarm_stats", which, replay_capacity=B * T * 2 + 7)
        last = {}
        step = env.step

        def recording_step(actions):
            out = step(actions)
            last["rewards"] = torch.stack([out[1][f"agent{i}"] for i in range(n)], dim=1).clone()
            last["actions"] = actions.clone()
            return out

        env.step = recording_step
        w0 = trainer.w.clone()
        stats = trainer.train_model_stepwise({"epsilon": 0.5, "epsilon_decay": 0.01, "min_epsilon": 0.05, "episodes": 2,
                                              "graphs_per_update": G, "update_target_every": 10})
        return trainer, stats, w0, last

    trainer, stats, w0, last = run()
    ring = trainer.replay_buffer.ring
    assert len(ring) == 2 * T * B and ring.position == 2 * T * B
    assert stats["ticks"] == 2 * T and stats["opt_steps"] == 2 * T          # B >= G: an update on every tick
    assert np.isfinite(stats["loss"]) and stats["loss"] > 0 and not torch.equal(trainer.w, w0)
    tail = torch.arange(2 * T * B - B, 2 * T * B, device=_dev(), dtype=torch.int64)
    got = sb.ops.replay_gather(ring, tail)
    assert torch.equal(got["rewards"], last["rewards"]) and torch.equal(got["actions"], last["actions"].to(torch.int32))
    assert torch.equal(got["next_state"], trainer.env.world.state)
    if which == "flocking":
        assert torch.equal(got["rewards"][:, 0], got["rewards"][:, n - 1])     # one collective reward per env
    # tick 20 was the last target sync (every 10 ticks); four more updates moved the online weights since
    assert not torch.equal(trainer.w, trainer.w_target)
    again, stats2, _, _ = run()
    assert torch.equal(again.w, trainer.w) and stats2["loss"] == stats["loss"]


def _flocking_pair(B, n, T, seed):
    """Two identical Flocking envs (explicit per-env start centres) + GoTo weights."""
    from helpers import load_params
    sb = _swarm()
    g = torch.Generator().manual_seed(seed)
    centers = torch.tensor([-1.0, 1.0]) + torch.tensor([-0.6, 0.6]) + 0.4 * torch.randn(B, 2, generator=g)
    envs = []
    for _ in range(2):
        sc = sb.FlockingScenario()
        env = sb.Environment(sc, num_envs=B, device=_dev(), max_steps=T, continuous_actions=False, seed=0, dict_spaces=True,
                             n_agents=n)
        sc.set_start_centers(centers)
        env.reset()
        envs.append(env)
    w = sb.pack_weights(load_params("GoTo", 0), _dev())
    return sb, envs[0], envs[1], w


@pytest.mark.parametrize("graph,n,B", [("complete", 7, 37), ("knn", 12, 37), ("complete", 2, 37),
                                       # the FLOCK, NT = 12 instantiation at 444 CTAs of 9-10 envs
                                       ("complete", 12, 4096)],
                         ids=["complete-7", "knn-12", "complete-2", "complete-12-4096"])
def test_fused_flocking_rollout_matches_env_stepping(graph, n, B):
    """swarm_rollout with the Flocking option (graph -> GAT-Q -> epsilon-greedy -> world step -> Flocking reward, T ticks in
    one launch) against Environment.step on a second FlockingScenario env driven with the traced actions: states, rewards,
    returns, replay pushes and the shaping memory agree bit for bit."""
    T = 20
    sb, env_a, env_b, w = _flocking_pair(B, n, T, seed=n)
    ops, L = sb.ops, sb._lib
    sc_a, sc_b = env_a.scenario, env_b.scenario
    cfg = ops.clone_config(env_a.world.cfg, graph_mode=L.GRAPH_KNN if graph == "knn" else L.GRAPH_COMPLETE, knn_k=min(5, n))
    ring = ops.ReplayRing(B * T, n, _dev())
    out = ops.rollout(cfg, w, env_a.world.state, T, trace=dict(actions=True, rewards=True, state=True), epsilon=0.3,
                      rng_seed=11, replay=ring, flocking=sc_a._spec(), shaping=sc_a.shaping)
    ret = torch.zeros(B, device=_dev())
    for t in range(T):
        _, rews, _, _ = env_b.step(out["trace_actions"][t])
        assert torch.equal(env_b.world.state, out["trace_state"][t]), f"state after tick {t}"
        r = rews["agent0"]
        assert torch.equal(out["trace_rewards"][t], r[:, None].expand(B, n)), f"reward of tick {t}"
        ret = ret + r
    assert torch.equal(sc_b.shaping, sc_a.shaping)
    assert torch.equal(out["returns"], ret[:, None].expand(B, n))
    got = ops.replay_gather(ring, torch.arange(B * T, device=_dev(), dtype=torch.int64))
    assert torch.equal(got["rewards"].view(T, B, n), out["trace_rewards"])
    assert torch.equal(got["next_state"].view(T, B, n, 4), out["trace_state"])
    # the option is validated: wrong scenario / missing shaping
    with pytest.raises(ValueError):
        ops.rollout(cfg, w, env_a.world.state, 1, flocking=sc_a._spec())
    oa = ops.clone_config(cfg, scenario=L.SCENARIO_OBSTACLE_AVOIDANCE)
    with pytest.raises(ValueError):
        ops.rollout(oa, w, env_a.world.state, 1, flocking=sc_a._spec(), shaping=sc_a.shaping)


def test_fused_batched_training_on_flocking():
    """DQNTrainer.train_model_batched on a Flocking env: the fused train tick pushes the Flocking reward (re-derived
    here by stepping a second env with the stored actions), and the CUDA-graph run equals the eager run bit for bit."""
    B, n, T, G = 64, 5, 15, 32

    def run(use_graph, episodes):
        sb, env, env_ref, _ = _flocking_pair(B, n, T, seed=9)
        sb.set_seed(3)
        trainer = sb.DQNTrainer(env, 3, "/tmp/swarm_models", "/tmp/swarm_stats", "Flocking", replay_capacity=B * T * 4)
        stats = trainer.train_model_batched({"epsilon": 0.4, "epsilon_decay": 0.01, "min_epsilon": 0.05, "episodes": episodes,
                                             "graphs_per_update": G, "update_target_every": 7, "cuda_graph": use_graph})
        return sb, trainer, env_ref, stats

    sb, trainer, env_ref, stats = run(False, 3)
    ring = trainer.replay_buffer.ring
    assert len(ring) == 3 * T * B and stats["opt_steps"] == 3 * T and np.isfinite(stats["loss"])
    first = sb.ops.replay_gather(ring, torch.arange(T * B, device=_dev(), dtype=torch.int64))     # episode 0
    for t in range(T):
        sl = slice(t * B, (t + 1) * B)
        assert torch.equal(first["state"][sl], env_ref.world.state), f"pre-step state of tick {t}"
        _, rews, _, _ = env_ref.step(first["actions"][sl])
        assert torch.equal(first["next_state"][sl], env_ref.world.state)
        assert torch.equal(first["rewards"][sl], rews["agent0"][:, None].expand(B, n)), f"reward of tick {t}"
    _, graphed, _, stats_g = run(True, 3)
    assert torch.equal(graphed.w, trainer.w) and torch.equal(graphed.w_target, trainer.w_target)
    assert stats_g["loss"] == stats["loss"]


def test_device_loop_training_on_flocking():
    """DQNTrainer.train_model_device on a Flocking env: the reset of flocking:93-121 (start centre from the counter RNG,
    grid at the desired distance, the two shaping memories) happens on the device inside the episode graph.  The
    pushed transitions of episode 0 are re-derived by stepping a second env from the same start states, and the
    CUDA-graph run equals the eager run bit for bit."""
    B, n, T, G = 64, 5, 12, 32
    cfgd = {"epsilon": 0.4, "epsilon_decay": 0.05, "min_epsilon": 0.05, "episodes": 3, "graphs_per_update": G,
            "update_target_every": 5}

    def run(use_graph):
        sb, env, env_ref, _ = _flocking_pair(B, n, T, seed=11)
        sb.set_seed(5)
        trainer = sb.DQNTrainer(env, 5, "/tmp/swarm_models", "/tmp/swarm_stats", "Flocking", replay_capacity=B * T * 4)
        stats = trainer.train_model_device(dict(cfgd, cuda_graph=use_graph))
        torch.cuda.synchronize()
        return sb, trainer, env_ref, stats

    sb, trainer, env_ref, stats = run(False)
    ring = trainer.replay_buffer.ring
    assert len(ring) == 3 * T * B and trainer.opt_step == 3 * T and torch.isfinite(stats).all()
    first = sb.ops.replay_gather(ring, torch.arange(T * B, device=_dev(), dtype=torch.int64))     # episode 0
    start = first["state"][:B]
    # the device reset: zero velocities, agents on the 0.15-spaced grid around a centre drawn from (-1, 1) + N((-0.6, 0.6), 0.4)
    assert (start[..., 2:] == 0).all()
    centres = start[..., :2].mean(dim=1).cpu()
    assert abs(centres[:, 0].mean().item() + 1.6) < 0.3 and abs(centres[:, 1].mean().item() - 1.6) < 0.3
    assert 0.2 < centres[:, 0].std().item() < 0.6
    dx = (start[:, 1, 0] - start[:, 0, 0]).cpu()
    assert torch.allclose(dx, torch.full_like(dx, 0.15), atol=1e-6)
    # rewards: the second env starts from the same states with the reset shaping memory and replays the stored actions
    env_ref.world.state.copy_(start)
    sb.ops.scenario_reward(env_ref.scenario._spec(), env_ref.world.state, env_ref.scenario.shaping, reset=True)
    for t in range(T):
        sl = slice(t * B, (t + 1) * B)
        assert torch.equal(first["state"][sl], env_ref.world.state), f"pre-step state of tick {t}"
        _, rews, _, _ = env_ref.step(first["actions"][sl])
        assert torch.equal(first["next_state"][sl], env_ref.world.state)
        assert torch.equal(first["rewards"][sl], rews["agent0"][:, None].expand(B, n)), f"reward of tick {t}"
    _, graphed, _, stats_g = run(True)
    assert torch.equal(graphed.w, trainer.w) and torch.equal(graphed.w_target, trainer.w_target)
    assert torch.equal(stats_g, stats)
