"""Device-driven DQN train tick of stacked GAT Q-networks (swarm_train_tick_stack, ops.StackTrainTick,
DQNTrainer.train_model_stack_device).

The tick is checked bit for bit against the public calls it composes: gatstack_forward (greedy actions), the exploration
draws of the counter RNG (a Python mirror of splitmix64 / rng_draw, csrc/tile_device.cuh), sim_step, scenario_reward,
replay_push, the slot draw (same mirror), dqn_grad_stack and adam_clip_step_stack.  Weights and moments are compared with
assert_close and the two tracks resynced every tick: the device forms Adam's bias corrections with its own double pow,
which may differ from the host's in the last bit."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M64 = (1 << 64) - 1


def _dev():
    return torch.device("cuda:0")


def _flocking_sd(seed, in_features=7):
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    pre = f"{seed}/"
    sd = {k[len(pre):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(pre)}
    if in_features == 5:
        sd["conv1.lin.weight"] = sd["conv1.lin.weight"][:, [0, 1, 2, 3, 6]].contiguous()
    return sd


def _splitmix64(x):
    x = (x + 0x9E3779B97F4A7C15) & M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M64
    return x ^ (x >> 31)


def _rng_draw(seed, env, tick, lane):
    return _splitmix64(_splitmix64(seed ^ ((env * 0xD1342543DE82EF95) & M64)) ^ ((tick * 0xA24BAED4963EE407) & M64) ^ lane)


def _explore(greedy, epsilon, seed, env_offset, tick):
    """train:164-165 on the device stream: one coin per env, then one uniform action per agent."""
    acts = greedy.cpu().clone()
    B, N = acts.shape
    eps = np.float32(epsilon)
    for b in range(B):
        coin = np.float32(_rng_draw(seed, env_offset + b, tick, 0xFFFF) >> 40) * np.float32(1.0 / 16777216.0)
        if coin < eps:
            for i in range(N):
                acts[b, i] = ((_rng_draw(seed, env_offset + b, tick, i) >> 32) * 9) >> 32
    return acts.to(greedy.device)


def _slots(seed, tick, G, ring_size):
    return torch.tensor([(_rng_draw(seed, g, tick, 0x5A17) * ring_size) >> 64 for g in range(G)], dtype=torch.int64)


# (name, world, reward, graph, k / radius, N, in_features)
CASES = [
    ("oa_world_knn5", "oa", None, "knn", 5, 12, 7),
    ("goto_world_radius", "goto", None, "radius", 0.35, 12, 7),
    ("flocking_complete", "goto", "flocking", "complete", 0, 12, 7),
    ("cohesion_in5_n9", "goto", "cohesion", "knn", 5, 9, 5),
    ("cohesion_in5_n9_radius", "goto", "cohesion", "radius", 0.35, 9, 5),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_stack_train_tick_matches_composed_calls(case):
    """Ten ticks over 'not enough samples' ticks, updates, the ring wrap-around and target syncs."""
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    dev = _dev()
    name, world, reward, graph, k, N, in_f = case
    B, G, capacity, every, T = 16, 32, 40, 3, 10
    rng_seed, sample_seed, env_offset, eps = 11, 5, 7, 0.4
    scen = L.SCENARIO_OBSTACLE_AVOIDANCE if world == "oa" else L.SCENARIO_GOTO
    gm = {"knn": L.GRAPH_KNN, "complete": L.GRAPH_COMPLETE, "radius": L.GRAPH_RADIUS}[graph]
    cfg = ops.make_config(scen, B, N, gm, int(k) if graph == "knn" else 5, graph_radius=float(k) if graph == "radius" else 0.35)
    spec = ops.stack_spec(3, 8, in_f)
    w = ops.pack_stack_weights(_flocking_sd(2, in_f), spec, dev)
    g = torch.Generator().manual_seed(3)
    base = torch.tensor([0.6, -0.6]) if world == "oa" else torch.tensor([0.3, -0.3])
    state = ops.reset_grid(cfg, (base + 0.15 * torch.randn(B, 2, generator=g)).to(dev))
    rs = shaping = None
    if reward == "flocking":
        rs = ops.reward_spec(L.REWARD_FLOCKING, B, N)
        shaping = torch.zeros(B, N, 2, device=dev)
        ops.scenario_reward(rs, state, shaping, reset=True)
    elif reward == "cohesion":
        rs = ops.reward_spec(L.REWARD_COHESION, B, N)

    ring = ops.ReplayRing(capacity, N, dev)
    tt = ops.StackTrainTick(cfg, spec, ring, graphs_per_update=G, update_target_every=every, rng_seed=rng_seed,
                            sample_seed=sample_seed, env_offset=env_offset, reward=rs, shaping=shaping)
    tt.load_cursor(0, 0, eps)
    w_t, m, v = w.clone(), torch.zeros_like(w), torch.zeros_like(w)
    returns, hits = torch.zeros(B, N, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)

    # the composed reference on copies
    st_c, w_c, wt_c, m_c, v_c = state.clone(), w.clone(), w.clone(), torch.zeros_like(w), torch.zeros_like(w)
    sh_c = shaping.clone() if shaping is not None else None
    ring_c = ops.ReplayRing(capacity, N, dev)
    ret_c, hits_c = torch.zeros(B, N, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
    gcfg = ops.clone_config(cfg, num_envs=G)
    opt, syncs, wrapped = 0, 0, False
    for tick in range(1, T + 1):
        grad_before = tt.grad_loss.clone()
        tt.tick(w, w_t, m, v, state, returns, hits)

        greedy = ops.gatstack_forward(cfg, spec, w_c, st_c, want_q=False, want_actions=True)
        acts = _explore(greedy, eps, rng_seed, env_offset, tick).to(torch.int32).contiguous()
        out = ops.sim_step(cfg, st_c, acts, want_obs=False)
        nxt = out["state"]
        if reward == "flocking":
            r = ops.scenario_reward(rs, nxt, sh_c).view(B, 1).expand(B, N).contiguous()
        elif reward == "cohesion":
            r = ops.scenario_reward(rs, nxt)
        else:
            r = out["rewards"]
        ret_c += r
        hits_c += ((out["flags"] & L.FLAG_HIT) != 0).sum(dim=1, dtype=torch.int32)
        wrapped = wrapped or ring_c.position + B > capacity
        ops.replay_push(cfg, ring_c, st_c, acts, r.contiguous(), nxt)
        st_c = nxt

        cur = tt.read_cursor()
        assert cur["tick"] == tick and ring.position == ring_c.position and ring.size == ring_c.size, tick
        assert torch.equal(state, st_c) and torch.equal(returns, ret_c) and torch.equal(hits, hits_c), tick
        for a, b in ((ring.state, ring_c.state), (ring.next_state, ring_c.next_state), (ring.actions, ring_c.actions),
                     (ring.rewards, ring_c.rewards)):
            assert torch.equal(a, b), tick
        if shaping is not None:
            assert torch.equal(shaping, sh_c), tick
        enough = len(ring_c) >= G
        assert cur["updating"] == int(enough)
        if enough:
            idx = _slots(sample_seed, tick, G, len(ring_c))
            assert torch.equal(tt.indices.cpu(), idx), tick
            grad_c, loss_c, _ = ops.dqn_grad_stack(gcfg, spec, w_c, wt_c, ring_c, idx.to(dev), G)
            assert torch.equal(tt.grad, grad_c) and torch.equal(tt.loss, loss_c), tick
            opt += 1
            sync = tick % every == 0
            syncs += sync
            ops.adam_clip_step_stack(spec, w_c, grad_c, m_c, v_c, opt, target=wt_c if sync else None)
        else:
            assert torch.equal(tt.grad_loss, grad_before), "a tick without an update leaves grad / loss untouched"
        assert cur["opt_step"] == opt
        for a, b in ((w, w_c), (w_t, wt_c), (m, m_c), (v, v_c)):
            torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-9)
        w_c.copy_(w); wt_c.copy_(w_t); m_c.copy_(m); v_c.copy_(v)     # keep the two tracks on identical weights
    assert opt == T - 1 and syncs >= 2 and wrapped
    assert (returns != 0).any() and not torch.equal(w, ops.pack_stack_weights(_flocking_sd(2, in_f), spec, dev))


def _trainer(sb, scen, B=64, steps=8):
    dev = _dev()
    if scen == "flocking":
        env = sb.make_env(sb.FlockingScenario(), num_envs=B, device=dev, continuous_actions=False, max_steps=steps,
                          dict_spaces=True, seed=0, n_agents=12)
        model = sb.StackedGCN.from_state_dict(_flocking_sd(7))
    else:
        env = sb.make_env(sb.CohesionScenario(), num_envs=B, device=dev, continuous_actions=False, max_steps=steps,
                          dict_spaces=True, seed=0, n_agents=9)
        torch.manual_seed(0)
        model = sb.StackedGCN(5, 8, 9, 3)
    return sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "t", replay_capacity=4096, model=model)


@pytest.mark.gpu
@pytest.mark.parametrize("scen", ["flocking", "cohesion"])
def test_train_model_stack_device_graph_equals_eager(scen):
    import swarm_b200 as sb
    B, steps, episodes = 64, 8, 4
    cfgd = {"episodes": episodes, "epsilon": 0.9, "epsilon_decay": 0.3, "min_epsilon": 0.05, "graphs_per_update": 32,
            "update_target_every": 5}
    out = []
    for use_graph in (False, True):
        tr = _trainer(sb, scen, B, steps)
        w0 = tr.w.clone()
        stats = tr.train_model_stack_device(dict(cfgd, cuda_graph=use_graph))
        torch.cuda.synchronize()
        out.append((tr.w.clone(), tr.w_target.clone(), stats, tr.opt_step, tr))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]) and torch.equal(out[0][2], out[1][2])
    stats, tr = out[0][2], out[0][4]
    assert out[0][3] == episodes * steps and out[1][3] == episodes * steps       # the ring holds >= G from tick 1
    eps = [0.9] + [max(0.05, 0.9 * float(np.exp(-0.3 * e))) for e in range(episodes - 1)]
    assert np.allclose(stats[:, 3].numpy(), np.array(eps, dtype=np.float32), rtol=1e-6)
    assert torch.isfinite(stats).all() and (stats[:, 2] > 0).all()
    assert not torch.equal(tr.w, w0) and torch.isfinite(tr.w).all()
    assert torch.equal(sb.ops.pack_stack_weights(tr.model.state_dict(), tr.stack_spec, _dev()), tr.w)
    if scen == "cohesion":
        # every episode starts from the state env.reset() leaves: the first tick of each episode pushed it as s
        tr.env.reset()
        start = tr.env.world.state
        ring = tr.replay_buffer.ring
        for e in range(episodes):
            slot = e * steps * B
            assert torch.equal(ring.state[slot:slot + B], start), e
    assert np.isfinite(tr.evaluate_policy(1))


@pytest.mark.gpu
def test_train_model_stack_device_scope():
    """A stack only; the world's own reward (GoTo here) trains too; the one-layer loop still refuses a stack."""
    import swarm_b200 as sb
    env = sb.make_env(sb.GoToPositionScenario(), num_envs=4, device=_dev(), continuous_actions=False, max_steps=4,
                      dict_spaces=True, seed=0, n_agents=5)
    cfg = {"episodes": 1, "epsilon": 0.5, "epsilon_decay": 0.1, "min_epsilon": 0.05}
    with pytest.raises(NotImplementedError, match="StackedGCN"):
        sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "t", replay_capacity=64).train_model_stack_device(cfg)
    tr = sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "t", replay_capacity=64, model=sb.StackedGCN(7, 8, 9, 2))
    with pytest.raises(NotImplementedError, match="train_model_stepwise"):
        tr.train_model_device(cfg)
    stats = tr.train_model_stack_device(dict(cfg, graphs_per_update=4))
    assert stats.shape == (1, 4) and tr.opt_step == 4


def test_stack_train_tick_argument_validation_without_device():
    import swarm_b200 as sb
    L, lib = sb._lib, sb._lib.lib()
    spec = sb.ops.stack_spec(3, 8, 7)
    B, N, G = 16, 12, 32
    cfg = sb.ops.make_config(L.SCENARIO_GOTO, B, N, L.GRAPH_COMPLETE)
    wb = int(lib.swarm_dqn_stack_workspace_bytes(C.byref(cfg), C.byref(spec), G))
    assert wb > 0

    def hyper(**kw):
        h = L.SwarmTrainHyper()
        h.lr, h.beta1, h.beta2, h.eps, h.max_norm = 1e-3, 0.9, 0.999, 1e-8, 1.0
        h.graphs_per_update, h.update_target_every, h.gamma, h.loss_scale = G, 200, 0.99, 1.0 / (G * N)
        for k_, v_ in kw.items():
            setattr(h, k_, v_)
        return h

    def tick(c=cfg, h=None, reward=None, ctl=8, ring=L.SwarmReplay(8, 8, 8, 8, 64), wsb=wb):
        h = h or hyper()
        return lib.swarm_train_tick_stack(C.byref(c), C.byref(spec), C.byref(h),
                                          C.addressof(reward) if reward is not None else None, 8, ctl, 8, 8, 8, 8, 8, 8, 8,
                                          C.byref(ring), 8, 8, 8, wsb, None)

    assert tick(ctl=None) == -1 and b"NULL" in lib.swarm_last_error()
    assert tick(ring=L.SwarmReplay(8, None, 8, 8, 64)) == -1 and b"replay ring" in lib.swarm_last_error()
    fs = sb.ops.reward_spec(L.REWARD_FLOCKING, B, N)
    assert tick(h=hyper(flocking=C.addressof(fs))) == -1 and b"hyper->flocking" in lib.swarm_last_error()
    assert tick(c=sb.ops.make_config(L.SCENARIO_GOTO, B, 129, L.GRAPH_COMPLETE)) == -2
    assert tick(c=sb.ops.make_config(L.SCENARIO_GOTO, B, 20, L.GRAPH_KNN, 5)) == -2
    assert b"n_agents <= 16" in lib.swarm_last_error()
    assert tick(wsb=wb - 1) == -1 and b"workspace too small" in lib.swarm_last_error()
    assert tick(ring=L.SwarmReplay(8, 8, 8, 8, B - 1)) == -1 and b"replay capacity" in lib.swarm_last_error()
    assert tick(reward=sb.ops.reward_spec(L.REWARD_COHESION, B + 1, N)) == -1 and b"disagree" in lib.swarm_last_error()
    oa = sb.ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B, N, L.GRAPH_COMPLETE)
    assert tick(c=oa, reward=sb.ops.reward_spec(L.REWARD_COHESION, B, N)) == -1 and b"GoTo world" in lib.swarm_last_error()
    assert tick(h=hyper(beta1=1.0)) == -1 and b"Adam" in lib.swarm_last_error()
    assert tick(h=hyper(graphs_per_update=0)) == -1
