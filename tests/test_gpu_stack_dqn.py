"""DQN training of stacked GAT Q-networks (swarm_dqn_stack_grad / swarm_adam_clip_stack_step, DQNTrainer(model=...)):
the conv1 .. convL form the reference ships as data/models/experiment_Flocking-seed_*.pth (conv2 / conv3 are comments in
train_gcn_dqn.py:54-55, 64-67).

Gradients are judged against float64 torch autograd through the oracle's GATConv (oracle/swarm_oracle.py gat_conv) stacked
as the network does, on the same graphs, with nn.MSELoss, using the bars of test_gpu_dqn.py: loss within 1e-5 relative,
TD within 2e-5 of max(|td|, 1), per tensor |g - g64| <= 1e-5 max|g64_tensor| + 2e-6 max|g64_all|, and no tensor more than
20x noisier than float32 autograd.  Clip + Adam is compared with torch.nn.utils.clip_grad_norm_ + torch.optim.Adam fed the
same gradients."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRAD_RTOL = 1e-5


def _dev():
    return torch.device("cuda:0")


def _flocking_sd(seed):
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    pre = f"{seed}/"
    return {k[len(pre):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(pre)}


def _random_sd(layers, hidden, in_features, seed):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for l in range(1, layers + 1):
        cin = in_features if l == 1 else hidden
        sd[f"conv{l}.att_src"] = 0.5 * torch.randn(1, 1, hidden, generator=g)
        sd[f"conv{l}.att_dst"] = 0.5 * torch.randn(1, 1, hidden, generator=g)
        sd[f"conv{l}.bias"] = 0.1 * torch.randn(hidden, generator=g)
        sd[f"conv{l}.lin.weight"] = (0.8 / cin ** 0.5) * torch.randn(hidden, cin, generator=g)
    sd["lin1.weight"] = (0.8 / hidden ** 0.5) * torch.randn(hidden, hidden, generator=g)
    sd["lin1.bias"] = 0.1 * torch.randn(hidden, generator=g)
    sd["lin2.weight"] = (0.8 / hidden ** 0.5) * torch.randn(9, hidden, generator=g)
    sd["lin2.bias"] = 0.1 * torch.randn(9, generator=g)
    return sd


def _five_feature(sd):
    sd = dict(sd)
    sd["conv1.lin.weight"] = sd["conv1.lin.weight"][:, [0, 1, 2, 3, 6]].contiguous()
    return sd


def _transitions(G, N, seed, scenario="go_to"):
    from test_gpu_dqn import _transitions as tr
    return tr(scenario, G, N, seed)


def _features(cfg, pos, vel, in_features):
    G, N, _ = pos.shape
    goal = torch.tensor([cfg.goal_x, cfg.goal_y], dtype=torch.float32).view(1, 1, 2).expand(G, N, 2)
    ids = torch.arange(N, dtype=torch.float32).view(1, N, 1).expand(G, N, 1)
    x = torch.cat([pos, vel, goal, ids], dim=2) if in_features == 7 else torch.cat([pos, vel, ids], dim=2)
    return x.reshape(G * N, in_features)


def _oracle_q(params, acts, x, ei):
    from oracle import swarm_oracle as so
    h, l = x, 1
    while f"conv{l}.lin.weight" in params:
        h = so.gat_conv(h, ei, params[f"conv{l}.lin.weight"], params[f"conv{l}.att_src"], params[f"conv{l}.att_dst"],
                        params[f"conv{l}.bias"])
        h = torch.tanh(h) if acts[l - 1] == "tanh" else torch.relu(h)
        l += 1
    h = torch.relu(h @ params["lin1.weight"].T + params["lin1.bias"])
    return h @ params["lin2.weight"].T + params["lin2.bias"]


def _oracle_loss_grads(cfg, sd_on, sd_tg, acts, in_features, trans, mode, k, dtype, gamma=0.99):
    """float64 (or float32) torch autograd of train_step_dqn for a stack on the batch's own graphs."""
    from oracle import batched_oracle as bo
    pos, vel, actions, rewards, pos2, vel2 = trans
    G, N, _ = pos.shape
    on = {k_: v.to(dtype).clone().requires_grad_(True) for k_, v in sd_on.items()}
    tg = {k_: v.to(dtype) for k_, v in sd_tg.items()}
    ei = bo.batch_edge_index(bo.graph_edges(pos, mode, k), N)
    ei2 = bo.batch_edge_index(bo.graph_edges(pos2, mode, k), N)
    values = _oracle_q(on, acts, _features(cfg, pos, vel, in_features).to(dtype), ei).gather(1, actions.reshape(-1, 1))
    with torch.no_grad():
        nxt = _oracle_q(tg, acts, _features(cfg, pos2, vel2, in_features).to(dtype), ei2).max(dim=1)[0]
    targets = rewards.reshape(-1).to(dtype) + gamma * nxt
    loss = nn.MSELoss()(values, targets.unsqueeze(1))
    loss.backward()
    td = (values.detach().reshape(-1) - targets).reshape(G, N)
    return loss.item(), {k_: v.grad.detach().clone() for k_, v in on.items()}, td


def _ring(sb, trans, capacity=None):
    from test_gpu_dqn import _ring_from
    return _ring_from(sb, *trans, capacity=capacity)


def _mode_cfg(sb, G, N, mode, k):
    L = sb._lib
    gm = {"complete": L.GRAPH_COMPLETE, "knn": L.GRAPH_KNN, "radius": L.GRAPH_RADIUS}[mode]
    return sb.ops.make_config(L.SCENARIO_GOTO, G, N, gm, int(k) if mode == "knn" else 5,
                              graph_radius=float(k) if mode == "radius" else 0.35)


def _check_grads(got, grads64, grads32, factor=1.0):
    gmax = max(v.abs().max().item() for v in grads64.values())
    for name, gref in grads64.items():
        g = got[name].reshape(gref.shape).double().cpu()
        err = (g - gref).abs().max().item()
        bound = factor * (GRAD_RTOL * gref.abs().max().item() + 2e-6 * gmax)
        assert err <= bound, f"{name}: gradient abs error {err:.3e} > bound {bound:.3e}"
        if grads32 is not None:
            err32 = (grads32[name].double() - gref).abs().max().item()
            assert err <= max(20 * err32, GRAD_RTOL * gref.abs().max().item()), f"{name}: far noisier than float32 autograd"


# (name, weights, layers, hidden, in_features, activations, graph, N, k (kNN k or radius), G)
CASES = [
    ("flock_complete_n12", "flock", 3, 8, 7, None, "complete", 12, 0, 32),
    ("flock_knn5_n12", "flock", 3, 8, 7, None, "knn", 12, 5, 32),
    ("flock_knn5_n5", "flock", 3, 8, 7, None, "knn", 5, 5, 32),
    ("flock_radius_n20", "flock", 3, 8, 7, None, "radius", 20, 0.3, 32),
    ("flock_complete_g1000_ragged", "flock", 3, 8, 7, None, "complete", 12, 0, 1000),
    ("flock_tanh_only", "flock", 3, 8, 7, ["tanh"] * 3, "complete", 12, 0, 32),
    ("gcn_l1_w32", "gcn", 1, 32, 7, ["tanh"], "complete", 12, 0, 32),
    ("l2_w16", "rand", 2, 16, 7, None, "complete", 9, 0, 32),
    ("l4_w32_n128", "rand", 4, 32, 7, None, "complete", 128, 0, 3),
    ("l2_w5_knn", "rand", 2, 5, 7, None, "knn", 8, 3, 40),
    ("l3_w13", "rand", 3, 13, 7, ["tanh", "relu", "tanh"], "radius", 16, 0.3, 32),
    ("in5_n9", "flock5", 3, 8, 5, None, "complete", 9, 0, 32),
    ("n40_three_per_cta", "rand", 2, 8, 7, None, "complete", 40, 0, 450),
    ("n2", "rand", 2, 8, 7, None, "complete", 2, 0, 200),
]


def _case_weights(src, layers, hidden, in_features):
    from helpers import load_params
    if src == "flock":
        return _flocking_sd(3), _flocking_sd(4)
    if src == "flock5":
        return _five_feature(_flocking_sd(3)), _five_feature(_flocking_sd(4))
    if src == "gcn":
        return load_params("GoTo", 3), load_params("GoTo", 4)
    return _random_sd(layers, hidden, in_features, 10 * layers + hidden), _random_sd(layers, hidden, in_features, 7)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_stack_grad_matches_float64_autograd(case):
    import swarm_b200 as sb
    ops = sb.ops
    name, src, layers, hidden, in_f, acts, mode, N, k, G = case
    acts = acts or (["tanh"] + ["relu"] * (layers - 1))
    sd_on, sd_tg = _case_weights(src, layers, hidden, in_f)
    trans = _transitions(G, N, seed=G + N + layers)
    cfg = _mode_cfg(sb, G, N, mode, k)
    loss64, g64, td64 = _oracle_loss_grads(cfg, sd_on, sd_tg, acts, in_f, trans, mode, k, torch.float64)
    _, g32, _ = _oracle_loss_grads(cfg, sd_on, sd_tg, acts, in_f, trans, mode, k, torch.float32)
    ring = _ring(sb, trans)
    spec = ops.stack_spec(layers, hidden, in_f, acts)
    w_on, w_tg = ops.pack_stack_weights(sd_on, spec, _dev()), ops.pack_stack_weights(sd_tg, spec, _dev())
    grad, loss, td = ops.dqn_grad_stack(cfg, spec, w_on, w_tg, ring, None, G, want_td=True)
    assert abs(loss.item() - loss64) <= GRAD_RTOL * abs(loss64), f"loss {loss.item()} vs {loss64}"
    assert (td.cpu().double() - td64).abs().max().item() <= 2e-5 * max(td64.abs().max().item(), 1.0), "TD errors differ"
    got = ops.unpack_stack_weights(grad.cpu(), spec)
    _check_grads(got, g64, g32)
    if src == "gcn":
        # the shipped one-layer GCN: the dedicated one-layer kernel agrees within twice the bar
        g1, l1, _ = ops.dqn_grad(cfg, sb.pack_weights(sd_on, _dev()), sb.pack_weights(sd_tg, _dev()), ring, None, G)
        _check_grads(sb.unpack_weights(g1.cpu()), g64, None)
        _check_grads({k_: got[k_] for k_ in g64}, {k_: sb.unpack_weights(g1.cpu())[k_].reshape(v.shape).double()
                                                   for k_, v in g64.items()}, None, factor=2.0)
        assert abs(l1.item() - loss.item()) <= 2 * GRAD_RTOL * abs(loss64)


@pytest.mark.gpu
@pytest.mark.parametrize("spec_args,mode,N,k", [((3, 8, 7), "complete", 12, 0), ((3, 8, 7), "knn", 12, 5),
                                                ((2, 13, 7), "radius", 20, 0.3), ((4, 32, 5), "knn", 9, 4),
                                                ((1, 32, 7), "complete", 30, 0)])
def test_td_uses_the_forward_bits(spec_args, mode, N, k):
    """td from the gradient kernel == values - (r + gamma * next) in float32 torch from swarm_gatstack_forward's Q."""
    import swarm_b200 as sb
    ops = sb.ops
    layers, hidden, in_f = spec_args
    G, gamma = 300, 0.99
    sd_on, sd_tg = _random_sd(layers, hidden, in_f, 1), _random_sd(layers, hidden, in_f, 2)
    trans = _transitions(G, N, seed=N + hidden, scenario="obstacle_avoidance")
    cfg = _mode_cfg(sb, G, N, mode, k)
    spec = ops.stack_spec(layers, hidden, in_f)
    w_on, w_tg = ops.pack_stack_weights(sd_on, spec, _dev()), ops.pack_stack_weights(sd_tg, spec, _dev())
    ring = _ring(sb, trans)
    _, _, td = ops.dqn_grad_stack(cfg, spec, w_on, w_tg, ring, None, G, gamma=gamma, want_td=True)
    pos, vel, actions, rewards, pos2, vel2 = trans
    q = ops.gatstack_forward(cfg, spec, w_on, torch.cat([pos, vel], 2).contiguous().to(_dev()))
    q2 = ops.gatstack_forward(cfg, spec, w_tg, torch.cat([pos2, vel2], 2).contiguous().to(_dev()))
    values = q.gather(2, actions.to(_dev()).unsqueeze(2)).squeeze(2)
    ref = values - (rewards.to(_dev()) + gamma * q2.max(dim=2)[0])
    assert torch.equal(td, ref)


@pytest.mark.gpu
def test_determinism_indexing_and_loss_scale():
    import swarm_b200 as sb
    ops = sb.ops
    G, N = 64, 12
    trans = _transitions(G, N, seed=5)
    ring = _ring(sb, trans)
    cfg = _mode_cfg(sb, G, N, "knn", 5)
    spec = ops.stack_spec(3, 8, 7)
    w_on, w_tg = ops.pack_stack_weights(_flocking_sd(0), spec, _dev()), ops.pack_stack_weights(_flocking_sd(1), spec, _dev())
    grad, loss, _ = ops.dqn_grad_stack(cfg, spec, w_on, w_tg, ring, None, G)
    grad2, loss2, _ = ops.dqn_grad_stack(cfg, spec, w_on, w_tg, ring, None, G)
    assert torch.equal(grad, grad2) and torch.equal(loss, loss2)
    # indexed call with permuted and repeated slots == the dense batch gathered the same way
    idx = torch.randint(0, G, (G,), generator=torch.Generator().manual_seed(3))
    gi, li, _ = ops.dqn_grad_stack(cfg, spec, w_on, w_tg, ring, idx.to(_dev()), G)
    dense = _ring(sb, tuple(t[idx] for t in trans))
    gd, ld, _ = ops.dqn_grad_stack(cfg, spec, w_on, w_tg, dense, None, G)
    assert torch.equal(gi, gd) and torch.equal(li, ld)
    # a quarter of the default loss scale: exactly a quarter of the loss and the gradient
    gq, lq, _ = ops.dqn_grad_stack(cfg, spec, w_on, w_tg, ring, None, G, loss_scale=0.25 / (G * N))
    assert torch.equal(gq, grad * 0.25) and torch.equal(lq, loss * 0.25)


@pytest.mark.gpu
def test_gradient_equals_the_module_autograd_path():
    """StackedGCN.forward (generic layer kernels under torch autograd) + nn.MSELoss + backward on the same batch."""
    import swarm_b200 as sb
    from oracle import batched_oracle as bo
    ops = sb.ops
    G, N, k = 32, 12, 5
    trans = _transitions(G, N, seed=11)
    pos, vel, actions, rewards, pos2, vel2 = trans
    cfg = _mode_cfg(sb, G, N, "knn", k)
    sd_on, sd_tg = _flocking_sd(2), _flocking_sd(5)
    spec = ops.stack_spec(3, 8, 7)
    w_on, w_tg = ops.pack_stack_weights(sd_on, spec, _dev()), ops.pack_stack_weights(sd_tg, spec, _dev())
    grad, loss, _ = ops.dqn_grad_stack(cfg, spec, w_on, w_tg, _ring(sb, trans), None, G)
    model = sb.StackedGCN.from_state_dict(sd_on).to(_dev())
    edges = bo.graph_edges(pos, "knn", k)
    batch = sb.Batch.from_data_list([sb.Data(x=_features(cfg, pos[g:g + 1], vel[g:g + 1], 7).to(_dev()),
                                             edge_index=edges[g].to(torch.int64).to(_dev())) for g in range(G)])
    q2 = ops.gatstack_forward(cfg, spec, w_tg, torch.cat([pos2, vel2], 2).contiguous().to(_dev()))
    targets = rewards.reshape(-1).to(_dev()) + 0.99 * q2.reshape(G * N, 9).max(dim=1)[0]
    values = model(batch).gather(1, actions.reshape(-1, 1).to(_dev()))
    mloss = nn.MSELoss()(values, targets.unsqueeze(1))
    mloss.backward()
    gmod = {n: p.grad.detach().double().cpu() for n, p in model.named_parameters()}
    assert abs(mloss.item() - loss.item()) <= GRAD_RTOL * abs(mloss.item())
    # two float32 evaluations, each within the bar of the exact gradient: they agree within twice the bar
    _check_grads(ops.unpack_stack_weights(grad.cpu(), spec), gmod, None, factor=2.0)


@pytest.mark.gpu
@pytest.mark.parametrize("layers,hidden,in_f", [(1, 32, 7), (2, 1, 7), (3, 8, 7), (4, 32, 7), (4, 8, 5)])
@pytest.mark.parametrize("max_norm", [1.0, 0.0])
def test_adam_clip_stack_matches_torch(layers, hidden, in_f, max_norm):
    import swarm_b200 as sb
    ops = sb.ops
    spec = ops.stack_spec(layers, hidden, in_f)
    model = sb.StackedGCN(in_f, hidden, 9, layers)
    model.load_state_dict(_random_sd(layers, hidden, in_f, 4))
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    w = ops.pack_stack_weights(model.state_dict(), spec, _dev())
    m, v, target = torch.zeros_like(w), torch.zeros_like(w), torch.zeros_like(w)
    norm_out = torch.zeros(1, device=_dev())
    g = torch.Generator().manual_seed(layers * 100 + hidden)
    names = [n for n, _ in model.named_parameters()]
    for step in range(1, 51):
        scale = [5.0, 0.01, 300.0, 1e-4, 1.0][step % 5]                  # clipped and un-clipped steps
        flat = torch.randn(w.numel(), generator=g) * scale
        parts = ops.unpack_stack_weights(flat, spec)
        for n, p_ in model.named_parameters():
            p_.grad = parts[n].reshape(p_.shape).clone()
        if max_norm > 0:
            ref_norm = torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm).item()
        else:
            ref_norm = torch.linalg.vector_norm(torch.stack([torch.linalg.vector_norm(p_.grad) for p_ in model.parameters()])).item()
        opt.step()
        sync = step in (2, 50)
        ops.adam_clip_step_stack(spec, w, flat.to(_dev()), m, v, step, max_norm=max_norm, target=target if sync else None,
                                 grad_norm=norm_out)
        assert abs(norm_out.item() - ref_norm) <= 1e-6 * ref_norm, f"step {step}: pre-clip norm"
        if sync:
            assert torch.equal(target, w)
        if step in (1, 2, 50):
            got_w = ops.unpack_stack_weights(w.cpu(), spec)
            got_m = ops.unpack_stack_weights(m.cpu(), spec)
            got_v = ops.unpack_stack_weights(v.cpu(), spec)
            # moments: relative to the larger of the tensor's and the whole vector's largest moment -- a width-1 tensor's
            # first moment can pass near zero, where the last bit of the clip coefficient (float32 norms in torch,
            # double sums here) dominates its relative error
            mmax = max(st_["exp_avg"].abs().max().item() for st_ in opt.state.values())
            vmax = max(st_["exp_avg_sq"].abs().max().item() for st_ in opt.state.values())
            for n, p_ in model.named_parameters():
                st = opt.state[p_]
                for what, got, ref, floor in (("weights", got_w[n], p_.detach(), 0.0), ("exp_avg", got_m[n], st["exp_avg"], mmax),
                                              ("exp_avg_sq", got_v[n], st["exp_avg_sq"], vmax)):
                    err = (got.reshape(ref.shape) - ref).abs().max().item()
                    assert err <= 1e-6 * max(ref.abs().max().item(), floor), f"step {step} {n} {what}: {err:.3e}"
    assert names[0] == "conv1.att_src"


def _fill_ring(sb, trainer, trans):
    G, N = trans[0].shape[:2]
    cfg = sb.ops.make_config(sb._lib.SCENARIO_GOTO, G, N)
    pos, vel, actions, rewards, pos2, vel2 = trans
    sb.ops.replay_push(cfg, trainer.replay_buffer.ring, torch.cat([pos, vel], 2).contiguous().to(_dev()),
                       actions.to(torch.int32).to(_dev()), rewards.contiguous().to(_dev()),
                       torch.cat([pos2, vel2], 2).contiguous().to(_dev()))


@pytest.mark.gpu
def test_trainer_steps_equal_direct_calls_and_oracle_loss():
    import swarm_b200 as sb
    ops = sb.ops
    N, G = 12, 32
    env = sb.make_env(sb.FlockingScenario(), num_envs=1, device=_dev(), continuous_actions=False, max_steps=10,
                      dict_spaces=True, seed=0, n_agents=N)
    model = sb.StackedGCN.from_state_dict(_flocking_sd(6))
    tr = sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "t", replay_capacity=256, model=model)
    assert tr.w.numel() == 409 and tr.exp_avg.numel() == 409 and tr._grad.numel() == 409
    assert torch.equal(tr.w, tr.w_target)
    trans = _transitions(48, N, seed=21)
    _fill_ring(sb, tr, trans)
    spec = tr.stack_spec
    cfg = ops.clone_config(tr.graph_cfg, num_envs=G)
    idx = torch.randint(0, 48, (G,), generator=torch.Generator().manual_seed(1)).to(_dev())
    w, wt, m, v = tr.w.clone(), tr.w_target.clone(), tr.exp_avg.clone(), tr.exp_avg_sq.clone()
    sub = tuple(t[idx.cpu()] for t in trans)
    acts = model.activations
    for step in range(1, 21):
        sd_on, sd_tg = ops.unpack_stack_weights(tr.w.cpu(), spec), ops.unpack_stack_weights(tr.w_target.cpu(), spec)
        loss = tr.train_step_dqn(G, ticks=step, update_target_every=7, indices=idx)
        g, _, _ = ops.dqn_grad_stack(cfg, spec, w, wt, tr.replay_buffer.ring, idx, G)
        ops.adam_clip_step_stack(spec, w, g, m, v, step, target=wt if step % 7 == 0 else None)
        for a, b in ((tr.w, w), (tr.w_target, wt), (tr.exp_avg, m), (tr.exp_avg_sq, v)):
            assert torch.equal(a, b), step
        loss64, _, _ = _oracle_loss_grads(cfg, sd_on, sd_tg, acts, 7, sub, "complete", 0, torch.float64)
        assert abs(loss - loss64) <= GRAD_RTOL * abs(loss64), f"step {step}: loss {loss} vs {loss64}"
    assert tr.opt_step == 20 and not torch.equal(tr.w, tr.w_target)
    tr.sync_modules()
    assert torch.equal(ops.pack_stack_weights(tr.model.state_dict(), spec, _dev()), tr.w)


@pytest.mark.gpu
@pytest.mark.parametrize("scen", ["flocking", "cohesion"])
def test_train_model_stepwise_with_a_stack(scen):
    import swarm_b200 as sb
    torch.manual_seed(0)
    if scen == "flocking":
        env = sb.make_env(sb.FlockingScenario(), num_envs=64, device=_dev(), continuous_actions=False, max_steps=8,
                          dict_spaces=True, seed=0, n_agents=12)
        model = sb.StackedGCN.from_state_dict(_flocking_sd(7))
    else:
        env = sb.make_env(sb.CohesionScenario(), num_envs=64, device=_dev(), continuous_actions=False, max_steps=8,
                          dict_spaces=True, seed=0, n_agents=9)
        model = sb.StackedGCN(5, 8, 9, 3)
    tr = sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "t", replay_capacity=1024, model=model)
    w0 = tr.w.clone()
    stats = tr.train_model_stepwise({"episodes": 3, "epsilon": 0.5, "epsilon_decay": 0.1, "min_epsilon": 0.05,
                                     "graphs_per_update": 32, "update_target_every": 5})
    assert tr.opt_step == 24 and stats["opt_steps"] == 24
    assert all(np.isfinite(tr.episode_losses)) and stats["loss"] > 0
    assert not torch.equal(tr.w, w0) and torch.isfinite(tr.w).all()
    assert np.isfinite(tr.evaluate_policy(1))


@pytest.mark.gpu
def test_train_model_checkpoint_loads_and_runs(tmp_path):
    import swarm_b200 as sb
    sb.set_seed(0)
    env = sb.make_env(sb.GoToPositionScenario(), num_envs=1, device=_dev(), continuous_actions=False, max_steps=40,
                      dict_spaces=True, seed=0, n_agents=5)
    tr = sb.DQNTrainer(env, 0, str(tmp_path / "models"), str(tmp_path / "stats"), "stack", replay_capacity=512,
                       model=sb.StackedGCN(7, 8, 9, 3))
    tr.train_model({"epsilon": 0.9, "epsilon_decay": 0.01, "min_epsilon": 0.05, "episodes": 1, "verbose": False,
                    "save": True})
    assert tr.opt_step == 40 - 31
    sd = torch.load(tmp_path / "models" / "experiment_stack-seed_0.pth")
    model = sb.StackedGCN.from_state_dict(sd).to(_dev())
    assert torch.equal(model.packed_stack_weights(_dev()), tr.w)
    env2 = sb.make_env(sb.GoToPositionScenario(), num_envs=1, device=_dev(), continuous_actions=False, max_steps=10,
                       dict_spaces=True, seed=1, n_agents=5)
    sim = sb.Simulator(env2, model, 1, "goto", 0, output_dir=str(tmp_path / "sim"), k=5)
    sim.run_simulation()
    assert len(sim.episode_rewards) == 1 and np.isfinite(sim.episode_rewards[0])


@pytest.mark.gpu
def test_trainer_rejects_what_a_stack_cannot_run():
    import swarm_b200 as sb
    env = sb.make_env(sb.GoToPositionScenario(), num_envs=4, device=_dev(), continuous_actions=False, max_steps=4,
                      dict_spaces=True, seed=0, n_agents=5)
    tr = sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "t", replay_capacity=64, model=sb.StackedGCN(7, 8, 9, 2))
    cfg = {"episodes": 1, "epsilon": 0.5, "epsilon_decay": 0.1, "min_epsilon": 0.05}
    with pytest.raises(NotImplementedError, match="train_model_stepwise"):
        tr.train_model_batched(cfg)
    with pytest.raises(NotImplementedError, match="train_model_stepwise"):
        tr.train_model_device(cfg)
    with pytest.raises(ValueError, match="input features"):
        sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "t", replay_capacity=64, model=sb.StackedGCN(5, 8, 9, 2))


def test_unpack_inverts_pack():
    import swarm_b200 as sb
    for layers, hidden, in_f in ((3, 8, 7), (1, 32, 7), (4, 5, 5)):
        sd = _random_sd(layers, hidden, in_f, 0)
        spec = sb.ops.stack_spec(layers, hidden, in_f)
        back = sb.ops.unpack_stack_weights(sb.ops.pack_stack_weights(sd, spec, "cpu"), spec)
        assert list(back) == list(sd)
        assert all(back[k].shape == sd[k].shape and torch.equal(back[k], sd[k]) for k in sd)
    sd = _flocking_sd(0)
    spec = sb.ops.stack_spec(3, 8, 7)
    back = sb.ops.unpack_stack_weights(sb.ops.pack_stack_weights(sd, spec, "cpu"), spec)
    assert set(back) == set(sd) and all(torch.equal(back[k], sd[k]) for k in sd)


def test_stack_dqn_argument_validation_without_device():
    import swarm_b200 as sb
    L, lib = sb._lib, sb._lib.lib()
    spec = sb.ops.stack_spec(3, 8, 7)
    cfg = sb.ops.make_config(L.SCENARIO_GOTO, 1, 12, L.GRAPH_COMPLETE)
    rs = L.SwarmReplay(8, 8, 8, 8, 64)
    wb = int(lib.swarm_dqn_stack_workspace_bytes(C.byref(cfg), C.byref(spec), 32))
    assert wb > 0

    def grad(c=cfg, s=spec, online=8, batch=rs, ws=8, wsb=wb, G=32):
        return lib.swarm_dqn_stack_grad(C.byref(c), C.byref(s), online, 8, C.byref(batch), None, G, 0.99, 0.01, 8, 8,
                                        None, ws, wsb, None)

    def adam(s=spec, w=8, step=1, beta1=0.9):
        return lib.swarm_adam_clip_stack_step(C.byref(s), w, 8, 8, 8, step, 1e-3, beta1, 0.999, 1e-8, 1.0, None, None, None)

    for field, value in (("n_layers", 0), ("n_layers", 5), ("hidden", 33), ("in_features", 6)):
        bad = sb.ops.stack_spec(3, 8, 7)
        setattr(bad, field, value)
        assert grad(s=bad) < 0 and adam(s=bad) < 0, field
        assert int(lib.swarm_dqn_stack_workspace_bytes(C.byref(cfg), C.byref(bad), 32)) == 0
    assert grad(c=sb.ops.make_config(L.SCENARIO_GOTO, 1, 129, L.GRAPH_COMPLETE)) < 0
    assert grad(c=sb.ops.make_config(L.SCENARIO_GOTO, 1, 20, L.GRAPH_KNN, 5)) == -2
    assert b"n_agents <= 16" in lib.swarm_last_error()
    assert grad(online=None) == -1 and b"NULL" in lib.swarm_last_error()
    assert grad(batch=L.SwarmReplay(8, None, 8, 8, 64)) == -1
    assert grad(ws=None) == -1
    assert grad(wsb=wb - 1) == -1 and b"workspace too small" in lib.swarm_last_error()
    assert grad(G=0) == -1
    assert adam(w=None) == -1
    assert adam(step=0) == -1 and b"1-based" in lib.swarm_last_error()
    assert adam(beta1=1.0) == -1 and b"Adam" in lib.swarm_last_error()
    # the largest shape fits one CTA's shared memory
    big = sb.ops.stack_spec(4, 32, 7)
    c128 = sb.ops.make_config(L.SCENARIO_GOTO, 1, 128, L.GRAPH_COMPLETE)
    assert int(lib.swarm_dqn_stack_workspace_bytes(C.byref(c128), C.byref(big), 4)) > 0
