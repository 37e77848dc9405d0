"""Argument validation of the C entry points, without a device: a table of malformed calls, each with the return code
and a message fragment it must give, and the workspace sizes the *_workspace_bytes calls report over a grid of
configs.  Where a call needs a non-NULL pointer, a fake address stands in; the calls run in a child process that sees
no CUDA device, so a call that wrongly got past its checks fails with SWARM_ERR_CUDA instead of launching a kernel."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

P = 8              # a fake device address: only ever passed to calls that must refuse it
BIG = 1 << 40      # a workspace size no check refuses


def _cases():
    """(id, call, expected return code, message fragment)."""
    import swarm_b200 as sb
    L, ops, lib = sb._lib, sb.ops, sb._lib.lib()
    GOTO, OA = L.SCENARIO_GOTO, L.SCENARIO_OBSTACLE_AVOIDANCE
    cfg = lambda n=12, graph=L.GRAPH_COMPLETE, k=10, B=4, **kw: ops.clone_config(ops.make_config(GOTO, B, n, graph, k), **kw)
    ref = C.byref
    ring = lambda cap=1000, state=P: L.SwarmReplay(state, P, P, P, cap)
    spec = lambda n_layers=3, hidden=8, in_features=7, act=None: _stack(ops, n_layers, hidden, in_features, act)
    rspec = lambda kind=L.REWARD_FLOCKING, B=4, n=12, **kw: ops.reward_spec(kind, B, n, **kw)

    def hyper(**kw):
        h = L.SwarmTrainHyper()
        h.lr, h.beta1, h.beta2, h.eps, h.max_norm = 1e-3, 0.9, 0.999, 1e-8, 1.0
        h.graphs_per_update, h.update_target_every, h.gamma, h.loss_scale = 32, 200, 0.99, 1.0
        for k, v in kw.items():
            setattr(h, k, v)
        return h

    def rollout(c, ticks=1, eps=0.0, replay=None, flocking=None, shaping=None):
        o = L.SwarmRolloutOptions()
        o.epsilon = eps
        if replay is not None:
            o.replay = C.pointer(replay)
        if flocking is not None:
            o.flocking = C.addressof(flocking)
        o.flocking_shaping = shaping
        return lib.swarm_rollout(ref(c), P, P, ticks, ref(o), None, None, None, None)

    def tick_grad(c=None, h=None, r=None, wsb=BIG):
        return lib.swarm_train_tick_grad(ref(c or cfg(B=64)), ref(h or hyper()), P, P, P, P, None, None,
                                         ref(r or ring()), None, P, P, P, wsb, None)

    def tick(c=None, h=None, r=None, exp_avg=P, wsb=BIG, peers=None):
        return lib.swarm_train_tick(ref(c or cfg(B=64)), ref(h or hyper()), P, P, P, exp_avg, P, P, None, None,
                                    ref(r or ring()), None, P, P, wsb, ref(peers) if peers else None, None)

    def flocking_hyper(c, shaping=None):
        fs = rspec(B=c.num_envs, n=c.n_agents)
        h = hyper(flocking=C.addressof(fs), flocking_shaping=shaping)
        h._keep = fs
        return h

    def scen(fn, s, state=P, shaping=P, reward=P, ws=P, wsb=BIG):
        if fn == "small":
            return lib.swarm_scenario_reward(ref(s) if s else None, state, shaping, reward, None, None)
        return lib.swarm_scenario_reward_large(ref(s) if s else None, state, shaping, reward, None, ws, wsb, None)

    def stack_roll(c, s=None, reward=None, shaping=P, wsb=BIG, ticks=1, large=False):
        fn = lib.swarm_rollout_stack_large if large else lib.swarm_rollout_stack
        return fn(ref(c), ref(s or spec()), P, P, ticks, ref(reward) if reward else None, shaping, None, None, P, wsb, None)

    def stack_tick(c=None, s=None, h=None, reward=None, r=None, wsb=BIG):
        c = c or cfg(B=64)
        return lib.swarm_train_tick_stack(ref(c), ref(s or spec()), ref(h or hyper()), ref(reward) if reward else None, P,
                                          P, P, P, P, P, P, None, None, ref(r or ring()), None, P, P, wsb, None)

    def dqn_stack(c=None, s=None, G=32, batch=None, wsb=BIG):
        return lib.swarm_dqn_stack_grad(ref(c or cfg()), ref(s or spec()), P, P, ref(batch or ring()), None, G, 0.99, 1.0,
                                        P, P, None, P, wsb, None)

    adam = lambda step=1, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, w=P: lib.swarm_adam_clip_step(
        w, P, P, P, step, lr, b1, b2, eps, 1.0, None, None, None)
    adam_stack = lambda s=None, step=1, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8: lib.swarm_adam_clip_stack_step(
        ref(s or spec()), P, P, P, P, step, lr, b1, b2, eps, 1.0, None, None, None)
    bad = lambda **kw: _stack(ops, **{**dict(n_layers=3, hidden=8, in_features=7, act=None), **kw})
    knn500, knn20 = cfg(500, L.GRAPH_KNN, 10, B=2), cfg(20, L.GRAPH_KNN, 5)
    nan = float("nan")
    return [
        # the cfg checks every entry point shares
        ("reset_grid/cfg_null", lambda: lib.swarm_reset_grid(None, P, P, None), -1, "cfg is NULL"),
        ("reset_grid/scenario", lambda: lib.swarm_reset_grid(ref(cfg(scenario=7)), P, P, None), -1, "unknown scenario"),
        ("reset_grid/num_envs", lambda: lib.swarm_reset_grid(ref(cfg(B=0)), P, P, None), -1, "num_envs"),
        ("reset_grid/buffers", lambda: lib.swarm_reset_grid(ref(cfg()), None, P, None), -1, "centers/state"),
        ("sim_step/too_large", lambda: lib.swarm_sim_step(ref(cfg(5000)), P, P, P, *[None] * 6), -2, "n_agents > 4096"),
        ("sim_step/contact", lambda: lib.swarm_sim_step(ref(cfg(64)), P, P, P, None, None, P, None, None, None), -2,
         "contact masks"),
        # kNN: k range, and the partial_sort branch above 128 agents
        ("graph_build/k_range", lambda: lib.swarm_graph_build(ref(cfg(5, L.GRAPH_KNN, 10)), P, P, None, None), -1,
         "selected index k out of range"),
        ("graph_build/partial_sort", lambda: lib.swarm_graph_build(ref(knn500), P, P, None, None), -2, "partial_sort"),
        ("graph_build/partial_sort_first", lambda: lib.swarm_graph_build(ref(knn500), None, None, None, None), -1, "state"),
        ("graph_build/radius", lambda: lib.swarm_graph_build(ref(cfg(graph=L.GRAPH_RADIUS)), P, P, None, None), -1,
         "swarm_graph_build_radius"),
        ("graph_build_radius/mode", lambda: lib.swarm_graph_build_radius(ref(cfg()), P, P, None, None), -1,
         "SWARM_GRAPH_RADIUS"),
        ("gatq_forward/large", lambda: lib.swarm_gatq_forward(ref(cfg(200)), P, P, P, None, None), -2, "n_agents > 128"),
        ("gatq_forward/no_output", lambda: lib.swarm_gatq_forward(ref(cfg()), P, P, None, None, None), -1, "no output"),
        ("gatq_forward_knn_large/mode", lambda: lib.swarm_gatq_forward_knn_large(ref(cfg(500)), P, P, P, P, None, None),
         -1, "SWARM_GRAPH_KNN"),
        ("gatq_forward_knn_large/smem", lambda: lib.swarm_gatq_forward_knn_large(
            ref(cfg(4096, L.GRAPH_KNN, 10, B=1)), P, P, P, P, None, None), -2, "shared memory"),
        ("graph_build_radius_csr/pass", lambda: lib.swarm_graph_build_radius_csr(
            ref(cfg(1024, L.GRAPH_RADIUS, B=2)), P, None, None, None, None), -1, "count pass"),
        ("gatq_forward_large/knn", lambda: lib.swarm_gatq_forward_large(ref(knn500), P, P, P, None, None), -1, "knn_large"),
        ("gatq_forward_large/too_large", lambda: lib.swarm_gatq_forward_large(
            ref(cfg(5000, L.GRAPH_RADIUS, B=1)), P, P, P, None, None), -2, "n_agents > 4096"),
        # swarm_rollout_large
        ("rollout_large/small", lambda: lib.swarm_rollout_large(ref(cfg(100)), P, P, 1, None, None, P, BIG, None), -1,
         "use swarm_rollout"),
        ("rollout_large/ticks_first", lambda: lib.swarm_rollout_large(ref(knn500), P, P, -1, None, None, P, BIG, None), -1,
         "ticks"),
        ("rollout_large/partial_sort", lambda: lib.swarm_rollout_large(ref(knn500), P, P, 1, None, None, P, BIG, None), -2,
         "partial_sort"),
        ("rollout_large/workspace", lambda: lib.swarm_rollout_large(
            ref(cfg(640, L.GRAPH_KNN, 10, B=2)), P, P, 1, None, None, P, 2 * 640 * 44 + 511, None), -1,
         "workspace too small"),
        ("rollout_large/workspace_null", lambda: lib.swarm_rollout_large(
            ref(cfg(600, L.GRAPH_RADIUS)), P, P, 1, None, None, None, BIG, None), -1, "workspace"),
        # swarm_rollout: options, replay ring, Flocking reward
        ("rollout/large", lambda: rollout(cfg(500)), -2, "n_agents > 128"),
        ("rollout/epsilon", lambda: rollout(cfg(), eps=2.0), -1, "epsilon"),
        ("rollout/ring_null", lambda: rollout(cfg(), replay=ring(state=None)), -1, "replay ring has NULL arrays"),
        ("rollout/ring_capacity", lambda: rollout(cfg(), replay=ring(cap=0)), -1, "capacity"),
        ("rollout/ring_overwrite", lambda: rollout(cfg(), ticks=300, replay=ring()), -1, "replay capacity"),
        ("rollout/flocking_kind", lambda: rollout(cfg(), flocking=rspec(L.REWARD_COHESION), shaping=P), -1,
         "Flocking reward spec"),
        ("rollout/flocking_world", lambda: rollout(cfg(scenario=OA), flocking=rspec()), -1, "GoTo world"),
        ("rollout/flocking_agents", lambda: rollout(cfg(1), flocking=rspec(n=1)), -1, "two agents"),
        ("rollout/flocking_shaping", lambda: rollout(cfg(), flocking=rspec()), -1, "shaping"),
        # replay ring calls
        ("replay_push/ring_null", lambda: lib.swarm_replay_push(ref(cfg()), None, 0, P, P, P, P, None), -1,
         "replay ring has NULL arrays"),
        ("replay_push/capacity", lambda: lib.swarm_replay_push(ref(cfg()), ref(ring(cap=0)), 0, P, P, P, P, None), -1,
         "no capacity"),
        ("replay_push/transition_first", lambda: lib.swarm_replay_push(ref(cfg()), ref(ring(cap=2)), 0, None, P, P, P,
                                                                       None), -1, "NULL transition array"),
        ("replay_push/num_envs", lambda: lib.swarm_replay_push(ref(cfg()), ref(ring(cap=2)), 0, P, P, P, P, None), -1,
         "num_envs exceeds the replay capacity"),
        ("replay_push/cursor", lambda: lib.swarm_replay_push(ref(cfg()), ref(ring()), -1, P, P, P, P, None), -1, "cursor"),
        ("replay_gather/cfg", lambda: lib.swarm_replay_gather(None, ref(ring()), P, 4, P, P, P, P, None), -1,
         "cfg is NULL"),
        ("replay_gather/ring_null", lambda: lib.swarm_replay_gather(ref(cfg()), ref(ring(state=None)), P, 4, P, P, P, P,
                                                                    None), -1, "replay ring has NULL arrays"),
        ("replay_gather/n_graphs", lambda: lib.swarm_replay_gather(ref(cfg()), ref(ring(cap=0)), P, -1, P, P, P, P, None),
         -1, "n_graphs"),
        # one-layer DQN update
        ("dqn_grad/n_graphs", lambda: lib.swarm_dqn_grad(ref(cfg()), P, P, ref(ring()), None, 0, 0.99, 1.0, P, P, None,
                                                         P, BIG, None), -1, "n_graphs"),
        ("dqn_grad/batch", lambda: lib.swarm_dqn_grad(ref(cfg()), P, P, ref(ring(state=None)), None, 32, 0.99, 1.0, P, P,
                                                      None, P, BIG, None), -1, "batch has NULL arrays"),
        ("dqn_grad/workspace", lambda: lib.swarm_dqn_grad(ref(cfg()), P, P, ref(ring()), None, 32, 0.99, 1.0, P, P, None,
                                                          P, 16, None), -1, "workspace too small"),
        ("adam/step", lambda: adam(step=0), -1, "1-based"),
        ("adam/null_first", lambda: adam(step=0, w=None), -1, "NULL argument"),
        ("adam/lr", lambda: adam(lr=-1.0), -1, "Adam"),
        ("adam/beta1", lambda: adam(b1=1.0), -1, "Adam"),
        ("adam/beta2", lambda: adam(b2=-0.1), -1, "Adam"),
        ("adam/eps_nan", lambda: adam(eps=nan), -1, "Adam"),
        ("tick_grad/graphs", lambda: tick_grad(h=hyper(graphs_per_update=0)), -1, "graphs_per_update"),
        ("tick_grad/target", lambda: tick_grad(h=hyper(update_target_every=0)), -1, "update_target_every"),
        ("tick_grad/adam", lambda: tick_grad(h=hyper(lr=nan)), -1, "Adam"),
        ("tick_grad/ring_null", lambda: tick_grad(r=ring(state=None)), -1, "replay ring has NULL arrays"),
        ("tick_grad/ring_capacity", lambda: tick_grad(r=ring(cap=0)), -1, "no capacity"),
        ("tick_grad/num_envs", lambda: tick_grad(r=ring(cap=10)), -1, "num_envs exceeds the replay capacity"),
        ("tick_grad/workspace", lambda: tick_grad(wsb=16), -1, "workspace too small"),
        ("tick_grad/flocking_world", lambda: tick_grad(c=cfg(B=64, scenario=OA), h=flocking_hyper(cfg(B=64))), -1,
         "GoTo world"),
        ("tick_grad/flocking_shaping", lambda: tick_grad(h=flocking_hyper(cfg(B=64))), -1, "shaping"),
        ("tick_apply/cfg", lambda: lib.swarm_train_tick_apply(None, ref(hyper()), P, P, P, P, P, P, 1000, None, None), -1,
         "cfg is NULL"),
        ("tick_apply/adam", lambda: lib.swarm_train_tick_apply(ref(cfg()), ref(hyper(beta2=1.0)), P, P, P, P, P, P, 1000,
                                                               None, None), -1, "Adam"),
        ("tick_apply/capacity", lambda: lib.swarm_train_tick_apply(ref(cfg()), ref(hyper()), P, P, P, P, P, P, 2, None,
                                                                   None), -1, "ring_capacity"),
        ("tick/exp_avg", lambda: tick(exp_avg=None), -1, "NULL argument"),
        ("tick/peers", lambda: tick(peers=_peers(L, 2, 5)), -1, "peer exchange"),
        ("tick/adam", lambda: tick(h=hyper(beta1=-0.5)), -1, "Adam"),
        ("tick/ring_null", lambda: tick(r=ring(state=None)), -1, "replay ring"),
        ("tick/num_envs", lambda: tick(r=ring(cap=10)), -1, "replay capacity"),
        ("tick/workspace", lambda: tick(wsb=16), -1, "workspace too small"),
        ("reset_random/std", lambda: lib.swarm_reset_random(ref(cfg()), ref(_reset(ops, GOTO, std_x=-1.0)), None, 0, None,
                                                            P, None), -1, "std"),
        ("reset_random/episode", lambda: lib.swarm_reset_random(ref(cfg()), ref(_reset(ops, GOTO)), None, -1, None, P,
                                                                None), -1, "episode"),
        ("episode_end/ctl", lambda: lib.swarm_episode_end(ref(cfg()), None, P, None, None, None, 0, 0.9, 0.01, 0.05, None),
         -1, "ctl/returns"),
        # Flocking / Cohesion rewards
        ("scenario_reward/spec_null", lambda: scen("small", None), -1, "spec is NULL"),
        ("scenario_reward/kind", lambda: scen("small", rspec(kind=5)), -1, "unknown reward kind"),
        ("scenario_reward/agents", lambda: scen("small", rspec(n=1)), -1, "two agents"),
        ("scenario_reward/large", lambda: scen("small", rspec(n=200)), -2, "n_agents <= 128"),
        ("scenario_reward/env_index", lambda: scen("small", rspec(env_index=4)), -1, "env_index"),
        ("scenario_reward/state", lambda: scen("small", rspec(), state=None), -1, "state is NULL"),
        ("scenario_reward/shaping", lambda: scen("small", rspec(), shaping=None), -1, "shaping"),
        ("scenario_reward/reward", lambda: scen("small", rspec(), reward=None), -1, "reward is NULL"),
        ("scenario_reward/cohesion_reset", lambda: scen("small", rspec(L.REWARD_COHESION, reset=1, sigma=0.0)), -1,
         "reset must be 0"),
        ("scenario_reward/cohesion_reward_first", lambda: scen("small", rspec(L.REWARD_COHESION, sigma=0.0), reward=None),
         -1, "reward is NULL"),
        ("scenario_reward/sigma", lambda: scen("small", rspec(L.REWARD_COHESION, sigma=0.0)), -1, "sigma"),
        ("scenario_reward_large/too_large", lambda: scen("large", rspec(n=5000)), -2, "n_agents <= 4096"),
        ("scenario_reward_large/sigma", lambda: scen("large", rspec(L.REWARD_COHESION, n=600, sigma=-1.0)), -1, "sigma"),
        ("scenario_reward_large/shaping", lambda: scen("large", rspec(n=600), shaping=None), -1, "shaping"),
        ("scenario_reward_large/workspace_null", lambda: scen("large", rspec(n=600), ws=None), -1, "workspace is NULL"),
        ("scenario_reward_large/workspace", lambda: scen("large", rspec(n=600), wsb=16), -1, "workspace too small"),
        # stacked networks: the spec
        ("gatstack_forward/cfg_null", lambda: lib.swarm_gatstack_forward(None, ref(spec()), P, P, P, None, None), -1,
         "cfg is NULL"),
        ("gatstack_forward/spec_null", lambda: lib.swarm_gatstack_forward(ref(cfg()), None, P, P, P, None, None), -1,
         "spec is NULL"),
        ("gatstack_forward/n_layers", lambda: lib.swarm_gatstack_forward(ref(cfg()), ref(bad(n_layers=5)), P, P, P, None,
                                                                         None), -1, "n_layers"),
        ("gatstack_forward/hidden", lambda: lib.swarm_gatstack_forward(ref(cfg()), ref(bad(hidden=33)), P, P, P, None,
                                                                       None), -2, "hidden"),
        ("gatstack_forward/in_features", lambda: lib.swarm_gatstack_forward(ref(cfg()), ref(bad(in_features=6)), P, P, P,
                                                                            None, None), -1, "in_features"),
        ("gatstack_forward/activation", lambda: lib.swarm_gatstack_forward(ref(cfg()), ref(bad(act=[0, 7, 1])), P, P, P,
                                                                           None, None), -1, "unknown activation"),
        ("gatstack_forward/knn", lambda: lib.swarm_gatstack_forward(ref(knn20), ref(spec()), P, P, P, None, None), -2,
         "n_agents <= 16"),
        ("gatstack_forward/cfg_first", lambda: lib.swarm_gatstack_forward(ref(cfg(scenario=7)), ref(bad(n_layers=0)), P, P,
                                                                          P, None, None), -1, "unknown scenario"),
        ("gatstack_forward_large/partial_sort", lambda: lib.swarm_gatstack_forward_large(
            ref(knn500), ref(spec()), P, P, P, P, None, P, BIG, None), -2, "partial_sort"),
        ("gatstack_forward_large/neighbours", lambda: lib.swarm_gatstack_forward_large(
            ref(cfg(640, L.GRAPH_KNN, 10, B=2)), ref(spec()), P, P, None, P, None, P, BIG, None), -1, "neighbours"),
        ("gatstack_forward_large/workspace", lambda: lib.swarm_gatstack_forward_large(
            ref(cfg(600)), ref(spec()), P, P, None, P, None, P, 16, None), -1, "workspace too small"),
        ("dqn_stack/n_graphs", lambda: dqn_stack(G=0), -1, "n_graphs"),
        ("dqn_stack/large", lambda: dqn_stack(c=cfg(200)), -2, "n_agents <= 128"),
        ("dqn_stack/agents", lambda: dqn_stack(c=cfg(1)), -2, "n_agents >= 2"),
        ("dqn_stack/spec", lambda: dqn_stack(s=bad(n_layers=5)), -1, "n_layers"),
        ("dqn_stack/batch", lambda: dqn_stack(batch=ring(state=None)), -1, "batch has NULL arrays"),
        ("dqn_stack/workspace", lambda: dqn_stack(wsb=16), -1, "workspace too small"),
        ("adam_stack/spec", lambda: adam_stack(s=bad(n_layers=5), step=0), -1, "n_layers"),
        ("adam_stack/hidden", lambda: adam_stack(s=bad(hidden=0)), -2, "hidden"),
        ("adam_stack/activation_not_checked", lambda: adam_stack(s=bad(act=[0, 7, 1]), step=0), -1, "1-based"),
        ("adam_stack/adam", lambda: adam_stack(b2=1.0), -1, "Adam"),
        ("adam_stack/eps", lambda: adam_stack(eps=-1.0), -1, "Adam"),
        # stacked rollouts: workspace and reward
        ("rollout_stack/workspace", lambda: stack_roll(cfg(), wsb=0), -1, "workspace too small"),
        ("rollout_stack/workspace_large", lambda: stack_roll(cfg(600), wsb=16), -1, "workspace too small"),
        ("rollout_stack/large_reward", lambda: stack_roll(cfg(600), reward=rspec(n=600)), -2,
         "implemented for n_agents <= 128"),
        ("rollout_stack/kind", lambda: stack_roll(cfg(), reward=rspec(kind=9)), -1, "unknown reward kind"),
        ("rollout_stack/world", lambda: stack_roll(cfg(scenario=OA), reward=rspec(L.REWARD_COHESION)), -1, "GoTo world"),
        ("rollout_stack/disagree", lambda: stack_roll(cfg(), reward=rspec(B=5)), -1, "disagree"),
        ("rollout_stack/agents", lambda: stack_roll(cfg(1), reward=rspec(n=1)), -1, "two agents"),
        ("rollout_stack/shaping", lambda: stack_roll(cfg(), reward=rspec(), shaping=None), -1, "shaping"),
        ("rollout_stack/sigma", lambda: stack_roll(cfg(), reward=rspec(L.REWARD_COHESION, sigma=0.0)), -1, "sigma"),
        ("rollout_stack/ticks", lambda: stack_roll(cfg(), ticks=-1), -1, "ticks"),
        ("rollout_stack_large/small", lambda: stack_roll(cfg(), large=True), -2, "swarm_rollout_stack"),
        ("rollout_stack_large/partial_sort", lambda: stack_roll(knn500, large=True), -2, "partial_sort"),
        ("rollout_stack_large/disagree", lambda: stack_roll(cfg(600), reward=rspec(n=601), large=True), -1, "disagree"),
        ("rollout_stack_large/sigma", lambda: stack_roll(cfg(600), reward=rspec(L.REWARD_COHESION, n=600, sigma=0.0),
                                                         large=True), -1, "sigma"),
        ("rollout_stack_large/workspace", lambda: stack_roll(cfg(600), reward=rspec(n=600), wsb=16, large=True), -1,
         "workspace too small"),
        ("rollout_stack_large/reward_workspace", lambda: stack_roll(
            cfg(600), reward=rspec(n=600), large=True,
            wsb=lib.swarm_rollout_stack_large_workspace_bytes(ref(cfg(600)), None)), -1, "workspace too small"),
        # the device-driven stacked tick
        ("tick_stack/adam", lambda: stack_tick(h=hyper(beta1=1.0)), -1, "Adam"),
        ("tick_stack/hyper_first", lambda: stack_tick(c=cfg(B=0), h=hyper(graphs_per_update=0)), -1, "graphs_per_update"),
        ("tick_stack/num_envs", lambda: stack_tick(c=cfg(B=0)), -1, "num_envs must be positive"),
        ("tick_stack/scenario_first", lambda: stack_tick(c=cfg(200, scenario=7)), -1, "unknown scenario"),
        ("tick_stack/large", lambda: stack_tick(c=cfg(200)), -2, "n_agents > 128"),
        ("tick_stack/spec", lambda: stack_tick(s=bad(in_features=3)), -1, "in_features"),
        ("tick_stack/knn", lambda: stack_tick(c=cfg(20, L.GRAPH_KNN, 5, B=64)), -2, "n_agents <= 16"),
        ("tick_stack/agents", lambda: stack_tick(c=cfg(1, B=64)), -2, "n_agents >= 2"),
        ("tick_stack/flocking", lambda: stack_tick(h=flocking_hyper(cfg(B=64))), -1, "hyper->flocking"),
        ("tick_stack/null", lambda: lib.swarm_train_tick_stack(ref(cfg(B=64)), ref(spec()), ref(hyper()), None, P, None,
                                                               P, P, P, P, P, None, None, ref(ring()), None, P, P, BIG,
                                                               None), -1, "NULL argument"),
        ("tick_stack/ring_null", lambda: stack_tick(r=ring(state=None)), -1, "replay ring has NULL arrays"),
        ("tick_stack/ring_capacity", lambda: stack_tick(r=ring(cap=0)), -1, "no capacity"),
        ("tick_stack/num_envs_capacity", lambda: stack_tick(r=ring(cap=63)), -1, "replay capacity"),
        ("tick_stack/workspace", lambda: stack_tick(wsb=16), -1, "workspace too small"),
        ("tick_stack/disagree", lambda: stack_tick(reward=rspec(L.REWARD_COHESION, B=65)), -1, "disagree"),
        ("tick_stack/world", lambda: stack_tick(c=cfg(B=64, scenario=OA), reward=rspec(L.REWARD_COHESION, B=64)), -1,
         "GoTo world"),
        ("tick_stack/sigma", lambda: stack_tick(reward=rspec(L.REWARD_COHESION, B=64, sigma=nan)), -1, "sigma"),
    ]


def _stack(ops, n_layers, hidden, in_features, act):
    s = ops.stack_spec(3, 8, 7)
    s.n_layers, s.hidden, s.in_features = n_layers, hidden, in_features
    if act is not None:
        for i, a in enumerate(act):
            s.activation[i] = a
    return s


def _reset(ops, scenario, **kw):
    sp = ops.reset_spec(scenario)
    for k, v in kw.items():
        setattr(sp, k, v)
    return sp


def _peers(L, world_size, rank):
    px = L.SwarmPeerExchange()
    px.world_size, px.rank = world_size, rank
    return px


GRID_NS = (2, 12, 128, 129, 600, 4096)
GRID_KS = (5, 10, 64)


def _workspace_grid():
    """Every *_workspace_bytes result on complete, kNN and radius graphs, N in GRID_NS, k in GRID_KS (kNN)."""
    import swarm_b200 as sb
    L, ops, lib = sb._lib, sb.ops, sb._lib.lib()
    spec = ops.stack_spec(3, 8, 7)
    out = {}
    for graph, ks in ((L.GRAPH_COMPLETE, (10,)), (L.GRAPH_KNN, GRID_KS), (L.GRAPH_RADIUS, (10,))):
        for n in GRID_NS:
            for k in ks:
                cfg = ops.make_config(L.SCENARIO_GOTO, 3, n, graph, k)
                ref = C.byref(cfg)
                flock = ops.reward_spec(L.REWARD_FLOCKING, 3, n)
                coh = ops.reward_spec(L.REWARD_COHESION, 3, n)
                out[f"{graph}/{n}/{k}"] = [int(v) for v in (
                    lib.swarm_rollout_large_workspace_bytes(ref),
                    lib.swarm_rollout_stack_workspace_bytes(ref),
                    lib.swarm_rollout_stack_large_workspace_bytes(ref, None),
                    lib.swarm_rollout_stack_large_workspace_bytes(ref, C.byref(flock)),
                    lib.swarm_rollout_stack_large_workspace_bytes(ref, C.byref(coh)),
                    lib.swarm_gatstack_large_workspace_bytes(ref, C.byref(spec)),
                    lib.swarm_dqn_workspace_bytes(ref, 32),
                    lib.swarm_dqn_stack_workspace_bytes(ref, C.byref(spec), 32),
                    lib.swarm_scenario_reward_large_workspace_bytes(C.byref(flock)),
                    lib.swarm_scenario_reward_large_workspace_bytes(C.byref(coh)))]
    return out


def _child_main():
    import swarm_b200 as sb
    lib = sb._lib.lib()
    calls = {}
    for name, call, _, _ in _cases():
        rc = int(call())
        calls[name] = [rc, lib.swarm_last_error().decode()]
    print(json.dumps({"calls": calls, "workspace": _workspace_grid()}))


@pytest.fixture(scope="module")
def results():
    import swarm_b200
    swarm_b200._build.build()
    code = (f"import sys; sys.path[:0] = {[ROOT, os.path.dirname(__file__)]!r}; import test_abi_rejections as t; "
            "t._child_main()")
    child = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                           capture_output=True, text=True)
    assert child.returncode == 0, child.stderr
    return json.loads(child.stdout.strip().splitlines()[-1])


def test_every_malformed_call_is_refused_with_its_code_and_message(results):
    failures = []
    for name, _, code, text in _cases():
        rc, msg = results["calls"][name]
        if rc != code or text not in msg:
            failures.append(f"{name}: got ({rc}, {msg!r}), want ({code}, ...{text!r}...)")
    assert not failures, "\n".join(failures)


def test_table_covers_every_entry_point_that_takes_a_cfg_spec_ring_or_adam_hyper_parameters():
    src = open(__file__).read()
    for fn in ("reset_grid", "sim_step", "graph_build", "graph_build_radius", "gatq_forward", "gatq_forward_knn_large",
               "graph_build_radius_csr", "gatq_forward_large", "rollout_large", "rollout", "replay_push", "replay_gather",
               "dqn_grad", "adam_clip_step", "train_tick_grad", "train_tick_apply", "train_tick", "reset_random",
               "episode_end", "scenario_reward", "scenario_reward_large", "gatstack_forward", "gatstack_forward_large",
               "dqn_stack_grad", "adam_clip_stack_step", "rollout_stack", "rollout_stack_large", "train_tick_stack"):
        assert re.search(rf"\blib\.swarm_{fn}\b", src), fn


def test_workspace_bytes_over_a_grid_of_configs(results):
    assert results["workspace"] == WORKSPACE_BYTES


# "graph/N/k": swarm_rollout_large, swarm_rollout_stack, swarm_rollout_stack_large (no reward, Flocking, Cohesion),
# swarm_gatstack_large (3 x 8 spec), swarm_dqn (32 graphs), swarm_dqn_stack (3 x 8 spec, 32 graphs) and
# swarm_scenario_reward_large (Flocking, Cohesion) workspace bytes, num_envs = 3
WORKSPACE_BYTES = {
    "0/2/10": [536, 1078, 0, 0, 0, 768, 215296, 52992, 24, 0],
    "0/12/10": [656, 1348, 0, 0, 0, 2560, 215296, 52992, 144, 0],
    "0/128/10": [2048, 4480, 0, 0, 0, 24832, 215296, 52992, 1536, 0],
    "0/129/10": [2060, 101376, 101376, 103180, 101632, 25088, 0, 0, 1548, 0],
    "0/600/10": [7712, 468736, 468736, 476192, 468992, 115456, 0, 0, 7200, 0],
    "0/4096/10": [49664, 3195392, 3195392, 3244800, 3195648, 786688, 0, 0, 49152, 0],
    "1/2/5": [656, 1078, 0, 0, 0, 0, 0, 0, 24, 0],
    "1/2/10": [776, 1078, 0, 0, 0, 0, 0, 0, 24, 0],
    "1/2/64": [2072, 1078, 0, 0, 0, 0, 0, 0, 24, 0],
    "1/12/5": [1376, 1348, 0, 0, 0, 2920, 215296, 52992, 144, 0],
    "1/12/10": [2096, 1348, 0, 0, 0, 3280, 215296, 52992, 144, 0],
    "1/12/64": [9872, 1348, 0, 0, 0, 0, 0, 0, 144, 0],
    "1/128/5": [9728, 4480, 0, 0, 0, 28672, 0, 0, 1536, 0],
    "1/128/10": [17408, 4480, 0, 0, 0, 32512, 0, 0, 1536, 0],
    "1/128/64": [100352, 4480, 0, 0, 0, 73984, 0, 0, 1536, 0],
    "1/129/5": [9800, 112926, 112926, 114730, 113182, 0, 0, 0, 1548, 0],
    "1/129/10": [17540, 124476, 124476, 126280, 124732, 0, 0, 0, 1548, 0],
    "1/129/64": [101132, 249984, 249984, 251788, 250240, 0, 0, 0, 1548, 0],
    "1/600/5": [43712, 522576, 522576, 530032, 522832, 133456, 0, 0, 7200, 0],
    "1/600/10": [79712, 576672, 576672, 584128, 576928, 0, 0, 0, 7200, 0],
    "1/600/64": [468512, 1159936, 1159936, 1167392, 1160192, 0, 0, 0, 7200, 0],
    "1/4096/5": [295424, 3564032, 3564032, 3613440, 3564288, 909568, 0, 0, 49152, 0],
    "1/4096/10": [541184, 3932672, 3932672, 3982080, 3932928, 1032448, 0, 0, 49152, 0],
    "1/4096/64": [3195392, 7913984, 7913984, 7963392, 7914240, 2359552, 0, 0, 49152, 0],
    "2/2/10": [536, 1078, 0, 0, 0, 768, 215296, 52992, 24, 0],
    "2/12/10": [656, 1348, 0, 0, 0, 2560, 215296, 52992, 144, 0],
    "2/128/10": [2048, 4480, 0, 0, 0, 24832, 0, 52992, 1536, 0],
    "2/129/10": [2060, 101376, 101376, 103180, 101632, 25088, 0, 0, 1548, 0],
    "2/600/10": [7712, 468736, 468736, 476192, 468992, 115456, 0, 0, 7200, 0],
    "2/4096/10": [49664, 3195392, 3195392, 3244800, 3195648, 786688, 0, 0, 49152, 0],
}
