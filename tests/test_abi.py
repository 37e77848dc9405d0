"""The C-ABI shared library: loads, exports every symbol include/swarm_b200.h declares, agrees with the
ctypes struct layouts, and validates arguments before touching a device (so these run without a GPU)."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "swarm_b200.h")


@pytest.fixture(scope="module")
def sb():
    import swarm_b200
    swarm_b200._build.build()
    return swarm_b200


def _declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(swarm_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(sb):
    names = _declared_functions()
    assert len(names) >= 15
    lib = C.CDLL(sb._build.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/swarm_b200.h but not exported"
    # and every declared function has a ctypes signature in the binding
    assert set(names) == set(sb._lib._SIGNATURES)


def test_only_c_abi_is_exported(sb):
    out = subprocess.run(["nm", "-D", "--defined-only", sb._build.LIB_PATH], capture_output=True, text=True).stdout
    exported = [l.split()[-1] for l in out.splitlines() if " T " in l]
    ours = [s for s in exported if s.startswith("swarm_")]
    assert sorted(ours) == _declared_functions()


def test_struct_layout_matches_header(sb, tmp_path):
    """sizeof / offsetof of the C structs, compiled with gcc from the header, equal the ctypes mirrors."""
    prog = tmp_path / "layout.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "swarm_b200.h"\nint main(){'
                    'printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(SwarmConfig), offsetof(SwarmConfig, num_envs),'
                    'offsetof(SwarmConfig, dt), offsetof(SwarmConfig, obstacle_weight), sizeof(SwarmTrace), sizeof(SwarmReplay),'
                    'sizeof(SwarmRolloutOptions), offsetof(SwarmRolloutOptions, replay), offsetof(SwarmRolloutOptions, env_offset));return 0;}')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    L = sb._lib
    exp = [C.sizeof(L.SwarmConfig), L.SwarmConfig.num_envs.offset, L.SwarmConfig.dt.offset,
           L.SwarmConfig.obstacle_weight.offset, C.sizeof(L.SwarmTrace), C.sizeof(L.SwarmReplay),
           C.sizeof(L.SwarmRolloutOptions), L.SwarmRolloutOptions.replay.offset, L.SwarmRolloutOptions.env_offset.offset]
    assert got == exp


def test_default_config_is_the_reference_world(sb):
    cfg = sb.ops.make_config(sb._lib.SCENARIO_OBSTACLE_AVOIDANCE, 3, 12)
    import numpy as np
    f = np.float32
    assert (cfg.num_envs, cfg.n_agents, cfg.knn_k) == (3, 12, 10)                    # simulator.py:19 ships k = 10
    assert (cfg.dt, cfg.drag, cfg.collision_force, cfg.contact_margin) == (f(0.1), f(0.25), f(100.0), f(1e-3))
    assert (cfg.agent_radius, cfg.landmark_radius) == (f(0.05), f(0.05))           # vmas default radius, not agent_radius=0.1
    assert (cfg.goal_x, cfg.goal_y, cfg.obstacle_x, cfg.obstacle_y) == (f(-0.8), f(0.8), f(-0.1), f(0.1))
    assert (cfg.hit_distance, cfg.penalty_distance, cfg.obstacle_weight, cfg.grid_spacing) == (f(0.2), f(1.0), f(2.5), 0.15)
    assert sb.ops.edges_per_env(cfg) == 12 * 11 + 1                                   # complete + (0,0), train:101-108
    cfg.graph_mode = sb._lib.GRAPH_KNN
    assert sb.ops.edges_per_env(cfg) == 2 * 10 * 12 + 1                               # simulator.py:15-24


def test_argument_validation_without_device(sb):
    lib = sb._lib.lib()
    cfg = sb.ops.make_config(sb._lib.SCENARIO_GOTO, 1, 5, sb._lib.GRAPH_KNN, 10)
    # k > n: torch.topk's error in the reference (simulator.py:19 with n_agents < 10)
    assert lib.swarm_graph_build(C.byref(cfg), 8, 8, None, None) == -1
    assert b"selected index k out of range" in lib.swarm_last_error()
    cfg.knn_k = 5
    assert lib.swarm_graph_build(C.byref(cfg), None, None, None, None) == -1
    cfg.n_agents = 5000
    assert lib.swarm_sim_step(C.byref(cfg), 8, 8, 8, None, None, None, None, None, None) == -2
    assert b"n_agents" in lib.swarm_last_error()
    cfg.n_agents = 500                       # large swarms: fused kernels refuse, kNN needs torch's partial_sort branch
    assert lib.swarm_rollout(C.byref(cfg), 8, 8, 1, None, None, None, None, None) == -2
    cfg.knn_k = 10
    assert lib.swarm_graph_build(C.byref(cfg), 8, 8, None, None) == -2 and b"partial_sort" in lib.swarm_last_error()
    cfg.n_agents, cfg.scenario = 5, 7
    assert lib.swarm_reset_grid(C.byref(cfg), 8, 8, None) == -1
    assert lib.swarm_adam_clip_step(8, 8, 8, 8, 0, 1e-3, 0.9, 0.999, 1e-8, 1.0, None, None, None) == -1   # step is 1-based
    assert lib.swarm_adam_clip_step(8, 8, 8, 8, 1, 1e-3, 1.5, 0.999, 1e-8, 1.0, None, None, None) == -1   # beta1 out of range
    assert lib.swarm_csr_workspace_bytes(10, 100) > 0 and lib.swarm_gatq_workspace_bytes(10) >= 10 * 36 * 4


def test_no_cpu_fallback(sb):
    import torch
    with pytest.raises(sb.SwarmError, match="CUDA"):
        sb.make_env(sb.GoToPositionScenario(), num_envs=1, device="cpu", continuous_actions=False, max_steps=5,
                    dict_spaces=True, seed=0, n_agents=5)
    with pytest.raises(sb.SwarmError):
        sb.ops.reset_grid(sb.ops.make_config(0, 2, 5), torch.zeros(2, 2))
    model = sb.GCN(7, 32, 9)
    with pytest.raises(sb.SwarmError, match="CUDA"):
        model(sb.Data(x=torch.zeros(5, 7), edge_index=torch.zeros(2, 3, dtype=torch.long)))
    # the oracle is test infrastructure: nothing in the product package imports it
    pkg = os.path.join(ROOT, "experiments-2025-acsos-marl-for-swarming-behaviors_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            assert "oracle" not in open(os.path.join(pkg, f)).read(), f"{f} mentions the oracle"


def test_training_struct_layouts_match_header(sb, tmp_path):
    """The device-driven training structs (SwarmTrainCtl is read and written by kernels AND by torch views in
    ops.TrainTick, so its byte layout is part of the contract)."""
    fields = [("SwarmTrainCtl", ["tick", "ring_cursor", "ring_size", "opt_step", "epsilon", "updating", "episode"]),
              ("SwarmTrainHyper", ["lr", "max_norm", "rng_seed", "env_offset", "graphs_per_update", "gamma", "loss_scale"]),
              ("SwarmResetSpec", ["base_x", "std_y", "seed", "env_offset", "shared_center"]),
              ("SwarmPeerExchange", ["data", "world_size", "rank"])]
    body = "".join(f'printf("%zu ", sizeof({s}));' + "".join(f'printf("%zu ", offsetof({s}, {f}));' for f in fs)
                   for s, fs in fields)
    prog = tmp_path / "layout2.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "swarm_b200.h"\nint main(){' + body + 'return 0;}')
    exe = tmp_path / "layout2"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    L = sb._lib
    exp = []
    for s, fs in fields:
        cls = getattr(L, s)
        exp.append(C.sizeof(cls))
        exp += [getattr(cls, f).offset for f in fs]
    assert got == exp
    assert C.sizeof(L.SwarmTrainCtl) == 48 and L.SwarmTrainCtl.epsilon.offset == 32 and L.SwarmTrainCtl.updating.offset == 36
    assert sb.ops.TrainTick.CTL_WORDS * 8 == C.sizeof(L.SwarmTrainCtl)


def test_training_argument_validation_without_device(sb):
    lib, L = sb._lib.lib(), sb._lib
    cfg = sb.ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, 64, 12)
    h = L.SwarmTrainHyper()
    h.lr, h.beta1, h.beta2, h.eps, h.max_norm = 1e-3, 0.9, 0.999, 1e-8, 1.0
    h.graphs_per_update, h.update_target_every, h.gamma, h.loss_scale = 32, 200, 0.99, 1.0
    ring = L.SwarmReplay(8, 8, 8, 8, 1000)
    args = lambda: (C.byref(cfg), C.byref(h), 8, 8, 8, 8, None, None, C.byref(ring), None, 8, 8, 8, 1 << 30, None)
    h.graphs_per_update = 0
    assert lib.swarm_train_tick_grad(*args()) == -1 and b"graphs_per_update" in lib.swarm_last_error()
    h.graphs_per_update, h.update_target_every = 32, 0
    assert lib.swarm_train_tick_grad(*args()) == -1 and b"update_target_every" in lib.swarm_last_error()
    h.update_target_every, h.beta2 = 200, 1.0
    assert lib.swarm_train_tick_grad(*args()) == -1 and b"Adam" in lib.swarm_last_error()
    h.beta2 = 0.999
    ring.capacity = 10                                                 # smaller than one tick's push
    assert lib.swarm_train_tick_grad(*args()) == -1 and b"capacity" in lib.swarm_last_error()
    ring.capacity = 1000
    assert lib.swarm_train_tick_grad(C.byref(cfg), C.byref(h), 8, 8, 8, 8, None, None, C.byref(ring), None, 8, 8, 8, 16,
                                     None) == -1 and b"workspace" in lib.swarm_last_error()
    # apply: ring capacity, peer exchange sanity
    assert lib.swarm_train_tick_apply(C.byref(cfg), C.byref(h), 8, 8, 8, 8, 8, 8, 10, None, None) == -1
    px = L.SwarmPeerExchange()
    px.world_size, px.rank = 2, 5
    assert lib.swarm_train_tick_apply(C.byref(cfg), C.byref(h), 8, 8, 8, 8, 8, 8, 1000, C.byref(px), None) == -1
    assert b"peer exchange" in lib.swarm_last_error()
    px.rank = 1                                                        # NULL peer buffers
    assert lib.swarm_train_tick_apply(C.byref(cfg), C.byref(h), 8, 8, 8, 8, 8, 8, 1000, C.byref(px), None) == -1
    # the one-call tick: both phases' checks
    one = lambda peers: lib.swarm_train_tick(C.byref(cfg), C.byref(h), 8, 8, 8, 8, 8, 8, None, None, C.byref(ring), None, 8, 8,
                                             1 << 30, peers, None)
    assert one(C.byref(px)) == -1 and b"peer exchange" in lib.swarm_last_error()
    h.graphs_per_update = 0
    assert one(None) == -1 and b"graphs_per_update" in lib.swarm_last_error()
    h.graphs_per_update = 32
    ring.capacity = 10
    assert one(None) == -1 and b"capacity" in lib.swarm_last_error()
    ring.capacity = 1000
    assert lib.swarm_train_tick(C.byref(cfg), C.byref(h), 8, 8, 8, 8, 8, 8, None, None, C.byref(ring), None, 8, 8, 16, None,
                                None) == -1 and b"workspace" in lib.swarm_last_error()
    # reset / episode end
    sp = sb.ops.reset_spec(L.SCENARIO_GOTO)
    assert (sp.base_x, sp.base_y, sp.mean_x, sp.mean_y) == (1.5, -1.5, pytest.approx(-0.6), pytest.approx(0.6))   # go_to:84-88
    sp.std_x = -1.0
    assert lib.swarm_reset_random(C.byref(cfg), C.byref(sp), None, 0, None, 8, None) == -1
    sp.std_x = 0.4
    assert lib.swarm_reset_random(C.byref(cfg), C.byref(sp), None, -1, None, 8, None) == -1
    assert lib.swarm_episode_end(C.byref(cfg), None, 8, None, None, None, 0, 0.9, 0.01, 0.05, None) == -1
    assert lib.swarm_episode_end(C.byref(cfg), 8, 8, None, None, 8, 0, 0.9, 0.01, 0.05, None) == -1     # stats without rows


def _largest_dqn_agents():
    """Largest n_agents that swarm_dqn_workspace_bytes(cfg, 32) accepts: complete, radius, kNN k = 5, kNN k = 10."""
    import swarm_b200 as sb
    lib, L = sb._lib.lib(), sb._lib
    out = []
    for graph, k in ((L.GRAPH_COMPLETE, 1), (L.GRAPH_RADIUS, 1), (L.GRAPH_KNN, 5), (L.GRAPH_KNN, 10)):
        ok = [n for n in range(k, 129)
              if lib.swarm_dqn_workspace_bytes(C.byref(sb.ops.make_config(L.SCENARIO_GOTO, 1, n, graph, k)), 32) > 0]
        out.append(max(ok))
    return out


def test_dqn_accepts_the_same_swarm_sizes_with_and_without_swarm_tc(sb):
    # the DQN gradient has one kernel: SWARM_TC=0 selects the bit-faithful forward only and leaves these limits alone
    # (checked in a child process started with the variable set, so no cached read of the environment can hide it)
    expected = [128, 120, 81, 79]
    assert _largest_dqn_agents() == expected
    code = f"import sys; sys.path[:0] = {[ROOT, os.path.dirname(__file__)]!r}; import test_abi; print(test_abi._largest_dqn_agents())"
    child = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, SWARM_TC="0"), capture_output=True, text=True,
                           check=True)
    assert child.stdout.strip().splitlines()[-1] == str(expected)


def test_reward_spec_layout_defaults_and_validation(sb, tmp_path):
    """SwarmRewardSpec (Flocking / Cohesion rewards): byte layout against the header, reference constants as defaults
    (flocking:10-21,96,142; cohesion:23) and argument checks that need no device."""
    fs = ["kind", "num_envs", "n_agents", "reset", "env_index", "goal_x", "goal_radius", "agent_radius", "pos_shaping",
          "dist_shaping", "desired_distance", "min_collision_distance", "collision_reward", "on_goal_bonus", "sigma"]
    body = 'printf("%zu ", sizeof(SwarmRewardSpec));' + "".join(f'printf("%zu ", offsetof(SwarmRewardSpec, {f}));' for f in fs)
    prog = tmp_path / "layout3.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "swarm_b200.h"\nint main(){' + body + 'return 0;}')
    exe = tmp_path / "layout3"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    L, lib = sb._lib, sb._lib.lib()
    assert got == [C.sizeof(L.SwarmRewardSpec)] + [getattr(L.SwarmRewardSpec, f).offset for f in fs]

    sp = sb.ops.reward_spec(L.REWARD_FLOCKING, 16, 5)
    assert (sp.kind, sp.num_envs, sp.n_agents, sp.reset, sp.env_index) == (0, 16, 5, 0, -1)
    assert (sp.goal_x, sp.goal_y) == (pytest.approx(-0.8), pytest.approx(0.8))
    assert (sp.pos_shaping, sp.dist_shaping, sp.on_goal_bonus, sp.collision_reward) == (10.0, 10.0, 50.0, -1.0)
    assert sp.desired_distance == pytest.approx(0.15) and sp.min_collision_distance == pytest.approx(0.005)
    assert sp.goal_radius == pytest.approx(0.05) and sp.agent_radius == pytest.approx(0.05) and sp.sigma == pytest.approx(0.15)
    with pytest.raises(TypeError):
        sb.ops.reward_spec(L.REWARD_FLOCKING, 16, 5, no_such_field=1.0)

    call = lambda s, shaping=8, reward=8: lib.swarm_scenario_reward(C.byref(s), 8, shaping, reward, None, None)
    assert lib.swarm_scenario_reward(None, 8, 8, 8, None, None) == -1
    assert call(sp, shaping=None) == -1 and b"shaping" in lib.swarm_last_error()
    assert call(sp, reward=None) == -1
    sp.reset = 1
    sp.n_agents = 1
    assert call(sp) == -1 and b"two agents" in lib.swarm_last_error()
    sp.n_agents = 129
    assert call(sp) == -2                                             # SWARM_ERR_UNSUPPORTED
    sp.n_agents, sp.env_index = 5, 16
    assert call(sp) == -1 and b"env_index" in lib.swarm_last_error()
    sp.env_index, sp.kind = -1, 7
    assert call(sp) == -1
    co = sb.ops.reward_spec(L.REWARD_COHESION, 16, 9)
    co.reset = 1
    assert call(co, shaping=None) == -1 and b"Cohesion" in lib.swarm_last_error()
    co.reset, co.sigma = 0, 0.0
    assert call(co, shaping=None) == -1 and b"sigma" in lib.swarm_last_error()
    co.sigma, co.num_envs, co.n_agents = 0.15, 1 << 28, 12
    assert call(co, shaping=None) == -2                               # beyond the kernel's 32-bit row index
    co.num_envs = 0
    assert call(co, shaping=None, reward=None) == 0                   # nothing to do


def test_gat_layer_argument_validation_without_device(sb):
    lib = sb._lib.lib()
    assert lib.swarm_gat_layer_workspace_bytes(100, 1000, 7, 8, 0) > 0
    assert lib.swarm_gat_layer_workspace_bytes(100, 1000, 7, 8, 1) > lib.swarm_gat_layer_workspace_bytes(100, 1000, 7, 8, 0)
    assert lib.swarm_gat_layer_workspace_bytes(100, 1000, 65, 8, 0) == -1 and b"<= 64" in lib.swarm_last_error()
    assert lib.swarm_gat_layer_workspace_bytes(100, 1000, 7, 0, 0) == -1
    fwd = lambda n, ci, co, w=8, ws=8, wb=1 << 30: lib.swarm_gat_layer_forward(n, ci, co, w, 8, 8, 8, 8, 8, 8, 8, ws, wb, None)
    assert fwd(10, 7, 65) == -2
    assert fwd(10, 0, 8) == -1
    assert fwd(10, 7, 8, w=None) == -1 and b"NULL" in lib.swarm_last_error()
    assert fwd(10, 7, 8, wb=16) == -1 and b"workspace" in lib.swarm_last_error()
    assert fwd(0, 7, 8, w=None) == 0                                   # nothing to do
    bwd = lambda n, E, src=8, gx=None, wb=1 << 30: lib.swarm_gat_layer_backward(
        n, E, 7, 8, 8, 8, 8, 8, 8, src, 8, 8, 8, 8, 8, 8, 8, 8, 8, gx, 8, wb, None)
    assert bwd(0, 0) == -1
    assert bwd(10, 5, src=None) == -1 and b"edge" in lib.swarm_last_error()
    assert bwd(10, 5, wb=64) == -1 and b"workspace" in lib.swarm_last_error()
    assert bwd(10, 1 << 31) == -2


def test_flocking_option_of_the_fused_tick_is_validated(sb):
    """SwarmRolloutOptions.flocking / SwarmTrainHyper.flocking: argument errors are reported before any launch."""
    lib, L = sb._lib.lib(), sb._lib
    cfg = sb.ops.make_config(L.SCENARIO_GOTO, 16, 5)
    spec = sb.ops.reward_spec(L.REWARD_FLOCKING, 16, 5)
    opts = L.SwarmRolloutOptions()
    opts.flocking = C.addressof(spec)
    roll = lambda c: lib.swarm_rollout(C.byref(c), 8, 8, 1, C.byref(opts), None, None, None, None)
    assert roll(cfg) == -1 and b"shaping" in lib.swarm_last_error()
    opts.flocking_shaping = 8
    oa = sb.ops.clone_config(cfg, scenario=L.SCENARIO_OBSTACLE_AVOIDANCE)
    assert roll(oa) == -1 and b"GoTo world" in lib.swarm_last_error()
    one = sb.ops.clone_config(cfg, n_agents=1)
    assert roll(one) == -1 and b"two agents" in lib.swarm_last_error()
    spec.kind = L.REWARD_COHESION
    assert roll(cfg) == -1 and b"Flocking reward spec" in lib.swarm_last_error()
    assert L.SwarmRolloutOptions.flocking.offset + 32 == C.sizeof(L.SwarmRolloutOptions)     # + knn_memo, knn_memo_entries
    opts2 = L.SwarmRolloutOptions()
    opts2.knn_memo, opts2.knn_memo_entries = 8, 1000                                        # not a power of two
    knn = sb.ops.make_config(L.SCENARIO_GOTO, 16, 5, L.GRAPH_KNN, 3)
    assert lib.swarm_rollout(C.byref(knn), 8, 8, 1, C.byref(opts2), None, None, None, None) == -1
    assert b"power of two" in lib.swarm_last_error()
    assert L.SwarmTrainHyper.flocking.offset + 16 == C.sizeof(L.SwarmTrainHyper)


def test_stack_spec_layout_weight_count_and_validation(sb, tmp_path):
    """SwarmStackSpec (multi-layer GAT Q-networks): byte layout against the header, the packed weight count against the
    checkpoints the reference ships for Flocking (conv1 7 -> 8, conv2 / conv3 8 -> 8, lin1 8 -> 8, lin2 8 -> 9), and the
    argument errors of the stack / large-swarm entry points, all without a device."""
    import numpy as np
    import torch
    L, lib = sb._lib, sb._lib.lib()
    src = tmp_path / "s.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "swarm_b200.h"\nint main(){printf("%zu %zu %zu\\n", '
                   'sizeof(SwarmStackSpec), offsetof(SwarmStackSpec, activation), offsetof(SwarmStackSpec, in_features));return 0;}')
    exe = tmp_path / "s"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(L.SwarmStackSpec), L.SwarmStackSpec.activation.offset, L.SwarmStackSpec.in_features.offset]
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    sd = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("0/")}
    spec = sb.ops.stack_spec(3, 8, 7)
    assert int(lib.swarm_stack_weight_count(C.byref(spec))) == sum(v.numel() for v in sd.values()) == 409
    assert list(spec.activation)[:3] == [L.ACT_TANH, L.ACT_RELU, L.ACT_RELU]
    packed = sb.ops.pack_stack_weights(sd, spec, "cpu")
    assert packed.numel() == 409 and torch.equal(packed[:8], sd["conv1.att_src"].reshape(-1))
    assert torch.equal(packed[-9:], sd["lin2.bias"])
    model = sb.StackedGCN.from_state_dict(sd)
    assert model.n_layers == 3 and model.stack_spec().hidden == 8 and model.stack_spec().in_features == 7
    with pytest.raises(ValueError, match="expected"):
        sb.ops.pack_stack_weights(sd, sb.ops.stack_spec(3, 8, 5), "cpu")
    bad = sb.ops.stack_spec(3, 8, 7)
    bad.n_layers = 5
    assert int(lib.swarm_stack_weight_count(C.byref(bad))) == 0
    cfg = sb.ops.make_config(L.SCENARIO_GOTO, 4, 12, L.GRAPH_COMPLETE)
    assert lib.swarm_gatstack_forward(C.byref(cfg), C.byref(bad), 8, 8, 8, None, None) == -1
    assert b"n_layers" in lib.swarm_last_error()
    assert lib.swarm_gatstack_forward(C.byref(cfg), C.byref(spec), 8, 8, None, None, None) == -1
    assert b"no output" in lib.swarm_last_error()
    knn20 = sb.ops.make_config(L.SCENARIO_GOTO, 4, 20, L.GRAPH_KNN, 5)
    assert lib.swarm_gatstack_forward(C.byref(knn20), C.byref(spec), 8, 8, 8, None, None) == -2
    assert lib.swarm_rollout_stack(C.byref(cfg), C.byref(spec), 8, 8, 1, None, None, None, None, 8, 0, None) == -1
    assert b"workspace too small" in lib.swarm_last_error()
    # large-swarm entry points
    rad = sb.ops.make_config(L.SCENARIO_GOTO, 2, 1024, L.GRAPH_RADIUS, graph_radius=0.35)
    assert lib.swarm_graph_build_radius_csr(C.byref(rad), 8, None, None, None, None) == -1
    assert b"count pass" in lib.swarm_last_error()
    assert lib.swarm_graph_build_radius_csr(C.byref(rad), 8, 8, 8, 8, None) == -1
    assert lib.swarm_graph_build_radius_csr(C.byref(cfg), 8, 8, None, None, None) == -1 and b"SWARM_GRAPH_RADIUS" in lib.swarm_last_error()
    knn = sb.ops.make_config(L.SCENARIO_GOTO, 2, 1024, L.GRAPH_KNN, 10)
    assert lib.swarm_gatq_forward_large(C.byref(knn), 8, 8, 8, None, None) == -1 and b"knn_large" in lib.swarm_last_error()
    assert lib.swarm_gatq_forward_large(C.byref(rad), 8, 8, None, None, None) == -1 and b"no output" in lib.swarm_last_error()
    assert int(lib.swarm_rollout_large_workspace_bytes(C.byref(rad))) == 2 * 1024 * 4 + 512
    assert int(lib.swarm_rollout_large_workspace_bytes(C.byref(knn))) == 2 * 1024 * 10 * 4 + 2 * 1024 * 4 + 512
    big = sb.ops.make_config(L.SCENARIO_GOTO, 1, 5000, L.GRAPH_RADIUS, graph_radius=0.35)
    assert lib.swarm_gatq_forward_large(C.byref(big), 8, 8, 8, None, None) == -2
