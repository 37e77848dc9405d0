"""The reference's OWN files, unmodified, on the CUDA product (SURVEY.md 8f rank 1: script-level drop-in).

`shim/` gives the module names `vmas` / `torch_geometric` to swarm_b200, `SWARM_DEVICE=cuda:0` serves the scripts'
hard-coded `device='cpu'` (train_gcn_dqn.py:262, tests/test_*.py:33) from the B200: tensors at the scripts' seams stay
host tensors, `env.step` is `swarm_sim_step`, `GATConv` is the CUDA layer (forward and backward).  The expected outputs
are what the SAME files produce on the CPU stand-ins of their dependencies (oracle/refstub; tests/golden/
make_reference_runs.py -> tests/golden/reference_runs.npz), which in turn reproduce the reference's shipped goldens
(tests/test_refstub.py).  The sources come from the git-ignored staging copy oracle/_ref (scripts/stage_reference.py).
"""
import os
import re

import numpy as np
import pytest
import torch

import refsrc
from helpers import npz

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(refsrc.reference_root() is None, reason="reference sources not staged")]

ENV = {"SWARM_DEVICE": "cuda:0"}


@pytest.mark.parametrize("exp,script,T", [("go_to", "tests/test_go_to_position.py", 50),
                                          ("obstacle_avoidance", "tests/test_obstacle_avoidance.py", 100)])
def test_reference_test_script_runs_unmodified(exp, script, T, tmp_path):
    """tests/test_go_to_position.py / test_obstacle_avoidance.py as __main__ (shipped constants: k = 10, agents 10 ...,
    seed 6967, 8 episodes): the CSV trees of its first two cases equal the ones the same script writes on the CPU
    stand-in."""
    wd = str(tmp_path)
    refsrc.write_models(wd)
    tree = os.path.join(wd, "data", "test_stats", exp, "seed_0")
    log = refsrc.run_reference_script("shim", script, wd, extra_env=ENV, timeout=900,
                                      stop_when=lambda _: os.path.exists(os.path.join(tree, "agents_12", "result.csv")))
    assert os.path.exists(os.path.join(tree, "agents_11", "result.csv")), log[-3000:]
    fix = npz("reference_runs.npz")
    exact = total = 0
    for n in (10, 11):
        got = refsrc.read_simulator_tree(os.path.join(tree, f"agents_{n}"))
        want = {k: fix[f"script/{exp}/agents_{n}/{k}"] for k in ("pos", "dist", "hits", "result")}
        assert got["pos"].shape == want["pos"].shape == (8, T, n, 2)
        # every episode starts from the reference's RNG stream (env seed -> reset draw -> GCN() constructor draws)
        assert (got["pos"][:, 0] == want["pos"][:, 0]).all(), "first tick differs: start centres / first actions"
        for e in range(8):
            total += 1
            same = bool((got["pos"][e] == want["pos"][e]).all())
            exact += int(same)
            if same:
                assert (got["hits"][e] == want["hits"][e]).all() and (got["dist"][e] == want["dist"][e]).all()
                assert np.allclose(got["result"][e], want["result"][e], rtol=1e-6)
    print(f"\n{script}: {exact}/{total} episodes bit-identical to the CPU stand-in run")
    assert exact >= EXPECT_SCRIPT[exp]


# measured on B200 (round 2); episodes that differ contain contact forces (log1p(exp(.)): SLEEF vs CUDA libm) or a
# greedy near-tie
EXPECT_SCRIPT = {"go_to": 0, "obstacle_avoidance": 0}


def test_reference_training_script_runs_unmodified(tmp_path):
    """src/training/train_gcn_dqn.py as __main__: its own DQNTrainer / GraphReplayBuffer / GCN classes, torch.optim.Adam
    and loss.backward() through the CUDA GATConv layer.  First two episodes of (seed 0, ObstacleAvoidance, 10 agents)
    against the CPU stand-in run: Python's `random` drives exploration and sampling identically, so the episode reward
    matches until a greedy near-tie, the loss to float32 accumulation accuracy."""
    wd = str(tmp_path)
    log = refsrc.run_reference_script("shim", "src/training/train_gcn_dqn.py", wd, extra_env=ENV, timeout=1500,
                                      stop_when=lambda s: len(re.findall(r"^Episode \d+, Loss", s, re.M)) >= 2)
    rows = re.findall(r"^Episode (\d+), Loss: ([-\d.e]+), Reward: ([-\d.e]+), Epsilon: ([-\d.e]+)", log, re.M)[:2]
    assert len(rows) == 2, log[-3000:]
    got = np.array([[float(v) for v in r] for r in rows])
    want = npz("reference_runs.npz")["train/ObstacleAvoidance/episodes"]
    print(f"\ntrain script: got {got.tolist()} want {want.tolist()}")
    assert "Device: cpu" in log and "Running seed 0 experiment ObstacleAvoidance" in log
    assert np.array_equal(got[:, [0, 3]], want[:, [0, 3]])                       # episode numbers, epsilon schedule
    assert abs(got[0, 2] - want[0, 2]) <= 1e-3 * abs(want[0, 2]), "episode-0 reward"
    assert abs(got[0, 1] - want[0, 1]) <= 1e-3 * abs(want[0, 1]), "episode-0 mean loss"
    assert abs(got[1, 1] - want[1, 1]) <= 5e-2 * abs(want[1, 1]), "episode-1 mean loss"


def _replay(ref, kind, n, monkeypatch):
    """The reference's scenario file on the shim's World (host-seam mode), replaying the fixture's seeds and actions."""
    import vmas
    monkeypatch.setenv("SWARM_DEVICE", "cuda:0")
    Scen = ref.flocking_scenario.FlockingScenario if kind == "flocking" else ref.cohesion_scenario.CohesionScenario
    seed = 100 + n
    env = vmas.make_env(Scen(), num_envs=1, device="cpu", continuous_actions=False, dict_spaces=True, wrapper=None,
                        max_steps=60 if n <= 12 else 30, seed=seed, n_agents=n)
    torch.manual_seed(seed + 1)
    env.reset()
    return env


@pytest.mark.parametrize("n", [2, 5, 7, 8, 9, 12, 40])
def test_reference_flocking_source_on_cuda_world_equals_kernels(n, monkeypatch):
    """flocking_scenario.py's reset_world_at / reward() torch code on the CUDA-stepped world == the fixture (same file on
    the CPU stand-in) == swarm_scenario_reward == the fused FLOCK rollout, bit for bit while no contact force has acted
    (afterwards positions agree to 1e-5 and the comparison of the three reward implementations continues on the SAME
    device state, still bit for bit)."""
    import swarm_b200 as sb
    from swarm_b200 import ops
    fix, pre = npz("reference_runs.npz"), f"flocking/n{n}/"
    dev = torch.device("cuda:0")
    with refsrc.reference_modules("shim") as ref:
        env = _replay(ref, "flocking", n, monkeypatch)
        world, agents = env.world, env.world.agents
        assert world.device.type == "cpu" and world.compute_device.type == "cuda" and not agents[0].state.pos.is_cuda
        pos0 = torch.cat([a.state.pos for a in agents]).numpy()
        assert np.array_equal(pos0, fix[pre + "pos0"])
        shp0 = np.stack([[float(a.previous_distance_to_goal), float(a.previous_distance_to_agents)] for a in agents])
        assert np.array_equal(shp0.astype(np.float32), fix[pre + "shaping0"])
        # the CUDA reward kernel's reset on the same state
        spec = ops.reward_spec(sb._lib.REWARD_FLOCKING, 1, n)
        shaping = torch.zeros(1, n, 2, device=dev)
        ops.scenario_reward(spec, world.state, shaping, reset=True)
        assert np.array_equal(shaping[0].cpu().numpy(), fix[pre + "shaping0"])
        # the fused rollout with the same action stream, from the same start
        actions = torch.from_numpy(fix[pre + "actions"].astype(np.int32))
        T = actions.shape[0]
        cfg = ops.make_config(sb._lib.SCENARIO_GOTO, 1, n)
        w0 = sb.pack_weights(__import__("helpers").load_params("go_to", 0), dev)
        fused = ops.rollout(cfg, w0, world.state.clone(), T, forced_actions=actions.view(T, 1, n).contiguous().to(dev),
                            trace=dict(state=True, rewards=True), flocking=spec, shaping=shaping.clone())
        touched = False
        for t in range(T):
            _, rewards, _, _ = env.step({f"agent{i}": actions[t, i:i + 1] for i in range(n)})
            pos = torch.cat([a.state.pos for a in agents]).numpy()
            d = np.linalg.norm(fix[pre + "pos"][t][:, None] - fix[pre + "pos"][t][None], axis=-1) + 9 * np.eye(n)
            r_ref = np.array([float(rewards[f"agent{i}"]) for i in range(n)], dtype=np.float32)
            r_kernel = ops.scenario_reward(spec, world.state, shaping)            # same device state, CUDA arithmetic
            assert np.all(r_ref == np.float32(r_kernel.item())), f"tick {t}: reference reward() vs swarm_scenario_reward"
            assert np.array_equal(fused["trace_state"][t, 0].cpu().numpy()[:, :2], pos), f"tick {t}: fused rollout state"
            assert np.all(np.float32(fused["trace_rewards"][t, 0, 0].item()) == r_ref), f"tick {t}: fused FLOCK reward"
            if not touched:
                assert np.array_equal(pos, fix[pre + "pos"][t]), f"tick {t}: contact-free positions must be bit-identical"
                assert np.array_equal(r_ref, fix[pre + "rewards"][t]), f"tick {t}: reward vs the CPU stand-in run"
            else:
                assert np.abs(pos - fix[pre + "pos"][t]).max() <= 1e-5
                assert np.allclose(r_ref, fix[pre + "rewards"][t], rtol=1e-4, atol=2e-3)
            touched |= bool(d.min() <= 0.1)                       # a contact force acts from the NEXT step on


@pytest.mark.parametrize("n", [2, 5, 9])
def test_reference_cohesion_source_on_cuda_world_equals_kernel(n, monkeypatch):
    """cohesion_scenario.py's reward() (incl. np.exp on a tensor, cohesion:80) on the CUDA-stepped world vs the fixture
    and vs swarm_scenario_reward on the same device state (expf: 1e-6 relative)."""
    import swarm_b200 as sb
    from swarm_b200 import ops
    fix, pre = npz("reference_runs.npz"), f"cohesion/n{n}/"
    with refsrc.reference_modules("shim") as ref:
        env = _replay(ref, "cohesion", n, monkeypatch)
        world, agents = env.world, env.world.agents
        assert np.array_equal(torch.cat([a.state.pos for a in agents]).numpy(), fix[pre + "pos0"])
        spec = ops.reward_spec(sb._lib.REWARD_COHESION, 1, n)
        actions = torch.from_numpy(fix[pre + "actions"].astype(np.int64))
        touched = False
        for t in range(actions.shape[0]):
            obs, rewards, _, _ = env.step({f"agent{i}": actions[t, i:i + 1] for i in range(n)})
            assert obs["agent0"].shape[-1] == 4
            pos = torch.cat([a.state.pos for a in agents]).numpy()
            r_ref = np.array([float(rewards[f"agent{i}"]) for i in range(n)], dtype=np.float32)
            r_kernel = ops.scenario_reward(spec, world.state)[0].cpu().numpy()
            assert np.allclose(r_kernel, r_ref, rtol=2e-6, atol=1e-7), f"tick {t}: swarm_scenario_reward vs reference reward()"
            if not touched:
                assert np.array_equal(pos, fix[pre + "pos"][t]) and np.array_equal(r_ref, fix[pre + "rewards"][t])
            else:
                assert np.abs(pos - fix[pre + "pos"][t]).max() <= 1e-5
            d = np.linalg.norm(fix[pre + "pos"][t][:, None] - fix[pre + "pos"][t][None], axis=-1) + 9 * np.eye(n)
            touched |= bool(d.min() <= 0.1)
