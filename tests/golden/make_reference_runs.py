"""Outputs of the reference's OWN Python files, run unmodified in this container on the CPU stand-ins of their two
dependencies (oracle/refstub: vmas / torch_geometric restated with the pinned oracle arithmetic).

    python tests/golden/make_reference_runs.py        ->  tests/golden/reference_runs.npz

Needs the reference sources (the copy build() stages into oracle/_ref).  What is recorded:

  flocking/n{N}/..., cohesion/n{N}/...
      FlockingScenario / CohesionScenario (src/scenarios/flocking_scenario.py, cohesion_scenario.py) stepped through
      vmas.make_env for T ticks with a seeded action stream that drives the agents together (contacts, the -1 collision
      term and the sigma branches of Cohesion are all exercised): start centre, actions, per-tick positions /
      velocities / the reward() value of every agent, and Flocking's shaping memory after reset and after every tick.
      This is the pin of oracle/scenario_rewards_oracle.py and of the CUDA reward kernels: the numbers come from the
      reference's reward() source, not from a restatement of it.
  script/{go_to,obstacle_avoidance}/agents_{n}/...
      tests/test_go_to_position.py / tests/test_obstacle_avoidance.py run as __main__ (shipped constants: kNN k = 10,
      agents 10 ..., seed 6967) until their first two (model, agents) cases have written their CSV trees.
  train/{experiment}/...
      src/training/train_gcn_dqn.py run as __main__ until seed 0 of its first experiment has printed two
      `Episode e, Loss: ..., Reward: ...` lines (shipped constants: 10 agents, 100-tick episodes).
"""
import os
import re
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import refsrc  # noqa: E402


def herding_actions(pos: torch.Tensor, gen: torch.Generator, p_random: float) -> torch.Tensor:
    """Flat 9-way actions that push every agent towards the swarm's centroid (u(1) = -1, u(2) = +1), a fraction
    replaced by uniform draws: squeezes the grid until contact forces and the collision terms fire."""
    c = pos.mean(dim=0, keepdim=True)
    d = c - pos
    ix = torch.where(d[:, 0].abs() < 0.02, 0, torch.where(d[:, 0] < 0, 1, 2))
    iy = torch.where(d[:, 1].abs() < 0.02, 0, torch.where(d[:, 1] < 0, 1, 2))
    a = ix * 3 + iy
    rnd = torch.randint(0, 9, a.shape, generator=gen)
    return torch.where(torch.rand(a.shape, generator=gen) < p_random, rnd, a)


def scenario_run(ref, vmas, kind: str, n: int, T: int, seed: int):
    Scen = ref.flocking_scenario.FlockingScenario if kind == "flocking" else ref.cohesion_scenario.CohesionScenario
    env = vmas.make_env(Scen(), num_envs=1, device="cpu", continuous_actions=False, dict_spaces=True, wrapper=None,
                        max_steps=T, seed=seed, n_agents=n)
    torch.manual_seed(seed + 1)
    env.reset()
    agents = env.world.agents
    out = {"pos0": torch.cat([a.state.pos for a in agents]).numpy().copy()}
    if kind == "flocking":
        out["shaping0"] = np.stack([[float(a.previous_distance_to_goal), float(a.previous_distance_to_agents)]
                                    for a in agents]).astype(np.float32)
    gen = torch.Generator().manual_seed(seed + 2)
    acts, poss, vels, rews, shp, obs_dim = [], [], [], [], [], None
    for t in range(T):
        pos = torch.cat([a.state.pos for a in agents])
        a = herding_actions(pos, gen, 0.3 if kind == "flocking" else 0.15)
        obs, rewards, done, _ = env.step({f"agent{i}": a[i:i + 1] for i in range(n)})
        obs_dim = obs["agent0"].shape[-1]
        acts.append(a.numpy())
        poss.append(torch.cat([ag.state.pos for ag in agents]).numpy().copy())
        vels.append(torch.cat([ag.state.vel for ag in agents]).numpy().copy())
        rews.append(np.array([float(torch.as_tensor(rewards[f"agent{i}"]).reshape(-1)[0]) for i in range(n)], dtype=np.float32))
        if kind == "flocking":
            shp.append(np.stack([[float(ag.previous_distance_to_goal), float(ag.previous_distance_to_agents)]
                                 for ag in agents]).astype(np.float32))
    out.update(actions=np.stack(acts).astype(np.int8), pos=np.stack(poss), vel=np.stack(vels), rewards=np.stack(rews),
               obs_dim=np.array(obs_dim))
    if kind == "flocking":
        out["shaping"] = np.stack(shp)
    return out


def main():
    torch.set_num_threads(1)
    out = {}
    with refsrc.reference_modules("refstub") as ref:
        import vmas
        for kind, sizes in (("flocking", (2, 5, 7, 8, 9, 12, 40)), ("cohesion", (2, 5, 9))):
            for n in sizes:
                run = scenario_run(ref, vmas, kind, n, T=60 if n <= 12 else 30, seed=100 + n)
                for k, v in run.items():
                    out[f"{kind}/n{n}/{k}"] = v
                r = run["rewards"]
                print(f"{kind} n={n}: reward range [{r.min():.3f}, {r.max():.3f}]", flush=True)

    for exp, script, T in (("go_to", "tests/test_go_to_position.py", 50),
                           ("obstacle_avoidance", "tests/test_obstacle_avoidance.py", 100)):
        with tempfile.TemporaryDirectory() as wd:
            refsrc.write_models(wd)
            tree = os.path.join(wd, "data", "test_stats", exp, "seed_0")
            refsrc.run_reference_script("refstub", script, wd,
                                        stop_when=lambda _: os.path.exists(os.path.join(tree, "agents_12", "result.csv")))
            for n in (10, 11):
                got = refsrc.read_simulator_tree(os.path.join(tree, f"agents_{n}"))
                assert got["pos"].shape == (8, T, n, 2), got["pos"].shape
                for k, v in got.items():
                    out[f"script/{exp}/agents_{n}/{k}"] = v
            print(f"script {exp}: agents_10 / agents_11 trees recorded", flush=True)

    with tempfile.TemporaryDirectory() as wd:
        log = refsrc.run_reference_script("refstub", "src/training/train_gcn_dqn.py", wd, timeout=1800,
                                          stop_when=lambda s: len(re.findall(r"^Episode \d+, Loss", s, re.M)) >= 2)
        rows = re.findall(r"^Episode (\d+), Loss: ([-\d.e]+), Reward: ([-\d.e]+), Epsilon: ([-\d.e]+)", log, re.M)[:2]
        first = re.search(r"Running seed (\d+) experiment (\w+)", log)
        assert len(rows) == 2 and first, log[-2000:]
        out[f"train/{first.group(2)}/episodes"] = np.array([[float(v) for v in r] for r in rows], dtype=np.float64)
        print(f"train {first.group(2)} seed {first.group(1)}: {rows}", flush=True)
    np.savez_compressed(os.path.join(HERE, "reference_runs.npz"), **out)


if __name__ == "__main__":
    main()
