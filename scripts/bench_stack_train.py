"""Time one DQN training tick of a stacked GAT Q-network: the device-driven tick of
``DQNTrainer.train_model_stack_device`` (one swarm_train_tick_stack call = rollout tick, slot draw + gradient, reduce,
clip + Adam; `--ticks` ticks captured in a CUDA graph and replayed) against ``DQNTrainer.train_model_stepwise`` (about ten
launches per tick from Python: greedy forward, torch exploration draws, env.step, the scenario's reward, replay push,
gradient, clip + Adam) on the same env.  CUDA events, median over `--windows` windows; every timed tick updates (the ring
is filled beyond G first).  Writes JSON with the card name, power limit and SM clock read in the same run.

    python scripts/bench_stack_train.py --out profiles/r6_stack_train.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, sm, sm_max = [x.strip() for x in out.splitlines()[0].split(",")]
        return {"nvidia_smi_name": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": sm_max}
    except Exception:
        return {"power_limit": "unknown", "sm_clock": "unknown"}


def _flocking_sd(seed):
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    pre = f"{seed}/"
    return {k[len(pre):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(pre)}


def _trainer(sb, scen, B, capacity):
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    if scen == "flocking":
        env = sb.make_env(sb.FlockingScenario(), num_envs=B, device=dev, continuous_actions=False, max_steps=100,
                          dict_spaces=True, seed=0, n_agents=12)
        model = sb.StackedGCN.from_state_dict(_flocking_sd(0))
    else:
        env = sb.make_env(sb.CohesionScenario(), num_envs=B, device=dev, continuous_actions=False, max_steps=100,
                          dict_spaces=True, seed=0, n_agents=9)
        model = sb.StackedGCN(5, 8, 9, 3)
    return sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "bench", replay_capacity=capacity, model=model)


def _device_tick_ms(sb, scen, B, G, ticks, windows):
    """The tick train_model_stack_device replays: StackTrainTick on the trainer's buffers, `ticks` ticks per graph."""
    ops, L = sb.ops, sb._lib
    tr = _trainer(sb, scen, B, max(4 * G, 4 * B))
    env, world, dev = tr.env, tr.env.world, tr.env.device
    env.reset()
    reward = shaping = None
    if scen == "flocking":
        reward, shaping = env.scenario._spec(), env.scenario.shaping
    else:
        reward = ops.reward_spec(L.REWARD_COHESION, B, env.n_agents, agent_radius=world.cfg.agent_radius,
                                 sigma=env.scenario.sigma)
    cfg = ops.clone_config(tr.graph_cfg, num_envs=B)
    tt = ops.StackTrainTick(cfg, tr.stack_spec, tr.replay_buffer.ring, graphs_per_update=G, update_target_every=200,
                            rng_seed=0, sample_seed=0, reward=reward, shaping=shaping)
    tt.load_cursor(0, 0, 0.5)
    returns = torch.zeros(B, env.n_agents, device=dev)
    hits = torch.zeros(B, dtype=torch.int32, device=dev)

    def tick():
        tt.tick(tr.w, tr.w_target, tr.exp_avg, tr.exp_avg_sq, world.state, returns, hits)

    for _ in range((G + B - 1) // B + 2):           # eager: the ring holds >= G slots, kernel attributes set
        tick()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.graph(graph, stream=side):
        for _ in range(ticks):
            tick()
    graph.replay()
    torch.cuda.synchronize()
    times = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        graph.replay()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) / ticks)
    cur = tt.read_cursor()
    assert cur["updating"] == 1 and torch.isfinite(tr.w).all()
    return float(np.median(times)), cur


def _stepwise_tick_ms(sb, scen, B, G, ticks, windows):
    """train_model_stepwise, one episode of `ticks` ticks per window (its reset included), after a filling episode."""
    tr = _trainer(sb, scen, B, max(4 * G, 4 * B))
    tr.env.max_steps = ticks
    cfg = {"episodes": 1, "epsilon": 0.5, "epsilon_decay": 0.0, "min_epsilon": 0.05, "graphs_per_update": G,
           "update_target_every": 200}
    tr.train_model_stepwise(cfg)
    torch.cuda.synchronize()
    times = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        tr.train_model_stepwise(cfg)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) / ticks)
    return float(np.median(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--ticks", type=int, default=100)
    ap.add_argument("--windows", type=int, default=7)
    args = ap.parse_args()
    import swarm_b200 as sb
    rows = []
    cases = [("flocking", B, G) for B in (64, 4096) for G in (32, 4096)] + [("cohesion", B, 32) for B in (64, 4096)]
    for scen, B, G in cases:
        dev_ms, cur = _device_tick_ms(sb, scen, B, G, args.ticks, args.windows)
        step_ms = _stepwise_tick_ms(sb, scen, B, G, max(args.ticks // 4, 10), args.windows)
        shape = ({"network": "Flocking checkpoint: 3 GATConv layers, width 8, 7 inputs", "n_agents": 12, "graph": "complete"}
                 if scen == "flocking" else
                 {"network": "StackedGCN(5, 8, 9, 3): 3 GATConv layers, width 8, 5 inputs", "n_agents": 9,
                  "graph": "complete"})
        r = dict(scenario=scen, num_envs=B, graphs_per_update=G, **shape, device_tick_ms=dev_ms,
                 stepwise_tick_ms=step_ms, speedup=step_ms / dev_ms, ticks_per_graph=args.ticks,
                 opt_steps_after=cur["opt_step"])
        print(json.dumps(r), flush=True)
        rows.append(r)
    res = {"device": torch.cuda.get_device_name(0), **_gpu_info(),
           "method": "CUDA events, median of windows.  device: one replay of a CUDA graph of `ticks_per_graph` "
                     "swarm_train_tick_stack calls (the tick of DQNTrainer.train_model_stack_device), every tick an "
                     "update.  stepwise: one DQNTrainer.train_model_stepwise episode (env.reset included) per window.  "
                     "Both per tick, epsilon 0.5.", "cases": rows}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
