"""Time stacked GAT Q-networks on large swarms: ops.rollout_stack above 128 agents (per tick [topk table ->] the one-launch
large stacked forward -> the large world step) beside the one-layer ops.rollout_large on the same shape, and the generic
route it replaces (StackedGCN.forward over the generic layer kernels on a materialised edge list + sim_step per tick).

Workloads: ObstacleAvoidance at 1 024 envs x 1 024 agents (C4, centres as bench_c4.py, seed 0) and 256 envs x 4 096
agents; the Flocking checkpoint seed 0 (tests/golden/flocking_models.npz); kNN k = 10, radius 0.35, complete.  CUDA
events, median of several windows after a warm-up.  The generic route's complete graph materialises N (N - 1) + 1 edges
per env, so it runs on as many envs as keep the edge list at <= 64 M edges; rates are per agent-step either way.
Writes JSON with the card name, power limit and SM clock read in the same run.

    python scripts/bench_stack_large.py --out profiles/r5_stack_large.json
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


def _smi(fields):
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def _window_ms(fn, windows):
    times = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), [round(t, 4) for t in times]


def run_case(sb, graph, B, N, ticks, generic_ticks, windows):
    ops, L = sb.ops, sb._lib
    dev = torch.device("cuda:0")
    gm = {"complete": L.GRAPH_COMPLETE, "knn": L.GRAPH_KNN, "radius": L.GRAPH_RADIUS}[graph]
    cfg = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B, N, gm, 10, graph_radius=0.35)
    g = torch.Generator().manual_seed(0)
    centers = (torch.tensor([0.6, -0.6]) + 0.1 * torch.randn(B, 2, generator=g)).to(dev)
    s0 = ops.reset_grid(cfg, centers)
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    sd = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("0/")}
    model = sb.StackedGCN.from_state_dict(sd).to(dev).eval()
    spec = model.stack_spec()
    w = model.packed_stack_weights(dev)
    m = np.load(os.path.join(ROOT, "tests", "golden", "models.npz"))
    pre = "ObstacleAvoidance/0/"
    w1 = sb.pack_weights({k[len(pre):]: torch.from_numpy(m[k]) for k in m.files if k.startswith(pre)}, dev)
    res = {"graph": graph, "num_envs": B, "n_agents": N, "ticks": ticks}

    state = s0.clone()
    ops.rollout_stack(cfg, spec, w, state, 2)
    torch.cuda.synchronize()

    def fused():
        state.copy_(s0)
        ops.rollout_stack(cfg, spec, w, state, ticks)
    ms, all_ms = _window_ms(fused, windows)
    res["stack_ms_per_tick"] = ms / ticks
    res["stack_agent_steps_per_s"] = B * N * ticks / (ms * 1e-3)
    res["stack_windows_ms"] = all_ms

    ops.rollout_large(cfg, w1, state, 2)
    torch.cuda.synchronize()

    def one_layer():
        state.copy_(s0)
        ops.rollout_large(cfg, w1, state, ticks)
    ms, all_ms = _window_ms(one_layer, windows)
    res["gcn_ms_per_tick"] = ms / ticks
    res["gcn_agent_steps_per_s"] = B * N * ticks / (ms * 1e-3)

    # the generic route on Bg envs
    e_per_env = N * (N - 1) + 1 if graph == "complete" else 2 * 10 * N + 1 if graph == "knn" else 40 * N
    Bg = max(1, min(B, (64 << 20) // e_per_env))
    cfg_g = ops.clone_config(cfg, num_envs=Bg)
    sg0 = s0[:Bg].clone()
    ids = torch.arange(N, device=dev, dtype=torch.float32).view(1, N, 1).expand(Bg, N, 1)
    goal = torch.tensor([cfg.goal_x, cfg.goal_y], device=dev).view(1, 1, 2).expand(Bg, N, 2)
    offs = (torch.arange(Bg, device=dev, dtype=torch.int64) * N).view(Bg, 1, 1)
    sg = sg0.clone()

    def generic_tick():
        if graph == "radius":
            row_ptr, src = ops.graph_build_radius_csr(cfg_g, sg)
            dst = torch.repeat_interleave(torch.arange(Bg * N, device=dev), (row_ptr[1:] - row_ptr[:-1]).long())
            ei = torch.stack([src.long(), dst])
        else:
            edges, _ = ops.graph_build(cfg_g, sg)
            ei = (edges.long() + offs).permute(1, 0, 2).reshape(2, -1)
        x = torch.cat([sg, goal, ids], 2).reshape(Bg * N, 7)
        with torch.no_grad():
            act = torch.argmax(model(sb.Data(x=x, edge_index=ei)), dim=1).to(torch.int32).view(Bg, N)
        ops.sim_step(cfg_g, sg, act, state_out=sg, want_obs=False)

    generic_tick()
    torch.cuda.synchronize()

    def generic():
        sg.copy_(sg0)
        for _ in range(generic_ticks):
            generic_tick()
    ms, all_ms = _window_ms(generic, windows)
    res["generic_envs"] = Bg
    res["generic_ticks"] = generic_ticks
    res["generic_ms_per_tick"] = ms / generic_ticks
    res["generic_agent_steps_per_s"] = Bg * N * generic_ticks / (ms * 1e-3)
    res["stack_over_generic"] = res["stack_agent_steps_per_s"] / res["generic_agent_steps_per_s"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--ticks", type=int, default=20)
    ap.add_argument("--generic-ticks", type=int, default=3)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="tiny shapes (a check of the script itself)")
    args = ap.parse_args()
    import swarm_b200 as sb
    if not torch.cuda.is_available():
        raise SystemExit("bench_stack_large.py needs a CUDA device")
    shapes = [(8, 256), (2, 1024)] if args.small else [(1024, 1024), (256, 4096)]
    out = {"gpu": torch.cuda.get_device_name(0), "power_limit": _smi("power.limit"),
           "sm_clock": _smi("clocks.sm"), "max_sm_clock": _smi("clocks.max.sm"),
           "network": "Flocking checkpoint seed 0 (3 x GATConv 7/8 -> 8, tanh/relu/relu)",
           "one_layer_network": "ObstacleAvoidance seed 0 (GCN, 7 -> 32)", "cases": []}
    for B, N in shapes:
        for graph in ("knn", "radius", "complete"):
            r = run_case(sb, graph, B, N, args.ticks, args.generic_ticks, args.windows)
            print(json.dumps(r), flush=True)
            out["cases"].append(r)
    out["sm_clock_after"] = _smi("clocks.sm")
    text = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
