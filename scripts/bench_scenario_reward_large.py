"""Time the large-swarm Flocking and Cohesion rewards: swarm_scenario_reward_large per tick, and the
swarm_rollout_stack_large tick with the Flocking reward against the same tick without a reward.

Workloads: 1 024 envs x 1 024 agents and 256 envs x 4 096 agents, agents on the start grid around random centres plus a
0.02 jitter (seed 0); the rollout runs the Flocking checkpoint seed 0 (tests/golden/flocking_models.npz) on the kNN
(k = 10), radius (0.35) and complete graphs.  CUDA events, median of several windows after a warm-up; the reward calls go
straight to the C entry point with preallocated buffers, so nothing but the two reward kernels is timed.  Flocking's
reward is all-pairs by definition: N (N - 1) exact square roots per env and tick, reported as pairs / s.  Writes JSON
with the card name, power limit and SM clock read in the same run.

    python scripts/bench_scenario_reward_large.py --out profiles/r7_scenario_reward_large.json
"""
import argparse
import ctypes as C
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


def _state(sb, B, N, dev):
    ops, L = sb.ops, sb._lib
    g = torch.Generator().manual_seed(0)
    centers = torch.tensor([-1.0, 1.0]) + torch.tensor([-0.6, 0.6]) + 0.4 * torch.randn(B, 2, generator=g)
    s = ops.reset_grid(ops.make_config(L.SCENARIO_GOTO, B, N), centers.to(dev))
    s[..., 0:2] += 0.02 * torch.randn(B, N, 2, generator=g).to(dev)
    return s


def reward_case(sb, kind, B, N, calls, windows):
    ops, L = sb.ops, sb._lib
    lib = L.lib()
    dev = torch.device("cuda:0")
    state = _state(sb, B, N, dev)
    flock = kind == "flocking"
    sp = ops.reward_spec(L.REWARD_FLOCKING if flock else L.REWARD_COHESION, B, N)
    shaping = torch.zeros(B, N, 2, device=dev)
    reward = torch.zeros(B if flock else B * N, device=dev)
    wb = int(lib.swarm_scenario_reward_large_workspace_bytes(C.byref(sp)))
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    if flock:
        ops.scenario_reward_large(sp, state, shaping, reset=True)

    def run():
        for _ in range(calls):
            rc = lib.swarm_scenario_reward_large(C.byref(sp), state.data_ptr(), shaping.data_ptr() if flock else None,
                                                 reward.data_ptr(), None, ws.data_ptr(), wb, stream)
            assert rc == 0, lib.swarm_last_error()

    run()
    torch.cuda.synchronize()
    ms, all_ms = _window_ms(run, windows)
    per = ms / calls
    pairs = B * N * (N - 1)
    return {"reward": kind, "num_envs": B, "n_agents": N, "ms_per_tick": round(per, 4),
            "pairs_per_s": float(f"{pairs / (per * 1e-3):.4g}"), "calls_per_window": calls, "window_ms": all_ms}


def rollout_case(sb, graph, B, N, ticks, windows):
    ops, L = sb.ops, sb._lib
    dev = torch.device("cuda:0")
    gm = {"complete": L.GRAPH_COMPLETE, "knn": L.GRAPH_KNN, "radius": L.GRAPH_RADIUS}[graph]
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N, gm, 10, graph_radius=0.35)
    s0 = _state(sb, B, N, dev)
    z = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    sd = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("0/")}
    model = sb.StackedGCN.from_state_dict(sd).to(dev).eval()
    spec = model.stack_spec()
    w = model.packed_stack_weights(dev)
    rs = ops.reward_spec(L.REWARD_FLOCKING, B, N)
    sh0 = torch.zeros(B, N, 2, device=dev)
    ops.scenario_reward_large(rs, s0, sh0, reset=True)
    state, shaping = s0.clone(), sh0.clone()
    returns = torch.zeros(B, N, device=dev)
    hits = torch.zeros(B, dtype=torch.int32, device=dev)
    out = {"graph": graph, "num_envs": B, "n_agents": N, "ticks_per_window": ticks}
    for label, reward in (("with_flocking_reward", rs), ("without_reward", None)):
        def run():
            ops.rollout_stack_large(cfg, spec, w, state, ticks, reward=reward, shaping=shaping if reward else None,
                                    returns=returns, hits=hits)
        state.copy_(s0); shaping.copy_(sh0)
        run()
        torch.cuda.synchronize()
        state.copy_(s0); shaping.copy_(sh0)
        ms, all_ms = _window_ms(run, windows)
        out[label] = {"ms_per_tick": round(ms / ticks, 4), "window_ms": all_ms}
    out["reward_share_of_tick"] = round(1.0 - out["without_reward"]["ms_per_tick"] / out["with_flocking_reward"]["ms_per_tick"], 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--quick", action="store_true", help="small shapes (a functional check of this script)")
    args = ap.parse_args()
    import swarm_b200 as sb
    shapes = [(1024, 1024), (256, 4096)] if not args.quick else [(4, 256)]
    res = {"device": torch.cuda.get_device_name(0), "power_limit_and_max_sm_clock": _smi("power.limit,clocks.max.sm"),
           "sm_clock_during_run": None, "reward": [], "rollout_tick": []}
    for B, N in shapes:
        for kind in ("flocking", "cohesion"):
            r = reward_case(sb, kind, B, N, calls=10 if not args.quick else 2, windows=args.windows)
            res["reward"].append(r)
            print(json.dumps(r), flush=True)
        for graph in ("knn", "radius", "complete"):
            r = rollout_case(sb, graph, B, N, ticks=5 if not args.quick else 2, windows=args.windows)
            res["rollout_tick"].append(r)
            print(json.dumps(r), flush=True)
    res["sm_clock_during_run"] = _smi("clocks.sm")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_and_max_sm_clock", "sm_clock_during_run")}))


if __name__ == "__main__":
    main()
