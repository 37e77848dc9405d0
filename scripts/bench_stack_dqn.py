"""Time one DQN update of a stacked GAT Q-network: the fused path (swarm_dqn_stack_grad: gradient kernel + reduce, then
swarm_adam_clip_stack_step) against the autograd path on the same batch (StackedGCN.forward on a Batch through the
generic layer kernels, .backward(), torch's clip_grad_norm_ + Adam).  CUDA events, median over several windows of
`--iters` updates after warm-up.  Writes JSON with the card name and power limit.

    python scripts/bench_stack_dqn.py --out profiles/r4_stack_dqn.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def _window_ms(fn, iters, windows):
    times = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) / iters)
    return float(np.median(times))


def run_case(sb, layers, hidden, N, mode, k, G, iters, windows):
    from oracle import batched_oracle as bo
    ops, L = sb.ops, sb._lib
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(0)
    sd = {}
    for l in range(1, layers + 1):
        cin = 7 if l == 1 else hidden
        sd[f"conv{l}.att_src"] = 0.5 * torch.randn(1, 1, hidden, generator=g)
        sd[f"conv{l}.att_dst"] = 0.5 * torch.randn(1, 1, hidden, generator=g)
        sd[f"conv{l}.bias"] = 0.1 * torch.randn(hidden, generator=g)
        sd[f"conv{l}.lin.weight"] = torch.randn(hidden, cin, generator=g) / cin ** 0.5
    sd["lin1.weight"] = torch.randn(hidden, hidden, generator=g) / hidden ** 0.5
    sd["lin1.bias"] = 0.1 * torch.randn(hidden, generator=g)
    sd["lin2.weight"] = torch.randn(9, hidden, generator=g) / hidden ** 0.5
    sd["lin2.bias"] = 0.1 * torch.randn(9, generator=g)
    gm = L.GRAPH_KNN if mode == "knn" else L.GRAPH_COMPLETE
    cfg = ops.make_config(L.SCENARIO_GOTO, G, N, gm, max(k, 1))
    pos = 0.5 * torch.randn(G, N, 2, generator=g)
    vel = 0.3 * torch.randn(G, N, 2, generator=g)
    pos2 = pos + 0.1 * vel
    actions = torch.randint(0, 9, (G, N), generator=g)
    rewards = torch.randn(G, N, generator=g)
    ring = ops.ReplayRing(G, N, dev)
    ops.replay_push(cfg, ring, torch.cat([pos, vel], 2).contiguous().to(dev), actions.to(torch.int32).to(dev),
                    rewards.contiguous().to(dev), torch.cat([pos2, vel], 2).contiguous().to(dev))
    spec = ops.stack_spec(layers, hidden, 7)
    w = ops.pack_stack_weights(sd, spec, dev)
    wt, m, v = w.clone(), torch.zeros_like(w), torch.zeros_like(w)
    grad = torch.empty_like(w)
    loss = torch.empty(1, device=dev)
    step = [0]

    def fused():
        step[0] += 1
        ops.dqn_grad_stack(cfg, spec, w, wt, ring, None, G, grad=grad, loss=loss)
        ops.adam_clip_step_stack(spec, w, grad, m, v, step[0])

    # autograd path on the same batch: targets from the kernel forward (constants), values through the module
    model = sb.StackedGCN.from_state_dict(sd).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    edges = bo.graph_edges(pos, mode, k)
    goal = torch.tensor([cfg.goal_x, cfg.goal_y]).view(1, 1, 2).expand(G, N, 2)
    ids = torch.arange(N, dtype=torch.float32).view(1, N, 1).expand(G, N, 1)
    x = torch.cat([pos, vel, goal, ids], 2)
    batch = sb.Batch.from_data_list([sb.Data(x=x[b_].to(dev), edge_index=edges[b_].to(torch.int64).to(dev))
                                     for b_ in range(G)])
    q2 = ops.gatstack_forward(cfg, spec, wt, torch.cat([pos2, vel], 2).contiguous().to(dev))
    targets = (rewards.reshape(-1).to(dev) + 0.99 * q2.reshape(G * N, 9).max(dim=1)[0]).unsqueeze(1)
    act = actions.reshape(-1, 1).to(dev)

    def autograd():
        opt.zero_grad()
        values = model(batch).gather(1, act)
        nn.MSELoss()(values, targets).backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()

    for fn in (fused, autograd):
        for _ in range(20):
            fn()
    torch.cuda.synchronize()
    fused_ms = _window_ms(fused, iters, windows)
    auto_iters = max(iters // 10, 20)
    auto_ms = _window_ms(autograd, auto_iters, windows)
    return {"layers": layers, "hidden": hidden, "in_features": 7, "n_agents": N, "graph": mode, "knn_k": k if mode == "knn" else None,
            "graphs_per_update": G, "fused_update_ms": fused_ms, "autograd_update_ms": auto_ms,
            "speedup": auto_ms / fused_ms, "fused_iters_per_window": iters, "autograd_iters_per_window": auto_iters,
            "windows": windows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--windows", type=int, default=7)
    args = ap.parse_args()
    import swarm_b200 as sb
    rows = []
    for layers, hidden, N, mode, k in ((3, 8, 12, "complete", 0), (3, 8, 12, "knn", 5), (2, 32, 12, "complete", 0)):
        for G in (32, 4096):
            r = run_case(sb, layers, hidden, N, mode, k, G, args.iters, args.windows)
            print(json.dumps(r), flush=True)
            rows.append(r)
    res = {"device": torch.cuda.get_device_name(0), "power_limit": _power_limit(),
           "method": "CUDA events, median of windows; one update = gradient + reduce + clip/Adam (fused) or "
                     "StackedGCN.forward + backward + clip_grad_norm_ + Adam (autograd)", "cases": rows}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
