"""Time the data-parallel DQN training tick of stacked GAT Q-networks on W = 1, 2, 4, 8 GPUs (as many as are visible):
one process per GPU, G = 32 graphs per rank, each tick ``StackTrainTick.grad_phase`` + ``apply_phase`` with the gradient
summed over the ranks either inside the grad phase's reduce launch through NVLink peer memory ("peer") or by an NCCL
all-reduce between the phases ("nccl") -- the two paths of ``DQNTrainer.train_model_stack_device``.  At W = 1 the
one-call ``swarm_train_tick_stack`` tick ("one_call") is the single-GPU baseline, and "peer" is a one-rank exchange
(every word pushed into the rank's own buffer and polled back).

CUDA events as in scripts/bench_stack_train.py: `--ticks` ticks captured in one CUDA graph, median over `--windows`
replays, every timed tick an update (the ring is filled beyond G first); each rank times its own stream and the slowest
rank's median is reported.  After each run the weights are compared across ranks bit for bit.  Writes JSON with the card
name, power limit and SM clock read in the same run.

    python scripts/bench_stack_train_multi.py --out profiles/r8_stack_train_multi.json
"""
import argparse
import json
import os
import socket
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (name, network, num_envs per rank): the Flocking checkpoint, and the widest stack (20 CTAs in the exchange)
CASES = [("flocking_ckpt_B64", "flocking", 64), ("flocking_ckpt_B4096", "flocking", 4096),
         ("stack_7_32_9_4_B64", "wide", 64)]
NETWORKS = {"flocking": "Flocking checkpoint: 3 GATConv layers, width 8, 7 inputs (409 weights)",
            "wide": "StackedGCN(7, 32, 9, 4): 4 GATConv layers, width 32, 7 inputs (5 033 weights)"}


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


def _time_case(sb, dist, rank, world, net, B, mode, ticks, windows, dev):
    """Median ms per tick on this rank, and whether the ranks' weights agree bit for bit afterwards."""
    from swarm_b200 import parallel
    ops, L = sb.ops, sb._lib
    N, G = 12, 32
    cfg = ops.make_config(L.SCENARIO_GOTO, B, N, L.GRAPH_COMPLETE)
    if net == "flocking":
        spec = ops.stack_spec(3, 8, 7)
        w = ops.pack_stack_weights(_flocking_sd(0), spec, dev)
    else:
        torch.manual_seed(0)
        model = sb.StackedGCN(7, 32, 9, 4)
        spec = model.stack_spec()
        w = ops.pack_stack_weights(model.state_dict(), spec, dev)
    rs = ops.reward_spec(L.REWARD_FLOCKING, B, N)
    g = torch.Generator().manual_seed(rank)
    state = ops.reset_grid(cfg, (torch.tensor([0.3, -0.3]) + 0.1 * torch.randn(B, 2, generator=g)).to(dev))
    shaping = torch.zeros(B, N, 2, device=dev)
    ops.scenario_reward(rs, state, shaping, reset=True)
    ring = ops.ReplayRing(max(4 * G, 4 * B), N, dev)
    w_t, m, v = w.clone(), torch.zeros_like(w), torch.zeros_like(w)
    returns = torch.zeros(B, N, device=dev)
    hits = torch.zeros(B, dtype=torch.int32, device=dev)
    tt = ops.StackTrainTick(cfg, spec, ring, graphs_per_update=G, update_target_every=200,
                            loss_scale=parallel.global_loss_scale(G, N), rng_seed=0, sample_seed=7919 * rank,
                            env_offset=rank * B, reward=rs, shaping=shaping)
    tt.load_cursor(0, 0, 0.5)
    if mode == "peer":
        tt.peers = parallel.PeerExchange(dev, stride=L.XCHG_STACK_STRIDE)

    def tick():
        if mode == "one_call":
            tt.tick(w, w_t, m, v, state, returns, hits)
            return
        tt.grad_phase(w, w_t, state, returns, hits)
        if mode == "nccl":
            dist.all_reduce(tt.grad_loss)
        tt.apply_phase(w, w_t, m, v)

    for _ in range((G + B - 1) // B + 2):           # eager: the ring holds >= G slots, kernel attributes set, NCCL warm
        tick()
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.graph(graph, stream=side):
        for _ in range(ticks):
            tick()
    graph.replay()
    torch.cuda.synchronize(dev)
    times = []
    for _ in range(windows):
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        graph.replay()
        b.record()
        torch.cuda.synchronize(dev)
        times.append(a.elapsed_time(b) / ticks)
    cur = tt.read_cursor()
    assert cur["updating"] == 1 and torch.isfinite(w).all()
    parts = [torch.empty_like(w) for _ in range(world)]
    dist.all_gather(parts, w)
    same = all(torch.equal(parts[0], p) for p in parts)
    meds = [None] * world
    dist.all_gather_object(meds, float(np.median(times)))
    del graph
    return meds, same


def _worker(rank, world, port, ticks, windows, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    try:
        import swarm_b200 as sb
        rows = []
        for name, net, B in CASES:
            for mode in (["one_call"] if world == 1 else []) + ["peer", "nccl"]:
                row = dict(case=name, network=NETWORKS[net], n_agents=12, graph="complete", reward="Flocking",
                           num_envs_per_rank=B, graphs_per_update_per_rank=32, world_size=world, mode=mode)
                try:
                    meds, same = _time_case(sb, dist, rank, world, net, B, mode, ticks, windows, dev)
                    row.update(tick_ms=max(meds), tick_ms_per_rank=meds, weights_bit_identical_across_ranks=same)
                except Exception as exc:        # e.g. no symmetric memory for a one-rank group: recorded, not hidden
                    row.update(tick_ms=None, error=repr(exc))
                if rank == 0:
                    print(json.dumps(row), flush=True)
                rows.append(row)
        dist.barrier()
        if rank == 0:
            with open(out, "w") as f:
                json.dump(rows, f)
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--ticks", type=int, default=100)
    ap.add_argument("--windows", type=int, default=7)
    args = ap.parse_args()
    import torch.multiprocessing as mp
    n = torch.cuda.device_count()
    if n < 1:
        raise SystemExit("no CUDA device: this benchmark times the B200 tick")
    rows = []
    with tempfile.TemporaryDirectory() as tmp:
        for world in [w for w in (1, 2, 4, 8) if w <= n]:
            part = os.path.join(tmp, f"w{world}.json")
            mp.spawn(_worker, args=(world, _free_port(), args.ticks, args.windows, part), nprocs=world, join=True)
            with open(part) as f:
                rows += json.load(f)
    res = {"device": torch.cuda.get_device_name(0), **_gpu_info(), "visible_gpus": n,
           "method": "CUDA events, median of windows (one replay of a CUDA graph of `ticks_per_graph` ticks each), "
                     "per tick, slowest rank's median; every timed tick an update; epsilon 0.5.  one_call: "
                     "swarm_train_tick_stack (one GPU).  peer: swarm_train_tick_stack_grad with the peer exchange + "
                     "swarm_train_tick_stack_apply.  nccl: swarm_train_tick_stack_grad + dist.all_reduce(grad_loss) + "
                     "swarm_train_tick_stack_apply.",
           "ticks_per_graph": args.ticks, "windows": args.windows, "cases": rows}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
