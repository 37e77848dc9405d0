#!/usr/bin/env python
"""bench.py -- agent-steps/s of the swarm hot path (world step + per-step graph + GAT-Q forward + greedy
argmax) on N B200s, next to the reference-structured CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1] / SURVEY.md 8d "C2"): ObstacleAvoidance, 12 agents, 4 096 envs per GPU,
complete graph + (0,0) self loop (E = 133), weights of experiment_ObstacleAvoidance-seed_0, start centres
(0.6,-0.6) + N(0, 0.1^2) from torch.Generator(cpu).manual_seed(rank).  One *step* = one 100-tick greedy
episode of all envs: reset_grid launch + one fused rollout launch (state stays on chip for the 100 ticks).
``value`` is timed with the inputs resident in HBM; ``e2e`` goes through the public API with pinned host
buffers (centres in, per-agent returns + per-env hit counts out) inside the timed region.
``--dump-outputs DIR`` writes what the last timed ``e2e`` step handed back to its caller (rank 0's envs) as
``DIR/state.npy`` f32[B,N,4], ``DIR/returns.npy`` f32[B,N] and ``DIR/hits.npy`` f64[B]: the inputs are seeded, so
two builds run with the same arguments can be compared output for output.  The ``e2e`` leg runs the same rollout from
the same centres as the ``value`` leg, whose returns and hits buffers instead accumulate over all its steps.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_AGENTS = 12
ENVS_PER_GPU = 4096
TICKS = 100
BYTES_PER_AGENT_STEP = 40.0       # SURVEY.md 8(d): fused step+graph+Q without a Q dump: state in/out 32 B, action 4 B, reward 4 B
FLOPS_PER_AGENT_STEP = 4200.0     # SURVEY.md 8(d): N = 12, complete graph
METRIC = "agent-steps/s (VMAS step + graph + GNN-Q fwd)"


def load_weights():
    models = np.load(os.path.join(ROOT, "tests", "golden", "models.npz"))
    pre = "ObstacleAvoidance/0/"
    return {k[len(pre):]: torch.from_numpy(models[k]) for k in models.files if k.startswith(pre)}


def draw_centers(seed: int, num_envs: int) -> torch.Tensor:
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.tensor([0.6, -0.6]) + 0.1 * torch.randn(num_envs, 2, generator=g)


# ----------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks line")
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [c for c in sm if c >= 0.5 * max(sm)] if sm else []
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU arms (oracle port of the reference's per-tick loop, num_envs = 1)
# ----------------------------------------------------------------------------------------------
def _cpu_episode(args):
    """One greedy episode of the single-env oracle; returns (agent_steps, seconds)."""
    seed, ticks = args
    torch.set_num_threads(1)
    from oracle import swarm_oracle as so
    params = load_weights()
    world = so.OracleWorld(so.OBSTACLE_AVOIDANCE, N_AGENTS, random=True)
    torch.manual_seed(seed)
    obs = world.reset()
    ei = so.graph_complete(N_AGENTS)
    t0 = time.perf_counter()
    for _ in range(ticks):
        x = so.node_features(obs)
        with torch.no_grad():
            actions = torch.argmax(so.gatq_forward(params, x, so.graph_complete(N_AGENTS)), dim=1)
        world.step(actions)
        obs = world.observations()
    return N_AGENTS * ticks, time.perf_counter() - t0


def cpu_baseline_single(target_seconds: float = 12.0):
    done, secs, ep = 0, 0.0, 0
    while secs < target_seconds:
        n, s = _cpu_episode((ep, TICKS))
        done += n
        secs += s
        ep += 1
    return {"value": done / secs, "unit": "agent-steps/s", "cores": 1, "kind": "port",
            "sample": f"{ep} greedy 100-tick episodes of one 12-agent ObstacleAvoidance env (complete graph), "
                      f"oracle/swarm_oracle.py, torch CPU 1 thread, {secs:.1f} s"}


def run_reference_arm(args):
    """--impl reference: the reference-structured CPU path (oracle port; vmas / torch_geometric are not
    installable here) on all host cores, one single-env process per core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    ticks = 25                                            # bounded sample: a quarter episode per process per step
    with ctx.Pool(cores) as pool:
        for w in range(args.warmup):
            pool.map(_cpu_episode, [(1000 * w + i, ticks) for i in range(cores)])
        t0 = time.perf_counter()
        total = 0
        for s in range(args.steps):
            res = pool.map(_cpu_episode, [(1000 * (s + 10) + i, ticks) for i in range(cores)])
            total += sum(r[0] for r in res)
        dt = time.perf_counter() - t0
    value = total / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(args.gpus), reference_arm_runs=(
                f"{cores} single-env CPU processes (num_envs = 1 each, as the reference runs), {ticks} greedy ticks per "
                "process per step from a fresh contact-free reset; same scenario / swarm size / graph / weights, not the "
                "4096-env batch (the reference cannot batch)")),
            "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": cores, "kind": "port",
                             "sample": f"per step: {cores} processes x {ticks} ticks of one 12-agent env each "
                                       "(reference-structured per-tick loop, oracle/swarm_oracle.py)"},
            "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def workload_config(n_gpus: int):
    return {"workload": "ObstacleAvoidance N=12, 4096 envs/GPU, complete graph + self loop (E=133), greedy GAT-Q "
                        "policy (experiment_ObstacleAvoidance-seed_0), one step = 100-tick episode of all envs",
            "envs_per_gpu": ENVS_PER_GPU, "n_agents": N_AGENTS, "ticks_per_step": TICKS, "graph": "complete",
            "l2": "flushed between timed steps (256 MiB write)", "parallelism": f"env-sharded x{n_gpus}, no collective"}


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import swarm_b200 as sb
    from swarm_b200 import ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    B, N, T = ENVS_PER_GPU, N_AGENTS, TICKS
    cfg = ops.make_config(sb._lib.SCENARIO_OBSTACLE_AVOIDANCE, B, N, sb._lib.GRAPH_COMPLETE)
    weights = sb.pack_weights(load_weights(), dev)
    centers_host = draw_centers(rank, B).pin_memory()
    centers = centers_host.to(dev)
    state = torch.empty(B, N, 4, device=dev)
    returns = torch.zeros(B, N, device=dev)
    hits = torch.zeros(B, dtype=torch.int32, device=dev)
    # end-to-end leg: the three results of a rollout (final states, returns, hits) live in ONE device allocation and come
    # back with ONE device->host copy into pinned memory
    pack = torch.empty(B * N * 4 + B * N + B, device=dev)
    pack_host = torch.empty(B * N * 4 + B * N + B).pin_memory()
    e_state = pack[:B * N * 4].view(B, N, 4)
    e_returns = pack[B * N * 4:B * N * 5].view(B, N)
    e_hits = pack[B * N * 5:].view(torch.int32)
    returns_host = pack_host[B * N * 4:B * N * 5].view(B, N)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step_resident():
        ops.reset_grid(cfg, centers, out=state)
        ops.rollout(cfg, weights, state, T, returns=returns, hits=hits)

    def step_e2e():
        c = centers_host.to(dev, non_blocking=True)
        pack[B * N * 4:].zero_()                               # returns and hits
        ops.reset_grid(cfg, c, out=e_state)
        ops.rollout(cfg, weights, e_state, T, returns=e_returns, hits=e_hits)
        pack_host.copy_(pack, non_blocking=True)               # what a caller of rollout() gets back: final states too
        stream.synchronize()
        return float(returns_host[0, 0])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, kernel_events=None):
        evs = []
        barrier()
        for _ in range(steps):
            flush.zero_()                                    # L2 flush, outside the timed events
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            evs.append((a, b))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        if dist is not None:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
        step_e2e()
    ms_res = timed(step_resident, args.steps)

    # the dominant kernel alone (rollout launch), CUDA events on the launching stream
    kev = []
    barrier()
    for _ in range(args.steps):
        ops.reset_grid(cfg, centers, out=state)
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        ops.rollout(cfg, weights, state, T, returns=returns, hits=hits)
        b.record(stream)
        kev.append((a, b))
    barrier()
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps
    ms_e2e = timed(step_e2e, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"state": pack_host[:B * N * 4].view(B, N, 4), "returns": returns_host,
                                         "hits": pack_host[B * N * 5:].view(torch.int32)})
    dqn_stats = measure_dqn(sb, ops, dev, cfg, weights, centers, dist, barrier, stream, rank, world)
    strong = None
    if world > 1:
        # strong-scaling point (SURVEY.md 8d C5): the SAME 4 096 envs in total, split over the ranks
        Bs = ENVS_PER_GPU // world
        scfg = ops.make_config(sb._lib.SCENARIO_OBSTACLE_AVOIDANCE, Bs, N, sb._lib.GRAPH_COMPLETE)
        sc = draw_centers(0, ENVS_PER_GPU)[rank * Bs:(rank + 1) * Bs].contiguous().to(dev)
        sstate = torch.empty(Bs, N, 4, device=dev)
        sret = torch.zeros(Bs, N, device=dev)
        shits = torch.zeros(Bs, dtype=torch.int32, device=dev)

        def step_strong():
            ops.reset_grid(scfg, sc, out=sstate)
            ops.rollout(scfg, weights, sstate, T, returns=sret, hits=shits)

        for _ in range(3):
            step_strong()
        ms_strong = timed(step_strong, args.steps)
        strong = {"scaling": "strong", "total_envs": Bs * world, "envs_per_gpu": Bs,
                  "value": Bs * world * N * T * args.steps / (ms_strong * 1e-3), "unit": "agent-steps/s",
                  "ms_per_step": ms_strong / args.steps}
    clocks = sampler.stop() if rank == 0 else None

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    agent_steps = world * B * N * T * args.steps
    value = agent_steps / (ms_res * 1e-3)
    e2e_value = agent_steps / (ms_e2e * 1e-3)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak_gbs, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    else:
        peak_gbs, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = BYTES_PER_AGENT_STEP * B * N * T / (kernel_ms * 1e-3) / 1e9
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    fp32_achieved = FLOPS_PER_AGENT_STEP * B * N * T / (kernel_ms * 1e-3) / 1e12
    line = {
        "metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(world),
        "e2e": {"value": e2e_value, "unit": "agent-steps/s", "h2d_bytes_per_step": B * 2 * 4,
                "d2h_bytes_per_step": B * N * 4 + B * 4 + B * N * 16, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": 2 * args.steps,
        # the dominant kernel keeps the state on chip for 100 ticks: it is bound by instruction issue on the CUDA cores,
        # not by HBM and not by the tensor pipe -- `roofline` states that bound (algorithmic FLOPs of the reference
        # computation, SURVEY.md 8d, against the FP32 FMA issue peak at the sampled clock); the HBM view of the same
        # launch is kept beside it
        "roofline": {"kernel": "tile_kernel<MODE_ROLLOUT>", "bound": "issue (fp32 CUDA cores)", "achieved": fp32_achieved,
                     "peak": fp32_peak, "unit": "TFLOP/s", "frac": fp32_achieved / fp32_peak,
                     "traffic": None, "kernel_ms": kernel_ms, "flops_per_agent_step": FLOPS_PER_AGENT_STEP,
                     "peak_source": f"148 SMs x 128 FMA lanes x 2 x {sm_mhz:.0f} MHz (sampled under load; not in "
                                    "MEASURED_PEAKS.json, which holds HBM and bf16 tensor peaks)",
                     "note": "algorithmic FLOPs = 4 200 per agent-step (reference op count, N = 12, complete graph); the "
                             "kernel itself executes fewer (attention in input space); traffic = DRAM bytes of one launch "
                             "from the committed ncu capture"},
        "roofline_hbm": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                         "peak_source": peak_src, "bytes_per_agent_step": BYTES_PER_AGENT_STEP,
                         "note": "40 B/agent-step algorithmic; only 36 B/agent/launch actually move (state in registers)"},
        "clocks": clocks,
    }
    line["roofline"]["traffic"] = ncu_dram_traffic_bytes()
    line["dqn"] = dqn_stats
    if strong is not None:
        line["strong_scaling_point"] = strong
    if world == 1:
        # side measurements must never cost the headline line: a failure is reported in place of the numbers
        for key, fn in (("memory_bound_kernels", lambda: measure_streaming_kernels(sb, ops, dev, peak_gbs)),
                        ("extra", lambda: measure_extra(sb, ops, dev))):
            try:
                line[key] = fn()
            except Exception as exc:                                   # noqa: BLE001
                line[key] = {"error": f"{type(exc).__name__}: {exc}"}
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline_single()
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(where: str, arrays: dict) -> None:
    """Each host tensor as ``where/<name>.npy``: float32 stays float32, integers become float64 (exact)."""
    os.makedirs(where, exist_ok=True)
    for name, t in arrays.items():
        a = t.numpy()
        np.save(os.path.join(where, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def measure_extra(sb, ops, dev):
    """The other BASELINE.json configurations, driver-run (SURVEY.md 8d): the kNN (evaluation-graph) variant of C2, the
    C3 sweep (65 536 envs, GoTo, N = 5 / 8 / 12, complete and kNN k = 5) and C4 (1 024 agents x 1 024 envs; kNN k = 10,
    radius 0.35, complete).
    Device-resident, CUDA events, greedy policy of the shipped seed-0 weights."""
    L = sb._lib
    models = np.load(os.path.join(ROOT, "tests", "golden", "models.npz"))

    def weights(pre):
        return sb.pack_weights({k[len(pre):]: torch.from_numpy(models[k]) for k in models.files if k.startswith(pre)}, dev)

    w_oa, w_goto = weights("ObstacleAvoidance/0/"), weights("GoTo/0/")

    def rollout_rate(scen, B, N, graph, k, ticks, reps=3, fresh_memo=True):
        # kNN rows: the memo table of boundary-tie patterns (ops.knn_memo_table) is cleared before every timed launch, so
        # the figure is that of a first encounter with these states, not of a replay of a remembered episode
        cfg = ops.make_config(scen, B, N, graph, k)
        centers = draw_centers(7, B).to(dev)
        state = ops.reset_grid(cfg, centers)
        ret = torch.zeros(B, N, device=dev)
        hits = torch.zeros(B, dtype=torch.int32, device=dev)
        w = w_oa if scen == L.SCENARIO_OBSTACLE_AVOIDANCE else w_goto
        ops.rollout(cfg, w, state, ticks, returns=ret, hits=hits)
        ms = 0.0
        for _ in range(reps):
            ops.reset_grid(cfg, centers, out=state)
            if graph == L.GRAPH_KNN and N <= 12 and fresh_memo:
                ops.knn_memo_table(dev, N, k, fresh=True)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ops.rollout(cfg, w, state, ticks, returns=ret, hits=hits)
            b.record()
            torch.cuda.synchronize(dev)
            ms += a.elapsed_time(b)
        return B * N * ticks * reps / (ms * 1e-3)

    out = {"unit": "agent-steps/s"}
    out["c2_knn_k5"] = rollout_rate(L.SCENARIO_OBSTACLE_AVOIDANCE, ENVS_PER_GPU, N_AGENTS, L.GRAPH_KNN, 5, TICKS)
    # the same launches with the memo table kept between them (what a Simulator running episode after episode sees)
    out["c2_knn_k5_warm_memo_table"] = rollout_rate(L.SCENARIO_OBSTACLE_AVOIDANCE, ENVS_PER_GPU, N_AGENTS, L.GRAPH_KNN, 5,
                                                    TICKS, fresh_memo=False)
    sweep = {}
    for n in (5, 8, 12):
        sweep[f"N{n}_complete"] = rollout_rate(L.SCENARIO_GOTO, 65536, n, L.GRAPH_COMPLETE, 5, 50)
        sweep[f"N{n}_knn_k5"] = rollout_rate(L.SCENARIO_GOTO, 65536, n, L.GRAPH_KNN, 5, 50)
    out["c3_goto_65536_envs"] = sweep
    # C4: large swarm, per-tick launches (topk table -> per-env Q -> world step)
    B4, N4, K4, T4 = 1024, 1024, 10, 10
    cfg4 = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B4, N4, L.GRAPH_KNN, K4)
    st4 = ops.reset_grid(cfg4, draw_centers(9, B4).to(dev))
    ops.rollout_large(cfg4, w_oa, st4, 2)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    ops.rollout_large(cfg4, w_oa, st4, T4)
    b.record()
    torch.cuda.synchronize(dev)
    out["c4_oa_1024x1024_knn_k10"] = {"agent_steps_per_s": B4 * N4 * T4 / (a.elapsed_time(b) * 1e-3),
                                      "ms_per_tick": a.elapsed_time(b) / T4}
    # C4 with the other two graphs SURVEY 8d names: radius r = 0.35 (uniform-grid broad phase) and the complete graph
    # (1.07e9 edges per tick if it were materialised); two launches per tick, no edge list
    for name, gm in (("radius_r0.35", L.GRAPH_RADIUS), ("complete", L.GRAPH_COMPLETE)):
        cfg = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B4, N4, gm, K4, graph_radius=0.35)
        st = ops.reset_grid(cfg, draw_centers(9, B4).to(dev))
        ops.rollout_large(cfg, w_oa, st, 2)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.rollout_large(cfg, w_oa, st, T4)
        b.record()
        torch.cuda.synchronize(dev)
        out[f"c4_oa_1024x1024_{name}"] = {"agent_steps_per_s": B4 * N4 * T4 / (a.elapsed_time(b) * 1e-3),
                                          "ms_per_tick": a.elapsed_time(b) / T4}
    # the shipped three-layer Flocking checkpoints (conv1-3 of width 8) on the C2 shape with the Flocking reward:
    # one forward launch + world step + reward kernel + totals per tick, launched from the library
    fz = np.load(os.path.join(ROOT, "tests", "golden", "flocking_models.npz"))
    sd = {k[2:]: torch.from_numpy(fz[k]) for k in fz.files if k.startswith("0/")}
    spec = ops.stack_spec(3, 8, 7)
    ws = ops.pack_stack_weights(sd, spec, dev)
    cfg = ops.make_config(L.SCENARIO_GOTO, ENVS_PER_GPU, N_AGENTS, L.GRAPH_KNN, 5)
    rs = ops.reward_spec(L.REWARD_FLOCKING, ENVS_PER_GPU, N_AGENTS)
    st = ops.reset_grid(cfg, draw_centers(7, ENVS_PER_GPU).to(dev))
    shaping = torch.zeros(ENVS_PER_GPU, N_AGENTS, 2, device=dev)
    ops.scenario_reward(rs, st, shaping, reset=True)
    ops.rollout_stack(cfg, spec, ws, st, 5, reward=rs, shaping=shaping)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    ops.rollout_stack(cfg, spec, ws, st, TICKS, reward=rs, shaping=shaping)
    b.record()
    torch.cuda.synchronize(dev)
    out["flocking_3layer_checkpoint_c2_shape_knn_k5"] = {
        "agent_steps_per_s": ENVS_PER_GPU * N_AGENTS * TICKS / (a.elapsed_time(b) * 1e-3),
        "us_per_tick": a.elapsed_time(b) * 1e3 / TICKS}
    return out


def ncu_dram_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of one rollout launch, from the committed `ncu --set full` summary
    of this same command (profiles/r2_ncu_rollout_c2.txt, else round 1's); None if the summary is missing."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_rollout_c2.txt")
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "r1_ncu_rollout_c2.txt")
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        total = 0.0
        for ln in open(path):
            if ln.startswith(("dram__bytes_read.sum =", "dram__bytes_write.sum =")):
                _, rhs = ln.split("=", 1)
                val, u = rhs.split()[:2]
                total += float(val) * unit[u]
        return total
    except (OSError, KeyError, ValueError):
        return None


def measure_streaming_kernels(sb, ops, dev, peak_gbs, envs=1 << 21):
    """The stand-alone HBM-bound kernels of the path at a working set far beyond L2 (25 M agents, 400 MB of state):
    achieved algorithmic GB/s against the measured HBM peak (SURVEY.md 8d bytes per agent-step)."""
    import ctypes as C
    L = sb._lib
    N = N_AGENTS
    cfg = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, envs, N)
    g = torch.Generator().manual_seed(0)
    centers = (torch.tensor([0.6, -0.6]) + 0.1 * torch.randn(envs, 2, generator=g)).to(dev)
    state = ops.reset_grid(cfg, centers)
    out_state = torch.empty_like(state)
    actions = torch.randint(0, 9, (envs, N), device=dev, dtype=torch.int32)
    rewards = torch.empty(envs, N, device=dev)
    flags = torch.empty(envs, N, dtype=torch.uint8, device=dev)
    obs = torch.empty(envs, N, 6, device=dev)
    dist_ = torch.empty(envs, N, 2, device=dev)
    E = ops.edges_per_env(cfg)
    edges = torch.empty(envs, 2, E, dtype=torch.int32, device=dev)
    ring = ops.ReplayRing(envs, N, dev)
    st = L.stream_ptr(dev)

    def step40():
        L.check(L.lib().swarm_sim_step(C.byref(cfg), L.ptr(state), L.ptr(actions), L.ptr(out_state), L.ptr(rewards), None, None,
                                       None, None, st))

    def step73():
        L.check(L.lib().swarm_sim_step(C.byref(cfg), L.ptr(state), L.ptr(actions), L.ptr(out_state), L.ptr(rewards),
                                       L.ptr(flags), None, L.ptr(obs), L.ptr(dist_), st))

    def complete():
        L.check(L.lib().swarm_graph_build(C.byref(cfg), L.ptr(state), L.ptr(edges), None, st))

    cases = [("swarm_sim_step (state+action -> state+reward)", step40, envs * N * 40.0),
             ("swarm_sim_step (+ observations, distances, flags)", step73, envs * N * 73.0),
             ("swarm_graph_build (complete graph export)", complete, envs * (N * 16.0 + 8.0 * E)),
             ("swarm_reset_grid", lambda: ops.reset_grid(cfg, centers, out=state), envs * (8.0 + 16.0 * N)),
             ("swarm_replay_push", lambda: ops.replay_push(cfg, ring, state, actions, rewards, out_state), envs * N * 77.0)]
    out = []
    for name, fn, nbytes in cases:
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(10):
            fn()
        b.record()
        torch.cuda.synchronize(dev)
        ms = a.elapsed_time(b) / 10
        gbs = nbytes / (ms * 1e-3) / 1e9
        out.append({"kernel": name, "ms": ms, "algorithmic_bytes": nbytes, "achieved": gbs, "unit": "GB/s",
                    "frac": gbs / peak_gbs})
    return out


def measure_dqn(sb, ops, dev, cfg, weights, centers, dist, barrier, stream, rank, world, ticks=100):
    """BASELINE.json configs[1]: full DQN train step on the same envs -- per tick one fused
    [Q -> eps-greedy -> step -> replay push] launch over all envs, one on-device draw of G whole-swarm transitions, one
    loss + backward, (gradient all-reduce,) clip + Adam (+ hard target sync every 200 ticks).  The tick counters live
    in device memory (swarm_train_tick_grad / _apply), so `ticks` ticks are captured once in a CUDA graph and
    replayed; the same ticks launched eagerly are timed next to it.  Reported for G = 32 (the reference's batch,
    train:175) and G = 4096 (one update touching as many transitions as one tick produces)."""
    from swarm_b200 import parallel
    B, N = cfg.num_envs, cfg.n_agents
    out = {}
    for G in (32, 4096):
        ring = ops.ReplayRing(1 << 20, N, dev)
        w = weights.clone()
        w_t = weights.clone()
        m, v = torch.zeros_like(w), torch.zeros_like(w)
        state = ops.reset_grid(cfg, centers)
        returns = torch.zeros(B, N, device=dev)
        hits = torch.zeros(B, dtype=torch.int32, device=dev)
        tt = ops.TrainTick(cfg, ring, graphs_per_update=G, update_target_every=200,
                           loss_scale=parallel.global_loss_scale(G, N), rng_seed=rank, sample_seed=1000 + rank,
                           env_offset=rank * B)
        tt.load_cursor(0, 0, 0.3)
        tt.peers = parallel.make_peer_exchange(dev)         # fused NVLink peer-memory all-reduce when available
        nccl = world > 1 and tt.peers is None

        def tick():
            if not nccl:
                tt.tick(w, w_t, m, v, state, returns, hits)
                return
            tt.grad_phase(w, w_t, state, returns, hits)
            dist.all_reduce(tt.grad_loss)
            tt.apply_phase(w, w_t, m, v)

        def timed(fn):
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            barrier()
            ms = a.elapsed_time(b)
            if dist is not None:
                t = torch.tensor([ms], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            return ms

        for _ in range(10):
            tick()
        ms_eager = timed(lambda: [tick() for _ in range(ticks)])
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(dev)
        side.wait_stream(stream)
        with torch.cuda.graph(graph, stream=side):
            for _ in range(ticks):
                tick()
        torch.cuda.synchronize(dev)
        graph.replay()                      # warm replay
        ms = timed(graph.replay)
        cur = tt.read_cursor()
        # replicas must stay bit-identical (train:131-133 semantics: one model): all-gather the packed weights after
        # the 10 + 2 * ticks + ticks data-parallel updates and compare them on every rank
        identical, digest = True, None
        if dist is not None:
            gathered = [torch.empty_like(w) for _ in range(world)]
            dist.all_gather(gathered, w)
            identical = all(torch.equal(gathered[0], x) for x in gathered)
            flag = torch.tensor([1 if identical else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            identical = bool(flag.item())
        import hashlib
        digest = hashlib.sha1(w.cpu().numpy().tobytes()).hexdigest()[:16]
        out[f"G{G}"] = {"weights_bit_identical_across_ranks": identical, "weights_sha1_16": digest, "ranks_compared": world,
"graphs_per_update_per_gpu": G, "updates_per_s": ticks / (ms * 1e-3),
                        "train_agent_steps_per_s": world * B * N * ticks / (ms * 1e-3),
                        "transitions_trained_per_s": world * G * ticks / (ms * 1e-3), "ms_per_tick": ms / ticks,
                        "ms_per_tick_eager": ms_eager / ticks, "kernels_per_tick": 5 if nccl else (3 if G <= 64 else 4),
                        "grad_allreduce": ("none" if world == 1 else ("nccl" if nccl else "one-shot push over NVLink peer memory inside the reduce + clip + Adam launch")),
                        "ticks_done": cur["tick"], "opt_steps_done": cur["opt_step"], "loss": float(tt.loss.item())}
    out["note"] = ("one train tick = rollout tick of all envs (eps 0.3) + replay push + on-device sample + TD target/loss/"
                   "backward + grad all-reduce (N>1) + clip + Adam (+ target sync every 200 ticks); %d ticks captured in "
                   "one CUDA graph (device-resident tick counters), eager launches timed beside it" % ticks)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed e2e step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    # stdout carries exactly ONE JSON line: everything else a library prints there (e.g. NCCL's version banner)
    # is diverted to stderr; the JSON line is written to the original descriptor at the end.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


_JSON_OUT = None


def emit(line: dict) -> None:
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


if __name__ == "__main__":
    main()
