"""Where the cycles of one rollout tick go, phase by phase (C2: ObstacleAvoidance, 4 096 envs x 12 agents, complete
graph, greedy, 100 ticks -- the launch bench.py times).

    python scripts/time_rollout_phases.py [--reps 5] [--out FILE]

Builds a second copy of the library whose tile kernel is compiled with -DSWARM_PHASE_CLOCKS (csrc/tile_tc_device.cuh):
lane 0 of every warp stamps clock64() at each phase boundary of the tick and sums the cycles per phase.  Only
tile_kernels.cu is recompiled; the other objects come from the regular build (package build/ directory), and the
result goes to build/phase/.  Prints, per phase, the median over all warps of the launch of cycles per tick, and the
launch time measured with CUDA events on the same instrumented kernel.  The stamps cost a few instructions and one
shared-memory round trip each, so the instrumented tick is somewhat slower than the plain one; the table is for the
split, bench.py for the rate.
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
import swarm_b200 as sb                                   # noqa: E402
from swarm_b200 import _build                             # noqa: E402

PHASES = ["publish + barrier", "attention", "projection round", "tanh + split + st", "lin1 round", "ReLU + split + st",
          "lin2 round + argmax", "world step + reward"]


def phase_library() -> str:
    _build.build()
    out_dir = os.path.join(_build.BUILD_DIR, "phase")
    lib = os.path.join(out_dir, "libswarm_b200_phase.so")
    if os.path.exists(lib) and all(os.path.getmtime(d) <= os.path.getmtime(lib) for d in _build._deps()):
        return lib
    os.makedirs(out_dir, exist_ok=True)
    src = os.path.join(_build.CSRC, "tile_kernels.cu")
    obj = os.path.join(out_dir, "tile_kernels.o")
    subprocess.run([_build._nvcc()] + _build.NVCC_FLAGS + ["-DSWARM_PHASE_CLOCKS", "-c", src, "-o", obj], check=True)
    objs = [obj] + [os.path.join(_build.BUILD_DIR, os.path.basename(s)[:-3] + ".o") for s in _build.sources() if s != src]
    subprocess.run([_build._nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs, check=True)
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", help="also write the table as JSON here")
    args = ap.parse_args()
    _build.LIB_PATH = phase_library()                     # every ops call below runs the instrumented library
    ops = sb.ops
    dev = torch.device("cuda:0")
    B, N, T = 4096, 12, 100
    cfg = ops.make_config(sb._lib.SCENARIO_OBSTACLE_AVOIDANCE, B, N, sb._lib.GRAPH_COMPLETE)
    models = np.load(os.path.join(ROOT, "tests", "golden", "models.npz"))
    pre = "ObstacleAvoidance/0/"
    w = sb.pack_weights({k[len(pre):]: torch.from_numpy(models[k]) for k in models.files if k.startswith(pre)}, dev)
    g = torch.Generator().manual_seed(0)
    centers = (torch.tensor([0.6, -0.6]) + 0.1 * torch.randn(B, 2, generator=g)).to(dev)
    returns = torch.zeros(B, N, device=dev)
    hits = torch.zeros(B, dtype=torch.int32, device=dev)
    fn = sb._lib.lib().swarm_phase_cycles
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int]
    warps = 148 * 4 * 4
    buf = np.zeros((warps, len(PHASES)), dtype=np.uint64)
    per_rep, ms = [], []
    for rep in range(args.reps + 1):
        state = ops.reset_grid(cfg, centers)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.rollout(cfg, w, state, T, returns=returns, hits=hits)
        b.record()
        torch.cuda.synchronize()
        got = fn(buf.ctypes.data, warps)
        assert got == warps
        if rep == 0:
            continue                                      # warm-up launch
        ms.append(a.elapsed_time(b))
        live = buf[buf.sum(axis=1) > 0].astype(np.float64) / T
        per_rep.append(np.median(live, axis=0))
    med = np.median(np.stack(per_rep), axis=0)
    total = float(med.sum())
    print(f"{torch.cuda.get_device_name(dev)}: C2 rollout, {int((buf.sum(axis=1) > 0).sum())} warps, "
          f"instrumented launch {np.median(ms):.3f} ms ({args.reps} launches)")
    print(f"{'phase':24s} {'cycles/tick':>12s} {'share':>7s}")
    for name, c in zip(PHASES, med):
        print(f"{name:24s} {c:12.0f} {100 * c / total:6.1f}%")
    print(f"{'tick':24s} {total:12.0f}")
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"device": torch.cuda.get_device_name(dev), "launch_ms": float(np.median(ms)),
                       "cycles_per_tick": {n: float(c) for n, c in zip(PHASES, med)}, "tick_cycles": total}, f, indent=1)


if __name__ == "__main__":
    main()
