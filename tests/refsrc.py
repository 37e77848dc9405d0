"""Locating and importing the reference's OWN Python files (unmodified) on top of a stand-in for its two pip
dependencies: ``oracle/refstub`` (CPU, pinned oracle arithmetic) or ``shim`` (the CUDA product).

The sources are not part of this repository: ``__graft_entry__.build()`` stages them from the reference checkout
(scripts/stage_reference.py) into the git-ignored ``oracle/_ref``, and they are read from there.  Where no checkout was
present at build time, the tests that execute them skip.
"""
import contextlib
import hashlib
import importlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGED = os.path.join(ROOT, "oracle", "_ref")
BACKENDS = {"refstub": os.path.join(ROOT, "oracle", "refstub"), "shim": os.path.join(ROOT, "shim")}
_REF_MODULES = ("go_to_position_scenario", "obstacle_avoidance_scenario", "flocking_scenario", "cohesion_scenario",
                "train_gcn_dqn", "simulator")


def reference_root():
    """Directory holding the reference's src/ and tests/ trees, or None."""
    if os.path.exists(os.path.join(STAGED, "MANIFEST.json")):
        manifest = json.load(open(os.path.join(STAGED, "MANIFEST.json")))
        for rel, digest in manifest.items():
            if hashlib.sha256(open(os.path.join(STAGED, rel), "rb").read()).hexdigest() != digest:
                raise AssertionError(f"staged reference file {rel} was modified after staging")
        return STAGED
    return None


def _purge():
    for name in list(sys.modules):
        if name in _REF_MODULES or name == "vmas" or name.startswith("vmas.") or name == "torch_geometric" or \
                name.startswith("torch_geometric."):
            del sys.modules[name]


@contextlib.contextmanager
def reference_modules(backend: str):
    """``with reference_modules("refstub") as ref: ref.flocking_scenario.FlockingScenario()`` -- the reference's files
    imported fresh with ``vmas`` / ``torch_geometric`` resolving to the chosen stand-in."""
    root = reference_root()
    if root is None:
        raise FileNotFoundError("reference sources not staged in oracle/_ref (build() stages them where the checkout exists)")
    paths = [BACKENDS[backend], os.path.join(root, "src", "scenarios"), os.path.join(root, "src", "training"),
             os.path.join(root, "src", "simulation")]
    saved = list(sys.path)
    _purge()
    sys.path[:0] = paths
    try:
        class _Ref:
            def __getattr__(self, name):
                if name not in _REF_MODULES:
                    raise AttributeError(name)
                return importlib.import_module(name)
        yield _Ref()
    finally:
        sys.path[:] = saved
        _purge()


def write_models(workdir: str) -> None:
    """``data/models/experiment_{GoTo,ObstacleAvoidance}-seed_{0..9}.pth`` (the files the reference scripts load,
    tests/test_go_to_position.py:45-46) rebuilt from tests/golden/models.npz."""
    import numpy as np
    import torch
    models = np.load(os.path.join(ROOT, "tests", "golden", "models.npz"))
    out = os.path.join(workdir, "data", "models")
    os.makedirs(out, exist_ok=True)
    groups = {}
    for k in models.files:
        exp, seed, key = k.split("/", 2)
        groups.setdefault((exp, seed), {})[key] = torch.from_numpy(models[k]).clone()
    for (exp, seed), sd in groups.items():
        torch.save(sd, os.path.join(out, f"experiment_{exp}-seed_{seed}.pth"))


def run_reference_script(backend: str, rel_script: str, workdir: str, stop_when, timeout: float = 600.0,
                         extra_env=None) -> str:
    """Run one of the reference's scripts UNMODIFIED as ``__main__`` in a subprocess (cwd = workdir, ``vmas`` /
    ``torch_geometric`` resolving to ``backend``) until ``stop_when(stdout_so_far)`` returns True, the script ends or
    ``timeout`` elapses; the scripts' full sweeps run for hours, the tests only need their first outputs.  Returns the
    captured stdout."""
    import subprocess
    import time
    root = reference_root()
    if root is None:
        raise FileNotFoundError("reference sources not staged")
    script = os.path.join(root, rel_script)
    boot = ("import sys, runpy; sys.path[:0] = [%r, %r]; runpy.run_path(%r, run_name='__main__')"
            % (BACKENDS[backend], ROOT, script))
    env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1", PYTHONUNBUFFERED="1")
    env.update(extra_env or {})
    log = os.path.join(workdir, "stdout.log")
    with open(log, "w") as fh:
        proc = subprocess.Popen([sys.executable, "-c", boot], cwd=workdir, env=env, stdout=fh, stderr=subprocess.STDOUT)
        t0 = time.time()
        try:
            while proc.poll() is None and time.time() - t0 < timeout:
                time.sleep(0.2)
                if stop_when(open(log).read()):
                    break
        finally:
            if proc.poll() is None:
                proc.kill()                      # the exact process we started
                proc.wait()
    return open(log).read()


def read_simulator_tree(where: str, episodes: int = 8):
    """The CSV tree Simulator.save_metrics_to_csv writes (simulator.py:111-166) as arrays:
    pos f32[E,T,n,2], dist f32[E,T], hits f32[E,T], result f64[E,4]."""
    import csv
    import numpy as np
    xs, ys, ds, hs = [], [], [], []
    for e in range(episodes):
        rx = list(csv.reader(open(f"{where}/positions/positions_episode_{e}_x.csv")))[1:]
        ry = list(csv.reader(open(f"{where}/positions/positions_episode_{e}_y.csv")))[1:]
        xs.append([[float(v) for v in r[1:]] for r in rx])
        ys.append([[float(v) for v in r[1:]] for r in ry])
        rd = list(csv.reader(open(f"{where}/data/distances_episode_{e}.csv")))[1:]
        ds.append([float(r[1]) for r in rd])
        hs.append([float(r[2]) for r in rd])
    res = [[float(v) for v in r[1:]] for r in list(csv.reader(open(f"{where}/result.csv")))[1:]]
    pos = np.stack([np.array(xs, dtype=np.float32), np.array(ys, dtype=np.float32)], axis=-1)
    return {"pos": pos, "dist": np.array(ds, dtype=np.float32), "hits": np.array(hs, dtype=np.float32),
            "result": np.array(res, dtype=np.float64)}
