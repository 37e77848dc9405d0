#!/usr/bin/env python
"""Stage the reference's own Python files for the script-level drop-in tests.

    python scripts/stage_reference.py [--src CHECKOUT] [--dst oracle/_ref]

Copies, byte for byte, `src/scenarios/*.py`, `src/simulation/simulator.py`, `src/training/train_gcn_dqn.py` and
`tests/test_*.py` of the reference checkout into `oracle/_ref/` (same relative layout).  The checkout is the one
BASELINE.json's `reference_path` names, or `$SWARM_REFERENCE` where it is set.  `__graft_entry__.build()` calls this
whenever that checkout exists.  The directory is git-ignored -- reference sources never enter this repository's
history -- but it is part of the working tree, so the staged copy goes wherever the built tree goes; there
`tests/test_gpu_reference_files.py` executes these files unmodified on top of `shim/` (the `vmas` / `torch_geometric`
module names backed by libswarm_b200.so).  A MANIFEST with the sha256 of every staged file is written next to them;
the tests check it so a stale or edited copy is noticed.
"""
import argparse
import hashlib
import json
import os
import shutil

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGED = os.path.join(ROOT, "oracle", "_ref")
FILES = ["src/__init__.py", "src/scenarios/__init__.py", "src/scenarios/go_to_position_scenario.py",
         "src/scenarios/obstacle_avoidance_scenario.py", "src/scenarios/flocking_scenario.py",
         "src/scenarios/cohesion_scenario.py", "src/simulation/__init__.py", "src/simulation/simulator.py",
         "src/training/__init__.py", "src/training/train_gcn_dqn.py", "tests/__init__.py",
         "tests/test_go_to_position.py", "tests/test_obstacle_avoidance.py"]


def reference_checkout() -> str:
    return os.environ.get("SWARM_REFERENCE") or json.load(open(os.path.join(ROOT, "BASELINE.json")))["reference_path"]


def stage(src: str = None, dst: str = STAGED) -> bool:
    src = src or reference_checkout()
    if not os.path.isdir(os.path.join(src, "src")):
        return False
    manifest = {}
    for rel in FILES:
        s = os.path.join(src, rel)
        if not os.path.exists(s):
            continue
        d = os.path.join(dst, rel)
        os.makedirs(os.path.dirname(d), exist_ok=True)
        shutil.copyfile(s, d)
        manifest[rel] = hashlib.sha256(open(d, "rb").read()).hexdigest()
    json.dump(manifest, open(os.path.join(dst, "MANIFEST.json"), "w"), indent=1, sort_keys=True)
    return True


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default=None, help="reference checkout (default: $SWARM_REFERENCE, else BASELINE.json)")
    ap.add_argument("--dst", default=STAGED)
    a = ap.parse_args()
    src = a.src or reference_checkout()
    print("staged" if stage(src, a.dst) else f"{src} not present: nothing staged")
