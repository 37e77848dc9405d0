"""The reference's OWN files, unmodified, on the CPU stand-ins of their two dependencies (oracle/refstub).

  * the stand-in is proven against the reference's shipped goldens: the reference's Simulator + scenario + GCN files on
    it reproduce data/test_stats/** bit for bit (with torch.topk's k forced to 5, the value the goldens were produced
    with -- the shipped simulator.py:19 says 10, SURVEY.md Appendix B);
  * the committed fixture tests/golden/reference_runs.npz (what the reference's Flocking / Cohesion reward() source
    and its scripts produce) is reproducible from the sources.
Skipped where build() found no reference checkout to stage into oracle/_ref.
"""
import os

import numpy as np
import pytest
import torch

import refsrc
from helpers import golden_eval, load_params, npz

pytestmark = pytest.mark.skipif(refsrc.reference_root() is None, reason="reference sources not staged")


@pytest.mark.parametrize("exp,n,m", [("go_to", 5, 0), ("go_to", 12, 7), ("obstacle_avoidance", 8, 2),
                                     ("obstacle_avoidance", 12, 5)])
def test_reference_files_on_refstub_reproduce_shipped_goldens(exp, n, m, tmp_path, monkeypatch):
    with refsrc.reference_modules("refstub") as ref:
        import vmas
        Scen = (ref.go_to_position_scenario.GoToPositionScenario if exp == "go_to"
                else ref.obstacle_avoidance_scenario.ObstacleAvoidanceScenario)
        orig = torch.topk
        monkeypatch.setattr(torch, "topk", lambda x, k, **kw: orig(x, 5, **kw))
        T = 50 if exp == "go_to" else 100
        env = vmas.make_env(Scen(), scenario_name="test_gcn_vmas", num_envs=1, device="cpu", continuous_actions=False,
                            dict_spaces=True, wrapper=None, seed=6967, n_agents=n, max_steps=T, random=True)
        model = ref.train_gcn_dqn.GCN(input_dim=7, hidden_dim=32, output_dim=9)
        model.load_state_dict(load_params(exp, m))
        model.eval()
        sim = ref.simulator.Simulator(env, model, 8, exp, 6967, output_dir=str(tmp_path))
        sim.run_simulation()
    got = refsrc.read_simulator_tree(str(tmp_path))
    gold = golden_eval(exp, m, n)
    assert (got["pos"] == gold["pos"]).all(), "positions written by the reference's Simulator differ from its shipped CSVs"
    assert (got["dist"] == gold["dist"]).all() and (got["hits"] == gold["hits"]).all()
    assert np.allclose(got["result"][:, 0], gold["result"][:, 0], rtol=1e-6)


def test_reference_runs_fixture_is_reproducible():
    """Re-run two Flocking / Cohesion cases of tests/golden/make_reference_runs.py and compare with the committed file."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_reference_runs",
                                                  os.path.join(refsrc.ROOT, "tests", "golden", "make_reference_runs.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    fix = npz("reference_runs.npz")
    with refsrc.reference_modules("refstub") as ref:
        import vmas
        for kind, n in (("flocking", 9), ("cohesion", 5)):
            run = mk.scenario_run(ref, vmas, kind, n, T=60, seed=100 + n)
            for k, v in run.items():
                assert np.array_equal(np.asarray(v), fix[f"{kind}/n{n}/{k}"]), f"{kind}/n{n}/{k} changed"
