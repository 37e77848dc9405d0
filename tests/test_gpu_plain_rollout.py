"""The plain rollout instantiation of the tile kernel (csrc/tile_kernels.cu, PLAIN: complete graph, greedy, nothing
traced) against the generic one, which a launch takes as soon as it asks for any per-tick trace.  Both run the same
arithmetic, so final states, returns and hit counts must agree bit for bit -- at the benchmark shape (4 096 envs, three
CTAs per SM), with more envs than one wave of three CTAs per SM holds (the four-CTA build: 592 balanced CTAs of 8-9 envs
at 5 000, 601 CTAs of 10 with a last CTA of 7 at 6 007), and with one env per CTA (48 CTAs; at B = 1 a single CTA
whose 116 inactive threads compute on env 0)."""
import pytest
import torch

from helpers import load_params

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("scenario,B", [("obstacle_avoidance", 4096), ("go_to", 4096), ("obstacle_avoidance", 8192),
                                        ("obstacle_avoidance", 1), ("go_to", 1), ("obstacle_avoidance", 48),
                                        ("obstacle_avoidance", 5000), ("obstacle_avoidance", 6007), ("go_to", 6007)])
def test_plain_rollout_equals_generic(scenario, B):
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    dev = torch.device("cuda:0")
    N, T = 12, 100
    scen = L.SCENARIO_GOTO if scenario == "go_to" else L.SCENARIO_OBSTACLE_AVOIDANCE
    w = sb.pack_weights(load_params("GoTo" if scenario == "go_to" else "ObstacleAvoidance", 0), dev)
    cfg = ops.make_config(scen, B, N, L.GRAPH_COMPLETE)
    g = torch.Generator().manual_seed(B)
    base = torch.tensor([0.9, -0.9]) if scenario == "go_to" else torch.tensor([0.6, -0.6])
    centers = (base + 0.1 * torch.randn(B, 2, generator=g)).to(dev)
    state0 = ops.reset_grid(cfg, centers)

    plain = ops.rollout(cfg, w, state0.clone(), T)
    generic = ops.rollout(cfg, w, state0.clone(), T, trace={"rewards": True})
    torch.cuda.synchronize()
    assert torch.equal(plain["state"], generic["state"])
    assert torch.equal(plain["returns"], generic["returns"])
    assert torch.equal(plain["hits"], generic["hits"])
    # the episode is not trivial: agents moved, and in the obstacle scenario some of them hit the obstacle (which takes
    # more than a handful of envs: the single GoTo swarm of B = 1 starts where the greedy action of every agent is 0)
    if B >= 48:
        assert not torch.equal(plain["state"], state0)
    if scenario == "obstacle_avoidance" and B >= 48:
        assert int(plain["hits"].sum()) > 0
