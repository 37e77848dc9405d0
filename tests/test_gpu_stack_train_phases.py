"""The stacked train tick as two phases (swarm_train_tick_stack_grad + swarm_train_tick_stack_apply, ops.StackTrainTick
grad_phase / apply_phase) on one GPU: the same bits as the one-call tick (swarm_train_tick_stack) over ten ticks of the
cases of test_gpu_stack_train_tick.py, eagerly and replayed from a CUDA graph, and -- where symmetric memory is
available -- the same values with a one-rank peer exchange as without one."""
import os
import socket
import sys

import pytest
import torch

from test_gpu_stack_train_tick import CASES, _flocking_sd

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _setup(case, dev):
    """A fresh tick (tt) and its tensors for one case of test_gpu_stack_train_tick.py: capacity 40 with B = 16 wraps the
    ring, G = 32 leaves tick 1 without an update, update_target_every = 3 syncs the target."""
    import swarm_b200 as sb
    ops, L = sb.ops, sb._lib
    name, world, reward, graph, k, N, in_f = case
    B, G, capacity, every = 16, 32, 40, 3
    scen = L.SCENARIO_OBSTACLE_AVOIDANCE if world == "oa" else L.SCENARIO_GOTO
    gm = {"knn": L.GRAPH_KNN, "complete": L.GRAPH_COMPLETE, "radius": L.GRAPH_RADIUS}[graph]
    cfg = ops.make_config(scen, B, N, gm, int(k) if graph == "knn" else 5, graph_radius=float(k) if graph == "radius" else 0.35)
    spec = ops.stack_spec(3, 8, in_f)
    w = ops.pack_stack_weights(_flocking_sd(2, in_f), spec, dev)
    g = torch.Generator().manual_seed(3)
    base = torch.tensor([0.6, -0.6]) if world == "oa" else torch.tensor([0.3, -0.3])
    state = ops.reset_grid(cfg, (base + 0.15 * torch.randn(B, 2, generator=g)).to(dev))
    rs = shaping = None
    if reward == "flocking":
        rs = ops.reward_spec(L.REWARD_FLOCKING, B, N)
        shaping = torch.zeros(B, N, 2, device=dev)
        ops.scenario_reward(rs, state, shaping, reset=True)
    elif reward == "cohesion":
        rs = ops.reward_spec(L.REWARD_COHESION, B, N)
    ring = ops.ReplayRing(capacity, N, dev)
    tt = ops.StackTrainTick(cfg, spec, ring, graphs_per_update=G, update_target_every=every, rng_seed=11, sample_seed=5,
                            env_offset=7, reward=rs, shaping=shaping)
    tt.load_cursor(0, 0, 0.4)
    t = dict(w=w, w_t=w.clone(), m=torch.zeros_like(w), v=torch.zeros_like(w), state=state,
             returns=torch.zeros(B, N, device=dev), hits=torch.zeros(B, dtype=torch.int32, device=dev), shaping=shaping)
    return tt, t


def _one_call(tt, t):
    tt.tick(t["w"], t["w_t"], t["m"], t["v"], t["state"], t["returns"], t["hits"])


def _phases(tt, t):
    tt.grad_phase(t["w"], t["w_t"], t["state"], t["returns"], t["hits"])
    tt.apply_phase(t["w"], t["w_t"], t["m"], t["v"])


def _snapshot(tt, t):
    """Everything a tick writes: weights, target, moments, grad + loss, cursor, replay ring, world, returns, hits."""
    out = {k: v.clone() for k, v in t.items() if v is not None}
    out.update(grad_loss=tt.grad_loss.clone(), ctl=tt.ctl.clone(), indices=tt.indices.clone(), ring_state=tt.ring.state.clone(),
               ring_next=tt.ring.next_state.clone(), ring_actions=tt.ring.actions.clone(),
               ring_rewards=tt.ring.rewards.clone())
    return out


def _assert_same(a, b, what):
    for k in a:
        assert torch.equal(a[k], b[k]), f"{what}: {k} differs"


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_phases_equal_the_one_call_tick(case):
    dev = torch.device("cuda:0")
    tt_a, a = _setup(case, dev)
    tt_b, b = _setup(case, dev)
    assert tt_b.peers is None
    updates = 0
    for tick in range(1, 11):
        _one_call(tt_a, a)
        _phases(tt_b, b)
        _assert_same(_snapshot(tt_a, a), _snapshot(tt_b, b), f"tick {tick}")
        updates += tt_b.read_cursor()["updating"]
    cur = tt_b.read_cursor()
    assert cur["tick"] == 10 and cur["opt_step"] == updates == 9          # tick 1: not enough samples


@pytest.mark.gpu
@pytest.mark.parametrize("case", [CASES[0], CASES[2]], ids=[CASES[0][0], CASES[2][0]])
def test_phases_replay_from_a_cuda_graph(case):
    """Three eager ticks, then three captured ticks replayed three times: the same bits as twelve eager ticks."""
    dev = torch.device("cuda:0")
    tt_a, a = _setup(case, dev)
    tt_b, b = _setup(case, dev)
    for _ in range(12):
        _phases(tt_a, a)
    for _ in range(3):
        _phases(tt_b, b)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.graph(graph, stream=side):
        for _ in range(3):
            _phases(tt_b, b)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize(dev)
    _assert_same(_snapshot(tt_a, a), _snapshot(tt_b, b), "graph")
    assert tt_b.read_cursor()["tick"] == 12


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _one_rank_worker(rank, port, out):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    try:
        import swarm_b200 as sb
        from swarm_b200 import parallel
        try:
            px = parallel.PeerExchange(dev, stride=sb._lib.XCHG_STACK_STRIDE)
        except Exception as exc:              # no symmetric memory on this machine
            torch.save({"skip": repr(exc)}, out)
            return
        res = {}
        for case in (CASES[1], CASES[3]):
            snaps = []
            for peers in (None, px):
                tt, t = _setup(case, dev)
                tt.peers = peers
                for _ in range(10):
                    _phases(tt, t)
                torch.cuda.synchronize(dev)
                snaps.append({k: v.cpu() for k, v in _snapshot(tt, t).items()})
            res[case[0]] = snaps
        torch.save(res, out)
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_one_rank_peer_exchange_equals_no_exchange(tmp_path):
    """A one-rank process group with a PeerExchange: the grad phase pushes each word into its own buffer, polls it and
    sums one rank -- the values of the call without peers (torch.equal: the exchange's +0.0 start may turn a -0.0
    gradient element into +0.0)."""
    import torch.multiprocessing as mp
    out = str(tmp_path / "res.pt")
    mp.spawn(_one_rank_worker, args=(_free_port(), out), nprocs=1, join=True)
    res = torch.load(out)
    if "skip" in res:
        pytest.skip(f"symmetric memory unavailable: {res['skip']}")
    for name, (plain, peer) in res.items():
        for k in plain:
            assert torch.equal(plain[k], peer[k]), f"{name}: {k} differs"
