"""Multi-GPU checks of data-parallel stacked training (skipped with fewer than two GPUs; uses every visible GPU, 2 ... 8):
swarm_train_tick_stack_grad sums the gradient over the ranks through NVLink peer memory inside its reduce launch.  For
the Flocking checkpoint (3 layers of width 8) and StackedGCN(7, 32, 9, 4) (20 CTAs in the exchange), 12 ticks with
G = 32 graphs per rank:
  * the peer, peer-in-a-CUDA-graph and NCCL modes leave every rank with the same bits;
  * peer equals peer-graph bit for bit, and peer equals NCCL bit for bit at 2 ranks (any order of two addends is the
    same sum; above 2 ranks NCCL's order is its own, so the comparison is a sanity bound);
  * at the first (updating) tick the exchanged gradient and loss equal one GPU's dqn_grad_stack over the union of all
    ranks' sampled transitions with loss_scale = 1 / (W G N), up to the summation order;
and DQNTrainer.train_model_stack_device trains Flocking and Cohesion envs on every rank, with peers and over NCCL."""
import os
import socket
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.dirname(os.path.abspath(__file__))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _net(sb, name, dev):
    """(cfg, spec, packed weights, reward spec) of one network: the Flocking checkpoint on the GoTo world with the
    Flocking reward, or a randomly initialised StackedGCN(7, 32, 9, 4) on the ObstacleAvoidance world's own reward."""
    from test_gpu_stack_train_tick import _flocking_sd
    ops, L = sb.ops, sb._lib
    B, N = 64, 12
    if name == "flocking":
        cfg = ops.make_config(L.SCENARIO_GOTO, B, N, L.GRAPH_COMPLETE)
        spec = ops.stack_spec(3, 8, 7)
        return cfg, spec, ops.pack_stack_weights(_flocking_sd(0), spec, dev), ops.reward_spec(L.REWARD_FLOCKING, B, N)
    torch.manual_seed(0)
    model = sb.StackedGCN(7, 32, 9, 4)
    spec = model.stack_spec()
    cfg = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, B, N, L.GRAPH_COMPLETE)
    return cfg, spec, ops.pack_stack_weights(model.state_dict(), spec, dev), None


def _union_check(sb, dist, world, cfg, spec, tt, w, w_t, G):
    """The exchanged grad + loss of this tick against dqn_grad_stack over every rank's G sampled transitions."""
    ops = sb.ops
    N = cfg.n_agents
    idx = tt.indices
    mine = [tt.ring.state[idx], tt.ring.next_state[idx], tt.ring.actions[idx], tt.ring.rewards[idx]]
    union = ops.ReplayRing(world * G, N, w.device)
    for t, dst in zip(mine, (union.state, union.next_state, union.actions, union.rewards)):
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t.contiguous())
        dst.copy_(torch.cat(parts))
    union.advance(world * G)
    gcfg = ops.clone_config(cfg, num_envs=world * G)
    grad, loss, _ = ops.dqn_grad_stack(gcfg, spec, w, w_t, union, None, world * G,
                                       loss_scale=1.0 / (world * G * N))
    got_g, got_l = tt.grad, tt.loss
    scale = grad.abs().max()
    assert ((got_g - grad).abs().max() / scale).item() <= 1e-5, "exchanged gradient != union gradient"
    assert ((got_l - loss).abs() / loss.abs()).item() <= 1e-5, "exchanged loss != union loss"


def _run_ticks(sb, dist, rank, world, net, mode, dev):
    from swarm_b200 import parallel
    ops = sb.ops
    G, T = 32, 12
    cfg, spec, w0, rs = _net(sb, net, dev)
    B, N = cfg.num_envs, cfg.n_agents
    g = torch.Generator().manual_seed(rank)
    base = torch.tensor([0.3, -0.3]) if rs is not None else torch.tensor([0.6, -0.6])
    state = ops.reset_grid(cfg, (base + 0.1 * torch.randn(B, 2, generator=g)).to(dev))
    shaping = None
    if rs is not None:
        shaping = torch.zeros(B, N, 2, device=dev)
        ops.scenario_reward(rs, state, shaping, reset=True)
    ring = ops.ReplayRing(4096, N, dev)
    w, w_t = w0.clone(), w0.clone()
    m, v = torch.zeros_like(w), torch.zeros_like(w)
    returns = torch.zeros(B, N, device=dev)
    hits = torch.zeros(B, dtype=torch.int32, device=dev)
    tt = ops.StackTrainTick(cfg, spec, ring, graphs_per_update=G, update_target_every=4,
                            loss_scale=parallel.global_loss_scale(G, N), rng_seed=3, sample_seed=100 + rank,
                            env_offset=rank * B, reward=rs, shaping=shaping)
    tt.load_cursor(0, 0, 0.3)
    if mode != "nccl":
        tt.peers = parallel.PeerExchange(dev, stride=sb._lib.XCHG_STACK_STRIDE)

    def tick(check_union=False):
        w_before, wt_before = (w.clone(), w_t.clone()) if check_union else (None, None)
        tt.grad_phase(w, w_t, state, returns, hits)
        if mode == "nccl":
            dist.all_reduce(tt.grad_loss)
        if check_union:
            _union_check(sb, dist, world, cfg, spec, tt, w_before, wt_before, G)
        tt.apply_phase(w, w_t, m, v)

    if mode == "peer_graph":
        for _ in range(3):
            tick()
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.graph(graph, stream=side):
            for _ in range(3):
                tick()
        for _ in range(3):
            graph.replay()
    else:
        for t in range(T):
            tick(check_union=(mode == "peer" and t == 0))
    torch.cuda.synchronize(dev)
    cur = tt.read_cursor()
    assert cur["tick"] == T and cur["opt_step"] == T, cur
    for x in (w, w_t, tt.grad_loss):
        parts = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(parts, x)
        assert all(torch.equal(parts[0], p) for p in parts), f"{net}/{mode}: ranks diverged"
    assert not torch.equal(w, w0)
    return w.clone(), w_t.clone(), tt.grad_loss.clone()


def _trainer_run(sb, dist, world, scen, dev):
    from test_gpu_stack_train_tick import _flocking_sd
    B, steps, episodes = 64, 8, 2
    if scen == "flocking":
        env = sb.make_env(sb.FlockingScenario(), num_envs=B, device=dev, continuous_actions=False, max_steps=steps,
                          dict_spaces=True, seed=0, n_agents=12)
        model = sb.StackedGCN.from_state_dict(_flocking_sd(7))
    else:
        env = sb.make_env(sb.CohesionScenario(), num_envs=B, device=dev, continuous_actions=False, max_steps=steps,
                          dict_spaces=True, seed=0, n_agents=9)
        torch.manual_seed(0)
        model = sb.StackedGCN(5, 8, 9, 3)
    tr = sb.DQNTrainer(env, 0, "/tmp/none", "/tmp/none", "t", replay_capacity=4096, model=model)
    w0 = tr.w.clone()
    stats = tr.train_model_stack_device({"episodes": episodes, "epsilon": 0.9, "epsilon_decay": 0.3, "min_epsilon": 0.05,
                                         "graphs_per_update": 32, "update_target_every": 5})
    torch.cuda.synchronize(dev)
    assert tr.opt_step == episodes * steps                      # the ring holds >= G from tick 1
    assert torch.isfinite(stats).all() and (stats[:, 2] > 0).all()
    assert not torch.equal(tr.w, w0) and torch.isfinite(tr.w).all()
    for x in (tr.w, tr.w_target):
        parts = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(parts, x)
        assert all(torch.equal(parts[0], p) for p in parts), f"trainer {scen}: ranks diverged"


def _worker(rank, world, port, out):
    import torch.distributed as dist
    sys.path[:0] = [ROOT, TESTS]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    try:
        import swarm_b200 as sb
        for net in ("flocking", "wide"):
            res = {mode: _run_ticks(sb, dist, rank, world, net, mode, dev) for mode in ("nccl", "peer", "peer_graph")}
            for x, y in zip(res["peer"], res["peer_graph"]):
                assert torch.equal(x, y), f"{net}: peer vs peer_graph differ: {(x - y).abs().max().item():.3e}"
            for x, y in zip(res["nccl"], res["peer"]):
                if world == 2:
                    assert torch.equal(x, y), f"{net}: nccl vs peer differ: {(x - y).abs().max().item():.3e}"
                else:       # as in test_gpu_multi.py: Adam's early steps amplify last-bit differences of the sum order
                    assert torch.allclose(x, y, rtol=1e-2, atol=5e-3), f"{net}: nccl vs peer: {(x - y).abs().max().item():.3e}"
        for peer_env in ("1", "0"):
            os.environ["SWARM_PEER_ALLREDUCE"] = peer_env
            for scen in ("flocking", "cohesion"):
                _trainer_run(sb, dist, world, scen, dev)
        os.environ.pop("SWARM_PEER_ALLREDUCE")
        dist.barrier()
    finally:
        dist.destroy_process_group()
    if rank == 0:
        open(out, "w").write("ok")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
def test_data_parallel_stacked_training(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "done")
    world = min(torch.cuda.device_count(), 8)
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert open(out).read() == "ok"
