"""DQN training at the reference's Python seam (src/training/train_gcn_dqn.py:25-48, 72-231).

``GraphReplayBuffer`` and ``DQNTrainer`` keep the reference's class / method names, argument meaning and
bookkeeping (epsilon schedule, target sync, CSV layout incl. its row quirk), while every tensor operation
runs in libswarm_b200.so: world step, replay push / sample, TD target, loss, backward, clip, Adam.

Two drivers:
  * ``DQNTrainer.train_model(config)``  -- the reference loop for ``num_envs = 1`` with the reference's Python
    ``random`` stream for exploration and sampling; reproduces the shipped ``data/stats/*.csv`` rows.
  * ``DQNTrainer.train_model_batched(config)`` -- B envs per tick with the device RNG, fused
    rollout-tick + replay push, G graphs per update (throughput mode); an episode's ticks replay from a CUDA graph.
  * ``DQNTrainer.train_model_device(config)`` -- as above with reset, epsilon schedule and episode statistics on
    the device too: one graph launch per episode, no host synchronisation until the run ends.

``DQNTrainer(..., model=StackedGCN(...))`` trains a stacked network (the conv1 .. convL form the reference ships as
data/models/experiment_Flocking-seed_*.pth) instead of the one-layer GCN: ``train_model`` and ``train_model_stepwise``
then run the stack's gradient kernel (``swarm_dqn_stack_grad``) and clip + Adam (``swarm_adam_clip_stack_step``), and
``train_model_stack_device`` is the stack's whole-run device loop -- one ``swarm_train_tick_stack`` call (four launches)
per tick, one CUDA-graph replay per episode -- for the GoTo, ObstacleAvoidance, Flocking and Cohesion rewards, on one GPU
or data-parallel over several (the gradient summed over the ranks through NVLink peer memory, or NCCL).
"""
from __future__ import annotations

import copy
import csv
import os
import random
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib, ops, parallel
from .gcn import GCN, StackedGCN
from .graph import Batch, Data, node_features, stack_observations
from .scenarios import CohesionScenario, FlockingScenario, _KernelScenario


class GraphReplayBuffer:
    """train:25-48 on a device ring.  ``push`` takes what the reference pushes (graph, actions, rewards,
    next graph) or raw states; ``sample`` draws with Python's ``random.sample`` exactly like the reference."""

    def __init__(self, capacity: int, n_agents: Optional[int] = None, device=None):
        self.capacity = int(capacity)
        self.ring: Optional[ops.ReplayRing] = None
        if n_agents is not None and device is not None:
            self.ring = ops.ReplayRing(self.capacity, n_agents, device)

    @property
    def position(self) -> int:
        return 0 if self.ring is None else self.ring.position

    def _ensure(self, n_agents: int, device) -> ops.ReplayRing:
        if self.ring is None:
            self.ring = ops.ReplayRing(self.capacity, n_agents, device)
        return self.ring

    @staticmethod
    def _state_of(g) -> torch.Tensor:
        x = g.x if hasattr(g, "x") else g
        return x[..., :4].reshape(1, -1, 4).contiguous()

    def push(self, graph_observation, actions, rewards, next_graph_observation) -> None:
        s, s2 = self._state_of(graph_observation), self._state_of(next_graph_observation)
        n, dev = s.shape[1], s.device
        ring = self._ensure(n, dev)
        cfg = ops.make_config(_lib.SCENARIO_GOTO, 1, n)
        a = torch.as_tensor(actions).reshape(1, n).to(device=dev, dtype=torch.int32)
        r = torch.as_tensor(rewards, dtype=torch.float32).reshape(1, n).to(dev)
        ops.replay_push(cfg, ring, s, a.contiguous(), r.contiguous(), s2)

    def sample_indices(self, batch_size: int) -> List[int]:
        # random.sample(self.buffer, k) consumes the Mersenne stream as a function of (len, k) only
        return random.sample(range(len(self)), batch_size)

    def sample(self, batch_size: int):
        """(Batch observations, actions int64[G*N], rewards f32[G*N], Batch next observations), train:38-45."""
        ring = self.ring
        idx = torch.tensor(self.sample_indices(batch_size), dtype=torch.int64, device=ring.state.device)
        b = ops.replay_gather(ring, idx)
        goal = getattr(self, "goal", (-0.8, 0.8))

        def graphs(state):
            G, N, _ = state.shape
            gl = torch.tensor(goal, dtype=torch.float32, device=state.device).view(1, 1, 2).expand(G, N, 2)
            x = node_features(torch.cat([state, gl], dim=2)).view(G, N, 7)
            cfg = ops.make_config(_lib.SCENARIO_GOTO, G, N, _lib.GRAPH_COMPLETE)
            edges, _ = ops.graph_build(cfg, state.contiguous())
            return Batch.from_data_list([Data(x=x[g_], edge_index=edges[g_].to(torch.int64)) for g_ in range(G)])

        return graphs(b["state"]), b["actions"].reshape(-1).long(), b["rewards"].reshape(-1), graphs(b["next_state"])

    def __len__(self) -> int:
        return 0 if self.ring is None else len(self.ring)


class DQNTrainer:
    """train:72-231.  ``env`` is a swarm_b200 Environment (``make_env``).  ``model``: a ``StackedGCN`` to train instead
    of the reference's ``GCN(n_input, 32, 9)``; its ``conv1`` must take ``observation dim + 1`` input features, and the
    target network starts as an exact copy of it."""

    def __init__(self, env, seed, models_path, stats_path, experiment, graph_mode: str = "complete", knn_k: int = 10,
                 replay_capacity: int = 1000000, model: Optional[StackedGCN] = None):
        self.env = env
        self.seed = seed
        self.models_path = models_path
        self.stats_path = stats_path
        self.experiment = experiment
        self.n_input = self.env.observation_space["agent0"].shape[0] + 1
        self.n_output = env.action_space["agent0"].n
        dev = env.device
        self.stack_spec = None
        if model is None:
            # constructors run on the CPU generator exactly like the reference (2 x 1 865 uniform draws)
            self.model = GCN(input_dim=self.n_input, hidden_dim=32, output_dim=self.n_output)
            self.target_model = GCN(input_dim=self.n_input, hidden_dim=32, output_dim=self.n_output)
            self.target_model.load_state_dict(self.model.state_dict())
        else:
            if not isinstance(model, StackedGCN):
                raise TypeError("model must be a StackedGCN")
            if model.conv1.in_channels != self.n_input:
                raise ValueError(f"model.conv1 takes {model.conv1.in_channels} input features, the environment's "
                                 f"observation gives {self.n_input} (observation dim + 1)")
            self.model = model
            self.target_model = copy.deepcopy(model)
            self.stack_spec = model.stack_spec()
        self.model.to(dev)
        self.target_model.to(dev)
        # packed device weights are the training state; the nn.Modules are refreshed from them on demand
        self.w = _lib.pack_weights(self.model.state_dict(), dev) if model is None else self.model.packed_stack_weights(dev)
        self.w_target = self.w.clone()
        self.exp_avg = torch.zeros_like(self.w)
        self.exp_avg_sq = torch.zeros_like(self.w)
        self.opt_step = 0
        self.lr, self.betas, self.eps, self.max_norm = 0.001, (0.9, 0.999), 1e-8, 1.0
        self.replay_buffer = GraphReplayBuffer(replay_capacity, env.n_agents, dev)
        gm = {"complete": _lib.GRAPH_COMPLETE, "knn": _lib.GRAPH_KNN}[graph_mode]
        self.graph_cfg = ops.clone_config(env.world.cfg, graph_mode=gm, knn_k=knn_k)
        self.episode_rewards: List[torch.Tensor] = []
        self.episode_losses: List[float] = []
        self.episode_obstacle_hits: List[float] = []
        self.rewards_buffer: List[torch.Tensor] = []
        self.obstacle_hits_buffer: List[float] = []
        self._grad = torch.empty_like(self.w)
        self._loss = torch.empty(1, dtype=torch.float32, device=dev)

    # -- reference API ---------------------------------------------------------------------------
    def create_graph_from_observations(self, observations: Dict[str, torch.Tensor]) -> Data:
        """train:94-110 (complete graph + (0,0)); edge list built by swarm_graph_build."""
        obs = stack_observations(observations)
        B, N, _ = obs.shape
        cfg = ops.clone_config(self.graph_cfg, num_envs=B)
        edges, _ = ops.graph_build(cfg, obs[:, :, :4].contiguous())
        offs = (torch.arange(B, device=obs.device, dtype=torch.int64) * N).view(B, 1, 1)
        ei = (edges.to(torch.int64) + offs).permute(1, 0, 2).reshape(2, -1).contiguous()
        return Data(x=node_features(obs), edge_index=ei)

    def sync_modules(self) -> None:
        """Copy the packed training weights back into the nn.Modules (for state_dict / torch.save)."""
        if self.stack_spec is not None:
            self.model.load_state_dict(ops.unpack_stack_weights(self.w, self.stack_spec))
            self.target_model.load_state_dict(ops.unpack_stack_weights(self.w_target, self.stack_spec))
            return
        self.model.load_state_dict(_lib.unpack_weights(self.w))
        self.target_model.load_state_dict(_lib.unpack_weights(self.w_target))

    def _dqn_grad(self, cfg, ring, indices, n_graphs, gamma) -> None:
        """Gradient + loss of one update into self._grad / self._loss, for the trained network's form."""
        if self.stack_spec is not None:
            ops.dqn_grad_stack(cfg, self.stack_spec, self.w, self.w_target, ring, indices, n_graphs, gamma=gamma,
                               grad=self._grad, loss=self._loss)
        else:
            ops.dqn_grad(cfg, self.w, self.w_target, ring, indices, n_graphs, gamma=gamma, grad=self._grad, loss=self._loss)

    def _adam_clip(self, target) -> None:
        """clip_grad_norm_ + Adam step self.opt_step on self._grad (train:125-126), optional target sync."""
        if self.stack_spec is not None:
            ops.adam_clip_step_stack(self.stack_spec, self.w, self._grad, self.exp_avg, self.exp_avg_sq, self.opt_step,
                                     self.lr, self.betas, self.eps, self.max_norm, target=target)
        else:
            ops.adam_clip_step(self.w, self._grad, self.exp_avg, self.exp_avg_sq, self.opt_step, self.lr, self.betas,
                               self.eps, self.max_norm, target=target)

    def _greedy_actions(self, cfg) -> torch.Tensor:
        """argmax_a Q_online for the world's current state, int32[B, N]."""
        if self.stack_spec is not None:
            return ops.gatstack_forward(cfg, self.stack_spec, self.w, self.env.world.state, want_q=False, want_actions=True)
        _, act = ops.gatq_forward(cfg, self.w, self.env.world.state, want_q=False)
        return act

    def _require_one_layer(self, what: str) -> None:
        if self.stack_spec is not None:
            raise NotImplementedError(f"{what} runs the fused train tick of the one-layer GCN; train a StackedGCN with "
                                      "train_model_stack_device or train_model_stepwise (or train_model for one env)")

    def train_step_dqn(self, batch_size, model=None, target_model=None, ticks=0, gamma=0.99, update_target_every=10,
                       indices: Optional[torch.Tensor] = None):
        """train:112-137.  ``model`` / ``target_model`` are accepted for signature parity; the packed weights
        of this trainer are what is trained."""
        if len(self.replay_buffer) < batch_size:
            print("Not enough samples in the replay buffer")
            return 0
        ring = self.replay_buffer.ring
        if indices is None:
            indices = torch.tensor(self.replay_buffer.sample_indices(batch_size), dtype=torch.int64, device=self.w.device)
        cfg = ops.clone_config(self.graph_cfg, num_envs=batch_size)
        self._dqn_grad(cfg, ring, indices, batch_size, gamma)
        self.opt_step += 1
        sync = (ticks % update_target_every == 0)
        if sync:
            print("Updating target model")
        self._adam_clip(self.w_target if sync else None)
        return self._loss.item()

    def _policy_actions(self) -> torch.Tensor:
        """argmax_a Q(s) for the env's current state with the online weights (train:161-162,167)."""
        cfg = ops.clone_config(self.graph_cfg, num_envs=self.env.num_envs)
        return self._greedy_actions(cfg)

    def _rewards_tensor(self, rewards) -> torch.Tensor:
        """The rewards of the tick just stepped as f32[B, n]: what the world-step kernel wrote for the two fused
        scenarios, else what the scenario's reward() returned (Flocking, Cohesion, a user's own)."""
        if isinstance(self.env.scenario, _KernelScenario):
            return self.env.world.last["rewards"]
        cols = [rewards[a.name] for a in self.env.agents] if isinstance(rewards, dict) else list(rewards)
        return torch.stack([c.reshape(-1).to(torch.float32) for c in cols], dim=1).contiguous()

    def train_model(self, config):
        """train:139-204 for num_envs = 1, Python ``random`` exploration/sampling like the reference."""
        if self.env.num_envs != 1:
            raise ValueError("train_model mirrors the reference's num_envs = 1 loop; use train_model_batched")
        initial_epsilon = config["epsilon"]
        epsilon_decay = config["epsilon_decay"]
        min_epsilon = config["min_epsilon"]
        episodes = config["episodes"]
        ticks = 0
        epsilon = initial_epsilon
        n = self.env.n_agents
        world = self.env.world
        for episode in range(episodes):
            self.env.reset()
            episode_loss = 0
            total_episode_reward = torch.zeros(n)
            for _ in range(self.env.max_steps):
                ticks += 1
                state = world.state.clone()
                if random.random() < epsilon:
                    actions = torch.tensor([random.randint(0, 8) for _ in range(n)], dtype=torch.int32,
                                           device=world.device).view(1, n)
                else:
                    actions = self._policy_actions()
                _, rewards, done, _ = self.env.step(actions)
                rewards_dev = self._rewards_tensor(rewards)
                ring = self.replay_buffer.ring
                ops.replay_push(world.cfg, ring, state, actions.contiguous(), rewards_dev, world.state)
                loss = self.train_step_dqn(32, self.model, self.target_model, ticks, update_target_every=200)
                episode_loss += loss
                total_episode_reward += (rewards_dev.reshape(n).cpu() / n)
            epsilon = max(min_epsilon, initial_epsilon * np.exp(-epsilon_decay * episode))
            average_loss = episode_loss / self.env.max_steps
            self.episode_losses.append(average_loss)
            self.rewards_buffer.append(total_episode_reward[0])
            if (episode + 1) % 10 == 0:
                self.episode_rewards.append(sum(self.rewards_buffer) / 10)
                self.rewards_buffer = []
                self.episode_obstacle_hits.append(sum(self.obstacle_hits_buffer) / 10)
                self.obstacle_hits_buffer = []
            if config.get("verbose", True):
                print(f"Episode {episode}, Loss: {average_loss}, Reward: {total_episode_reward.sum().item()}, Epsilon: {epsilon}")
        self.sync_modules()
        if config.get("save", True):
            os.makedirs(self.models_path, exist_ok=True)
            torch.save(self.model.state_dict(), f"{self.models_path}/experiment_{self.experiment}-seed_{self.seed}.pth")
            self.save_metrics_to_csv()

    def train_model_batched(self, config) -> Dict[str, float]:
        """B envs per tick, G graphs per update (throughput mode).  Same schedule as train:139-204 (epsilon per
        episode, hard target sync every ``update_target_every`` ticks), device RNG for exploration and sampling.

        Every tick is the pair ``swarm_train_tick_grad`` (fused [Q -> eps-greedy -> step -> replay push], index draw,
        TD target / loss / backward) + ``swarm_train_tick_apply`` (clip + Adam + target sync), with one gradient
        all-reduce in between when data-parallel.  The tick counters live on the device, so with
        ``config["cuda_graph"]`` (default on) the ticks of one episode are captured once in a CUDA graph and each
        episode is a single graph launch.  A ``FlockingScenario`` env trains on its collective reward: the tick kernel
        then evaluates the Flocking reward on the GoTo world and keeps the scenario's shaping memory up to date."""
        self._require_one_layer("train_model_batched")
        flock = isinstance(self.env.scenario, FlockingScenario)
        if not flock and not isinstance(self.env.scenario, _KernelScenario):
            raise NotImplementedError("the fused train tick computes the GoTo / ObstacleAvoidance / Flocking rewards in the "
                                      "kernel; train other scenarios with train_model / train_model_stepwise")
        env, world = self.env, self.env.world
        B, n, dev = env.num_envs, env.n_agents, env.device
        G = int(config.get("graphs_per_update", 32))
        episodes = config["episodes"]
        epsilon = config["epsilon"]
        use_graph = bool(config.get("cuda_graph", True))
        ring = self.replay_buffer.ring
        cfg = ops.clone_config(self.graph_cfg, num_envs=B)
        rank = torch.distributed.get_rank() if parallel.world_size() > 1 else 0
        # env-sharded data parallelism: G graphs per rank, loss = mean over the global batch, gradient summed
        # over ranks, identical clip + Adam everywhere (weights stay replicated; target sync is local)
        tt = ops.TrainTick(cfg, ring, graphs_per_update=G, update_target_every=int(config.get("update_target_every", 200)),
                           gamma=float(config.get("gamma", 0.99)), loss_scale=parallel.global_loss_scale(G, n),
                           lr=self.lr, betas=self.betas, eps=self.eps, max_norm=self.max_norm, rng_seed=self.seed,
                           sample_seed=int(config.get("sample_seed", self.seed)) + 7919 * rank,
                           env_offset=int(config.get("env_offset", rank * B)),
                           flocking=env.scenario._spec() if flock else None,
                           shaping=env.scenario.shaping if flock else None)
        parallel.require_equal_shards(B, ring.size, ring.position, ring.capacity, G)
        parallel.broadcast_weights(self.w)
        self.w_target.copy_(self.w)
        tt.load_cursor(int(config.get("start_tick", 0)), self.opt_step, epsilon)
        returns = torch.zeros(B, n, dtype=torch.float32, device=dev)
        hits = torch.zeros(B, dtype=torch.int32, device=dev)
        multi = parallel.world_size() > 1
        # data-parallel: the gradient all-reduce runs inside the clip + Adam kernel over NVLink peer memory when
        # symmetric memory is available, else as an NCCL all-reduce between the two phases
        tt.peers = parallel.make_peer_exchange(dev)
        nccl = multi and tt.peers is None

        def tick():
            if not nccl:
                tt.tick(self.w, self.w_target, self.exp_avg, self.exp_avg_sq, world.state, returns, hits)
                return
            tt.grad_phase(self.w, self.w_target, world.state, returns, hits)
            torch.distributed.all_reduce(tt.grad_loss)
            tt.apply_phase(self.w, self.w_target, self.exp_avg, self.exp_avg_sq)

        graph = None
        stats = {}
        for episode in range(episodes):
            env.reset()
            returns.zero_()
            hits.zero_()
            tt.set_epsilon(epsilon)
            if use_graph and graph is None and episode > 0:
                # capture after one eager episode (kernel attributes set, NCCL communicator warm)
                torch.cuda.synchronize(dev)
                graph = torch.cuda.CUDAGraph()
                side = torch.cuda.Stream(dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.graph(graph, stream=side):
                    for _ in range(env.max_steps):
                        tick()
                graph.replay()
            elif graph is not None:
                graph.replay()
            else:
                for _ in range(env.max_steps):
                    tick()
            epsilon = max(config["min_epsilon"], config["epsilon"] * np.exp(-config["epsilon_decay"] * episode))
            cur = tt.read_cursor()
            stats = {"episode": episode, "mean_return_agent0": float(returns[:, 0].mean() / n),
                     "loss": float(tt.loss.item()) if cur["opt_step"] else 0.0, "hits_per_env": float(hits.float().mean()),
                     "ticks": cur["tick"], "opt_steps": cur["opt_step"]}
            self.opt_step = cur["opt_step"]
            self.episode_losses.append(stats["loss"])
            self.rewards_buffer.append(torch.tensor(stats["mean_return_agent0"]))
            if (episode + 1) % 10 == 0:
                self.episode_rewards.append(sum(self.rewards_buffer) / 10)
                self.rewards_buffer = []
            if config.get("verbose", False):
                print(stats)
        self._grad.copy_(tt.grad)
        self._loss.copy_(tt.loss)
        self.sync_modules()
        return stats

    def train_model_stepwise(self, config) -> Dict[str, float]:
        """B envs per tick for ANY scenario (Flocking, user-written): the reference's loop body (train:153-178) batched
        over the envs with the scenario's own ``reward()``.  Per tick: greedy Q forward -> one exploration draw per env
        (train:164) -> ``env.step`` -> replay push of the B transitions -> G slot indices -> ``swarm_dqn_grad`` ->
        ``swarm_adam_clip_step`` (hard target sync every ``update_target_every`` ticks).  Exploration and sampling use a
        torch device generator.  This is the general path (about ten launches per tick, no CUDA graph);
        ``train_model_batched`` is the fused one for GoTo / ObstacleAvoidance."""
        env, world = self.env, self.env.world
        B, n, dev = env.num_envs, env.n_agents, env.device
        G = int(config.get("graphs_per_update", 32))
        every = int(config.get("update_target_every", 200))
        gamma = float(config.get("gamma", 0.99))
        gen = torch.Generator(device=dev)
        gen.manual_seed(int(config.get("sample_seed", self.seed)))
        ring = self.replay_buffer.ring
        cfg = ops.clone_config(self.graph_cfg, num_envs=B)
        gcfg = ops.clone_config(self.graph_cfg, num_envs=G)
        if ring.capacity < B:
            raise ValueError("the replay ring must hold at least one tick of transitions")
        epsilon = config["epsilon"]
        ticks = int(config.get("start_tick", 0))
        stats: Dict[str, float] = {}
        for episode in range(config["episodes"]):
            env.reset()
            returns = torch.zeros(B, n, dtype=torch.float32, device=dev)
            loss_sum = torch.zeros(1, dtype=torch.float32, device=dev)
            updates = 0
            for _ in range(env.max_steps):
                ticks += 1
                state = world.state.clone()
                greedy = self._greedy_actions(cfg)
                explore = torch.rand(B, 1, device=dev, generator=gen) < epsilon
                rnd = torch.randint(0, 9, (B, n), device=dev, generator=gen, dtype=torch.int32)
                actions = torch.where(explore, rnd, greedy.view(B, n).to(torch.int32)).contiguous()
                _, rewards, _, _ = env.step(actions)
                rewards_dev = self._rewards_tensor(rewards)
                ops.replay_push(cfg, ring, state, actions, rewards_dev, world.state)
                returns += rewards_dev
                if len(ring) >= G:
                    idx = torch.randint(0, len(ring), (G,), device=dev, generator=gen, dtype=torch.int64)
                    self._dqn_grad(gcfg, ring, idx, G, gamma)
                    self.opt_step += 1
                    self._adam_clip(self.w_target if ticks % every == 0 else None)
                    loss_sum += self._loss
                    updates += 1
            epsilon = max(config["min_epsilon"], config["epsilon"] * np.exp(-config["epsilon_decay"] * episode))
            stats = {"episode": episode, "mean_return_agent0": float(returns[:, 0].mean() / n),
                     "loss": float(loss_sum.item()) / max(updates, 1), "ticks": ticks, "opt_steps": self.opt_step}
            self.episode_losses.append(stats["loss"])
            self.rewards_buffer.append(torch.tensor(stats["mean_return_agent0"]))
            if (episode + 1) % 10 == 0:
                self.episode_rewards.append(sum(self.rewards_buffer) / 10)
                self.rewards_buffer = []
            if config.get("verbose", False):
                print(stats)
        self.sync_modules()
        return stats

    def train_model_device(self, config) -> torch.Tensor:
        """Whole training run on the device: every episode is ONE replay of a CUDA graph holding
        [swarm_reset_random -> max_steps x (swarm_train_tick_grad, gradient all-reduce, swarm_train_tick_apply) ->
        swarm_episode_end]; start centres, exploration, replay sampling, the epsilon schedule and the per-episode
        statistics (train:179-199) all live on the device and the host only reads the statistics at the end.
        Per-env start centres come from the counter RNG (``shared_center`` reproduces the reference's one draw per
        reset).  Returns stats f32[episodes, 4] = (mean agent-0 return / N, hits per env, last loss, epsilon)."""
        self._require_one_layer("train_model_device")
        flock = isinstance(self.env.scenario, FlockingScenario)
        if not (flock or isinstance(self.env.scenario, _KernelScenario)):
            raise NotImplementedError("the whole-run device loop resets GoTo / ObstacleAvoidance / Flocking worlds on the "
                                      "device; train other scenarios with train_model_stepwise")
        env, world = self.env, self.env.world
        B, n, dev = env.num_envs, env.n_agents, env.device
        G = int(config.get("graphs_per_update", 32))
        episodes = int(config["episodes"])
        ring = self.replay_buffer.ring
        cfg = ops.clone_config(self.graph_cfg, num_envs=B)
        rank = torch.distributed.get_rank() if parallel.world_size() > 1 else 0
        multi = parallel.world_size() > 1
        tt = ops.TrainTick(cfg, ring, graphs_per_update=G, update_target_every=int(config.get("update_target_every", 200)),
                           gamma=float(config.get("gamma", 0.99)), loss_scale=parallel.global_loss_scale(G, n),
                           lr=self.lr, betas=self.betas, eps=self.eps, max_norm=self.max_norm, rng_seed=self.seed,
                           sample_seed=int(config.get("sample_seed", self.seed)) + 7919 * rank,
                           env_offset=int(config.get("env_offset", rank * B)),
                           flocking=env.scenario._spec() if flock else None,
                           shaping=env.scenario.shaping if flock else None)
        spec = ops.reset_spec(cfg.scenario, random=bool(getattr(env.scenario, "random", True)),
                              seed=int(config.get("reset_seed", self.seed)), env_offset=tt.hyper.env_offset,
                              shared_center=bool(config.get("shared_center", False)), flocking=flock)
        flock_spec = env.scenario._spec() if flock else None
        parallel.require_equal_shards(B, ring.size, ring.position, ring.capacity, G)
        parallel.broadcast_weights(self.w)
        self.w_target.copy_(self.w)
        tt.load_cursor(int(config.get("start_tick", 0)), self.opt_step, config["epsilon"], 0)
        returns = torch.zeros(B, n, dtype=torch.float32, device=dev)
        hits = torch.zeros(B, dtype=torch.int32, device=dev)
        stats = torch.zeros(episodes, 4, dtype=torch.float32, device=dev)

        tt.peers = parallel.make_peer_exchange(dev)
        nccl = multi and tt.peers is None

        def episode():
            ops.reset_random(cfg, spec, world.state, ctl=tt.ctl)
            if flock:
                # previous_distance_to_goal / previous_distance_to_agents as reset_world_at leaves them
                # (flocking:101-121), on the device: the same reset launch the host-side reset_world_at issues
                ops.scenario_reward(flock_spec, world.state, env.scenario.shaping, reset=True)
            for _ in range(env.max_steps):
                if not nccl:
                    tt.tick(self.w, self.w_target, self.exp_avg, self.exp_avg_sq, world.state, returns, hits)
                    continue
                tt.grad_phase(self.w, self.w_target, world.state, returns, hits)
                torch.distributed.all_reduce(tt.grad_loss)
                tt.apply_phase(self.w, self.w_target, self.exp_avg, self.exp_avg_sq)
            tt.episode_end(returns, hits, stats, config["epsilon"], config["epsilon_decay"], config["min_epsilon"])

        _run_episodes(episode, episodes, bool(config.get("cuda_graph", True)), dev)
        cur = tt.read_cursor()
        self.opt_step = cur["opt_step"]
        self._grad.copy_(tt.grad)
        self._loss.copy_(tt.loss)
        self.sync_modules()
        out = stats.cpu()
        self.episode_losses.extend(out[:, 2].tolist())
        return out

    def train_model_stack_device(self, config) -> torch.Tensor:
        """``train_model_device`` for a stacked network: every episode is ONE replay of a CUDA graph holding
        [reset -> max_steps x swarm_train_tick_stack -> swarm_episode_end] (after one eager episode; ``cuda_graph``
        False runs every episode eagerly), four launches per tick and no host synchronisation until the run ends.  The
        reward is the world's own (GoTo / ObstacleAvoidance), Flocking's (its shaping memory reset on the device with
        the world) or Cohesion's.  GoTo / ObstacleAvoidance / Flocking start from ``swarm_reset_random``; Cohesion starts
        from its fixed table, so its reset is a device copy of the state one ``env.reset()`` leaves.  Data-parallel (one
        process per GPU, envs sharded as in ``train_model_device``): G graphs per rank, the loss is the mean over the
        global batch, and each tick is ``swarm_train_tick_stack_grad`` (which sums the gradient over the ranks through
        NVLink peer memory) + ``swarm_train_tick_stack_apply``, with an NCCL all-reduce in between where peer memory is
        unavailable or SWARM_PEER_ALLREDUCE=0; the weights stay identical on every rank.  Returns stats
        f32[episodes, 4] = (mean agent-0 return / N, hits per env, last loss, epsilon)."""
        if self.stack_spec is None:
            raise NotImplementedError("train_model_stack_device trains a StackedGCN; the one-layer GCN has "
                                      "train_model_device")
        env, world = self.env, self.env.world
        flock = isinstance(env.scenario, FlockingScenario)
        cohesion = isinstance(env.scenario, CohesionScenario)
        if not (flock or cohesion or isinstance(env.scenario, _KernelScenario)):
            raise NotImplementedError("the stacked device loop covers the GoTo, ObstacleAvoidance, Flocking and Cohesion "
                                      "rewards; train other scenarios with train_model_stepwise")
        B, n, dev = env.num_envs, env.n_agents, env.device
        G = int(config.get("graphs_per_update", 32))
        episodes = int(config["episodes"])
        ring = self.replay_buffer.ring
        cfg = ops.clone_config(self.graph_cfg, num_envs=B)
        rank = torch.distributed.get_rank() if parallel.world_size() > 1 else 0
        multi = parallel.world_size() > 1
        reward = shaping = None
        if flock:
            reward, shaping = env.scenario._spec(), env.scenario.shaping
        elif cohesion:
            reward = ops.reward_spec(_lib.REWARD_COHESION, B, n, agent_radius=world.cfg.agent_radius,
                                     sigma=env.scenario.sigma)
        tt = ops.StackTrainTick(cfg, self.stack_spec, ring, graphs_per_update=G,
                                update_target_every=int(config.get("update_target_every", 200)),
                                gamma=float(config.get("gamma", 0.99)), loss_scale=parallel.global_loss_scale(G, n),
                                lr=self.lr, betas=self.betas, eps=self.eps, max_norm=self.max_norm, rng_seed=self.seed,
                                sample_seed=int(config.get("sample_seed", self.seed)) + 7919 * rank,
                                env_offset=int(config.get("env_offset", rank * B)), reward=reward, shaping=shaping)
        if cohesion:
            env.reset()
            start = world.state.clone()

            def reset():
                world.state.copy_(start)
        else:
            spec = ops.reset_spec(cfg.scenario, random=bool(getattr(env.scenario, "random", True)),
                                  seed=int(config.get("reset_seed", self.seed)), env_offset=tt.hyper.env_offset,
                                  shared_center=bool(config.get("shared_center", False)), flocking=flock)

            def reset():
                ops.reset_random(cfg, spec, world.state, ctl=tt.ctl)
                if flock:
                    ops.scenario_reward(reward, world.state, shaping, reset=True)
        parallel.require_equal_shards(B, ring.size, ring.position, ring.capacity, G)
        parallel.broadcast_weights(self.w)
        self.w_target.copy_(self.w)
        tt.load_cursor(int(config.get("start_tick", 0)), self.opt_step, config["epsilon"], 0)
        returns = torch.zeros(B, n, dtype=torch.float32, device=dev)
        hits = torch.zeros(B, dtype=torch.int32, device=dev)
        stats = torch.zeros(episodes, 4, dtype=torch.float32, device=dev)
        tt.peers = parallel.make_peer_exchange(dev, stride=_lib.XCHG_STACK_STRIDE)
        nccl = multi and tt.peers is None

        def episode():
            reset()
            for _ in range(env.max_steps):
                if not multi:
                    tt.tick(self.w, self.w_target, self.exp_avg, self.exp_avg_sq, world.state, returns, hits)
                    continue
                tt.grad_phase(self.w, self.w_target, world.state, returns, hits)
                if nccl:
                    torch.distributed.all_reduce(tt.grad_loss)
                tt.apply_phase(self.w, self.w_target, self.exp_avg, self.exp_avg_sq)
            tt.episode_end(returns, hits, stats, config["epsilon"], config["epsilon_decay"], config["min_epsilon"])

        _run_episodes(episode, episodes, bool(config.get("cuda_graph", True)), dev)
        self.opt_step = tt.read_cursor()["opt_step"]
        self._grad.copy_(tt.grad)
        self._loss.copy_(tt.loss)
        self.sync_modules()
        out = stats.cpu()
        self.episode_losses.extend(out[:, 2].tolist())
        return out

    def evaluate_policy(self, eval_episodes):
        """train:206-223 (greedy episodes, mean agent-0 return)."""
        total = 0
        n = self.env.n_agents
        cfg = ops.clone_config(self.graph_cfg, num_envs=self.env.num_envs)
        if self.stack_spec is not None:
            return self._evaluate_stack(cfg, eval_episodes)
        for _ in range(eval_episodes):
            self.env.reset()
            flock = isinstance(self.env.scenario, FlockingScenario)
            out = ops.rollout(cfg, self.w, self.env.world.state, self.env.max_steps,
                              trace=dict(rewards=True, flags=True, dist=True),
                              flocking=self.env.scenario._spec() if flock else None,
                              shaping=self.env.scenario.shaping if flock else None)
            self.env.steps += self.env.max_steps
            self.env.world.adopt_rollout(out)
            total += out["returns"][0, 0].item()
        return total / eval_episodes

    def _evaluate_stack(self, cfg, eval_episodes):
        """evaluate_policy for a stacked network: ``swarm_rollout_stack`` with the scenario's reward (the world's own,
        Flocking with its shaping memory, or Cohesion's per-agent reward)."""
        total = 0
        env = self.env
        for _ in range(eval_episodes):
            env.reset()
            reward = shaping = None
            if isinstance(env.scenario, FlockingScenario):
                reward, shaping = env.scenario._spec(), env.scenario.shaping
            elif isinstance(env.scenario, CohesionScenario):
                reward = ops.reward_spec(_lib.REWARD_COHESION, env.num_envs, env.n_agents,
                                         agent_radius=env.world.cfg.agent_radius, sigma=env.scenario.sigma)
            elif not isinstance(env.scenario, _KernelScenario):
                raise NotImplementedError("evaluate_policy of a StackedGCN covers the GoTo, ObstacleAvoidance, Flocking and "
                                          "Cohesion rewards")
            out = ops.rollout_stack(cfg, self.stack_spec, self.w, env.world.state, env.max_steps, reward=reward,
                                    shaping=shaping)
            env.steps += env.max_steps
            env.world.version += 1                 # the state moved under the world: version-keyed caches drop
            env.world._download()
            total += out["returns"][0, 0].item()
        return total / eval_episodes

    def save_metrics_to_csv(self):
        """train:225-231, including its row quirk (Loss column = episode_losses[i // 10])."""
        os.makedirs(self.stats_path, exist_ok=True)
        with open(f"{self.stats_path}/experiment_{self.experiment}-seed_{self.seed}.csv", mode="w", newline="") as file:
            writer = csv.writer(file)
            writer.writerow(["Episode", "Reward", "Loss"])
            for i in range(len(self.episode_losses)):
                if (i + 1) % 10 == 0:
                    writer.writerow([i, self.episode_rewards[i // 10].item(), self.episode_losses[i // 10]])


def _run_episodes(episode, episodes: int, cuda_graph: bool, dev) -> None:
    """Run ``episode()`` ``episodes`` times: with ``cuda_graph`` (and more than one episode) once eagerly -- kernel
    attributes set, an NCCL communicator warm -- then captured once and replayed for the others."""
    done = 0
    if cuda_graph and episodes > 1:
        episode()
        done = 1
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.graph(graph, stream=side):
            episode()
        for _ in range(episodes - 1):            # capture records, it does not execute
            graph.replay()
        done = episodes
    for _ in range(episodes - done):
        episode()


def set_seed(seed):
    """train:233-239."""
    random.seed(seed)
    torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed_all(seed)
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False
