"""Thin tensor-level wrappers over the C ABI (include/swarm_b200.h).

Tensors are only containers for device memory here: every function validates shapes/dtypes, passes raw
pointers plus the current CUDA stream to libswarm_b200.so and returns the output tensors.  Nothing
is computed in PyTorch.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from ._lib import SwarmConfig, SwarmReplay, SwarmRolloutOptions, SwarmTrace, check, lib, ptr, stream_ptr


def make_config(scenario: int, num_envs: int, n_agents: int, graph_mode: int = _lib.GRAPH_COMPLETE,
                knn_k: int = 10, graph_radius: float = 0.35) -> SwarmConfig:
    cfg = _lib.default_config(scenario, num_envs, n_agents)
    cfg.graph_radius = graph_radius
    cfg.graph_mode = graph_mode
    cfg.knn_k = knn_k
    return cfg


def clone_config(cfg: SwarmConfig, **updates) -> SwarmConfig:
    out = SwarmConfig()
    C.memmove(C.byref(out), C.byref(cfg), C.sizeof(SwarmConfig))
    for k, v in updates.items():
        setattr(out, k, v)
    return out


def edges_per_env(cfg: SwarmConfig) -> int:
    return int(lib().swarm_edges_per_env(C.byref(cfg)))


def _expect(t: torch.Tensor, dtype: torch.dtype, numel: int, name: str) -> None:
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if t.numel() != numel:
        raise ValueError(f"{name}: expected {numel} elements, got {t.numel()}")


def reset_grid(cfg: SwarmConfig, centers: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """centers f32[B,2] -> state f32[B,N,4]."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(centers, torch.float32, B * 2, "centers")
    state = out if out is not None else torch.empty(B, N, 4, dtype=torch.float32, device=centers.device)
    _expect(state, torch.float32, B * N * 4, "state")
    check(lib().swarm_reset_grid(C.byref(cfg), ptr(centers), ptr(state), stream_ptr(centers.device)))
    return state


def sim_step(cfg: SwarmConfig, state: torch.Tensor, actions: torch.Tensor, *, state_out: Optional[torch.Tensor] = None,
             want_obs: bool = True, want_contact: bool = False) -> Dict[str, torch.Tensor]:
    """One world step.  state f32[B,N,4], actions int32[B,N] -> dict(state, rewards, flags, [contact], [obs])."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(actions, torch.int32, B * N, "actions")
    dev = state.device
    out_state = state_out if state_out is not None else torch.empty_like(state)
    rewards = torch.empty(B, N, dtype=torch.float32, device=dev)
    flags = torch.empty(B, N, dtype=torch.uint8, device=dev)
    contact = torch.empty(B, N, dtype=torch.int32, device=dev) if want_contact else None
    obs = torch.empty(B, N, 6, dtype=torch.float32, device=dev) if want_obs else None
    dist = torch.empty(B, N, 2, dtype=torch.float32, device=dev)
    check(lib().swarm_sim_step(C.byref(cfg), ptr(state), ptr(actions), ptr(out_state), ptr(rewards), ptr(flags),
                               ptr(contact), ptr(obs), ptr(dist), stream_ptr(dev)))
    res = {"state": out_state, "rewards": rewards, "flags": flags, "dist": dist}
    if contact is not None:
        res["contact"] = contact
    if obs is not None:
        res["obs"] = obs
    return res


def graph_build(cfg: SwarmConfig, state: torch.Tensor, want_neighbours: bool = False
                ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """edges int32[B,2,E] (env-local ids) and, for kNN, the topk index table int32[B,N,k].  Radius graphs (extension)
    return the padded edge block int32[B,2,N(N-1)+1] (-1 past the env's edge count) and the counts int32[B]."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    E = edges_per_env(cfg)
    edges = torch.empty(B, 2, E, dtype=torch.int32, device=state.device)
    if cfg.graph_mode == _lib.GRAPH_RADIUS:
        counts = torch.empty(B, dtype=torch.int32, device=state.device)
        check(lib().swarm_graph_build_radius(C.byref(cfg), ptr(state), ptr(edges), ptr(counts), stream_ptr(state.device)))
        return edges, counts
    nbr = None
    if want_neighbours and cfg.graph_mode == _lib.GRAPH_KNN:
        nbr = torch.empty(B, N, cfg.knn_k, dtype=torch.int32, device=state.device)
    check(lib().swarm_graph_build(C.byref(cfg), ptr(state), ptr(edges), ptr(nbr), stream_ptr(state.device)))
    return edges, nbr


def gatq_forward(cfg: SwarmConfig, weights: torch.Tensor, state: torch.Tensor, want_q: bool = True,
                 want_actions: bool = True) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """Structured GCN.forward on the per-env graph: q f32[B,N,9], greedy actions int32[B,N]."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(weights, torch.float32, _lib.W_COUNT, "weights")
    dev = state.device
    q = torch.empty(B, N, 9, dtype=torch.float32, device=dev) if want_q else None
    act = torch.empty(B, N, dtype=torch.int32, device=dev) if want_actions else None
    check(lib().swarm_gatq_forward(C.byref(cfg), ptr(weights), ptr(state), ptr(q), ptr(act), stream_ptr(dev)))
    return q, act


class ReplayRing:
    """Device replay ring of whole-swarm transitions (GraphReplayBuffer, train:25-48), state-only SoA."""

    def __init__(self, capacity: int, n_agents: int, device):
        self.capacity, self.n_agents = int(capacity), int(n_agents)
        self.state = torch.zeros(capacity, n_agents, 4, dtype=torch.float32, device=device)
        self.next_state = torch.zeros(capacity, n_agents, 4, dtype=torch.float32, device=device)
        self.actions = torch.zeros(capacity, n_agents, dtype=torch.uint8, device=device)
        self.rewards = torch.zeros(capacity, n_agents, dtype=torch.float32, device=device)
        self.position = 0          # next slot to write (train:30,36)
        self.size = 0              # len(buffer)

    def struct(self) -> SwarmReplay:
        return SwarmReplay(ptr(self.state), ptr(self.next_state), ptr(self.actions), ptr(self.rewards), self.capacity)

    def advance(self, n: int) -> None:
        self.position = (self.position + n) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def __len__(self) -> int:
        return self.size


_KNN_MEMO: Dict[Tuple[str, int, int], torch.Tensor] = {}
KNN_MEMO_ENTRIES = 1 << 17          # 1 MB: stays L2 resident


def knn_memo_table(device, n_agents: int, knn_k: int, fresh: bool = False) -> torch.Tensor:
    """The cached memo table of kNN boundary-tie patterns for (device, n_agents, knn_k) (SwarmRolloutOptions.knn_memo);
    ``fresh`` clears it."""
    key = (str(torch.device(device)), int(n_agents), int(knn_k))
    t = _KNN_MEMO.get(key)
    if t is None:
        t = torch.zeros(KNN_MEMO_ENTRIES, dtype=torch.int64, device=device)
        _KNN_MEMO[key] = t
    elif fresh:
        t.zero_()
    return t


def rollout(cfg: SwarmConfig, weights: torch.Tensor, state: torch.Tensor, ticks: int, *,
            forced_actions: Optional[torch.Tensor] = None, returns: Optional[torch.Tensor] = None,
            hits: Optional[torch.Tensor] = None, trace: Optional[Dict[str, bool]] = None,
            epsilon: float = 0.0, rng_seed: int = 0, rng_tick0: int = 0, env_offset: int = 0,
            replay: Optional[ReplayRing] = None, flocking: Optional["_lib.SwarmRewardSpec"] = None,
            shaping: Optional[torch.Tensor] = None, knn_memo="auto") -> Dict[str, torch.Tensor]:
    """Fused (epsilon-)greedy rollout, in place on ``state``.  ``trace`` names the per-tick records to keep
    (any of state, actions, q, rewards, flags, contact, edges, dist).  With ``replay`` every tick's B
    transitions are pushed into the ring (and its cursor advanced).  With ``flocking`` (a Flocking reward spec, cfg =
    the GoTo world) the reward of every tick is the Flocking collective reward and ``shaping`` f32[B,N,2] carries the
    ``previous_*`` memory in and out.  ``knn_memo``: the memo table of kNN boundary-tie patterns (``"auto"`` = one
    cached int64 table per (device, n_agents, knn_k), ``None`` = no table, or a caller-owned zero-initialised int64
    tensor with a power-of-two length); it only saves time, results never depend on it."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(weights, torch.float32, _lib.W_COUNT, "weights")
    dev = state.device
    if isinstance(knn_memo, str):
        knn_memo = knn_memo_table(dev, N, cfg.knn_k) if (cfg.graph_mode == _lib.GRAPH_KNN and N <= 12) else None
    if forced_actions is not None:
        _expect(forced_actions, torch.int32, ticks * B * N, "forced_actions")
    if returns is None:
        returns = torch.zeros(B, N, dtype=torch.float32, device=dev)
    if hits is None:
        hits = torch.zeros(B, dtype=torch.int32, device=dev)
    _expect(returns, torch.float32, B * N, "returns")
    _expect(hits, torch.int32, B, "hits")
    out: Dict[str, torch.Tensor] = {"state": state, "returns": returns, "hits": hits}
    tr = None
    if trace:
        tr = SwarmTrace()
        E = edges_per_env(cfg)
        shapes = {"state": ((ticks, B, N, 4), torch.float32), "actions": ((ticks, B, N), torch.int32),
                  "q": ((ticks, B, N, 9), torch.float32), "rewards": ((ticks, B, N), torch.float32),
                  "flags": ((ticks, B, N), torch.uint8), "contact": ((ticks, B, N), torch.int32),
                  "edges": ((ticks, B, 2, E), torch.int32), "dist": ((ticks, B, N, 2), torch.float32)}
        for name, on in trace.items():
            if not on:
                continue
            shape, dt = shapes[name]
            t = torch.empty(shape, dtype=dt, device=dev)
            setattr(tr, name, ptr(t))
            out["trace_" + name] = t
    opts = SwarmRolloutOptions()
    opts.forced_actions = ptr(forced_actions)
    opts.epsilon = float(epsilon)
    opts.rng_seed = int(rng_seed) & 0xFFFFFFFFFFFFFFFF
    opts.rng_tick0 = int(rng_tick0)
    opts.env_offset = int(env_offset)
    if flocking is not None:
        if shaping is None:
            raise ValueError("Flocking needs the shaping buffer f32[B,N,2]")
        _expect(shaping, torch.float32, B * N * 2, "shaping")
        opts.flocking = C.addressof(flocking)
        opts.flocking_shaping = ptr(shaping)
        out["shaping"] = shaping
    if knn_memo is not None:
        _expect(knn_memo, torch.int64, knn_memo.numel(), "knn_memo")
        opts.knn_memo = ptr(knn_memo)
        opts.knn_memo_entries = knn_memo.numel()
    rstruct = None
    if replay is not None:
        if replay.n_agents != N:
            raise ValueError("replay ring was built for a different n_agents")
        rstruct = replay.struct()
        opts.replay = C.pointer(rstruct)
        opts.replay_cursor = replay.position
    check(lib().swarm_rollout(C.byref(cfg), ptr(weights), ptr(state), int(ticks), C.byref(opts), ptr(returns),
                              ptr(hits), C.byref(tr) if tr is not None else None, stream_ptr(dev)))
    if replay is not None:
        replay.advance(ticks * B)
    return out


def replay_push(cfg: SwarmConfig, ring: ReplayRing, state: torch.Tensor, actions: torch.Tensor,
                rewards: torch.Tensor, next_state: torch.Tensor) -> None:
    """GraphReplayBuffer.push for the B envs of cfg (train:32-36)."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(next_state, torch.float32, B * N * 4, "next_state")
    _expect(actions, torch.int32, B * N, "actions")
    _expect(rewards, torch.float32, B * N, "rewards")
    rs = ring.struct()
    check(lib().swarm_replay_push(C.byref(cfg), C.byref(rs), ring.position, ptr(state), ptr(actions), ptr(rewards),
                                  ptr(next_state), stream_ptr(state.device)))
    ring.advance(B)


def replay_gather(ring: ReplayRing, indices: torch.Tensor) -> Dict[str, torch.Tensor]:
    """GraphReplayBuffer.sample materialisation (train:38-45) for the given slot indices int64[G]."""
    if indices.dtype != torch.int64:
        raise TypeError("indices must be int64")
    G, N, dev = indices.numel(), ring.n_agents, ring.state.device
    cfg = make_config(_lib.SCENARIO_GOTO, max(G, 1), N)
    out = {"state": torch.empty(G, N, 4, dtype=torch.float32, device=dev),
           "actions": torch.empty(G, N, dtype=torch.int32, device=dev),
           "rewards": torch.empty(G, N, dtype=torch.float32, device=dev),
           "next_state": torch.empty(G, N, 4, dtype=torch.float32, device=dev)}
    rs = ring.struct()
    check(lib().swarm_replay_gather(C.byref(cfg), C.byref(rs), ptr(indices), G, ptr(out["state"]), ptr(out["actions"]),
                                    ptr(out["rewards"]), ptr(out["next_state"]), stream_ptr(dev)))
    return out


def dqn_grad(cfg: SwarmConfig, online: torch.Tensor, target: torch.Tensor, batch: ReplayRing,
             indices: Optional[torch.Tensor], n_graphs: int, gamma: float = 0.99, loss_scale: Optional[float] = None,
             want_td: bool = False, grad: Optional[torch.Tensor] = None, loss: Optional[torch.Tensor] = None
             ) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
    """train_step_dqn's loss + gradient (train:116-124) over n_graphs transitions of ``batch`` (slots
    ``indices`` if given).  Returns (grad f32[1673], loss f32[1], td f32[G,N] or None)."""
    N, dev = cfg.n_agents, online.device
    _expect(online, torch.float32, _lib.W_COUNT, "online weights")
    _expect(target, torch.float32, _lib.W_COUNT, "target weights")
    if indices is not None:
        if indices.dtype != torch.int64 or indices.numel() != n_graphs:
            raise TypeError("indices must be int64[n_graphs]")
    if loss_scale is None:
        loss_scale = 1.0 / (n_graphs * N)
    grad = grad if grad is not None else torch.empty(_lib.W_COUNT, dtype=torch.float32, device=dev)
    loss = loss if loss is not None else torch.empty(1, dtype=torch.float32, device=dev)
    td = torch.empty(n_graphs, N, dtype=torch.float32, device=dev) if want_td else None
    wb = int(lib().swarm_dqn_workspace_bytes(C.byref(cfg), n_graphs))
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    rs = batch.struct()
    check(lib().swarm_dqn_grad(C.byref(cfg), ptr(online), ptr(target), C.byref(rs), ptr(indices), n_graphs, float(gamma),
                               float(loss_scale), ptr(grad), ptr(loss), ptr(td), ptr(ws), wb, stream_ptr(dev)))
    return grad, loss, td


def adam_clip_step(weights: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
                   step: int, lr: float = 1e-3, betas: Tuple[float, float] = (0.9, 0.999), eps: float = 1e-8,
                   max_norm: float = 1.0, target: Optional[torch.Tensor] = None,
                   grad_norm: Optional[torch.Tensor] = None) -> None:
    """clip_grad_norm_(max_norm) + torch.optim.Adam step on the packed weights, in place (train:125-126);
    optionally copies the new weights into ``target`` (train:131-133)."""
    for name, t in (("weights", weights), ("grad", grad), ("exp_avg", exp_avg), ("exp_avg_sq", exp_avg_sq)):
        _expect(t, torch.float32, _lib.W_COUNT, name)
    check(lib().swarm_adam_clip_step(ptr(weights), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq), int(step), float(lr),
                                     float(betas[0]), float(betas[1]), float(eps), float(max_norm), ptr(target),
                                     ptr(grad_norm), stream_ptr(weights.device)))


def reset_spec(scenario: int, random: bool = True, seed: int = 0, env_offset: int = 0,
               shared_center: bool = False, flocking: bool = False) -> _lib.SwarmResetSpec:
    """Start-centre distribution of the scenario's reset_world_at (go_to:84-88, oa:100-102; ``flocking``:
    flocking_scenario.py:94-98, position_range (-1, 1) + N((-0.6, 0.6), 0.4))."""
    sp = _lib.SwarmResetSpec()
    if flocking:
        sp.base_x, sp.base_y, sp.mean_x, sp.mean_y, sp.std_x, sp.std_y = -1.0, 1.0, -0.6, 0.6, 0.4, 0.4
    elif scenario == _lib.SCENARIO_GOTO:
        sp.base_x, sp.base_y, sp.mean_x, sp.mean_y, sp.std_x, sp.std_y = 1.5, -1.5, -0.6, 0.6, 0.4, 0.4
    else:
        sp.base_x, sp.base_y, sp.mean_x, sp.mean_y = 0.6, -0.6, 0.0, 0.0
        sp.std_x = sp.std_y = 0.1 if random else 0.0
    sp.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    sp.env_offset = int(env_offset)
    sp.shared_center = 1 if shared_center else 0
    return sp


def reward_spec(kind: int, num_envs: int, n_agents: int, **overrides) -> _lib.SwarmRewardSpec:
    """Reference constants of the Flocking / Cohesion reward (flocking:10-21, cohesion:10-23); keyword overrides."""
    sp = _lib.SwarmRewardSpec()
    lib().swarm_default_reward_spec(C.byref(sp), kind, num_envs, n_agents)
    for k, v in overrides.items():
        if not hasattr(sp, k):
            raise TypeError(f"SwarmRewardSpec has no field {k!r}")
        setattr(sp, k, v)
    return sp


def scenario_reward(spec: _lib.SwarmRewardSpec, state: torch.Tensor, shaping: Optional[torch.Tensor] = None, *,
                    reset: bool = False, env_index: Optional[int] = None, want_terms: bool = False):
    """swarm_scenario_reward on state f32[B,N,4].  Flocking: shaping f32[B,N,2] is updated in place; returns the
    collective reward f32[B] (None for a reset call).  Cohesion: returns f32[B,N].  ``want_terms`` adds f32[B,N,4].
    Above 128 agents (up to 4 096) it runs ``scenario_reward_large``."""
    return _scenario_reward(spec, state, shaping, reset, env_index, want_terms, spec.n_agents > 128)


def scenario_reward_large(spec: _lib.SwarmRewardSpec, state: torch.Tensor, shaping: Optional[torch.Tensor] = None, *,
                          reset: bool = False, env_index: Optional[int] = None, want_terms: bool = False):
    """``scenario_reward`` through swarm_scenario_reward_large (any 2 <= N <= 4 096; its workspace allocated here)."""
    return _scenario_reward(spec, state, shaping, reset, env_index, want_terms, True)


def _scenario_reward(spec, state, shaping, reset, env_index, want_terms, large):
    B, N = spec.num_envs, spec.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    dev = state.device
    flocking = spec.kind == _lib.REWARD_FLOCKING
    if flocking:
        if shaping is None:
            raise ValueError("Flocking needs the shaping buffer f32[B,N,2]")
        _expect(shaping, torch.float32, B * N * 2, "shaping")
    call = _lib.SwarmRewardSpec.from_buffer_copy(spec)
    call.reset = 1 if reset else 0
    call.env_index = -1 if env_index is None else int(env_index)
    reward = None
    if not reset:
        reward = torch.zeros(B, dtype=torch.float32, device=dev) if flocking else \
            torch.zeros(B, N, dtype=torch.float32, device=dev)
    terms = torch.zeros(B, N, 4, dtype=torch.float32, device=dev) if (want_terms and not reset) else None
    if large:
        wb = int(lib().swarm_scenario_reward_large_workspace_bytes(C.byref(call)))
        ws = torch.empty(wb, dtype=torch.uint8, device=dev) if wb > 0 else None
        check(lib().swarm_scenario_reward_large(C.byref(call), ptr(state), ptr(shaping) if flocking else None, ptr(reward),
                                                ptr(terms), ptr(ws), wb, stream_ptr(dev)))
    else:
        check(lib().swarm_scenario_reward(C.byref(call), ptr(state), ptr(shaping) if flocking else None, ptr(reward),
                                          ptr(terms), stream_ptr(dev)))
    return (reward, terms) if want_terms else reward


def reset_random(cfg: SwarmConfig, spec: _lib.SwarmResetSpec, state: torch.Tensor, *, ctl: Optional[torch.Tensor] = None,
                 episode: int = 0, centers_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Device-side reset_world_at for every env: start centres from the counter RNG (episode number from the device
    cursor ``ctl`` when given), agents on the grid, velocities zero."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    if centers_out is not None:
        _expect(centers_out, torch.float32, B * 2, "centers_out")
    check(lib().swarm_reset_random(C.byref(cfg), C.byref(spec), ptr(ctl), int(episode), ptr(centers_out), ptr(state),
                                   stream_ptr(state.device)))
    return state


class _TrainCursor:
    """The device cursor of a device-driven train tick (``TrainTick``, ``StackTrainTick``): the tick number, replay
    cursor / fill, optimiser step and epsilon held in a 48-byte device struct that the kernels advance themselves, the
    hyper-parameters, and the host-side bookkeeping around them.  Subclasses hold ``loss``, the last update's loss."""

    CTL_WORDS = 6      # int64 words: tick, ring_cursor, ring_size, opt_step, (epsilon f32 | updating i32), episode

    def __init__(self, cfg: SwarmConfig, ring: ReplayRing, graphs_per_update: int, update_target_every: int, gamma: float,
                 loss_scale: Optional[float], lr: float, betas, eps: float, max_norm: float, rng_seed: int,
                 sample_seed: int, env_offset: int):
        dev = ring.state.device
        self.cfg, self.ring = cfg, ring
        G = int(graphs_per_update)
        h = _lib.SwarmTrainHyper()
        h.lr, h.beta1, h.beta2, h.eps, h.max_norm = float(lr), float(betas[0]), float(betas[1]), float(eps), float(max_norm)
        h.rng_seed = int(rng_seed) & 0xFFFFFFFFFFFFFFFF
        h.sample_seed = int(sample_seed) & 0xFFFFFFFFFFFFFFFF
        h.env_offset = int(env_offset)
        h.graphs_per_update, h.update_target_every = G, int(update_target_every)
        h.gamma = float(gamma)
        h.loss_scale = float(loss_scale) if loss_scale is not None else 1.0 / (G * cfg.n_agents)
        self.hyper = h
        assert C.sizeof(_lib.SwarmTrainCtl) == 8 * self.CTL_WORDS
        self.ctl = torch.zeros(self.CTL_WORDS, dtype=torch.int64, device=dev)
        self.indices = torch.zeros(G, dtype=torch.int64, device=dev)
        self._rstruct = ring.struct()

    # -- cursor <-> host bookkeeping ---------------------------------------------------------------
    def load_cursor(self, tick: int, opt_step: int, epsilon: float, episode: int = 0) -> None:
        """Write the host-side counters (tick, ring position / size, optimiser step, epsilon) into the device cursor."""
        words = torch.tensor([int(tick), self.ring.position, self.ring.size, int(opt_step), 0, int(episode)],
                             dtype=torch.int64)
        words.view(torch.float32)[8] = float(epsilon)
        self.ctl.copy_(words)

    def set_epsilon(self, epsilon: float) -> None:
        self.ctl.view(torch.float32)[8:9].fill_(float(epsilon))

    def read_cursor(self) -> Dict[str, float]:
        """Read the device cursor back (one small D2H copy) and update the ring's host-side position / size."""
        words = self.ctl.cpu()
        self.ring.position, self.ring.size = int(words[1]), int(words[2])
        return {"tick": int(words[0]), "opt_step": int(words[3]), "epsilon": float(words.view(torch.float32)[8]),
                "updating": int(words.view(torch.int32)[9]), "episode": int(words[5])}

    def episode_end(self, returns: torch.Tensor, hits: Optional[torch.Tensor], stats: Optional[torch.Tensor],
                    epsilon0: float, epsilon_decay: float, min_epsilon: float) -> None:
        """End-of-episode bookkeeping on the device (swarm_episode_end): stats row, accumulators zeroed, epsilon
        schedule (train:179-199), episode counter."""
        max_ep = 0 if stats is None else stats.shape[0]
        check(lib().swarm_episode_end(C.byref(self.cfg), ptr(self.ctl), ptr(returns), ptr(hits), ptr(self.loss), ptr(stats),
                                      max_ep, float(epsilon0), float(epsilon_decay), float(min_epsilon),
                                      stream_ptr(returns.device)))


class TrainTick(_TrainCursor):
    """Device-driven train tick (swarm_train_tick_grad / swarm_train_tick_apply): one iteration of the loop body of
    train_gcn_dqn.py:153-178 for all B envs, with the tick number, replay cursor / fill, optimiser step and epsilon
    held in a 48-byte device struct that the kernels advance themselves.  No launch argument changes from tick to
    tick, so ``grad_phase`` / ``apply_phase`` can be captured in a CUDA graph and replayed (``DQNTrainer``)."""

    def __init__(self, cfg: SwarmConfig, ring: ReplayRing, *, graphs_per_update: int = 32, update_target_every: int = 200,
                 gamma: float = 0.99, loss_scale: Optional[float] = None, lr: float = 1e-3, betas=(0.9, 0.999),
                 eps: float = 1e-8, max_norm: float = 1.0, rng_seed: int = 0, sample_seed: int = 0, env_offset: int = 0,
                 flocking: Optional["_lib.SwarmRewardSpec"] = None, shaping: Optional[torch.Tensor] = None):
        super().__init__(cfg, ring, graphs_per_update, update_target_every, gamma, loss_scale, lr, betas, eps, max_norm,
                         rng_seed, sample_seed, env_offset)
        dev = ring.state.device
        G = int(graphs_per_update)
        h = self.hyper
        if flocking is not None:
            # the tick's reward is the Flocking collective reward; `shaping` f32[B,N,2] is its memory (in / out)
            if shaping is None:
                raise ValueError("Flocking needs the shaping buffer f32[B,N,2]")
            _expect(shaping, torch.float32, cfg.num_envs * cfg.n_agents * 2, "shaping")
            self._flocking, self._shaping = _lib.SwarmRewardSpec.from_buffer_copy(flocking), shaping   # kept alive
            h.flocking = C.addressof(self._flocking)
            h.flocking_shaping = ptr(shaping)
        # gradient and loss share one buffer so that a data-parallel trainer all-reduces both in one collective
        self.grad_loss = torch.zeros(_lib.W_COUNT + 1, dtype=torch.float32, device=dev)
        self.grad = self.grad_loss[:_lib.W_COUNT]
        self.loss = self.grad_loss[_lib.W_COUNT:]
        gcfg = clone_config(cfg, num_envs=G)
        self._ws_bytes = int(lib().swarm_dqn_workspace_bytes(C.byref(gcfg), G))
        self.workspace = torch.empty(max(self._ws_bytes, 256), dtype=torch.uint8, device=dev)
        self.peers = None          # parallel.PeerExchange: fuse the gradient all-reduce into apply_phase

    # -- the two phases -------------------------------------------------------------------------------
    def grad_phase(self, weights: torch.Tensor, target: torch.Tensor, state: torch.Tensor, returns: torch.Tensor,
                   hits: torch.Tensor) -> None:
        dev = state.device
        check(lib().swarm_train_tick_grad(C.byref(self.cfg), C.byref(self.hyper), ptr(self.ctl), ptr(weights), ptr(target),
                                          ptr(state), ptr(returns), ptr(hits), C.byref(self._rstruct), ptr(self.indices),
                                          ptr(self.grad), ptr(self.loss), ptr(self.workspace), self._ws_bytes,
                                          stream_ptr(dev)))

    def apply_phase(self, weights: torch.Tensor, target: torch.Tensor, exp_avg: torch.Tensor,
                    exp_avg_sq: torch.Tensor) -> None:
        """clip + Adam (+ target sync) and cursor advance.  With ``self.peers`` set (``parallel.PeerExchange``) the
        gradient + loss are first summed over the ranks inside the same kernel through NVLink peer memory."""
        peers = C.byref(self.peers.struct) if self.peers is not None else None
        check(lib().swarm_train_tick_apply(C.byref(self.cfg), C.byref(self.hyper), ptr(self.ctl), ptr(weights), ptr(target),
                                           ptr(exp_avg), ptr(exp_avg_sq), ptr(self.grad_loss), self.ring.capacity, peers,
                                           stream_ptr(weights.device)))

    def tick(self, weights: torch.Tensor, target: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
             state: torch.Tensor, returns: torch.Tensor, hits: torch.Tensor) -> None:
        """``grad_phase`` + ``apply_phase`` as one library call (swarm_train_tick): the same bits, one launch less per
        tick for small update batches (the partial gradients are summed inside the clip + Adam kernel).  For trainers
        that need nothing between the phases: one GPU, or ``self.peers`` set."""
        peers = C.byref(self.peers.struct) if self.peers is not None else None
        check(lib().swarm_train_tick(C.byref(self.cfg), C.byref(self.hyper), ptr(self.ctl), ptr(weights), ptr(target),
                                     ptr(exp_avg), ptr(exp_avg_sq), ptr(state), ptr(returns), ptr(hits),
                                     C.byref(self._rstruct), ptr(self.indices), ptr(self.grad_loss), ptr(self.workspace),
                                     self._ws_bytes, peers, stream_ptr(state.device)))


class StackTrainTick(_TrainCursor):
    """``TrainTick`` for a stacked network (swarm_train_tick_stack): one call per tick runs the rollout tick, the slot
    draw + gradient, the partial-sum reduce and clip + Adam (+ target sync) with the cursor on the device, so the ticks
    of an episode capture into a CUDA graph.  ``reward``: None for the world's own reward (GoTo / ObstacleAvoidance), or
    a Flocking / Cohesion ``reward_spec`` on the GoTo world (Flocking: ``shaping`` f32[B,N,2] is its memory, in / out).
    Data-parallel trainers run the tick as ``grad_phase`` + ``apply_phase`` (swarm_train_tick_stack_grad /
    swarm_train_tick_stack_apply): with ``self.peers`` set (``parallel.PeerExchange`` of ``_lib.XCHG_STACK_STRIDE``
    words) the gradient phase sums ``grad_loss`` over the ranks itself, otherwise the trainer all-reduces ``grad_loss``
    between the phases."""

    def __init__(self, cfg: SwarmConfig, spec, ring: ReplayRing, *, graphs_per_update: int = 32,
                 update_target_every: int = 200, gamma: float = 0.99, loss_scale: Optional[float] = None, lr: float = 1e-3,
                 betas=(0.9, 0.999), eps: float = 1e-8, max_norm: float = 1.0, rng_seed: int = 0, sample_seed: int = 0,
                 env_offset: int = 0, reward: Optional["_lib.SwarmRewardSpec"] = None,
                 shaping: Optional[torch.Tensor] = None):
        super().__init__(cfg, ring, graphs_per_update, update_target_every, gamma, loss_scale, lr, betas, eps, max_norm,
                         rng_seed, sample_seed, env_offset)
        dev = ring.state.device
        G = int(graphs_per_update)
        self.spec = spec
        self._reward = _lib.SwarmRewardSpec.from_buffer_copy(reward) if reward is not None else None    # kept alive
        self._shaping = shaping
        if shaping is not None:
            _expect(shaping, torch.float32, cfg.num_envs * cfg.n_agents * 2, "shaping")
        self.count = int(lib().swarm_stack_weight_count(C.byref(spec)))
        self.grad_loss = torch.zeros(self.count + 1, dtype=torch.float32, device=dev)
        self.grad = self.grad_loss[:self.count]
        self.loss = self.grad_loss[self.count:]
        self._ws_bytes = int(lib().swarm_dqn_stack_workspace_bytes(C.byref(cfg), C.byref(spec), G))
        self.workspace = torch.empty(max(self._ws_bytes, 256), dtype=torch.uint8, device=dev)
        self.peers = None          # parallel.PeerExchange: sum grad_loss over the ranks inside grad_phase

    def _expect_weights(self, **tensors) -> None:
        for name, t in tensors.items():
            _expect(t, torch.float32, self.count, name)

    # -- the two phases -------------------------------------------------------------------------------
    def grad_phase(self, weights: torch.Tensor, target: torch.Tensor, state: torch.Tensor, returns: torch.Tensor,
                   hits: torch.Tensor) -> None:
        """Rollout tick, slot draw + gradient and the partial-sum reduce; with ``self.peers`` set, ``grad_loss`` then
        holds the sum over the ranks."""
        self._expect_weights(weights=weights, target=target)
        peers = None
        if self.peers is not None:
            if self.peers.stride != _lib.XCHG_STACK_STRIDE:        # the kernel writes SWARM_XCHG_STACK_STRIDE-word slots
                raise ValueError(f"a stacked tick exchanges through a PeerExchange of stride {_lib.XCHG_STACK_STRIDE}, "
                                 f"got {self.peers.stride}")
            peers = C.byref(self.peers.struct)
        check(lib().swarm_train_tick_stack_grad(C.byref(self.cfg), C.byref(self.spec), C.byref(self.hyper),
                                                C.addressof(self._reward) if self._reward is not None else None,
                                                ptr(self._shaping), ptr(self.ctl), ptr(weights), ptr(target), ptr(state),
                                                ptr(returns), ptr(hits), C.byref(self._rstruct), ptr(self.indices),
                                                ptr(self.grad_loss), ptr(self.workspace), self._ws_bytes, peers,
                                                stream_ptr(state.device)))

    def apply_phase(self, weights: torch.Tensor, target: torch.Tensor, exp_avg: torch.Tensor,
                    exp_avg_sq: torch.Tensor) -> None:
        """clip + Adam on ``grad_loss`` (+ target sync) and the cursor advance."""
        self._expect_weights(weights=weights, target=target, exp_avg=exp_avg, exp_avg_sq=exp_avg_sq)
        check(lib().swarm_train_tick_stack_apply(C.byref(self.cfg), C.byref(self.spec), C.byref(self.hyper), ptr(self.ctl),
                                                 ptr(weights), ptr(target), ptr(exp_avg), ptr(exp_avg_sq),
                                                 ptr(self.grad_loss), self.ring.capacity, stream_ptr(weights.device)))

    def tick(self, weights: torch.Tensor, target: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
             state: torch.Tensor, returns: torch.Tensor, hits: torch.Tensor) -> None:
        """Both phases as one library call (swarm_train_tick_stack), without the peer exchange: the same bits as
        ``grad_phase`` + ``apply_phase``, for one GPU."""
        self._expect_weights(weights=weights, target=target, exp_avg=exp_avg, exp_avg_sq=exp_avg_sq)
        check(lib().swarm_train_tick_stack(C.byref(self.cfg), C.byref(self.spec), C.byref(self.hyper),
                                           C.addressof(self._reward) if self._reward is not None else None,
                                           ptr(self._shaping), ptr(self.ctl), ptr(weights), ptr(target), ptr(exp_avg),
                                           ptr(exp_avg_sq), ptr(state), ptr(returns), ptr(hits), C.byref(self._rstruct),
                                           ptr(self.indices), ptr(self.grad_loss), ptr(self.workspace), self._ws_bytes,
                                           stream_ptr(state.device)))


def csr_from_edges(edge_index: torch.Tensor, n_nodes: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """edge_index int64[2,E] -> (row_ptr int32[n+1], src int32[E], perm int32[E]), edges grouped by target,
    each group in edge-list order."""
    if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.shape[0] != 2:
        raise TypeError("edge_index must be int64[2, E]")
    dev = edge_index.device
    E = edge_index.shape[1]
    ei = edge_index.contiguous()
    row_ptr = torch.empty(n_nodes + 1, dtype=torch.int32, device=dev)
    src = torch.empty(E, dtype=torch.int32, device=dev)
    perm = torch.empty(E, dtype=torch.int32, device=dev)
    wb = int(lib().swarm_csr_workspace_bytes(n_nodes, E))
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    check(lib().swarm_csr_from_edges(n_nodes, E, ptr(ei[0]), ptr(ei[1]), ptr(row_ptr), ptr(src), ptr(perm), ptr(ws), wb,
                                     stream_ptr(dev)))
    return row_ptr, src, perm


def gatq_forward_csr(weights: torch.Tensor, x: torch.Tensor, row_ptr: torch.Tensor, src: torch.Tensor,
                     want_q: bool = True, want_actions: bool = False):
    """Generic GCN.forward: x f32[n,7] + CSR-by-target -> q f32[n,9] (and / or greedy actions int32[n])."""
    n = x.shape[0]
    _expect(x, torch.float32, n * 7, "x")
    _expect(weights, torch.float32, _lib.W_COUNT, "weights")
    _expect(row_ptr, torch.int32, n + 1, "row_ptr")
    dev = x.device
    q = torch.empty(n, 9, dtype=torch.float32, device=dev) if want_q else None
    act = torch.empty(n, dtype=torch.int32, device=dev) if want_actions else None
    wb = int(lib().swarm_gatq_workspace_bytes(n))
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    check(lib().swarm_gatq_forward_csr(n, ptr(weights), ptr(x.contiguous()), ptr(row_ptr), ptr(src), ptr(q), ptr(act),
                                       ptr(ws), wb, stream_ptr(dev)))
    if want_q and want_actions:
        return q, act
    return q if want_q else act


def gatq_forward_knn_large(cfg: SwarmConfig, weights: torch.Tensor, state: torch.Tensor, neighbours: torch.Tensor,
                           want_q: bool = True, want_actions: bool = False):
    """GCN.forward on the kNN graph of a large swarm straight from the topk table (one CTA per env, no edge list)."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(weights, torch.float32, _lib.W_COUNT, "weights")
    _expect(neighbours, torch.int32, B * N * cfg.knn_k, "neighbours")
    dev = state.device
    q = torch.empty(B, N, 9, dtype=torch.float32, device=dev) if want_q else None
    act = torch.empty(B, N, dtype=torch.int32, device=dev) if want_actions else None
    check(lib().swarm_gatq_forward_knn_large(C.byref(cfg), ptr(weights), ptr(state), ptr(neighbours), ptr(q), ptr(act),
                                             stream_ptr(dev)))
    if want_q and want_actions:
        return q, act
    return q if want_q else act


def gatq_forward_large(cfg: SwarmConfig, weights: torch.Tensor, state: torch.Tensor, want_q: bool = True,
                       want_actions: bool = False):
    """GCN.forward on the radius / complete graph of a swarm of any size without an edge list (one CTA per env,
    uniform-grid broad phase for the radius graph, attention in input space)."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(weights, torch.float32, _lib.W_COUNT, "weights")
    dev = state.device
    q = torch.empty(B, N, 9, dtype=torch.float32, device=dev) if want_q else None
    act = torch.empty(B, N, dtype=torch.int32, device=dev) if want_actions else None
    check(lib().swarm_gatq_forward_large(C.byref(cfg), ptr(weights), ptr(state), ptr(q), ptr(act), stream_ptr(dev)))
    if want_q and want_actions:
        return q, act
    return q if want_q else act


def graph_build_radius_csr(cfg: SwarmConfig, state: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Radius graph of swarms of any size as a CSR grouped by target: (row_ptr int32[B*N+1], src int32[E]) with global
    node ids, sources ascending per target, node 0's (0, 0) last -- what csr_from_edges makes of the edge list.  Two
    library passes (count, fill) with the prefix sum in between as tensor plumbing."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    dev = state.device
    deg = torch.empty(B * N, dtype=torch.int32, device=dev)
    check(lib().swarm_graph_build_radius_csr(C.byref(cfg), ptr(state), ptr(deg), None, None, stream_ptr(dev)))
    row_ptr = torch.zeros(B * N + 1, dtype=torch.int32, device=dev)
    total = torch.cumsum(deg, 0, dtype=torch.int64)
    if int(total[-1]) > 2 ** 31 - 1:
        raise _lib.SwarmError("the radius graph has more than 2^31 - 1 edges")
    row_ptr[1:] = total.to(torch.int32)
    src = torch.empty(max(int(total[-1]), 1), dtype=torch.int32, device=dev)
    check(lib().swarm_graph_build_radius_csr(C.byref(cfg), ptr(state), None, ptr(row_ptr), ptr(src), stream_ptr(dev)))
    return row_ptr, src[:int(total[-1])]


def stack_spec(n_layers: int, hidden: int, in_features: int = 7, activations=None) -> "_lib.SwarmStackSpec":
    """Multi-layer GAT Q-network description; ``activations`` per conv layer ("tanh" / "relu"), default the reference's
    commented forward (train:61-67): tanh after conv1, relu after the others."""
    sp = _lib.SwarmStackSpec()
    sp.n_layers, sp.hidden, sp.in_features = int(n_layers), int(hidden), int(in_features)
    acts = activations or (["tanh"] + ["relu"] * (n_layers - 1))
    if len(acts) != n_layers:
        raise ValueError("one activation per conv layer")
    for l, a in enumerate(acts):
        sp.activation[l] = {"tanh": _lib.ACT_TANH, "relu": _lib.ACT_RELU}[a]
    return sp


def pack_stack_weights(state_dict, spec, device) -> torch.Tensor:
    """state dict with the reference's key names (conv{l}.att_src / att_dst / bias / lin.weight, lin1.*, lin2.*; the
    layout of data/models/experiment_Flocking-seed_*.pth) -> the packed float32 vector of SwarmStackSpec."""
    parts = []
    H = spec.hidden
    for l in range(1, spec.n_layers + 1):
        cin = spec.in_features if l == 1 else H
        w = state_dict[f"conv{l}.lin.weight"]
        if tuple(w.shape) != (H, cin):
            raise ValueError(f"conv{l}.lin.weight has shape {tuple(w.shape)}, expected {(H, cin)}")
        parts += [state_dict[f"conv{l}.att_src"].reshape(-1), state_dict[f"conv{l}.att_dst"].reshape(-1),
                  state_dict[f"conv{l}.bias"].reshape(-1), w.reshape(-1)]
    parts += [state_dict["lin1.weight"].reshape(-1), state_dict["lin1.bias"].reshape(-1),
              state_dict["lin2.weight"].reshape(-1), state_dict["lin2.bias"].reshape(-1)]
    packed = torch.cat([p.detach().to(torch.float32).cpu() for p in parts]).contiguous()
    if packed.numel() != int(lib().swarm_stack_weight_count(C.byref(spec))):
        raise ValueError("state dict does not match the stack spec")
    return packed.to(device)


def unpack_stack_weights(packed: torch.Tensor, spec) -> Dict[str, torch.Tensor]:
    """The inverse of ``pack_stack_weights``: packed float32 vector -> state dict with the reference's key names and
    shapes (``conv{l}.att_src`` / ``att_dst`` [1,1,H], ``conv{l}.bias`` [H], ``conv{l}.lin.weight`` [H,Cin], ``lin1.*``,
    ``lin2.*``), as views of ``packed``."""
    H, out, off = spec.hidden, {}, 0

    def take(key, shape):
        nonlocal off
        n = 1
        for s_ in shape:
            n *= s_
        out[key] = packed[off:off + n].reshape(shape)
        off += n

    for l in range(1, spec.n_layers + 1):
        take(f"conv{l}.att_src", (1, 1, H))
        take(f"conv{l}.att_dst", (1, 1, H))
        take(f"conv{l}.bias", (H,))
        take(f"conv{l}.lin.weight", (H, spec.in_features if l == 1 else H))
    take("lin1.weight", (H, H))
    take("lin1.bias", (H,))
    take("lin2.weight", (9, H))
    take("lin2.bias", (9,))
    if off != packed.numel():
        raise ValueError(f"packed weights have {packed.numel()} floats, the stack spec needs {off}")
    return out


def dqn_grad_stack(cfg: SwarmConfig, spec, online: torch.Tensor, target: torch.Tensor, batch: ReplayRing,
                   indices: Optional[torch.Tensor], n_graphs: int, gamma: float = 0.99, loss_scale: Optional[float] = None,
                   want_td: bool = False, grad: Optional[torch.Tensor] = None, loss: Optional[torch.Tensor] = None
                   ) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
    """train_step_dqn's loss + gradient (train:116-124) for a stacked network over n_graphs transitions of ``batch``
    (slots ``indices`` if given), in one gradient launch + one reduce launch.  Returns (grad f32[count] in packed stack
    order, loss f32[1], td f32[G,N] or None)."""
    N, dev = cfg.n_agents, online.device
    count = int(lib().swarm_stack_weight_count(C.byref(spec)))
    _expect(online, torch.float32, count, "online weights")
    _expect(target, torch.float32, count, "target weights")
    if indices is not None:
        if indices.dtype != torch.int64 or indices.numel() != n_graphs:
            raise TypeError("indices must be int64[n_graphs]")
    if loss_scale is None:
        loss_scale = 1.0 / (n_graphs * N)
    grad = grad if grad is not None else torch.empty(count, dtype=torch.float32, device=dev)
    loss = loss if loss is not None else torch.empty(1, dtype=torch.float32, device=dev)
    _expect(grad, torch.float32, count, "grad")
    td = torch.empty(n_graphs, N, dtype=torch.float32, device=dev) if want_td else None
    wb = int(lib().swarm_dqn_stack_workspace_bytes(C.byref(cfg), C.byref(spec), n_graphs))
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    rs = batch.struct()
    check(lib().swarm_dqn_stack_grad(C.byref(cfg), C.byref(spec), ptr(online), ptr(target), C.byref(rs), ptr(indices),
                                     n_graphs, float(gamma), float(loss_scale), ptr(grad), ptr(loss), ptr(td), ptr(ws), wb,
                                     stream_ptr(dev)))
    return grad, loss, td


def adam_clip_step_stack(spec, weights: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
                         step: int, lr: float = 1e-3, betas: Tuple[float, float] = (0.9, 0.999), eps: float = 1e-8,
                         max_norm: float = 1.0, target: Optional[torch.Tensor] = None,
                         grad_norm: Optional[torch.Tensor] = None) -> None:
    """clip_grad_norm_(max_norm) + torch.optim.Adam step on a stack's packed weights, in place (train:125-126);
    optionally copies the new weights into ``target`` (train:131-133) and the pre-clip norm into ``grad_norm``."""
    count = int(lib().swarm_stack_weight_count(C.byref(spec)))
    for name, t in (("weights", weights), ("grad", grad), ("exp_avg", exp_avg), ("exp_avg_sq", exp_avg_sq)):
        _expect(t, torch.float32, count, name)
    if target is not None:
        _expect(target, torch.float32, count, "target")
    check(lib().swarm_adam_clip_stack_step(C.byref(spec), ptr(weights), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq), int(step),
                                           float(lr), float(betas[0]), float(betas[1]), float(eps), float(max_norm),
                                           ptr(target), ptr(grad_norm), stream_ptr(weights.device)))


def gatstack_forward(cfg: SwarmConfig, spec, weights: torch.Tensor, state: torch.Tensor, want_q: bool = True,
                     want_actions: bool = False):
    """A whole multi-layer GAT Q-network forward on the per-env graph in one launch: q f32[B,N,9], actions int32[B,N].
    Above 128 agents it runs ``gatstack_forward_large`` (kNN: after the topk table of ``graph_build``)."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(weights, torch.float32, int(lib().swarm_stack_weight_count(C.byref(spec))), "weights")
    dev = state.device
    q = torch.empty(B, N, 9, dtype=torch.float32, device=dev) if want_q else None
    act = torch.empty(B, N, dtype=torch.int32, device=dev) if want_actions else None
    if N > 128:
        gatstack_forward_large(cfg, spec, weights, state, q=q, actions=act)
    else:
        check(lib().swarm_gatstack_forward(C.byref(cfg), C.byref(spec), ptr(weights), ptr(state), ptr(q), ptr(act),
                                           stream_ptr(dev)))
    if want_q and want_actions:
        return q, act
    return q if want_q else act


def gatstack_forward_large(cfg: SwarmConfig, spec, weights: torch.Tensor, state: torch.Tensor,
                           neighbours: Optional[torch.Tensor] = None, q: Optional[torch.Tensor] = None,
                           actions: Optional[torch.Tensor] = None) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """The stacked forward of ``swarm_gatstack_forward_large`` (one CTA per env, any N <= 4096) into the given ``q``
    f32[B,N,9] / ``actions`` int32[B,N]; on the kNN graph ``neighbours`` is the topk table int32[B,N,k] of
    ``swarm_graph_build`` (as ``graph_build(..., want_neighbours=True)`` returns it), built here when not given."""
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(weights, torch.float32, int(lib().swarm_stack_weight_count(C.byref(spec))), "weights")
    if q is not None:
        _expect(q, torch.float32, B * N * 9, "q")
    if actions is not None:
        _expect(actions, torch.int32, B * N, "actions")
    dev = state.device
    if cfg.graph_mode == _lib.GRAPH_KNN:
        if neighbours is None:
            # the topk table alone (swarm_graph_build without the edge list)
            neighbours = torch.empty(B, N, cfg.knn_k, dtype=torch.int32, device=dev)
            check(lib().swarm_graph_build(C.byref(cfg), ptr(state), None, ptr(neighbours), stream_ptr(dev)))
        _expect(neighbours, torch.int32, B * N * cfg.knn_k, "neighbours")
    wb = int(lib().swarm_gatstack_large_workspace_bytes(C.byref(cfg), C.byref(spec)))
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    check(lib().swarm_gatstack_forward_large(C.byref(cfg), C.byref(spec), ptr(weights), ptr(state), ptr(neighbours), ptr(q),
                                             ptr(actions), ptr(ws), wb, stream_ptr(dev)))
    return q, actions


def rollout_stack(cfg: SwarmConfig, spec, weights: torch.Tensor, state: torch.Tensor, ticks: int,
                  reward: Optional["_lib.SwarmRewardSpec"] = None, shaping: Optional[torch.Tensor] = None,
                  returns: Optional[torch.Tensor] = None, hits: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """Greedy rollout of a stacked network, in place on ``state``: per tick forward -> world step -> reward (the world's,
    or the Flocking / Cohesion reward of ``reward``) -> running totals, all launched from the library.  Above 128 agents
    a Flocking / Cohesion reward runs through ``rollout_stack_large``."""
    if cfg.n_agents > 128 and reward is not None:
        return rollout_stack_large(cfg, spec, weights, state, ticks, reward, shaping, returns, hits)
    return _rollout_stack(cfg, spec, weights, state, ticks, reward, shaping, returns, hits, False)


def rollout_stack_large(cfg: SwarmConfig, spec, weights: torch.Tensor, state: torch.Tensor, ticks: int,
                        reward: Optional["_lib.SwarmRewardSpec"] = None, shaping: Optional[torch.Tensor] = None,
                        returns: Optional[torch.Tensor] = None, hits: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """``rollout_stack`` through swarm_rollout_stack_large (129 <= N <= 4 096, any reward): per tick [topk table ->] the
    large stacked forward -> world step -> [large scenario reward] with returns += the tick's reward."""
    return _rollout_stack(cfg, spec, weights, state, ticks, reward, shaping, returns, hits, True)


def _rollout_stack(cfg, spec, weights, state, ticks, reward, shaping, returns, hits, large):
    B, N = cfg.num_envs, cfg.n_agents
    _expect(state, torch.float32, B * N * 4, "state")
    _expect(weights, torch.float32, int(lib().swarm_stack_weight_count(C.byref(spec))), "weights")
    dev = state.device
    if returns is None:
        returns = torch.zeros(B, N, dtype=torch.float32, device=dev)
    if hits is None:
        hits = torch.zeros(B, dtype=torch.int32, device=dev)
    if shaping is not None:
        _expect(shaping, torch.float32, B * N * 2, "shaping")
    rptr = C.addressof(reward) if reward is not None else None
    if large:
        wb = int(lib().swarm_rollout_stack_large_workspace_bytes(C.byref(cfg), rptr))
        ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
        fn = lib().swarm_rollout_stack_large
    else:
        wb = int(lib().swarm_rollout_stack_workspace_bytes(C.byref(cfg)))
        ws = torch.empty(wb, dtype=torch.uint8, device=dev)
        fn = lib().swarm_rollout_stack
    check(fn(C.byref(cfg), C.byref(spec), ptr(weights), ptr(state), int(ticks), rptr, ptr(shaping), ptr(returns), ptr(hits),
             ptr(ws), wb, stream_ptr(dev)))
    out = {"state": state, "returns": returns, "hits": hits}
    if shaping is not None:
        out["shaping"] = shaping
    return out


def gatconv_forward_csr(weights: torch.Tensor, x: torch.Tensor, row_ptr: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
    """The GATConv layer alone: x f32[n,7] + CSR-by-target -> f32[n,32] (aggregate + bias)."""
    n = x.shape[0]
    _expect(x, torch.float32, n * 7, "x")
    _expect(weights, torch.float32, _lib.W_COUNT, "weights")
    out = torch.empty(n, 32, dtype=torch.float32, device=x.device)
    wb = int(lib().swarm_gatq_workspace_bytes(n))
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=x.device)
    check(lib().swarm_gatconv_forward_csr(n, ptr(weights), ptr(x.contiguous()), ptr(row_ptr), ptr(src), ptr(out), ptr(ws), wb,
                                          stream_ptr(x.device)))
    return out


def gatq_backward_csr(weights: torch.Tensor, x: torch.Tensor, edge_index: torch.Tensor, grad_q: torch.Tensor,
                      by_target: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None,
                      conv_only: bool = False) -> torch.Tensor:
    """Gradient of GCN.forward w.r.t. the packed weights for an arbitrary graph: x f32[n,7], edge_index int64[2,E],
    grad_q f32[n,9] -> f32[1673].  ``by_target`` = (row_ptr, src, perm) of the forward's grouping, if already built.
    ``conv_only``: the GATConv layer alone, grad_q = d(conv output) f32[n,32]."""
    n = x.shape[0]
    E = edge_index.shape[1]
    _expect(x, torch.float32, n * 7, "x")
    _expect(weights, torch.float32, _lib.W_COUNT, "weights")
    _expect(grad_q, torch.float32, n * (32 if conv_only else 9), "grad_q")
    dev = x.device
    row_ptr, src, perm = by_target if by_target is not None else csr_from_edges(edge_index, n)
    row_ptr_s, tgt_s, perm_s = csr_from_edges(edge_index.flip(0).contiguous(), n)
    grad = torch.empty(_lib.W_COUNT, dtype=torch.float32, device=dev)
    wb = int(lib().swarm_gatq_backward_workspace_bytes(n, E))
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    fn = lib().swarm_gatconv_backward_csr if conv_only else lib().swarm_gatq_backward_csr
    check(fn(n, E, ptr(weights), ptr(x.contiguous()), ptr(row_ptr), ptr(src), ptr(perm), ptr(row_ptr_s), ptr(tgt_s),
             ptr(perm_s), ptr(grad_q.contiguous()), ptr(grad), ptr(ws), wb, stream_ptr(dev)))
    return grad


def gat_layer_forward(lin_weight: torch.Tensor, att_src: torch.Tensor, att_dst: torch.Tensor, bias: torch.Tensor,
                      x: torch.Tensor, row_ptr: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
    """One GATConv(in, out, heads=1) layer of any width <= 64: x f32[n,in] + CSR-by-target -> f32[n,out]."""
    n, ci = x.shape
    co = lin_weight.shape[0]
    _expect(lin_weight, torch.float32, co * ci, "lin_weight")
    for name, t in (("att_src", att_src), ("att_dst", att_dst), ("bias", bias)):
        _expect(t, torch.float32, co, name)
    _expect(row_ptr, torch.int32, n + 1, "row_ptr")
    dev = x.device
    out = torch.empty(n, co, dtype=torch.float32, device=dev)
    wb = int(lib().swarm_gat_layer_workspace_bytes(n, 0, ci, co, 0))
    if wb < 0:
        check(-1 if "must be" in lib().swarm_last_error().decode() else -2)
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    check(lib().swarm_gat_layer_forward(n, ci, co, ptr(lin_weight.contiguous()), ptr(att_src.contiguous()),
                                        ptr(att_dst.contiguous()), ptr(bias.contiguous()), ptr(x.contiguous()), ptr(row_ptr),
                                        ptr(src), ptr(out), ptr(ws), wb, stream_ptr(dev)))
    return out


def gat_layer_backward(lin_weight: torch.Tensor, att_src: torch.Tensor, att_dst: torch.Tensor, x: torch.Tensor,
                       edge_index: torch.Tensor, grad_out: torch.Tensor, want_grad_x: bool = True,
                       by_target: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None):
    """Backward of gat_layer_forward: -> (grad_lin_weight f32[out,in], grad_att_src f32[out], grad_att_dst f32[out],
    grad_bias f32[out], grad_x f32[n,in] or None)."""
    n, ci = x.shape
    co = lin_weight.shape[0]
    E = edge_index.shape[1]
    _expect(grad_out, torch.float32, n * co, "grad_out")
    dev = x.device
    row_ptr, src, perm = by_target if by_target is not None else csr_from_edges(edge_index, n)
    row_ptr_s, tgt_s, perm_s = csr_from_edges(edge_index.flip(0).contiguous(), n)
    gw = torch.empty(co, ci, dtype=torch.float32, device=dev)
    gas, gad, gb = (torch.empty(co, dtype=torch.float32, device=dev) for _ in range(3))
    gx = torch.empty(n, ci, dtype=torch.float32, device=dev) if want_grad_x else None
    wb = int(lib().swarm_gat_layer_workspace_bytes(n, E, ci, co, 1))
    if wb < 0:
        check(-2)
    ws = torch.empty(max(wb, 1), dtype=torch.uint8, device=dev)
    check(lib().swarm_gat_layer_backward(n, E, ci, co, ptr(lin_weight.contiguous()), ptr(att_src.contiguous()),
                                         ptr(att_dst.contiguous()), ptr(x.contiguous()), ptr(row_ptr), ptr(src), ptr(perm),
                                         ptr(row_ptr_s), ptr(tgt_s), ptr(perm_s), ptr(grad_out.contiguous()), ptr(gw),
                                         ptr(gas), ptr(gad), ptr(gb), ptr(gx), ptr(ws), wb, stream_ptr(dev)))
    return gw, gas, gad, gb, gx


def rollout_large(cfg: SwarmConfig, weights: torch.Tensor, state: torch.Tensor, ticks: int,
                  returns: Optional[torch.Tensor] = None, hits: Optional[torch.Tensor] = None,
                  trace_state: bool = False, fused: bool = True) -> Dict[str, torch.Tensor]:
    """Greedy rollout for large swarms (n_agents > 128): per tick graph_build -> CSR grouping -> generic GAT-Q
    forward (argmax) -> world step, all on the device; the per-tick glue (node features, edge offsets, reward
    accumulation) is tensor plumbing.  In place on ``state``."""
    B, N = cfg.num_envs, cfg.n_agents
    dev = state.device
    if returns is None:
        returns = torch.zeros(B, N, dtype=torch.float32, device=dev)
    if hits is None:
        hits = torch.zeros(B, dtype=torch.int32, device=dev)
    ids = torch.arange(N, device=dev, dtype=torch.float32).view(1, N, 1).expand(B, N, 1)
    goal = torch.tensor([cfg.goal_x, cfg.goal_y], dtype=torch.float32, device=dev).view(1, 1, 2).expand(B, N, 2)
    offs = (torch.arange(B, device=dev, dtype=torch.int64) * N).view(B, 1, 1)
    trace = []
    static_csr = None
    if fused and not trace_state and 128 < N <= 4096:
        # the whole tick sequence from the library (swarm_rollout_large): [topk table ->] per-env Q + argmax -> world
        # step with returns / hits accumulated by the step kernel; no tensor op between the launches.  The library
        # refuses a swarm its kernels do not take (SWARM_ERR_UNSUPPORTED) before it launches anything.
        wb = int(lib().swarm_rollout_large_workspace_bytes(C.byref(cfg)))
        ws = torch.empty(wb, dtype=torch.uint8, device=dev)
        rc = lib().swarm_rollout_large(C.byref(cfg), ptr(weights), ptr(state), int(ticks), ptr(returns), ptr(hits), ptr(ws),
                                       wb, stream_ptr(dev))
        if rc != _lib.ERR_UNSUPPORTED:
            check(rc)
            return {"state": state, "returns": returns, "hits": hits}
    # kNN: the per-env fused forward straight from the topk table while the library takes the env, else the CSR path
    fused_knn = fused and cfg.graph_mode == _lib.GRAPH_KNN
    nbr = torch.empty(B, N, cfg.knn_k, dtype=torch.int32, device=dev) if fused_knn else None
    act = torch.empty(B, N, dtype=torch.int32, device=dev) if fused_knn else None
    for _ in range(ticks):
        if fused_knn:
            # topk table only (no edge list), then the per-env fused forward
            check(lib().swarm_graph_build(C.byref(cfg), ptr(state), None, ptr(nbr), stream_ptr(dev)))
            rc = lib().swarm_gatq_forward_knn_large(C.byref(cfg), ptr(weights), ptr(state), ptr(nbr), None, ptr(act),
                                                    stream_ptr(dev))
            fused_knn = rc != _lib.ERR_UNSUPPORTED
        if fused_knn:
            check(rc)
            out = sim_step(cfg, state, act, state_out=state, want_obs=False)
            returns += out["rewards"]
            hits += ((out["flags"] & _lib.FLAG_HIT) != 0).sum(dim=1, dtype=torch.int32)
            if trace_state:
                trace.append(state.clone())
            continue
        if cfg.graph_mode == _lib.GRAPH_COMPLETE and static_csr is not None:
            row_ptr, src = static_csr
        elif cfg.graph_mode == _lib.GRAPH_RADIUS:
            row_ptr, src = graph_build_radius_csr(cfg, state)         # bit-faithful generic path: CSR straight from the grid
        else:
            edges, _ = graph_build(cfg, state)
            ei = (edges.to(torch.int64) + offs).permute(1, 0, 2).reshape(2, -1).contiguous()
            row_ptr, src, _ = csr_from_edges(ei, B * N)
            if cfg.graph_mode == _lib.GRAPH_COMPLETE:
                static_csr = (row_ptr, src)
        x = torch.cat([state, goal, ids], dim=2).reshape(B * N, 7)
        act = gatq_forward_csr(weights, x, row_ptr, src, want_q=False, want_actions=True).view(B, N)
        out = sim_step(cfg, state, act, state_out=state, want_obs=False)
        returns += out["rewards"]
        hits += ((out["flags"] & _lib.FLAG_HIT) != 0).sum(dim=1, dtype=torch.int32)
        if trace_state:
            trace.append(state.clone())
    res = {"state": state, "returns": returns, "hits": hits}
    if trace_state:
        res["trace_state"] = torch.stack(trace)
    return res
