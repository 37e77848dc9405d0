"""Batched CPU oracle (TEST INFRASTRUCTURE -- see oracle/__init__.py).

"B envs" is defined as B independent copies of the reference's ``num_envs = 1`` execution (the reference
code itself is only valid for batch_dim == 1: obstacle_avoidance_scenario.py:149 branches on a tensor,
train_gcn_dqn.py:96,168,171 squeeze / .item()).  This module vectorises oracle/swarm_oracle.py over the
env axis with the same separately-rounded torch ops; tests/test_oracle_golden.py proves it equal, bit for
bit, to B runs of the single-env oracle.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from . import swarm_oracle as so


def reset_grid(scenario: str, centers: torch.Tensor, n_agents: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """centers f32[B,2] -> pos f32[B,N,2] (generate_grid per env), vel zeros."""
    pos = torch.stack([so.generate_grid(c, n_agents) for c in centers])
    return pos, torch.zeros_like(pos)


def step(scenario: str, pos: torch.Tensor, vel: torch.Tensor, actions: torch.Tensor) -> Dict[str, torch.Tensor]:
    """One world step for B envs.  pos/vel f32[B,N,2], actions int64[B,N]."""
    B, N, _ = pos.shape
    u = so.decode_action(actions.to(torch.int64))                      # [B,N,2]
    forces = [torch.zeros(B, 2) + u[:, i] for i in range(N)]
    goal = torch.tensor(list(so.GOAL_POS)).expand(B, 2)
    obstacle = torch.tensor(list(so.OBSTACLE_POS)).expand(B, 2)
    dist_min = torch.tensor(so.SPHERE_RADIUS) + torch.tensor(so.SPHERE_RADIUS)
    contact = torch.zeros(B, N, dtype=torch.int64)
    agent_contact = torch.zeros(B, N, dtype=torch.bool)              # any partner, also where the mask has no bit
    obstacle_contact = torch.zeros(B, N, dtype=torch.bool)

    if scenario == so.OBSTACLE_AVOIDANCE:
        for i in range(N):
            f = so.constraint_force(obstacle, pos[:, i])
            forces[i] = forces[i] + (-f)
            obstacle_contact[:, i] = torch.linalg.vector_norm(obstacle - pos[:, i], dim=-1) <= dist_min
    for i in range(N):
        for j in range(i + 1, N):
            f = so.constraint_force(pos[:, i], pos[:, j])
            forces[i] = forces[i] + f
            forces[j] = forces[j] + (-f)
            hit = torch.linalg.vector_norm(pos[:, i] - pos[:, j], dim=-1) <= dist_min
            agent_contact[:, i] |= hit
            agent_contact[:, j] |= hit
            if i < 63 and j < 63:
                contact[:, i] |= hit.to(torch.int64) << j
                contact[:, j] |= hit.to(torch.int64) << i

    new_pos, new_vel = [], []
    for i in range(N):
        v = vel[:, i] * (1 - so.DRAG)
        accel = forces[i] / 1.0
        v = v + accel * so.DT
        new_vel.append(v)
        new_pos.append(pos[:, i] + v * so.DT)
    new_pos = torch.stack(new_pos, dim=1)
    new_vel = torch.stack(new_vel, dim=1)

    d_goal = torch.linalg.vector_norm(new_pos - goal.unsqueeze(1), dim=-1)             # [B,N]
    flags = torch.zeros(B, N, dtype=torch.uint8)
    flags |= obstacle_contact.to(torch.uint8) * 1
    if scenario == so.GOTO:
        collective = 0
        for i in range(N):
            collective = collective + (-d_goal[:, i])
        rewards = collective.unsqueeze(1).expand(B, N).clone()
        d_obs = torch.zeros(B, N)
    else:
        d_obs = so.get_distance(new_pos, obstacle.unsqueeze(1))
        avoid = torch.where(d_obs <= so.PENALTY_DISTANCE, -(so.PENALTY_DISTANCE - d_obs), torch.zeros(()))
        rewards = (-d_goal) + so.OBSTACLE_WEIGHT * avoid
        flags |= (d_obs <= so.HIT_DISTANCE).to(torch.uint8) * 2
        flags |= (d_obs <= so.PENALTY_DISTANCE).to(torch.uint8) * 4
    return {"pos": new_pos, "vel": new_vel, "rewards": rewards, "flags": flags, "contact": contact,
            "agent_contact": agent_contact, "d_goal": d_goal, "d_obs": d_obs}


def node_features(pos: torch.Tensor, vel: torch.Tensor) -> torch.Tensor:
    """f32[B,N,7] = [pos, vel, goal, agent id]."""
    B, N, _ = pos.shape
    goal = torch.tensor(list(so.GOAL_POS)).view(1, 1, 2).expand(B, N, 2)
    ids = torch.arange(N).float().view(1, N, 1).expand(B, N, 1)
    return torch.cat([pos, vel, goal, ids], dim=2)


def knn_table(pos: torch.Tensor, k: int) -> torch.Tensor:
    """topk index rows int64[B,N,k]: per env and node i, topk(||p_j - p_i||, k, largest=False)."""
    diff = pos.unsqueeze(1) - pos.unsqueeze(2)             # [B, i, j, 2] = p_j - p_i
    dist = torch.linalg.norm(diff, dim=-1)
    return torch.topk(dist, k, dim=-1, largest=False).indices


def edges_from_knn(nbr: torch.Tensor) -> torch.Tensor:
    """int64[B,N,k] -> env-local edges int64[B,2,2kN+1] in simulator.py:20-24 order."""
    B, N, k = nbr.shape
    i = torch.arange(N).view(1, N, 1).expand(B, N, k)
    src = torch.stack([i, nbr], dim=-1).reshape(B, -1)     # (i, a), (a, i) interleaved
    dst = torch.stack([nbr, i], dim=-1).reshape(B, -1)
    zero = torch.zeros(B, 1, dtype=torch.int64)
    return torch.stack([torch.cat([src, zero], 1), torch.cat([dst, zero], 1)], dim=1)


def edges_complete(B: int, N: int) -> torch.Tensor:
    return so.graph_complete(N).unsqueeze(0).expand(B, 2, -1).contiguous()


def edges_radius(pos: torch.Tensor, radius: float) -> torch.Tensor:
    """EXTENSION (no reference counterpart, SURVEY.md Appendix C): the complete builder of train_gcn_dqn.py:94-110
    filtered by distance.  For i < j with ||p_j - p_i|| <= radius (float32 norm as in simulator.py:18): (i -> j),
    (j -> i) in (i, j) order, then (0 -> 0).  Returns the padded block int64[B,2,N(N-1)+1] with -1 past each env's
    edge count (batch_edge_index drops the padding)."""
    B, N, _ = pos.shape
    cap = N * (N - 1) + 1
    out = torch.full((B, 2, cap), -1, dtype=torch.int64)
    r = torch.tensor(radius, dtype=torch.float32)
    for b in range(B):
        e = []
        for i in range(N):
            d = torch.linalg.norm(pos[b] - pos[b, i], dim=1)          # ||p_j - p_i|| for every j
            for j in range(i + 1, N):
                if d[j] <= r:
                    e.append([i, j])
                    e.append([j, i])
        e.append([0, 0])
        ei = torch.tensor(e, dtype=torch.int64).t()
        out[b, :, :ei.shape[1]] = ei
    return out


def batch_edge_index(edges: torch.Tensor, N: int) -> torch.Tensor:
    """env-local int64[B,2,E] -> Batch.from_data_list edge_index int64[2,B*E] (columns holding -1 are padding of the
    variable-length radius lists and are dropped; env order and in-env order are kept)."""
    B = edges.shape[0]
    off = (torch.arange(B) * N).view(B, 1, 1)
    ei = (edges + off).permute(1, 0, 2).reshape(2, -1)
    keep = edges.permute(1, 0, 2).reshape(2, -1)[0] >= 0
    return ei[:, keep] if not bool(keep.all()) else ei


def gatq(params: Dict[str, torch.Tensor], pos: torch.Tensor, vel: torch.Tensor, edges: torch.Tensor) -> torch.Tensor:
    """Q f32[B,N,9] for B envs with env-local edges int64[B,2,E]."""
    B, N, _ = pos.shape
    x = node_features(pos, vel).reshape(B * N, 7)
    return so.gatq_forward(params, x, batch_edge_index(edges, N)).reshape(B, N, 9)


def graph_edges(pos: torch.Tensor, graph_mode: str, k) -> torch.Tensor:
    """``k`` is the neighbour count for "knn" and the radius for "radius"."""
    B, N, _ = pos.shape
    if graph_mode == "knn":
        return edges_from_knn(knn_table(pos, k))
    if graph_mode == "radius":
        return edges_radius(pos, float(k))
    return edges_complete(B, N)


def rollout(scenario: str, params: Dict[str, torch.Tensor], pos: torch.Tensor, vel: torch.Tensor, ticks: int,
            graph_mode: str = "complete", k: int = 5, forced_actions: Optional[torch.Tensor] = None
            ) -> Dict[str, torch.Tensor]:
    """Greedy rollout of B envs; returns per-tick traces (pre-step Q / edges / actions, post-step rest)."""
    tr = {key: [] for key in ("pos", "vel", "q", "actions", "rewards", "flags", "contact", "edges", "d_goal", "d_obs")}
    for t in range(ticks):
        edges = graph_edges(pos, graph_mode, k)
        with torch.no_grad():
            q = gatq(params, pos, vel, edges)
        actions = torch.argmax(q, dim=2)
        if forced_actions is not None:
            actions = torch.where(forced_actions[t] >= 0, forced_actions[t].to(torch.int64), actions)
        out = step(scenario, pos, vel, actions)
        pos, vel = out["pos"], out["vel"]
        tr["edges"].append(edges)
        tr["q"].append(q)
        tr["actions"].append(actions)
        for key in ("pos", "vel", "rewards", "flags", "contact", "d_goal", "d_obs"):
            tr[key].append(out[key])
    return {key: torch.stack(v) for key, v in tr.items()}
