"""ctypes binding of libswarm_b200.so (the C ABI declared in include/swarm_b200.h).

There is no CPU fallback: every compute call goes through the CUDA library, and loading fails loudly
when it has not been built (``python -m swarm_b200._build`` / ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import _build

SCENARIO_GOTO = 0
SCENARIO_OBSTACLE_AVOIDANCE = 1
GRAPH_COMPLETE = 0
GRAPH_KNN = 1
GRAPH_RADIUS = 2
FLAG_OBSTACLE_CONTACT = 1
FLAG_HIT = 2
FLAG_PENALTY = 4
W_COUNT = 1673
ABI_VERSION = 9
ERR_UNSUPPORTED = -2     # SWARM_ERR_UNSUPPORTED: the library does not implement this call's shape
XCHG_STRIDE = 1680
XCHG_STACK_STRIDE = 5040

# state-dict tensors in packed order (include/swarm_b200.h SWARM_W_*)
WEIGHT_KEYS = ("conv1.lin.weight", "conv1.att_src", "conv1.att_dst", "conv1.bias",
               "lin1.weight", "lin1.bias", "lin2.weight", "lin2.bias")
WEIGHT_SHAPES = ((32, 7), (1, 1, 32), (1, 1, 32), (32,), (32, 32), (32,), (9, 32), (9,))


class SwarmConfig(C.Structure):
    _fields_ = [
        ("grid_spacing", C.c_double),
        ("num_envs", C.c_int32), ("n_agents", C.c_int32), ("scenario", C.c_int32),
        ("graph_mode", C.c_int32), ("knn_k", C.c_int32),
        ("dt", C.c_float), ("drag", C.c_float), ("collision_force", C.c_float),
        ("contact_margin", C.c_float), ("agent_radius", C.c_float), ("landmark_radius", C.c_float),
        ("goal_x", C.c_float), ("goal_y", C.c_float), ("obstacle_x", C.c_float), ("obstacle_y", C.c_float),
        ("hit_distance", C.c_float), ("penalty_distance", C.c_float), ("obstacle_weight", C.c_float),
        ("graph_radius", C.c_float),
    ]


class SwarmTrace(C.Structure):
    _fields_ = [("state", C.c_void_p), ("actions", C.c_void_p), ("q", C.c_void_p), ("rewards", C.c_void_p),
                ("flags", C.c_void_p), ("contact", C.c_void_p), ("edges", C.c_void_p), ("dist", C.c_void_p)]


class SwarmReplay(C.Structure):
    _fields_ = [("state", C.c_void_p), ("next_state", C.c_void_p), ("actions", C.c_void_p), ("rewards", C.c_void_p),
                ("capacity", C.c_int64)]


class SwarmRolloutOptions(C.Structure):
    _fields_ = [("forced_actions", C.c_void_p), ("epsilon", C.c_float), ("rng_seed", C.c_uint64),
                ("rng_tick0", C.c_int64), ("replay", C.POINTER(SwarmReplay)), ("replay_cursor", C.c_int64),
                ("env_offset", C.c_int64), ("flocking", C.c_void_p), ("flocking_shaping", C.c_void_p),
                ("knn_memo", C.c_void_p), ("knn_memo_entries", C.c_int64)]


class SwarmStackSpec(C.Structure):
    """Multi-layer GAT Q-network (include/swarm_b200.h SwarmStackSpec)."""
    _fields_ = [("n_layers", C.c_int32), ("hidden", C.c_int32), ("in_features", C.c_int32),
                ("activation", C.c_int32 * 4), ("pad", C.c_int32)]


ACT_TANH, ACT_RELU = 0, 1


class SwarmTrainCtl(C.Structure):
    """Host mirror of the 48-byte device struct (only used to document / check the layout)."""
    _fields_ = [("tick", C.c_int64), ("ring_cursor", C.c_int64), ("ring_size", C.c_int64), ("opt_step", C.c_int64),
                ("epsilon", C.c_float), ("updating", C.c_int32), ("episode", C.c_int64)]


class SwarmTrainHyper(C.Structure):
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("max_norm", C.c_double), ("rng_seed", C.c_uint64), ("sample_seed", C.c_uint64),
                ("env_offset", C.c_int64), ("graphs_per_update", C.c_int32), ("update_target_every", C.c_int32),
                ("gamma", C.c_float), ("loss_scale", C.c_float), ("flocking", C.c_void_p), ("flocking_shaping", C.c_void_p)]


class SwarmResetSpec(C.Structure):
    _fields_ = [("base_x", C.c_float), ("base_y", C.c_float), ("mean_x", C.c_float), ("mean_y", C.c_float),
                ("std_x", C.c_float), ("std_y", C.c_float), ("seed", C.c_uint64), ("env_offset", C.c_int64),
                ("shared_center", C.c_int32), ("pad", C.c_int32)]


class SwarmRewardSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("num_envs", C.c_int32), ("n_agents", C.c_int32), ("reset", C.c_int32),
                ("env_index", C.c_int64), ("goal_x", C.c_float), ("goal_y", C.c_float), ("goal_radius", C.c_float),
                ("agent_radius", C.c_float), ("pos_shaping", C.c_float), ("dist_shaping", C.c_float),
                ("desired_distance", C.c_float), ("min_collision_distance", C.c_float), ("collision_reward", C.c_float),
                ("on_goal_bonus", C.c_float), ("sigma", C.c_float), ("pad", C.c_float)]


REWARD_FLOCKING, REWARD_COHESION = 0, 1


class SwarmPeerExchange(C.Structure):
    _fields_ = [("data", C.c_void_p * 16), ("world_size", C.c_int32), ("rank", C.c_int32)]


class SwarmError(RuntimeError):
    pass


_LIB: Optional[C.CDLL] = None

_SIGNATURES = {
    "swarm_abi_version": (C.c_int, []),
    "swarm_last_error": (C.c_char_p, []),
    "swarm_default_config": (None, [C.POINTER(SwarmConfig), C.c_int32, C.c_int32, C.c_int32]),
    "swarm_edges_per_env": (C.c_int64, [C.POINTER(SwarmConfig)]),
    "swarm_reset_grid": (C.c_int, [C.POINTER(SwarmConfig), C.c_void_p, C.c_void_p, C.c_void_p]),
    "swarm_sim_step": (C.c_int, [C.POINTER(SwarmConfig)] + [C.c_void_p] * 9),
    "swarm_graph_build": (C.c_int, [C.POINTER(SwarmConfig)] + [C.c_void_p] * 4),
    "swarm_graph_build_radius": (C.c_int, [C.POINTER(SwarmConfig)] + [C.c_void_p] * 4),
    "swarm_stack_weight_count": (C.c_int64, [C.POINTER(SwarmStackSpec)]),
    "swarm_gatstack_forward": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec)] + [C.c_void_p] * 5),
    "swarm_gatstack_large_workspace_bytes": (C.c_int64, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec)]),
    "swarm_gatstack_forward_large": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec)] + [C.c_void_p] * 6
                                     + [C.c_int64, C.c_void_p]),
    "swarm_rollout_stack_workspace_bytes": (C.c_int64, [C.POINTER(SwarmConfig)]),
    "swarm_rollout_stack": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec), C.c_void_p, C.c_void_p, C.c_int32,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "swarm_rollout_stack_large_workspace_bytes": (C.c_int64, [C.POINTER(SwarmConfig), C.c_void_p]),
    "swarm_rollout_stack_large": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec), C.c_void_p, C.c_void_p,
                                            C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_int64, C.c_void_p]),
    "swarm_dqn_stack_workspace_bytes": (C.c_int64, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec), C.c_int32]),
    "swarm_dqn_stack_grad": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec), C.c_void_p, C.c_void_p,
                                       C.POINTER(SwarmReplay), C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "swarm_adam_clip_stack_step": (C.c_int, [C.POINTER(SwarmStackSpec), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                             C.c_void_p, C.c_void_p, C.c_void_p]),
    "swarm_graph_build_radius_csr": (C.c_int, [C.POINTER(SwarmConfig)] + [C.c_void_p] * 5),
    "swarm_gatq_forward_large": (C.c_int, [C.POINTER(SwarmConfig)] + [C.c_void_p] * 5),
    "swarm_gatq_forward": (C.c_int, [C.POINTER(SwarmConfig)] + [C.c_void_p] * 5),
    "swarm_gatq_workspace_bytes": (C.c_int64, [C.c_int32]),
    "swarm_gatq_forward_csr": (C.c_int, [C.c_int32] + [C.c_void_p] * 6 + [C.c_void_p, C.c_int64, C.c_void_p]),
    "swarm_gatq_forward_knn_large": (C.c_int, [C.POINTER(SwarmConfig)] + [C.c_void_p] * 6),
    "swarm_rollout_large_workspace_bytes": (C.c_int64, [C.POINTER(SwarmConfig)]),
    "swarm_rollout_large": (C.c_int, [C.POINTER(SwarmConfig), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int64, C.c_void_p]),
    "swarm_gatconv_forward_csr": (C.c_int, [C.c_int32] + [C.c_void_p] * 6 + [C.c_int64, C.c_void_p]),
    "swarm_gatconv_backward_csr": (C.c_int, [C.c_int32, C.c_int64] + [C.c_void_p] * 11 + [C.c_int64, C.c_void_p]),
    "swarm_gat_layer_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32]),
    "swarm_gat_layer_forward": (C.c_int, [C.c_int32, C.c_int32, C.c_int32] + [C.c_void_p] * 9 + [C.c_int64, C.c_void_p]),
    "swarm_gat_layer_backward": (C.c_int, [C.c_int32, C.c_int64, C.c_int32, C.c_int32] + [C.c_void_p] * 17 +
                                 [C.c_int64, C.c_void_p]),
    "swarm_gatq_backward_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int64]),
    "swarm_gatq_backward_csr": (C.c_int, [C.c_int32, C.c_int64] + [C.c_void_p] * 11 + [C.c_int64, C.c_void_p]),
    "swarm_csr_workspace_bytes": (C.c_int64, [C.c_int32, C.c_int64]),
    "swarm_csr_from_edges": (C.c_int, [C.c_int32, C.c_int64] + [C.c_void_p] * 6 + [C.c_int64, C.c_void_p]),
    "swarm_rollout": (C.c_int, [C.POINTER(SwarmConfig), C.c_void_p, C.c_void_p, C.c_int32,
                                C.POINTER(SwarmRolloutOptions), C.c_void_p, C.c_void_p, C.POINTER(SwarmTrace),
                                C.c_void_p]),
    "swarm_replay_push": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmReplay), C.c_int64] + [C.c_void_p] * 5),
    "swarm_replay_gather": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmReplay), C.c_void_p, C.c_int32]
                            + [C.c_void_p] * 5),
    "swarm_dqn_workspace_bytes": (C.c_int64, [C.POINTER(SwarmConfig), C.c_int32]),
    "swarm_dqn_grad": (C.c_int, [C.POINTER(SwarmConfig), C.c_void_p, C.c_void_p, C.POINTER(SwarmReplay), C.c_void_p,
                                 C.c_int32, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int64, C.c_void_p]),
    "swarm_adam_clip_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_double,
                                       C.c_double, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "swarm_train_tick_grad": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmTrainHyper)] + [C.c_void_p] * 6
                              + [C.POINTER(SwarmReplay)] + [C.c_void_p] * 4 + [C.c_int64, C.c_void_p]),
    "swarm_default_reward_spec": (None, [C.POINTER(SwarmRewardSpec), C.c_int32, C.c_int32, C.c_int32]),
    "swarm_scenario_reward": (C.c_int, [C.POINTER(SwarmRewardSpec)] + [C.c_void_p] * 5),
    "swarm_scenario_reward_large_workspace_bytes": (C.c_int64, [C.POINTER(SwarmRewardSpec)]),
    "swarm_scenario_reward_large": (C.c_int, [C.POINTER(SwarmRewardSpec)] + [C.c_void_p] * 5 + [C.c_int64, C.c_void_p]),
    "swarm_reset_random": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmResetSpec), C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "swarm_episode_end": (C.c_int, [C.POINTER(SwarmConfig)] + [C.c_void_p] * 5 + [C.c_int64, C.c_double, C.c_double,
                                                                                 C.c_double, C.c_void_p]),
    "swarm_train_tick_apply": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmTrainHyper)] + [C.c_void_p] * 6
                               + [C.c_int64, C.POINTER(SwarmPeerExchange), C.c_void_p]),
    "swarm_train_tick": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmTrainHyper)] + [C.c_void_p] * 8
                         + [C.POINTER(SwarmReplay)] + [C.c_void_p] * 3 + [C.c_int64, C.POINTER(SwarmPeerExchange),
                                                                          C.c_void_p]),
    "swarm_train_tick_stack": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec), C.POINTER(SwarmTrainHyper)]
                               + [C.c_void_p] * 10 + [C.POINTER(SwarmReplay)] + [C.c_void_p] * 3
                               + [C.c_int64, C.c_void_p]),
    "swarm_train_tick_stack_grad": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec), C.POINTER(SwarmTrainHyper)]
                                    + [C.c_void_p] * 8 + [C.POINTER(SwarmReplay)] + [C.c_void_p] * 3
                                    + [C.c_int64, C.POINTER(SwarmPeerExchange), C.c_void_p]),
    "swarm_train_tick_stack_apply": (C.c_int, [C.POINTER(SwarmConfig), C.POINTER(SwarmStackSpec),
                                               C.POINTER(SwarmTrainHyper)] + [C.c_void_p] * 6 + [C.c_int64, C.c_void_p]),
}


def lib() -> C.CDLL:
    """Load (once) the CUDA library.  Raises if it is missing -- there is no fallback path."""
    global _LIB
    if _LIB is None:
        path = _build.LIB_PATH
        if not os.path.exists(path):
            raise SwarmError(
                f"{path} is missing: build the sm_100a CUDA extension first "
                "(python -c 'import __graft_entry__ as g; g.build()'); swarm_b200 has no CPU fallback")
        handle = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError if the ABI is incomplete
            fn.restype = res
            fn.argtypes = args
        if handle.swarm_abi_version() != ABI_VERSION:
            raise SwarmError("libswarm_b200.so ABI version mismatch; rebuild")
        _LIB = handle
    return _LIB


def offload_device() -> Optional[torch.device]:
    """``SWARM_DEVICE`` (e.g. ``cuda`` or ``cuda:0``): the B200 that serves scripts which ask for ``device="cpu"``.

    The reference scripts hard-code ``device = 'cpu'`` (train_gcn_dqn.py:262, tests/test_*.py:33).  With SWARM_DEVICE set
    such a script runs UNMODIFIED: tensors at its seams (observations, rewards, ``agent.state.pos``, ``Data.x``,
    model parameters) stay host tensors as it asked, while ``env.step`` and ``GATConv`` / ``GCN`` execute in
    libswarm_b200.so on this device (host<->device copies at the seam).  Without it, a CPU device raises: there is no
    CPU implementation to fall back to."""
    name = os.environ.get("SWARM_DEVICE", "").strip()
    if not name:
        return None
    dev = torch.device(name)
    if dev.type != "cuda":
        raise SwarmError(f"SWARM_DEVICE must name a CUDA device, got {name!r}")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().swarm_last_error().decode()
        if rc == -1:
            # mirrors the exceptions torch / vmas raise for bad arguments
            raise (RuntimeError if "out of range" in msg else ValueError)(msg)
        raise SwarmError(f"swarm_b200 error {rc}: {msg}")


def default_config(scenario: int, num_envs: int, n_agents: int) -> SwarmConfig:
    cfg = SwarmConfig()
    lib().swarm_default_config(C.byref(cfg), scenario, num_envs, n_agents)
    return cfg


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise SwarmError("swarm_b200 kernels take CUDA tensors only (no CPU fallback)")
    if not t.is_contiguous():
        raise SwarmError("swarm_b200 kernels take contiguous tensors")
    return t.data_ptr()


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def pack_weights(state_dict, device=None) -> torch.Tensor:
    """Flatten a reference GCN state dict (train_gcn_dqn.py:50-57 key set) into the packed float[1673]."""
    parts = []
    for key, shape in zip(WEIGHT_KEYS, WEIGHT_SHAPES):
        t = state_dict[key]
        if tuple(t.shape) != shape:
            raise ValueError(f"{key}: expected shape {shape}, got {tuple(t.shape)}")
        parts.append(t.detach().reshape(-1).to(torch.float32))
    w = torch.cat(parts).contiguous()
    return w.to(device) if device is not None else w


def unpack_weights(packed: torch.Tensor):
    out, off = {}, 0
    for key, shape in zip(WEIGHT_KEYS, WEIGHT_SHAPES):
        n = 1
        for s in shape:
            n *= s
        out[key] = packed[off:off + n].reshape(shape)
        off += n
    return out
