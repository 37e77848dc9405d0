"""Multi-GPU plumbing: one process per GPU, envs sharded across ranks, no data-path collective for rollouts.

The reference is single-process (SURVEY.md 2b); the only exchange the sharded DQN needs is the all-reduce of
the 1 673-float Q-network gradient per update (6 692 B, latency bound) plus one weight broadcast at start.
Every rank then applies the identical clip + Adam step to the identical reduced gradient, so the online and
target weights stay replicated and the hard target sync (train:131-133) is a local copy.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib


@dataclass(frozen=True)
class EnvShard:
    """Contiguous env range [offset, offset + count) owned by ``rank`` out of ``total`` envs."""
    rank: int
    world: int
    total: int
    offset: int
    count: int


def shard_envs(total: int, rank: int, world: int) -> EnvShard:
    """Split ``total`` envs into ``world`` contiguous ranges whose sizes differ by at most one."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of size {world}")
    if total < world:
        raise ValueError(f"cannot shard {total} envs over {world} ranks")
    base, extra = divmod(total, world)
    count = base + (1 if rank < extra else 0)
    offset = rank * base + min(rank, extra)
    return EnvShard(rank, world, total, offset, count)


def init_from_env(backend: Optional[str] = None) -> Tuple[int, int, int]:
    """(rank, world, local_rank) from the torchrun environment; initialises the process group when
    WORLD_SIZE > 1 (NCCL on GPUs, gloo otherwise)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        kwargs = {}
        if backend == "nccl":
            torch.cuda.set_device(local)
            kwargs["device_id"] = torch.device("cuda", local)
        dist.init_process_group(backend, **kwargs)
    return rank, world, local


def world_size() -> int:
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def broadcast_weights(packed: torch.Tensor, src: int = 0) -> torch.Tensor:
    """Initial weight broadcast so that every rank starts from rank ``src``'s Q-network."""
    if world_size() > 1:
        dist.broadcast(packed, src=src)
    return packed


def allreduce_gradient(grad: torch.Tensor, loss: Optional[torch.Tensor] = None) -> None:
    """Sum the per-rank partial gradients (each already scaled by 1 / global node count) in place.  With
    ``loss`` the per-rank partial losses are summed in the same collective round."""
    if world_size() == 1:
        return
    if loss is None:
        dist.all_reduce(grad, op=dist.ReduceOp.SUM)
        return
    buf = torch.cat([grad.reshape(-1), loss.reshape(-1)])
    dist.all_reduce(buf, op=dist.ReduceOp.SUM)
    grad.copy_(buf[:grad.numel()].reshape(grad.shape))
    loss.copy_(buf[grad.numel():].reshape(loss.shape))


def global_loss_scale(local_graphs: int, n_agents: int) -> float:
    """1 / (total nodes of the update over all ranks): the mean of train:122 taken over the global batch."""
    return 1.0 / (local_graphs * world_size() * n_agents)


def require_equal_shards(num_envs: int, ring_size: int, ring_position: int, ring_capacity: int,
                         graphs_per_update: int) -> None:
    """The data-parallel tick decides on the device whether a tick updates (ring fill >= G, train:113-115) and every
    rank must take the same decision: a rank that exchanges gradients while a peer skips would wait for words that
    never arrive (fused peer exchange) or apply Adam alone (NCCL path).  So all ranks must run the same number of
    envs per tick and start from the same ring state.  Raises ValueError otherwise (``shard_envs`` with a remainder
    gives unequal counts: pad or trim the env total to a multiple of the world size)."""
    if world_size() <= 1:
        return
    mine = [int(num_envs), int(ring_size), int(ring_position), int(ring_capacity), int(graphs_per_update)]
    gathered = [None] * world_size()
    dist.all_gather_object(gathered, mine)
    if any(g != gathered[0] for g in gathered):
        raise ValueError("data-parallel DQN needs the same (num_envs, replay fill, cursor, capacity, graphs_per_update) on "
                         f"every rank; got {gathered}")


class PeerExchange:
    """Symmetric (peer-mapped) receive buffers for the fused one-shot PUSH all-reduce of the data-parallel ticks: every
    rank allocates uint64[2][world][stride] with ``torch.distributed._symmetric_memory`` and maps all peers' copies over
    NVLink; the exchanging kernel writes its partial gradient (value + epoch per 8-byte word) into its slot of every
    peer's buffer, polls its own local buffer for the peers' words and sums the partials in rank order.  ``stride`` is
    ``_lib.XCHG_STRIDE`` for the one-layer GCN (``swarm_train_tick_apply``) and ``_lib.XCHG_STACK_STRIDE`` for stacked
    networks (``swarm_train_tick_stack_grad``).  PyTorch only provides the allocation / rendezvous plumbing."""

    def __init__(self, device, group=None, stride: int = _lib.XCHG_STRIDE):
        import torch.distributed._symmetric_memory as symm_mem
        group = group if group is not None else dist.group.WORLD
        world = dist.get_world_size(group)
        if world > 16:
            raise ValueError("PeerExchange supports up to 16 ranks")
        self.stride = int(stride)
        self.buf = symm_mem.empty(2 * world * self.stride, dtype=torch.int64, device=device)
        self.buf.zero_()
        self.handle = symm_mem.rendezvous(self.buf, group)
        st = _lib.SwarmPeerExchange()
        st.world_size, st.rank = self.handle.world_size, self.handle.rank
        for r, base in enumerate(self.handle.buffer_ptrs):
            st.data[r] = base
        self.struct = st
        torch.cuda.synchronize(device)
        dist.barrier(group)            # every rank's buffer is zeroed before anybody's kernel can write into it


def make_peer_exchange(device, stride: int = _lib.XCHG_STRIDE) -> Optional["PeerExchange"]:
    """PeerExchange (of ``stride`` words per rank and parity) when data-parallel on GPUs with symmetric memory
    available, else None (the trainer then keeps the NCCL all-reduce between the two tick phases).
    SWARM_PEER_ALLREDUCE=0 forces the NCCL path."""
    if world_size() <= 1 or os.environ.get("SWARM_PEER_ALLREDUCE", "1") == "0":
        return None
    try:
        return PeerExchange(device, stride=stride)
    except Exception as exc:           # no NVLink peer mapping / symmetric memory on this box
        import warnings
        warnings.warn(f"peer-memory gradient exchange unavailable ({exc!r}); using the NCCL all-reduce")
        return None
