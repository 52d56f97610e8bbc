"""Data-parallel sharding of the update step across the GPUs of one node.

The path shards by sample row (SURVEY.md 8e): every rank holds a replica of the
embedding table, the nets and the optimizer state, processes its own rows, and
the ranks exchange exactly one thing -- the summed weight gradients (critic every
step, actor on policy steps) plus the loss scalars -- with an all-reduce before
the (identical) optimizer step.  Local loss terms are already scaled by
1/N_global on the device, so SUM over ranks gives the single-device gradient.

One process per GPU (torchrun).  torch.distributed supplies rendezvous, the weight broadcast and a
NCCL fallback; the per-step gradient exchange itself runs inside the step's CUDA graph as kernels that
read the peers' staging buffers over NVLink (``PeerComm`` -> ``recnn_comm_*`` in include/recnn_b200.h).
"""
from __future__ import annotations

import ctypes
import os
import warnings

import torch
import torch.distributed as dist

from . import _lib
from .nn.arena import param_arena


class PeerComm:
    """cudaIpc-mapped staging buffers of all ranks + the in-kernel all-reduce that uses them."""

    def __init__(self, group, device, capacity_floats):
        L = _lib.lib()
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.device = torch.device(device)
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(L.recnn_comm_create(self.rank, self.world, int(capacity_floats), ctypes.byref(self.handle)))
            nbytes = L.recnn_comm_handle_bytes()
            mine = ctypes.create_string_buffer(nbytes)
            _lib.check(L.recnn_comm_local_handle(self.handle, mine))
            everyone = [None] * self.world
            dist.all_gather_object(everyone, bytes(mine.raw), group=group)
            status = L.recnn_comm_connect(self.handle, b"".join(everyone))
            # all ranks must agree, otherwise some would wait in a kernel for peers that use NCCL
            ok = [None] * self.world
            dist.all_gather_object(ok, int(status), group=group)
            if any(ok):
                msg = L.recnn_b200_last_error().decode() if status else "a peer could not map the staging buffers"
                L.recnn_comm_destroy(self.handle)
                self.handle = None
                raise _lib.RecnnError("peer-memory communicator unavailable: " + msg)

    @property
    def ptr(self):
        return self.handle.value

    def all_reduce(self, t: torch.Tensor):
        """In-place sum over the ranks (fp32, contiguous); same bits on every rank."""
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
        _lib.check(_lib.lib().recnn_comm_allreduce(self.handle, t.data_ptr(), t.numel(),
                                                   torch.cuda.current_stream(t.device).cuda_stream))
        return t

    def close(self):
        if self.handle is not None:
            _lib.lib().recnn_comm_destroy(self.handle)
            self.handle = None


def shard_rows(n_rows: int, rank: int, world: int):
    """Contiguous, balanced row range of this rank (first ``n_rows % world`` ranks get one more)."""
    base, extra = divmod(n_rows, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def broadcast_nets(nets: dict, group=None, src: int = 0):
    """Make every replica bit-identical to rank ``src`` (one broadcast per net arena)."""
    for name in sorted(nets):
        dist.broadcast(param_arena(nets[name]), src=src, group=group)


def enable_data_parallel(agent_or_nets, group=None, sync_weights=True):
    """Turn on gradient all-reduce for an Algo (or a nets dict).  Must be called on every
    rank after the nets are on their CUDA device."""
    if not dist.is_initialized():
        raise RuntimeError("torch.distributed is not initialised")
    nets = agent_or_nets.nets if hasattr(agent_or_nets, "nets") else agent_or_nets
    world = dist.get_world_size(group)
    if sync_weights:
        broadcast_nets(nets, group)
    policy = nets["policy_net"]
    comm = None
    arena = param_arena(policy)
    if world > 1 and arena.is_cuda and os.environ.get("RECNN_B200_COMM", "peer") != "nccl":
        try:
            comm = PeerComm(group, arena.device, max(param_arena(m).numel() for m in nets.values()))
        except _lib.RecnnError as exc:     # e.g. no peer access between the GPUs: NCCL between the phases instead
            warnings.warn("recnn_b200: %s; falling back to NCCL all-reduces between the step's phases" % exc)
    policy.__dict__["_recnn_dp"] = (group, world, comm)
    for eng in policy.__dict__.get("_recnn_engines", {}).values():
        eng.set_data_parallel(group, world, comm)
    return agent_or_nets
