"""Multi-GPU use of the learner, limited to where the path shards (SURVEY 8e, BASELINE.json configs[3], configs[4]).

* single agent, B = 256: replicas only (one agent per rank, nothing to exchange);
* population of independent agents: `partition_agents` assigns agents to ranks, no communication;
* large-batch data parallel: `DataParallelSAC` averages the critic gradients, then the actor + temperature gradients,
  across ranks (two dependent all-reduces per step: the actor phase needs the stepped critics, sac_imp.py:109-118).

One process per GPU; `torch.distributed` is only plumbing (NCCL over NVLink on GPUs, gloo in the CPU tests).
"""
import ctypes

import numpy as np
import torch
import torch.distributed as dist

from . import _native as N
from .sac_imp import _loss_dict


def partition_agents(n_agents, world_size, rank):
    """Agents owned by `rank`: contiguous, sizes differ by at most one, every agent owned exactly once."""
    base, extra = divmod(int(n_agents), int(world_size))
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))


def allreduce_mean_(tensors, group=None):
    """In-place mean over the ranks of `group` of every tensor in `tensors` (no-op without an initialised group)."""
    if not (dist.is_available() and dist.is_initialized()):
        return tensors
    world = dist.get_world_size(group)
    if world == 1:
        return tensors
    for t in tensors:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        t.div_(world)
    return tensors


class DataParallelSAC:
    """update_parameters for one replicated agent whose minibatch is split over the ranks.

    Every rank holds the same weights / optimizer state and its own replay shard; a step is
        backward(critics) on B_local rows -> all-reduce mean of the q1|q2 gradient slab -> Adam + Polyak
        backward(actor, temperature)      -> all-reduce mean of the policy slab and the log_alpha gradient -> Adam
    so the result equals the single-GPU update on the concatenated batch (mean of equal-sized means) up to fp32
    reassociation.  `agent` is a `sac_imp.SAC` on this rank's GPU.
    """

    def __init__(self, agent, group=None, exchange="peer"):
        """exchange: 'peer' = the library's own fused exchange (flag barrier + ONE kernel that sums the replicas' gradient slabs over
        NVLink peer memory in rank order and applies Adam; needs all ranks on one node) -- 'nccl' = torch.distributed all-reduce of
        the slabs followed by the element-wise apply kernel (the round-1 path, kept for A/B timing and multi-node use)."""
        self.agent, self.group = agent, group
        self.exchange = True           # False: skip the exchange (measurement of its share only; the replicas then diverge)
        world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        rank = dist.get_rank(group) if world > 1 else 0
        self.world, self.rank = world, rank
        self.mode = exchange
        if exchange == "peer":
            lib = N.lib()
            mine = ctypes.create_string_buffer(64)
            N.check(lib.sacb_dp_ipc_handle(agent._h, mine))
            handles = [None] * world
            if world > 1:
                dist.all_gather_object(handles, bytes(mine.raw), group=group)      # plumbing only: 64 bytes per rank
            else:
                handles[0] = bytes(mine.raw)
            blob = ctypes.create_string_buffer(b"".join(handles), 64 * world)
            N.check(lib.sacb_dp_connect(agent._h, rank, world, blob))
            if world > 1:
                dist.barrier(group=group)      # every rank has mapped its peers before the first flag is written
            self.exchange_kind = "fused: flag barrier in NVLink peer memory + one kernel summing the replicas' gradient slabs (peer loads) with Adam + Polyak applied in the same pass"
        else:
            self.exchange_kind = "ncclAllReduce (torch.distributed) on the library's stream + element-wise Adam apply"
        self._bufs = {}
        for phase in (0, 1, 2):
            ptr, n = ctypes.c_void_p(), ctypes.c_int64()
            N.check(N.lib().sacb_dp_grad_buffer(agent._h, phase, ctypes.byref(ptr), ctypes.byref(n)))
            self._bufs[phase] = torch.as_tensor(N.DevArray(ptr.value, (n.value,), agent), device=f"cuda:{agent._cfg.device}")
        sp = ctypes.c_void_p()
        N.check(N.lib().sacb_get_stream(agent._h, ctypes.byref(sp)))
        # the library's own stream as a torch stream: the all-reduces are enqueued on it between backward and apply (NCCL orders
        # itself against the current stream with events), so a step runs without any host synchronisation
        self._stream = torch.cuda.ExternalStream(sp.value, device=f"cuda:{agent._cfg.device}")

    def gradient_slabs(self, phase):
        """Device tensors (aliases of the arena) that are averaged after `phase`: 0 -> [q1|q2], 1 -> [policy, log_alpha block]."""
        return [self._bufs[0]] if phase == 0 else [self._bufs[1], self._bufs[2]]

    def update_parameters(self, batch_size_local, *, idx=None, eps=None, staged=False, sync=True):
        """idx / eps: test hooks as in `SAC.update_parameters`; staged=True: the rank's indices were pre-staged on the device
        (`sacb_stage_indices`); sync=False returns None without reading the losses (throughput mode)."""
        a, lib = self.agent, N.lib()
        a.replay_buffer._flush()
        a._publish_alias_writes()
        if staged:
            ix, n_local = None, int(batch_size_local)
        else:
            ix = a.replay_buffer._draw(batch_size_local) if idx is None else np.ascontiguousarray(idx, np.int64)
            n_local = ix.size
        e_next = e_cur = None
        if eps is not None:
            e_next, e_cur = N.f32(eps[0]), N.f32(eps[1])
        with torch.cuda.stream(self._stream):
            for phase in (0, 1):
                N.check(lib.sacb_dp_backward(a._h, phase, n_local, N.ptr(ix, ctypes.c_int64) if (phase == 0 and ix is not None) else None, N.ptr(e_next), N.ptr(e_cur)))
                if self.mode == "peer" and self.exchange:
                    N.check(lib.sacb_dp_exchange_apply(a._h, phase))          # barrier + peer-memory reduction + Adam in one kernel
                else:
                    if self.exchange:
                        allreduce_mean_(self.gradient_slabs(phase), self.group)   # same stream: ordered behind the backward, ahead of the apply
                    N.check(lib.sacb_dp_apply(a._h, phase))
        a._alpha_is_float = False
        if not sync:
            return None
        losses = np.zeros(3, np.float32)
        if self.mode == "peer" and self.exchange:      # the finish kernels averaged the replicas' loss scalars through peer memory
            N.check(lib.sacb_dp_get_losses(a._h, N.ptr(losses)))
            return _loss_dict(losses)
        N.check(lib.sacb_get_losses(a._h, 0, N.ptr(losses)))
        t = torch.from_numpy(losses.copy()).to(self._bufs[0].device)
        with torch.cuda.stream(self._stream):
            allreduce_mean_([t], self.group)
        self._stream.synchronize()
        return _loss_dict(t.tolist())
