"""Multi-GPU plumbing: one process per GPU, torch.distributed (NCCL on the B200 box, gloo in CPU tests).

Extraction shards by utterance and needs no collective (SURVEY 8e).  Cloak + GRL training is data parallel with one
flat-bucket gradient all-reduce per step; per-speaker statistics need one all-gather of the utterance partials' merge,
and their gradient one all-gather of dstats and one integer all-reduce of the min / max tie weights.
"""
from __future__ import annotations

from typing import Iterable, Sequence

import numpy as np
import torch
import torch.distributed as dist


def shard_by_length(lengths: Sequence[int], world_size: int, bucket: int = 8000) -> list[np.ndarray]:
    """Length-bucketed, balanced assignment of utterances to ranks.

    Utterances are sorted into buckets of `bucket` samples (0.5 s at 16 kHz), then dealt longest-first to the rank
    with the least samples so far; every rank gets the same mix of lengths and (almost) the same total audio.
    Returns, per rank, the utterance indices in ascending order."""
    lengths = np.asarray(lengths, dtype=np.int64)
    order = np.lexsort((np.arange(len(lengths)), -(lengths // bucket)))
    load = np.zeros(world_size, dtype=np.int64)
    parts: list[list[int]] = [[] for _ in range(world_size)]
    for i in order:
        r = int(np.argmin(load))
        parts[r].append(int(i))
        load[r] += lengths[i]
    return [np.sort(np.asarray(p, dtype=np.int64)) for p in parts]


def allreduce_gradients(params: Iterable[torch.nn.Parameter], group=None, average: bool = True) -> int:
    """All-reduce the gradients of `params` as ONE flat fp32 bucket (5 MB for the GRL model: latency-bound on NVLink,
    so a single collective beats per-tensor calls).  Parameters without a gradient contribute zeros so every rank
    reduces the same layout.  Returns the number of elements reduced."""
    params = [p for p in params if p.requires_grad]
    if not params or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return 0
    grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in params]
    flat = torch.cat([g.reshape(-1).float() for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    if average:
        flat /= dist.get_world_size(group)
    off = 0
    for p, g in zip(params, grads):
        n = g.numel()
        chunk = flat[off:off + n].view_as(g).to(g.dtype)
        if p.grad is None:
            p.grad = chunk.clone()
        else:
            p.grad.copy_(chunk)
        off += n
    return off


class FlatGradients:
    """One persistent fp32 buffer that IS the gradients: every trainable parameter's `.grad` is a view into it (same
    sizes and strides as the parameter, so channels_last weights keep their layout).  Autograd accumulates into existing
    `.grad` tensors in place, so after backward the buffer holds every gradient back to back -- the data-parallel
    exchange is ONE all-reduce of `flat` with no `torch.cat` before it and no copy-back after it, `zero()` is one memset,
    and all three are fixed-address operations that a CUDA graph can capture together with backward and the optimizer.

    Do not call `optimizer.zero_grad(set_to_none=True)` while this is in use: it would detach the views (`check()` tells)."""

    def __init__(self, params: Iterable[torch.nn.Parameter], early: Iterable[torch.nn.Parameter] = ()):
        """`early`: parameters whose gradients are complete first in backward (the layers nearest the loss).  They are laid
        out at the front of the buffer as their own bucket, so that bucket can be reduced on a side stream while backward
        still runs through the earlier layers (`allreduce_early` / `allreduce_late`)."""
        params = [p for p in params if p.requires_grad]
        early_ids = {id(p) for p in early}
        self.params = [p for p in params if id(p) in early_ids] + [p for p in params if id(p) not in early_ids]
        self.n_early_params = sum(1 for p in params if id(p) in early_ids)
        if not self.params:
            raise ValueError("no trainable parameters")
        if any(p.dtype != torch.float32 for p in self.params):
            raise ValueError("FlatGradients holds fp32 gradients (the reference trains in fp32)")
        dev = self.params[0].device
        self.offsets = []
        total = 0
        for p in self.params:
            self.offsets.append(total)
            total += p.numel()
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.early_numel = sum(p.numel() for p in self.params[:self.n_early_params])
        for p, off in zip(self.params, self.offsets):
            dense = p.is_contiguous() or p.is_contiguous(memory_format=torch.channels_last)
            p.grad = (torch.as_strided(self.flat, p.size(), p.stride(), off) if dense
                      else self.flat[off:off + p.numel()].view(p.shape))

    def zero(self) -> None:
        self.flat.zero_()

    def check(self) -> bool:
        """True while every .grad still aliases the buffer."""
        base = self.flat.data_ptr()
        return all(p.grad is not None and p.grad.data_ptr() == base + 4 * off for p, off in zip(self.params, self.offsets))

    def _reduce(self, t: torch.Tensor, group, average: bool) -> int:
        if t.numel() == 0 or not dist.is_initialized() or dist.get_world_size(group) == 1:
            return 0
        world = dist.get_world_size(group)
        if average and dist.get_backend(group) == "nccl":
            dist.all_reduce(t, op=dist.ReduceOp.AVG, group=group)              # the division happens inside the collective
        else:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
            if average:
                t.mul_(1.0 / world)
        return t.numel()

    def allreduce(self, group=None, average: bool = True) -> int:
        """Sum (mean) the buffer over the ranks in place; returns the number of elements exchanged (0 on one rank)."""
        return self._reduce(self.flat, group, average)

    def allreduce_early(self, group=None, average: bool = True) -> int:
        """The bucket of the `early` parameters (call it as soon as their gradients are complete)."""
        return self._reduce(self.flat[:self.early_numel], group, average)

    def allreduce_late(self, group=None, average: bool = True) -> int:
        """Everything behind the early bucket."""
        return self._reduce(self.flat[self.early_numel:], group, average)


def broadcast_parameters(module: torch.nn.Module, src: int = 0, group=None) -> None:
    """Make every rank start from rank `src`'s parameters and buffers."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    for t in list(module.parameters()) + list(module.buffers()):
        dist.broadcast(t.data, src=src, group=group)


def merge_speaker_partials(count: torch.Tensor, mean: torch.Tensor, m2: torch.Tensor, mn: torch.Tensor, mx: torch.Tensor,
                           group=None):
    """Chan merge of per-rank per-speaker (count, mean, M2, min, max) partials, each (n_spk, F) with the same speaker
    rows on every rank: all-gather, then merge in rank order (deterministic).  Returns merged (count, mean, std, min, max)."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        world = dist.get_world_size(group)
        packed = torch.stack([count, mean, m2, mn, mx])
        gathered = [torch.empty_like(packed) for _ in range(world)]
        dist.all_gather(gathered, packed, group=group)
    else:
        gathered = [torch.stack([count, mean, m2, mn, mx])]
    n, mu, s2, lo, hi = (gathered[0][i].clone() for i in range(5))
    for part in gathered[1:]:
        nb, mb, sb, lb, hb = (part[i] for i in range(5))
        tot = n + nb
        safe = torch.where(tot > 0, tot, torch.ones_like(tot))
        d = mb - mu
        mu = mu + d * (nb / safe)
        s2 = s2 + sb + d * d * (n * nb / safe)
        n = tot
        lo, hi = torch.minimum(lo, lb), torch.maximum(hi, hb)
    std = torch.sqrt(s2 / torch.where(n > 0, n, torch.ones_like(n)))
    return n, mu, std, lo, hi


def sum_in_rank_order(t: torch.Tensor, group=None) -> torch.Tensor:
    """Sum of `t` over the ranks: one all-gather, then additions in rank order, so every rank holds the same bits and
    repeated runs do too (a float all-reduce leaves the order to the collective).  `t` itself on one rank."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return t
    gathered = [torch.empty_like(t) for _ in range(dist.get_world_size(group))]
    dist.all_gather(gathered, t.contiguous(), group=group)
    total = gathered[0]
    for part in gathered[1:]:
        total += part
    return total


def allreduce_exact_sum(t: torch.Tensor, group=None) -> torch.Tensor:
    """In-place SUM all-reduce of an integer tensor (exact, so the order does not matter); nothing on one rank."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


# ---- host placement: the end-to-end (host buffer) path is bound by PCIe and by the host's memory fabric --------------
def bind_host_to_gpu(device_index: int) -> dict | None:
    """Pin the calling thread to the CPUs NVML reports as local to the GPU and prefer that NUMA node for the memory it
    allocates from now on (pinned staging buffers are first-touched by this thread).  Call it before allocating pinned
    host memory.  Returns {"cpus": [...], "node": n} or None when the platform exposes no topology (then nothing changes)."""
    import ctypes
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = device_index
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if device_index < len(ids) and ids[device_index].isdigit():
                phys = int(ids[device_index])
        handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(handle, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if not cpus or len(cpus) == len(allowed):
            return None                                            # one domain: nothing to choose
        os.sched_setaffinity(0, cpus)
        node = None
        for entry in os.listdir(f"/sys/devices/system/cpu/cpu{cpus[0]}"):
            if entry.startswith("node") and entry[4:].isdigit():
                node = int(entry[4:])
        if node is not None:
            libc = ctypes.CDLL(None, use_errno=True)
            nodemask = ctypes.c_ulong(1 << node)
            MPOL_PREFERRED, SYS_set_mempolicy = 1, 238            # x86_64
            libc.syscall(SYS_set_mempolicy, MPOL_PREFERRED, ctypes.byref(nodemask), ctypes.c_ulong(64))
        return {"cpus": cpus, "node": node}
    except Exception:
        return None
