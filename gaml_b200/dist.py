"""Read-id sharding across ranks (one process per GPU) — SURVEY.md §8e.

Every read's term is independent given the walks, so each rank scores the contiguous read-id block it
holds and the only exchange is the per-set partial {integer part, 2^-40 units, floored, -inf terms, nan terms}:
40 bytes per read set per evaluation. The partials are ALL-GATHERED and every rank adds them exactly (128-bit
integers, `gaml_combine_partials`), so the total is bit-identical for any number of ranks and independent of the
collective's internal order; `torch.distributed` (NCCL over NVLink on the GPU box, gloo in CPU tests) is only the
plumbing.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np


def shard_bounds(n_reads: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous read-id block of `rank` (pairs stay together because a pair shares one read id)."""
    per = (n_reads + world - 1) // world
    return min(rank * per, n_reads), min((rank + 1) * per, n_reads)


class PartialGatherer:
    """All-gather of the per-rank partial vector with preallocated pinned/device staging buffers
    (the exchange is latency bound: nothing is allocated per evaluation)."""

    def __init__(self, n_doubles: int, device=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.n = n_doubles
        self.device = device
        if self.world > 1:
            pin = device is not None and torch.cuda.is_available()
            self.h_in = torch.empty(n_doubles, dtype=torch.float64, pin_memory=pin)
            self.h_out = torch.empty(self.world * n_doubles, dtype=torch.float64, pin_memory=pin)
            dev = device if device is not None else "cpu"
            self.d_in = torch.empty(n_doubles, dtype=torch.float64, device=dev)
            self.d_out = torch.empty(self.world * n_doubles, dtype=torch.float64, device=dev)

    def __call__(self, partials: np.ndarray) -> np.ndarray:
        """[n] float64 of this rank -> [world, n] on every rank."""
        if self.world == 1:
            return np.asarray(partials, dtype=np.float64)[None, :]
        self.h_in.numpy()[:] = partials
        self.d_in.copy_(self.h_in, non_blocking=True)
        self.dist.all_gather_into_tensor(self.d_out, self.d_in)
        self.h_out.copy_(self.d_out, non_blocking=True)
        if self.device is not None and self.torch.cuda.is_available():
            self.torch.cuda.current_stream().synchronize()
        return self.h_out.numpy().reshape(self.world, self.n).copy()


def allgather_partials(partials: np.ndarray, device=None) -> np.ndarray:
    """One-shot form of PartialGatherer (allocates): [n] float64 of this rank -> [world, n] on every rank."""
    import torch
    import torch.distributed as dist
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return np.asarray(partials, dtype=np.float64)[None, :]
    t = torch.from_numpy(np.ascontiguousarray(partials, dtype=np.float64))
    if device is not None:
        t = t.to(device)
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return torch.stack(out).cpu().numpy()


def sharded_calc_prob(pc, paths: Sequence[Sequence[int]], device=None, gatherer: "PartialGatherer" = None):
    """CalcProb over all ranks' shards: local partials -> all-gather -> exact combine (same value on every rank)."""
    part, tl = pc.calc_prob_partial(paths)
    g = gatherer(part) if gatherer is not None else allgather_partials(part, device)
    return pc.combine(g, g.shape[0], tl)


def allgather_keys(keys: np.ndarray, device=None) -> np.ndarray:
    """All-gather of a uint64 array whose length differs per rank: the lengths first, then the arrays padded to the
    longest -> every rank's keys concatenated in rank order (the same array on every rank)."""
    import torch
    import torch.distributed as dist
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return keys
    world = dist.get_world_size()
    dev = device if device is not None else "cpu"
    n = torch.tensor([len(keys)], dtype=torch.int64, device=dev)
    ns = [torch.empty_like(n) for _ in range(world)]
    dist.all_gather(ns, n)
    ns = [int(x.item()) for x in ns]
    buf = torch.zeros(max(max(ns), 1), dtype=torch.int64)   # the words as int64: every backend gathers those
    buf[:len(keys)] = torch.from_numpy(keys.view(np.int64))
    buf = buf.to(dev)
    out = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(out, buf)
    return np.concatenate([o.cpu().numpy()[:k] for o, k in zip(out, ns)]).view(np.uint64)


def sharded_calc_prob_batch(pc, packed, device=None):
    """A candidate batch over all ranks' shards (gaml_calc_prob_batch_shard), penalised paired sets included: this shard's
    partials and thinned coverage keys -> per penalised set an all-gather of the keys and their import -> all-gather of the
    partials -> exact combine. Every rank passes the same candidates and gets the same (probs [n], total_lens [n],
    zeros [n, sets, 2]), bit-identical to an unsharded gaml_calc_prob_batch."""
    from .workload import KIND_PAIRED
    part, tls = pc.calc_prob_batch_shard_packed(packed)
    for s, info in enumerate(pc.sets):
        spec = info["spec"]
        if spec.kind == KIND_PAIRED and spec.penalty_constant != 0:
            pc.batch_penalty_import(s, allgather_keys(pc.batch_penalty_export(s), device))
    g = allgather_partials(part.reshape(-1), device)
    probs, zeros = pc.combine_batch_partials(g.reshape((g.shape[0],) + part.shape))
    return probs, tls, zeros


class ResultExchange:
    """Host shared-memory segment for the ranks' 64-byte result lines (gaml_set_result_exchange): rank 0 creates and
    zeroes it, the others attach; `torch.distributed` is used only to hand the name round and as the setup barrier.
    After attach(pc) every evaluation's all-gather is done by the kernels' publishing blocks writing into this segment."""

    MAX_SETS = 8

    def __init__(self, rank: int, world: int, name: str = None):
        import mmap
        import os
        import torch.distributed as dist
        self.rank, self.world = rank, world
        self.bytes = max(2 * world * self.MAX_SETS * 64, mmap.PAGESIZE)
        self.bytes = (self.bytes + mmap.PAGESIZE - 1) // mmap.PAGESIZE * mmap.PAGESIZE
        names = [name or f"/dev/shm/gaml_b200_exch_{os.getpid()}"]
        if dist.is_initialized() and world > 1:
            dist.broadcast_object_list(names, src=0)
        self.path = names[0]
        if rank == 0:
            with open(self.path, "wb") as f:
                f.write(b"\0" * self.bytes)
        if dist.is_initialized() and world > 1:
            dist.barrier()
        self.fd = os.open(self.path, os.O_RDWR)
        self.map = mmap.mmap(self.fd, self.bytes, mmap.MAP_SHARED, mmap.PROT_READ | mmap.PROT_WRITE)
        if dist.is_initialized() and world > 1:
            dist.barrier()
        if rank == 0:
            os.unlink(self.path)   # stays alive while mapped

    def attach(self, pc) -> None:
        pc.set_result_exchange(self.map, self.rank, self.world)


class PeerExchange:
    """Result exchange over NVLink peer memory (gaml_peer_exchange_*): every rank creates its device buffer, the 64-byte
    CUDA IPC handles are all-gathered with `torch.distributed` (plumbing), every rank maps the others' buffers. After
    attach(pc) an evaluation's all-gather is a 64-byte peer store per rank from the publishing block plus the chain's
    last kernel waiting for the lines in its own buffer."""

    def __init__(self, rank: int, world: int):
        self.rank, self.world = rank, world

    def attach(self, pc) -> None:
        import torch.distributed as dist
        handle, _ptr = pc.peer_exchange_create(self.rank, self.world)
        handles = [None] * self.world
        if dist.is_initialized() and self.world > 1:
            dist.all_gather_object(handles, handle)
        else:
            handles[0] = handle
        pc.peer_exchange_open(handles=handles)
        if dist.is_initialized() and self.world > 1:
            dist.barrier()   # nobody evaluates before every rank has mapped every buffer


class NcclExchange:
    """Result exchange as one ncclAllReduce(sum, fp64) per evaluation on the library's stream (gaml_nccl_exchange_init)."""

    def __init__(self, rank: int, world: int):
        self.rank, self.world = rank, world

    def attach(self, pc) -> None:
        import torch.distributed as dist
        from . import api
        ids = [api.nccl_unique_id() if self.rank == 0 else None]
        if dist.is_initialized() and self.world > 1:
            dist.broadcast_object_list(ids, src=0)
        pc.nccl_exchange_init(ids[0], self.rank, self.world)
        if dist.is_initialized() and self.world > 1:
            dist.barrier()
