"""Data parallelism of the hot path: rays are independent, so each rank processes its own contiguous slice of the
global batch with replicated parameters, and the only exchange is the average of a flat gradient arena (hash tables + MLP
weights) per step.  Replaces the reference's DistributedDataParallel wrap with find_unused_parameters=True and 25 MiB
buckets (nerfstudio/pipelines/base_pipeline.py:305-307): same result (sum / world_size).

On one box the arena lives in symmetric memory and the collective is this package's kernel over NVLink peer memory
(csrc/peer_reduce.cu: two-shot, reduction inside the NVSwitch when multicast is available, average fused); otherwise NCCL.

The arena is reduced in two pieces so that the collective hides behind compute: the main hash table's gradient (64 MiB
of the 88 MiB at BASELINE config 2 / 3) is final as soon as the field's backward kernels are enqueued - autograd runs
them BEFORE the two proposal rounds' backward - so its reduction starts right there on a communication stream and
overlaps with the proposal backward; only the small remainder (proposal table + MLPs) is reduced after the last kernel.
"""
from __future__ import annotations

import os

from typing import Iterable, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist
from torch import Tensor, nn

from ._lib import NeuradarB200Error


def shard_bounds(num_rays: int, world_size: int, rank: int, granule: int = 1) -> Tuple[int, int]:
    """Contiguous slice [start, end) of a global ray batch owned by `rank`.

    `granule` keeps camera patches (1024 rays) or radar scans (256 rays) whole: the decoders downstream consume
    them as units (SURVEY.md 8e).  Granules are dealt as evenly as possible, earlier ranks get the remainder."""
    if num_rays % granule != 0:
        raise ValueError(f"num_rays={num_rays} is not a multiple of granule={granule}")
    units = num_rays // granule
    base, rem = divmod(units, world_size)
    start = rank * base + min(rank, rem)
    end = start + base + (1 if rank < rem else 0)
    return start * granule, end * granule


def _world() -> int:
    if not dist.is_available() or not dist.is_initialized():
        return 1
    return dist.get_world_size()


class PeerMemory:
    """A flat fp32 buffer in symmetric memory (every rank's copy is mapped into every process of the box) plus a zeroed
    flag area, for `nrb_peer_all_reduce` (csrc/peer_reduce.cu).  Built on torch.distributed._symmetric_memory, which only
    provides the mapping; the collective is this package's kernel."""

    def __init__(self, numel: int, device):
        import ctypes as C

        import torch.distributed._symmetric_memory as symm

        self.world, self.rank, pg = dist.get_world_size(), dist.get_rank(), dist.group.WORLD
        self.flat = symm.empty(numel, dtype=torch.float32, device=device)
        self.flags = symm.empty(256, dtype=torch.int32, device=device)  # 4 slots x 64 words (peer_reduce.cu: kSlotWords)
        self.flat.zero_()
        self.flags.zero_()
        h_flat, h_flags = symm.rendezvous(self.flat, pg), symm.rendezvous(self.flags, pg)
        bufs = [h_flat.get_buffer(p, (numel,), torch.float32).data_ptr() for p in range(self.world)]
        sigs = [h_flags.get_buffer(p, (256,), torch.int32).data_ptr() for p in range(self.world)]
        self._handles = (h_flat, h_flags)
        # NVLS: the W replicas of the arena behind one multicast address, when the fabric offers it (NRB_PEER_MULTICAST=0: no)
        self.multicast_ptr = 0
        if os.environ.get("NRB_PEER_MULTICAST", "1") != "0":
            try:
                # (with two ranks the switch has nothing to save; measured slower than the unicast form)
                base = int(h_flat.multicast_ptr or 0) if self.world > 2 else 0
                self.multicast_ptr = base + int(getattr(h_flat, "offset", 0)) if base else 0
            except Exception:  # noqa: BLE001
                self.multicast_ptr = 0
        self.buffer_ptrs = (C.c_uint64 * self.world)(*bufs)
        self.flag_ptrs = (C.c_uint64 * self.world)(*sigs)
        torch.cuda.synchronize(device)
        dist.barrier()  # every rank's flags are zero before anyone's first collective

    def all_reduce(self, slot: int, offset: int, n: int, scale: float, max_ctas: int = 0) -> None:
        """In place over floats [offset, offset + n) of every rank's buffer, on the current stream."""
        from . import _lib

        _lib.call("nrb_peer_all_reduce", self.buffer_ptrs, self.flag_ptrs, self.multicast_ptr, self.rank, self.world, slot, offset,
                  n, float(scale), max_ctas, _lib.stream_ptr())


def peer_memory_or_none(numel: int, device) -> Optional[PeerMemory]:
    """Symmetric memory for the arena when this is a single-box NCCL job of at most 8 ranks (NRB_PEER_REDUCE=0 disables)."""
    if (os.environ.get("NRB_PEER_REDUCE", "1") == "0" or _world() == 1 or torch.device(device).type != "cuda"
            or dist.get_backend() != "nccl" or dist.get_world_size() > 8):
        return None
    if int(os.environ.get("LOCAL_WORLD_SIZE", dist.get_world_size())) != dist.get_world_size():
        return None  # more than one box: the ranks do not share an NVSwitch domain
    pm = None
    try:
        pm = PeerMemory(numel, device)
    except Exception as e:  # noqa: BLE001 - no peer mapping on this system: NCCL carries the collective
        import warnings

        warnings.warn(f"neuradar_b200: peer-memory all-reduce unavailable ({type(e).__name__}: {str(e)[:120]}); using NCCL")
    # every rank must take the same route: agree on the outcome
    ok = torch.tensor([1 if pm is not None else 0], device=device, dtype=torch.int32)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    return pm if int(ok.item()) == 1 else None


def padded_numel(n: int) -> int:
    """Floats a view of `n` elements takes in a flat gradient buffer: 16-byte aligned for the scatters' vector atomics."""
    return (n + 3) // 4 * 4


class OverlappedReduce:
    """All-reduce of one flat gradient buffer whose first `n_early` elements become final early in the backward pass.

    `start_early()` (called by the backward of the kernel that produced those gradients, on the stream it ran on) launches
    their all-reduce on a side stream; `finish()` reduces the rest and joins.  Without an early call `finish()` reduces
    everything in one collective.  Single process: no-ops.  States: idle -> (start_early) in flight -> (finish) idle; a
    second `start_early()` in flight raises, as the write that caused it would never be exchanged.  The constructor is a
    collective point: it creates the side stream and the early piece's communicator, so the backward creates nothing."""

    def __init__(self, flat: Tensor, n_early: int = 0, peer: Optional[PeerMemory] = None):
        self.flat, self.n_early = flat, int(n_early)
        self.peer = peer  # the buffer lives in symmetric memory: this package's NVLink kernel instead of NCCL
        self._work = None  # idle; in flight: the early collective (True on the peer-memory route)
        overlap = self.n_early > 0 and _world() > 1 and flat.is_cuda
        self._stream = torch.cuda.Stream(device=flat.device) if overlap else None
        self._early_group = self._cta_limited_group() if overlap and peer is None else None  # None: the default one

    early_ctas = int(os.environ.get("NRB_EARLY_REDUCE_CTAS", "8"))
    """CTAs NCCL may use for the EARLY collective.  It runs beside the proposal backward, which it slows down in proportion
    to the SMs it occupies (B200 x8, 64 MiB: 16+ CTAs by default, 0.28 ms alone, +0.15 ms on the overlapped kernels;
    8 CTAs: 0.50 ms alone, still well inside the 1.3 ms it has to hide in; profiles/r2_nccl_probe_n8.txt)."""

    def _cta_limited_group(self):
        """A second NCCL communicator over the same ranks whose kernels are limited to `early_ctas` CTAs (None: default)."""
        if self.early_ctas <= 0 or dist.get_backend() != "nccl":
            return None
        try:
            opts = dist.ProcessGroupNCCL.Options()
            opts.config.max_ctas = self.early_ctas
            opts.config.min_ctas = 1
            return dist.new_group(backend="nccl", pg_options=opts)
        except Exception:  # noqa: BLE001 - an older torch / NCCL without communicator configs: use the default one
            return None

    def use_nccl(self) -> None:
        """Reduce with NCCL although the buffer is in symmetric memory.  A collective point, like the constructor."""
        self.peer = None
        if self._stream is not None:
            self._early_group = self._cta_limited_group()

    peer_ctas = int(os.environ.get("NRB_PEER_CTAS", "0"))
    """CTAs of the peer-memory kernel (0 = measured defaults, profiles/r2_peer_reduce_probe.txt): with in-switch reduction
    (NVLS multicast) 8 CTAs already saturate the links (8 x B200: 24 MiB in 71 us, 64 MiB in 159 us; more CTAs are slower);
    without it the early piece gets 16 CTAs and the exposed tail all of them."""

    def _peer_ctas(self, early: bool) -> int:
        if self.peer_ctas > 0:
            return self.peer_ctas
        if self.peer.multicast_ptr:
            return 8
        return 16 if early else 0

    def start_early(self) -> None:
        if self.n_early <= 0 or _world() == 1:
            return
        if self._work is not None:
            raise NeuradarB200Error("early gradients written again while their all-reduce was in flight: under data "
                                    "parallelism one backward per all_reduce() (no gradient accumulation, no second backward)")
        if not self.flat.is_cuda:
            self._work = dist.all_reduce(self.flat[: self.n_early], op=dist.ReduceOp.SUM, async_op=True)
            return
        self._stream.wait_stream(torch.cuda.current_stream(self.flat.device))
        with torch.cuda.stream(self._stream):
            if self.peer is not None:  # (already averaged: finish() returns 1)
                self.peer.all_reduce(0, 0, self.n_early, 1.0 / self.peer.world, self._peer_ctas(True))
                self._work = True
            else:
                self._work = dist.all_reduce(self.flat[: self.n_early], op=dist.ReduceOp.SUM, group=self._early_group,
                                             async_op=True)

    def finish(self, group=None) -> float:
        """Sum over ranks; returns the factor that still has to be applied for the average: 1 / world_size after NCCL (the
        caller applies it or hands it to the optimiser), 1 after the peer-memory kernel (which averages in place)."""
        if group is not None and group is not dist.group.WORLD:
            raise ValueError("only the default process group is supported")
        world = _world()
        if world == 1:
            return 1.0
        early, self._work = self._work, None
        lo = self.n_early if early is not None else 0
        if self.peer is not None:  # sums AND averages in place (the x 1/world rides in the kernel)
            self.peer.all_reduce(1, lo, self.flat.numel() - lo, 1.0 / world, self._peer_ctas(False))
        else:
            dist.all_reduce(self.flat[lo:], op=dist.ReduceOp.SUM)
            if early is not None:
                early.wait()  # the current stream waits for the early collective
        if early is not None and self._stream is not None:
            torch.cuda.current_stream(self.flat.device).wait_stream(self._stream)
        return 1.0 if self.peer is not None else 1.0 / world


def order_early_first(params: Sequence[nn.Parameter], early: Optional[Iterable[nn.Parameter]]) -> Tuple[List[nn.Parameter], int]:
    """Reorder `params` so that the `early` ones come first; returns (ordered, number of early parameters)."""
    ids = {id(p) for p in (early or [])}
    first = [p for p in params if id(p) in ids]
    return first + [p for p in params if id(p) not in ids], len(first)


class GradArena:
    """One contiguous fp32 buffer that holds the gradient of every trainable parameter as a view.

    `param.grad` is pointed into the arena, so autograd accumulates straight into it, `zero()` is one memset and
    `all_reduce()` is one or two collectives (see OverlappedReduce).  Parameters that receive no gradient in a step
    (e.g. the never-evaluated first proposal field) simply contribute zeros, which is what DDP's find_unused_parameters
    does.  `direct_scatter=True` additionally lets the backward kernels add straight into the arena
    (`param._nrb_grad_sink`, functional.grad_sink_of) instead of returning a temporary to autograd.  `early` names the
    parameters (hash tables with a direct sink) whose gradient is complete when their backward kernel has run; they lead
    the buffer and that kernel's backward starts their reduction (`param._nrb_grad_ready`).  A gradient a parameter
    already has when the arena is built is copied into its view.

    Contract: gradients must stay views of the arena.  `optimizer.zero_grad()` / `module.zero_grad()` default to
    set_to_none=True and would detach them; `zero()` and `all_reduce()` therefore re-link (`relink()`).  Under data
    parallelism with `early`, exactly one backward runs per `all_reduce()`, and every rank runs it."""

    def __init__(self, params: Iterable[nn.Parameter], skip_unused: Optional[List[nn.Parameter]] = None,
                 direct_scatter: bool = False, early: Optional[Iterable[nn.Parameter]] = None):
        skip = {id(p) for p in (skip_unused or [])}
        params = [p for p in params if p.requires_grad and id(p) not in skip]
        if not params:
            raise ValueError("no trainable parameters")
        self.params, n_first = order_early_first(params, early if direct_scatter else None)
        dev = self.params[0].device
        if any(p.dtype != torch.float32 or p.device != dev for p in self.params):
            raise ValueError("GradArena expects fp32 parameters on one device")
        sizes = [padded_numel(p.numel()) for p in self.params]
        self.offsets = [sum(sizes[:i]) for i in range(len(sizes))]
        total, n_early = sum(sizes), sum(sizes[:n_first])
        peer = peer_memory_or_none(total, dev)
        self.flat = peer.flat if peer is not None else torch.zeros((total,), device=dev, dtype=torch.float32)
        self.reducer = OverlappedReduce(self.flat, n_early, peer)
        self._views = [self.flat[off : off + p.numel()].view_as(p) for p, off in zip(self.params, self.offsets)]
        for i, (p, view) in enumerate(zip(self.params, self._views)):
            if p.grad is not None:
                view.copy_(p.grad)
            p.grad = view
            if direct_scatter:
                p._nrb_grad_sink = view
                if i < n_first:
                    p._nrb_grad_ready = self.reducer.start_early

    @property
    def nbytes(self) -> int:
        return self.flat.numel() * 4

    @property
    def peer(self) -> Optional[PeerMemory]:  # None: NCCL (or a single process)
        return self.reducer.peer

    def relink(self) -> int:
        """Point every `param.grad` back into the arena; returns how many had been detached.  A gradient that was replaced
        is copied into its view.  One that was set to None counts as zero, unless the parameter has a sink: the backward
        kernels add into the sink whatever `.grad` is, so its view already holds the gradient."""
        fixed = 0
        for p, view in zip(self.params, self._views):
            if p.grad is not None and p.grad.data_ptr() == view.data_ptr():
                continue
            sink = getattr(p, "_nrb_grad_sink", None) is not None
            if p.grad is not None:
                view.copy_(p.grad)
            elif not sink:
                view.zero_()
            p.grad = view
            if sink:
                p._nrb_grad_sink = view
            fixed += 1
        return fixed

    def zero(self) -> None:
        self.flat.zero_()
        for p, view in zip(self.params, self._views):  # after the memset a detached gradient simply counts as zero
            if p.grad is None or p.grad.data_ptr() != view.data_ptr():
                p.grad = view

    def reduce(self, group=None) -> float:
        """Re-link, then sum over the ranks of the default process group; returns the factor that makes it the average."""
        self.relink()
        return self.reducer.finish(group)

    def all_reduce(self, group=None, average: bool = True) -> None:
        mult = self.reduce(group)
        if average and mult != 1.0:
            self.flat.mul_(mult)
        elif not average and self.peer is not None and _world() > 1:
            self.flat.mul_(float(_world()))  # (the peer-memory kernel averages in place)
