"""Multi-GPU plumbing of the rasterization() hot path.

(1) View-axis data parallelism (SURVEY.md section 8e): every rank holds the full (replicated) set of Gaussian
parameters and renders its own camera views; the only coupling is the sum of the parameter gradients -- ONE
all-reduce of the 59 floats / Gaussian (means 3 | quats 4 | scales 3 | opacities 1 | SH 48 -> 236 B), done by
our own kernel over NVSwitch multicast / peer memory (``NvlsGradArena``, csrc/nvls.cu) or by NCCL / gloo
(``all_reduce_gaussian_grads``).
(2) The row collectives of the reference's ``distributed=True`` mode (Gaussian-sharded,
/root/reference/gsplat/distributed.py:117-272): ``all_gather_rows`` (Seam A, cameras) and the differentiable
uneven ``all_to_all_rows`` (Seam B, projected Gaussians), used by ``rendering.rasterization``.

Launch: one process per GPU (torchrun / ``cli`` below, the reference's spawner restated from
/root/reference/gsplat/distributed.py:319-375).
"""
from __future__ import annotations

import math
import os
from typing import Callable, Dict, Iterable, List, Optional, Sequence

import torch

from ._cabi import stream as _raw_stream
import torch.distributed as dist
from torch import Tensor


def shard_views(n_views: int, rank: Optional[int] = None, world_size: Optional[int] = None) -> List[int]:
    """Indices of the camera views rank ``rank`` renders: ``rank::world_size`` (round robin)."""
    rank = dist.get_rank() if rank is None else rank
    world_size = dist.get_world_size() if world_size is None else world_size
    return list(range(rank, n_views, world_size))


class GradBucket:
    """Flat fp32 buffer the gradients of all parameter tensors are packed into for a single collective."""

    def __init__(self, params: Sequence[Tensor]):
        self.params = list(params)
        self.sizes = [p.numel() for p in self.params]
        dev = self.params[0].device
        self.flat = torch.zeros(sum(self.sizes), device=dev, dtype=torch.float32)

    def pack(self) -> Tensor:
        o = 0
        for p, n in zip(self.params, self.sizes):
            if p.grad is None:
                self.flat[o : o + n].zero_()
            else:
                self.flat[o : o + n].copy_(p.grad.reshape(-1))
            o += n
        return self.flat

    def unpack(self, scale: Optional[float] = None) -> None:
        """Copy the (reduced) flat buffer back into the ``.grad`` tensors.  ``scale=None`` uses the factor stored
        by ``all_reduce_gaussian_grads(average=True, async_op=True)`` (1.0 otherwise)."""
        if scale is None:
            scale = getattr(self, "_scale", 1.0)
        self._scale = 1.0
        o = 0
        for p, n in zip(self.params, self.sizes):
            g = self.flat[o : o + n].view_as(p)
            if scale != 1.0:
                g = g * scale
            if p.grad is None:
                p.grad = g.clone()
            else:
                p.grad.copy_(g)
            o += n


def all_reduce_gaussian_grads(
    params: Sequence[Tensor], bucket: Optional[GradBucket] = None, average: bool = False, group=None,
    async_op: bool = False, coalesced: bool = False,
):
    """Sum (or average) the ``.grad`` of the replicated Gaussian parameters over all ranks with one
    all-reduce.  Returns the bucket (and the work handle when ``async_op``); call ``bucket.unpack()``
    after ``work.wait()`` in the async case.

    ``coalesced=True``: no staging buffer -- the gradient tensors themselves are reduced in place inside
    one coalesced launch (``torch.distributed._coalescing_manager``: a single NCCL group call on NVLink);
    parameters without a gradient get a zero gradient first so that every rank issues the same calls."""
    if coalesced:
        grads = []
        for p in params:
            if p.grad is None:
                p.grad = torch.zeros_like(p)
            elif not p.grad.is_contiguous():
                p.grad = p.grad.contiguous()
            grads.append(p.grad)
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            if str(dist.get_backend(group)).lower() == "nccl":
                with dist._coalescing_manager(group=group, device=grads[0].device, async_ops=False):
                    for g in grads:
                        dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group)
            else:  # gloo (CPU tests) has no coalescing: same calls, one by one
                for g in grads:
                    dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group)
            if average:
                inv = 1.0 / dist.get_world_size(group)
                for g in grads:
                    g.mul_(inv)
        return None
    if bucket is None:
        bucket = GradBucket(params)
    flat = bucket.pack()
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        bucket.unpack()
        return (bucket, None) if async_op else bucket
    work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=async_op)
    scale = 1.0 / dist.get_world_size(group) if average else 1.0
    if async_op:
        bucket._scale = scale
        return bucket, work
    bucket.unpack(scale)
    return bucket


class NvlsGradArena:
    """The gradients of the replicated Gaussian parameters in ONE symmetric fp32 buffer (same layout on every
    rank, bound to an NVSwitch multicast address) plus the in-place all-reduce over it done by our own kernel
    (csrc/nvls.cu: in-switch ``multimem.ld_reduce`` + ``multimem.st``; include/gsplat_b200.h
    gsb200_nvls_allreduce_f32).  Allocation / handle exchange is torch's symmetric-memory plumbing.

        arena = NvlsGradArena({"means": means, "quats": quats, "scales": scales, "opacities": opac, "sh": sh})
        ops.set_gradient_allocator(arena.allocator)      # the fused backward writes into the arena directly
        loss.backward(); arena.all_reduce()              # p.grad are views of the arena afterwards

    Raises RuntimeError when the GPUs have no multicast support (fall back to all_reduce_gaussian_grads)."""

    ALIGN = 64  # floats (256 B) between segment starts

    def __init__(
        self, named_params: Dict[str, Tensor], group=None, blocks: int = 128, algo: Optional[str] = None,
        row_sparse: bool = True,
    ):
        import torch.distributed._symmetric_memory as symm_mem

        from ._cabi import lib

        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        self.params = dict(named_params)
        self.blocks = int(blocks)
        dev = next(iter(self.params.values())).device
        self.offsets, o = {}, 0
        for k, p in self.params.items():
            if p.dtype != torch.float32:
                raise TypeError("NvlsGradArena holds float32 gradients")
            self.offsets[k] = o
            o += (p.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        # row-sparse mode: every parameter is [N, ...] over the same N gaussians; one bit per gaussian and rank
        # ("its gradient rows are not all zero here") lives in the same symmetric buffer, behind the gradients
        rows = {int(p.shape[0]) for p in self.params.values() if p.dim() >= 1}
        self.n_rows = rows.pop() if len(rows) == 1 and all(p.dim() >= 1 for p in self.params.values()) else None
        self.row_sparse = bool(row_sparse) and self.n_rows is not None and self.n_rows > 0
        self.bitmap_off = o
        if self.row_sparse:
            o += ((self.n_rows + 31) // 32 + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        self.numel = max(o, self.ALIGN)
        need_pad = self.blocks * self.world * 4
        if symm_mem.get_signal_pad_size() < need_pad:
            symm_mem.set_signal_pad_size(need_pad)
        self.flat = symm_mem.empty(self.numel, dtype=torch.float32, device=dev)
        self.hdl = symm_mem.rendezvous(self.flat, self.group.group_name)
        # world == 2: plain peer loads / stores move 1x the payload per direction, the multicast scheme 1.5x
        self.algo = algo or ("p2p" if self.world == 2 else "nvls")
        if self.algo not in ("p2p", "nvls"):
            raise ValueError(f"unknown all-reduce algorithm {self.algo!r}")
        if self.algo == "nvls" and int(self.hdl.multicast_ptr) == 0:
            raise RuntimeError("NvlsGradArena: no NVLS multicast support on this system")
        if int(self.hdl.signal_pad_size) < need_pad:
            raise RuntimeError("NvlsGradArena: signal pad too small for the requested number of blocks")
        self.flat.zero_()
        self.views = {k: self.flat[self.offsets[k] : self.offsets[k] + p.numel()].view(p.shape) for k, p in self.params.items()}
        self._handed_out = set()  # segments given to a backward kernel since the last all_reduce() / reset()
        self._lib = lib()
        self.bits, self._bits_requests = None, 0
        if self.row_sparse:
            import ctypes

            nw = (self.n_rows + 31) // 32
            self.bits = self.flat[self.bitmap_off : self.bitmap_off + nw].view(torch.int32)
            names = list(self.params)
            self._seg_off = (ctypes.c_int64 * len(names))(*[self.offsets[k] for k in names])
            self._seg_w = (ctypes.c_int32 * len(names))(*[self.params[k].numel() // self.n_rows for k in names])
            self.stats = torch.zeros(1, dtype=torch.int64, device=dev)

    def allocator(self, name: str, like: Optional[Tensor]) -> Optional[Tensor]:
        if name == "seen_bits":
            # asked for once per fused backward: the bitmap describes the gradients only if exactly one backward
            # wrote into the arena since the last all_reduce()
            self._bits_requests += 1
            return self.bits
        v = self.views.get(name)
        if v is None or v.shape != like.shape:
            return None
        p = self.params.get(name)
        if p is not None and p.grad is not None and p.grad.data_ptr() == v.data_ptr():
            # gradient accumulation across backward passes: the segment still holds the accumulated .grad, so this
            # backward must write elsewhere (autograd then adds it in); the arena expects zero_grad(set_to_none=True)
            return None
        if name in self._handed_out:
            # a second fused rasterization() in the same backward graph (several renders summed into one loss): the
            # backward kernels WRITE their outputs, so the same segment twice would overwrite the first gradient
            # before autograd adds the two.  The second request gets ordinary memory; autograd accumulates.
            return None
        self._handed_out.add(name)
        # a FRESH tensor object over the arena segment: autograd adopts a gradient as .grad without copying only
        # when nothing else references that tensor object
        return v.detach()

    def reset(self) -> None:
        """Forget which segments were handed out (call after optimizer.zero_grad() when a step is abandoned
        without all_reduce())."""
        self._handed_out.clear()
        self._bits_requests = 0

    def all_reduce(self) -> None:
        """Sums the .grad of all registered parameters over the ranks, in place in the arena."""
        from ._cabi import check

        self._handed_out.clear()
        # the row bitmap is trustworthy only when ONE fused backward produced every gradient that was written in place;
        # gradients that arrive from elsewhere (e.g. opacities through torch) are zero on unseen rows by construction
        sparse = self.row_sparse and self._bits_requests == 1
        self._bits_requests = 0
        for k, p in self.params.items():
            v = self.views[k]
            if p.grad is None:
                v.zero_()
            elif p.grad.data_ptr() != v.data_ptr():
                v.copy_(p.grad)  # produced elsewhere (e.g. opacities): staged
            p.grad = v
        st = _raw_stream()
        pads, pad_bytes = int(self.hdl.signal_pad_ptrs_dev), int(self.hdl.signal_pad_size)
        self.last_kind = ("rows-" if sparse else "") + self.algo
        if sparse:
            rc = self._lib.gsb200_rows_allreduce_f32(
                int(self.hdl.multicast_ptr) if self.algo == "nvls" else None, int(self.hdl.buffer_ptrs_dev), len(self.params),
                self._seg_off, self._seg_w, self.n_rows, self.bitmap_off, self.rank, self.world, pads, pad_bytes, self.blocks,
                self.stats.data_ptr(), st,
            )
        elif self.algo == "nvls":
            rc = self._lib.gsb200_nvls_allreduce_f32(
                int(self.hdl.multicast_ptr), self.numel, self.rank, self.world, pads, pad_bytes, self.blocks, st
            )
        else:
            rc = self._lib.gsb200_p2p_allreduce_f32(
                int(self.hdl.buffer_ptrs_dev), self.numel, self.rank, self.world, pads, pad_bytes, self.blocks, st
            )
        check(rc, f"{self.last_kind}_allreduce")


def render_views_dp(
    rasterize: Callable[..., tuple], gaussians: Dict[str, Tensor], viewmats: Tensor, Ks: Tensor, width: int, height: int,
    **kwargs,
):
    """Renders this rank's share (``rank::world``) of the C views in ``viewmats`` [C,4,4] / ``Ks`` [C,3,3]
    with the replicated ``gaussians`` (keys: means, quats, scales, opacities, colors).  Returns
    (render_colors, render_alphas, meta, view_ids)."""
    ids = shard_views(viewmats.shape[0]) if (dist.is_available() and dist.is_initialized()) else list(range(viewmats.shape[0]))
    idx = torch.as_tensor(ids, device=viewmats.device, dtype=torch.long)
    rc, ra, meta = rasterize(
        gaussians["means"], gaussians["quats"], gaussians["scales"], gaussians["opacities"], gaussians["colors"],
        viewmats.index_select(0, idx), Ks.index_select(0, idx), width, height, **kwargs,
    )
    return rc, ra, meta, ids


# ------------------------------------------------------------------------------------------------
# Reference-semantics ``distributed=True`` (gaussian-sharded rendering): every rank owns a shard of the
# Gaussians and a set of cameras.  Seam A: cameras are all-gathered so that each rank projects ITS Gaussians
# onto ALL cameras; Seam B: the projected Gaussians are exchanged all-to-all so that each rank ends up with
# ALL Gaussians projected onto ITS cameras, and composites those.  Both seams are differentiable (the
# backward of an all-gather is a reduce-scatter-like gather of gradients, of an all-to-all the reverse
# all-to-all).  Reference: /root/reference/gsplat/cuda/csrc/DistributedCollectives.cpp:299-453,
# csrc/Rendering.cpp:852-874,1217-1262; Python helpers /root/reference/gsplat/distributed.py:25-272.


def all_gather_ints(value: int, device, group=None) -> List[int]:
    """One integer from every rank (non-differentiable bookkeeping: counts of gaussians / cameras)."""
    world = dist.get_world_size(group)
    if world == 1:
        return [int(value)]
    mine = torch.tensor([int(value)], dtype=torch.int64, device=device)
    out = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(out, mine, group=group)
    return [int(t.item()) for t in out]


def all_gather_int_lists(values: Sequence[int], device, group=None) -> List[List[int]]:
    """The same-length integer list of every rank (e.g. per-destination row counts), rank-major."""
    world = dist.get_world_size(group)
    if world == 1:
        return [list(map(int, values))]
    mine = torch.tensor(list(map(int, values)), dtype=torch.int64, device=device)
    out = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(out, mine, group=group)
    return [t.tolist() for t in out]


def all_gather_rows(tensors: Sequence[Tensor], counts: Sequence[int], group=None) -> List[Tensor]:
    """Differentiable all-gather of several row-aligned tensors [n_r, ...] (n_r = counts[rank]) in ONE
    collective: columns are concatenated, rows padded to max(counts), gathered, trimmed.  Returns the
    tensors with sum(counts) rows, rank-major."""
    world = dist.get_world_size(group)
    if world == 1:
        return list(tensors)
    import torch.distributed.nn.functional as distF

    n = tensors[0].shape[0]
    widths = [t[0].numel() if n else int(t.numel() // max(n, 1)) for t in tensors]
    flat = torch.cat([t.reshape(n, -1) for t in tensors], dim=-1)
    cap = max(counts)
    if n < cap:
        flat = torch.cat([flat, flat.new_zeros((cap - n, flat.shape[1]))], dim=0)
    if flat.requires_grad:
        parts = distF.all_gather(flat, group=group)
    else:
        parts = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(parts, flat.contiguous(), group=group)
    full = torch.cat([p[:c] for p, c in zip(parts, counts)], dim=0)
    outs = []
    for chunk, t in zip(torch.split(full, widths, dim=-1), tensors):
        outs.append(chunk.reshape((-1,) + tuple(t.shape[1:])))
    return outs


def all_to_all_rows(
    tensors: Sequence[Tensor], send_counts: Sequence[int], recv_counts: Sequence[int], group=None
) -> List[Tensor]:
    """Differentiable all-to-all of several row-aligned tensors in ONE collective: rows
    [sum(send_counts[:j]), +send_counts[j]) go to rank j; returns tensors with sum(recv_counts) rows,
    source-rank-major.  Integer tensors are exchanged exactly (no gradient)."""
    world = dist.get_world_size(group)
    if world == 1:
        return list(tensors)
    import torch.distributed.nn.functional as distF

    n = tensors[0].shape[0]
    assert sum(send_counts) == n, (send_counts, n)
    outs: List[Optional[Tensor]] = [None] * len(tensors)
    for is_float in (True, False):
        idx = [i for i, t in enumerate(tensors) if t.is_floating_point() == is_float]
        if not idx:
            continue
        group_t = [tensors[i] for i in idx]
        widths = [int(t.numel() // max(n, 1)) if n else int(math.prod(t.shape[1:])) for t in group_t]
        flat = torch.cat([t.reshape(n, -1) for t in group_t], dim=-1).contiguous()
        send = list(flat.split(list(send_counts), dim=0))
        uneven_ok = str(dist.get_backend(group)).lower() == "nccl"
        if not uneven_ok:
            # gloo (CPU tests) only exchanges equally sized chunks: pad every chunk to the global maximum
            cap_t = torch.tensor([max(list(send_counts) + list(recv_counts))], dtype=torch.int64, device=flat.device)
            dist.all_reduce(cap_t, op=dist.ReduceOp.MAX, group=group)
            cap = int(cap_t.item())
            send = [torch.cat([x, x.new_zeros((cap - x.shape[0], x.shape[1]))], dim=0) if x.shape[0] < cap else x for x in send]
            recv = [flat.new_empty((cap, flat.shape[1])) for _ in recv_counts]
        else:
            recv = [flat.new_empty((c, flat.shape[1])) for c in recv_counts]
        if is_float and flat.requires_grad:
            recv = list(distF.all_to_all(recv, send, group=group))
        elif uneven_ok:
            dist.all_to_all(recv, [x.contiguous() for x in send], group=group)
        else:
            # gloo has no all_to_all: everyone gathers everyone's padded chunks and keeps its own column
            stacked = torch.stack(send, dim=0).contiguous()  # [world, cap, w]
            gathered = [torch.empty_like(stacked) for _ in range(world)]
            dist.all_gather(gathered, stacked, group=group)
            me = dist.get_rank(group)
            recv = [g[me] for g in gathered]
        if not uneven_ok:
            recv = [r[:c] for r, c in zip(recv, recv_counts)]
        full = torch.cat(recv, dim=0)
        for i, chunk, t in zip(idx, torch.split(full, widths, dim=-1), group_t):
            outs[i] = chunk.reshape((-1,) + tuple(t.shape[1:]))
    return outs  # type: ignore[return-value]


def camera_major_to_local(t: Tensor, C_local: int, N_world: Sequence[int]) -> Tensor:
    """[sum_i C_local * N_i, ...] received rank-major (rank i contributes its N_i gaussians for each of our
    C_local cameras) -> [C_local, sum_i N_i, ...]."""
    parts, o = [], 0
    for n_i in N_world:
        parts.append(t[o : o + C_local * n_i].reshape((C_local, n_i) + tuple(t.shape[1:])))
        o += C_local * n_i
    return torch.cat(parts, dim=1)


# ---- the reference's helper names (gsplat/distributed.py:25-272), same arguments and results, over the collectives above
def all_gather_int32(world_size: int, value, device: Optional[torch.device] = None) -> List:
    """One 32-bit integer from every rank (a list of ints for an int input, of 0-d tensors for a tensor input).
    Reference: gsplat/distributed.py:25-67.  Not differentiable."""
    if world_size == 1:
        return [value]
    if isinstance(value, int):
        assert device is not None, "device is required for scalar input"
        return [int(v) for v in all_gather_ints(value, device)]
    mine = value.reshape(1)
    out = [torch.empty_like(mine) for _ in range(world_size)]
    dist.all_gather(out, mine)
    return [t.reshape(()) for t in out]


def all_to_all_int32(world_size: int, values: Sequence, device: Optional[torch.device] = None) -> List:
    """Rank r sends values[j] to rank j and receives one integer from every rank (gsplat/distributed.py:70-114)."""
    if world_size == 1:
        return list(values)
    assert len(values) == world_size, "The length of values should be equal to world_size"
    scalars = [isinstance(v, int) for v in values]
    if any(scalars):
        assert device is not None, "device is required for scalar input"
    dev = device if device is not None else next(v.device for v in values if not isinstance(v, int))
    table = all_gather_int_lists([int(v) for v in values], dev)  # table[src][dst]
    me = dist.get_rank()
    got = [table[src][me] for src in range(world_size)]
    return [g if is_int else torch.tensor(g, dtype=torch.int, device=dev) for g, is_int in zip(got, scalars)]


def all_gather_tensor_list(world_size: int, tensor_list: Sequence[Tensor]) -> List[Tensor]:
    """Differentiable all-gather of row-aligned tensors [(N, *), ...] -> [(N * world_size, *), ...], rank-major
    (gsplat/distributed.py:117-182).  Every rank must pass the same N."""
    if world_size == 1:
        return list(tensor_list)
    n = len(tensor_list[0])
    for t in tensor_list:
        assert len(t) == n, "All tensors should have the same first dimension size"
    return all_gather_rows(list(tensor_list), [n] * world_size)


def all_to_all_tensor_list(
    world_size: int, tensor_list: Sequence[Tensor], splits: Sequence, output_splits: Optional[Sequence] = None
) -> List[Tensor]:
    """Differentiable all-to-all of row-aligned tensors: the first splits[j] rows... go to rank j
    (gsplat/distributed.py:185-272).  ``output_splits`` = all_to_all_int32(world_size, splits) when omitted."""
    if world_size == 1:
        return list(tensor_list)
    n = len(tensor_list[0])
    for t in tensor_list:
        assert len(t) == n, "All tensors should have the same first dimension size"
    assert len(splits) == world_size, "The length of splits should be equal to world_size"
    send = [int(s) for s in splits]
    if output_splits is None:
        output_splits = all_to_all_int32(world_size, send, device=tensor_list[0].device)
    return all_to_all_rows(list(tensor_list), send, [int(r) for r in output_splits])


def _distributed_worker(local_rank: int, world: int, fn: Callable, args) -> None:
    """Spawn target of :func:`cli` (module level: the spawn start method pickles it; the reference keeps its
    ``_distributed_worker`` at module level for the same reason, gsplat/distributed.py:275-316)."""
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29511")
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", rank=local_rank, world_size=world)
    try:
        fn(local_rank, local_rank, world, args)
    finally:
        dist.barrier()
        dist.destroy_process_group()


def cli(fn: Callable, args, verbose: bool = False) -> None:
    """Spawn one process per visible GPU and run ``fn(local_rank, world_rank, world_size, args)``
    (single node).  Under torchrun (RANK set) the process group is created from the environment."""
    if "RANK" in os.environ:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl")
        try:
            fn(local, dist.get_rank(), dist.get_world_size(), args)
        finally:
            dist.barrier()
            dist.destroy_process_group()
        return
    world = torch.cuda.device_count()
    if world <= 1:
        fn(0, 0, 1, args)
        return

    torch.multiprocessing.spawn(_distributed_worker, args=(world, fn, args), nprocs=world, join=True)
