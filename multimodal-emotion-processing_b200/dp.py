"""Data-parallel training plumbing: batch sharding and a bucketed gradient all-reduce that is
overlapped with backward.  The reference has no multi-GPU code (``device = cuda:0`` everywhere,
others/realformer.py:16); this is the new exchange step SURVEY.md §8(e) asks for.

One process per GPU (``torch.distributed``, NCCL over NVLink/NVSwitch; gloo on CPU for tests).
Every op of the model is per-sample and the losses are means over equal shards, so averaging the
per-rank gradients reproduces the single-process full-batch gradient up to fp32 summation order.

Mechanics: parameters are packed into flat float32 buckets in the order their gradients become
ready (observed during the first backward, like DDP's bucket rebuild; parameters that never
receive a gradient, e.g. the first-layer ``c`` of each chain, are left out identically on all
ranks).  The fused blocks accumulate ALL their parameter gradients into one zero-filled buffer;
a block declares that buffer's layout (``module.mmemo_grad_unit()``) and the reducer places the
whole unit in a bucket with the block's own offsets, so the block's buffer IS a bucket region
(``ops.register_zbuf_dest``): the buckets are zero-filled once per backward, no block fills or
copies anything, and ``p.grad`` of every block parameter is a view of its bucket (one writer per
region and backward — a shared block's second use goes through autograd's normal accumulation).
Other gradients are copied into their slots by a post-accumulate hook.  When a bucket is full its
all-reduce is issued asynchronously on a side stream, so it overlaps the rest of backward, also
under CUDA-graph capture.  ``finish()`` joins the collectives.  The loss is pre-scaled by 1/world
so a SUM reduction yields the average (gloo has no AVG).

Transport: on CUDA the buckets are carved out of ONE symmetric-memory allocation
(``torch.distributed._symmetric_memory``: same layout on every rank, peer and NVLS multicast
mappings) and reduced by libmmemo's own two-shot kernel (csrc/allreduce.cu) on a side stream:
``multimem.ld_reduce`` lets the NVSwitch sum a slice across all replicas, ``multimem.st``
broadcasts it back.  Its CTAs (256 threads, <= 96 registers, no shared memory) fit next to a
persistent GEMM or attention CTA on the same SM; the LayerNorm backward fills the register file,
so while a bucket is in flight the one-CTA-per-SM kernels of the compute stream shrink their
grids by ``symm_sm_reserve`` SMs (``mmemo_stream_set_sm_budget``) instead of queueing statically
partitioned work behind the collective.  Measured on 2 GPUs (profiles/r02_dp_sweep_2gpu.log):
step with / without the collectives 1.62 / 1.53 ms, against 1.55 ms on one GPU.
``transport="nccl"`` (and every CPU/gloo run) uses ``dist.all_reduce`` per bucket.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import os

import torch
import torch.distributed as dist

_NO_COMM = os.environ.get("MMEMO_DP_NO_COMM") == "1"   # debug: measure the bucket plumbing alone


def shard_bounds(n: int, rank: int, world: int, align: int = 1) -> slice:
    """Contiguous, equal, ``align``-aligned shard of ``range(n)`` for ``rank``.  ``align=2`` keeps
    the R-Drop pairs (rows 2i, 2i+1; Ren-MME/run.py:143-146,332-333) on one rank."""
    if n % (world * align) != 0:
        raise ValueError(f"batch {n} is not divisible into {world} shards aligned to {align}")
    per = n // world
    return slice(rank * per, (rank + 1) * per)


def shard_batch(batch, rank: int, world: int, align: int = 1):
    """Slice every tensor of a (nested) batch along dim 0."""
    if torch.is_tensor(batch):
        return batch[shard_bounds(batch.shape[0], rank, world, align)]
    if isinstance(batch, dict):
        return {k: shard_batch(v, rank, world, align) for k, v in batch.items()}
    if isinstance(batch, (list, tuple)):
        return type(batch)(shard_batch(v, rank, world, align) for v in batch)
    return batch


class _Unit:
    """The parameters of one fused module whose gradients are accumulated into ONE contiguous
    zero-filled buffer by its backward (``module.mmemo_grad_unit()``, e.g. the full
    Attention_Block: five weight gradients + LayerNorm / bias / gate gradients).  A unit is placed
    in a bucket as a whole, with the module's own internal offsets, so that the module's buffer is
    a bucket region and none of its gradients is copied."""
    __slots__ = ("key", "members", "total")

    def __init__(self, key, members, total):
        self.key, self.members, self.total = key, list(members), int(total)

    def numel(self) -> int:
        return self.total


class _Bucket:
    __slots__ = ("flat", "params", "offsets", "pending", "work", "todo", "base", "units")

    ALIGN = 1024        # bucket length granularity (floats)

    @classmethod
    def layout(cls, params: Sequence[torch.nn.Parameter], world: int = 1):
        """Slot offsets and padded length.  The length is a multiple of 4 floats x world (the
        all-reduce kernel gives every rank a 16-byte-aligned 1/world slice): 1024 for the usual
        power-of-two worlds, lcm(1024, 4*world) otherwise."""
        import math
        align = math.lcm(cls.ALIGN, 4 * max(world, 1))
        offsets, n = [], 0
        for p in params:          # an entry is a parameter or a _Unit (offset = start of its region)
            offsets.append(n)
            n += (p.numel() + 31) // 32 * 32          # 128-byte aligned slots
        return offsets, (n + align - 1) // align * align

    def __init__(self, entries: Sequence, flat: Optional[torch.Tensor] = None,
                 base: int = 0, world: int = 1):
        starts, n = self.layout(entries, world)
        self.params, self.offsets, self.units = [], [], []
        for e, o in zip(entries, starts):
            if isinstance(e, _Unit):
                self.units.append((e, o))
                for p, rel in e.members:
                    self.params.append(p)
                    self.offsets.append(o + rel)
            else:
                self.params.append(e)
                self.offsets.append(o)
        p0 = self.params[0]
        self.flat = (torch.zeros(n, dtype=torch.float32, device=p0.device) if flat is None
                     else flat[base:base + n])
        self.base = base    # offset of this bucket inside the shared symmetric buffer
        self.pending = len(self.params)
        self.work = None
        self.todo = []      # (parameter, slot view) pairs whose gradient still has to be copied in


class GradReducer:
    def __init__(self, model: torch.nn.Module, world_size: Optional[int] = None,
                 bucket_bytes: int = 8 << 20, group=None, zero_copy: bool = True,
                 sm_reserve: int = 16, reserve_launches: int = 5, transport: str = "auto",
                 comm_blocks: int = 16, symm_sm_reserve: int = 16):
        self.model = model
        self.group = group
        self.world = world_size if world_size is not None else dist.get_world_size(group)
        self.bucket_bytes = bucket_bytes
        self.enabled = True
        self.no_comm = _NO_COMM
        self.zero_copy = zero_copy
        self.buckets: List[_Bucket] = []
        # SMs left to the NCCL kernel of a bucket for the next `reserve_launches` GEMM launches after
        # the all-reduce is issued (set sm_reserve to NCCL_MAX_CTAS; 0 disables)
        on_cuda = next(model.parameters()).is_cuda
        if transport not in ("auto", "nccl", "symm"):
            raise ValueError(f"unknown transport {transport!r}")
        # "auto": libmmemo's symmetric-memory all-reduce on CUDA, the process group's otherwise
        self.transport = "nccl" if (transport == "nccl" or not on_cuda) else "symm"
        self._requested_transport = transport
        self.comm_blocks = comm_blocks
        self._symm = None           # (handle, comm stream) once the buckets are built
        self._flat_all = None       # the one symmetric buffer all buckets are views of
        self._nccl_sm_reserve = sm_reserve if on_cuda else 0
        # (the symmetric-memory kernel: `symm_sm_reserve` SMs, 0 = share the SMs with the GEMMs)
        self._symm_sm_reserve = symm_sm_reserve if on_cuda else 0
        self.sm_reserve = self._nccl_sm_reserve if self.transport == "nccl" else self._symm_sm_reserve
        self.reserve_launches = reserve_launches
        self._slot: Dict[torch.nn.Parameter, tuple] = {}
        self._order: List[torch.nn.Parameter] = []
        self._built = False
        self._hooks = [p.register_post_accumulate_grad_hook(self._on_grad)
                       for p in model.parameters() if p.requires_grad]

    # -- bucket construction ---------------------------------------------------------------
    def _build(self) -> None:
        """Pack the parameters that received a gradient, in readiness order, into buckets."""
        # fused modules declare gradient units (see _Unit); a unit enters the order where its first
        # gradient became ready, with the members that actually receive gradients
        got = set(self._order)
        unit_of: Dict[torch.nn.Parameter, _Unit] = {}
        if self.zero_copy and self._order:
            for m in self.model.modules():
                fn = getattr(m, "mmemo_grad_unit", None)
                if fn is None:
                    continue
                key, members, total = fn()
                members = [(p, off) for p, off in members if p in got]
                if key in got and members and not any(p in unit_of for p, _ in members):
                    u = _Unit(key, members, total)
                    for p, _ in members:
                        unit_of[p] = u
        entries, seen = [], set()
        for p in self._order:
            u = unit_of.get(p)
            if u is None:
                entries.append(p)
            elif id(u) not in seen:
                seen.add(id(u))
                entries.append(u)
        groups, cur, size = [], [], 0
        for e in entries:
            cur.append(e)
            size += e.numel() * 4
            if size >= self.bucket_bytes:
                groups.append(cur)
                cur, size = [], 0
        if cur:
            groups.append(cur)
        flat, bases = None, [0] * len(groups)
        if self.transport == "symm" and groups:
            first = groups[0][0]
            flat, bases = self._try_symmetric([_Bucket.layout(g, self.world)[1] for g in groups],
                                              (first.key if isinstance(first, _Unit) else first).device)
        self._flat_all = flat
        self.buckets = [_Bucket(g, flat, base, self.world) for g, base in zip(groups, bases)]
        for bi, b in enumerate(self.buckets):
            from . import ops
            for u, off in b.units:
                # the module's whole gradient buffer is this bucket region
                ops.register_zbuf_dest(u.key, b.flat, off, u.total)
            for p, off in zip(b.params, b.offsets):
                self._slot[p] = (bi, off)
        self._built = True

    def _try_symmetric(self, sizes: List[int], device):
        """Symmetric buckets when every rank can set them up; otherwise ALL ranks switch to the
        process group's all-reduce (a transport choice between two GPU paths, agreed collectively —
        e.g. GPUs without peer access, or a torch build without symmetric memory)."""
        import sys
        flat, bases, err = None, [0] * len(sizes), None
        # vote on what every rank can check locally (import, device, peer access) BEFORE entering
        # the collective rendezvous: a rank that failed here would otherwise leave the others
        # hanging inside symm_mem.rendezvous
        try:
            import torch.distributed._symmetric_memory as symm_mem  # noqa: F401
            if device.type != "cuda":
                raise RuntimeError("symmetric memory needs CUDA tensors")
            me = device.index if device.index is not None else torch.cuda.current_device()
            for peer in range(torch.cuda.device_count()):
                if peer != me and not torch.cuda.can_device_access_peer(me, peer):
                    raise RuntimeError(f"no peer access between GPU {me} and GPU {peer}")
        except Exception as ex:      # noqa: BLE001
            err = ex
        ok = torch.tensor([0.0 if err is not None else 1.0], device=device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
        if float(ok.item()) == 1.0:
            try:
                flat, bases = self._alloc_symmetric(sizes, device)
            except Exception as ex:  # noqa: BLE001 - any setup failure means "not available here"
                err = ex
            ok = torch.tensor([0.0 if err is not None else 1.0], device=device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            if float(ok.item()) == 1.0:
                return flat, bases
        if self._requested_transport == "symm":
            raise RuntimeError(f"symmetric-memory gradient transport unavailable: {err!r}")
        if dist.get_rank(self.group) == 0:
            print(f"[mmemo_b200.dp] symmetric memory unavailable ({err!r}); using the process "
                  "group's all-reduce", file=sys.stderr)
        self._symm = None
        self.transport = "nccl"
        self.sm_reserve = self._nccl_sm_reserve
        return None, [0] * len(sizes)

    def _alloc_symmetric(self, sizes: List[int], device):
        """One symmetric allocation for all buckets + rendezvous (collective, first step only)."""
        import torch.distributed._symmetric_memory as symm_mem
        group = self.group if self.group is not None else dist.group.WORLD
        bases, total = [], 0
        for n in sizes:
            bases.append(total)
            total += n
        flat = symm_mem.empty(total, dtype=torch.float32, device=device)
        flat.zero_()
        handle = symm_mem.rendezvous(flat, group)
        if handle.world_size != self.world:
            raise RuntimeError("symmetric-memory group size does not match the reducer's world size")
        # our flag slots live in the upper half of the signal pad (torch's own barriers use the
        # lower part); one slot per (block, peer)
        self._slot_base = handle.signal_pad_size // 8
        if (self._slot_base + self.comm_blocks * self.world) * 4 > handle.signal_pad_size:
            raise RuntimeError("signal pad too small for comm_blocks x world flags")
        torch.cuda.synchronize(device)
        dist.barrier(group)
        self._symm = (handle, torch.cuda.Stream(device=device))
        return flat, bases

    def _launch_symm(self, b: _Bucket) -> None:
        """Issue the in-place all-reduce of one bucket on the side stream."""
        from . import ops
        handle, comm = self._symm
        comm.wait_stream(torch.cuda.current_stream())
        ops._call("mmemo_allreduce_sum_f32", handle.multicast_ptr or None, handle.buffer_ptrs_dev,
                  handle.signal_pad_ptrs_dev, self._slot_base, b.base, b.flat.numel(), handle.rank,
                  self.world, self.comm_blocks, comm.cuda_stream)

    @property
    def uses_multicast(self) -> bool:
        return self._symm is not None and bool(self._symm[0].multicast_ptr)

    def bucket_layout(self) -> List[List[int]]:
        """[[numel, ...] per bucket] — identical on every rank (asserted by the tests)."""
        return [[p.numel() for p in b.params] for b in self.buckets]

    # -- hooks -----------------------------------------------------------------------------
    def _on_grad(self, p: torch.nn.Parameter) -> None:
        if not self.enabled or self.world == 1:
            return
        if p.grad is None:
            # an autograd node handed this parameter an undefined gradient (e.g. the first-layer
            # ``c`` of a chain, which has no previous scores): the hook fires but nothing was
            # accumulated — identical on every rank, so the parameter simply stays out of the buckets
            return
        if not self._built:
            self._order.append(p)
            return
        bi, off = self._slot[p]
        b = self.buckets[bi]
        if p.grad.data_ptr() != b.flat.data_ptr() + 4 * off:     # not produced in place
            b.todo.append((p, b.flat[off:off + p.numel()].view_as(p)))
        b.pending -= 1
        if b.pending == 0:
            if b.todo:   # one multi-tensor copy for all small gradients of the bucket
                torch._foreach_copy_([v for _, v in b.todo], [q.grad for q, _ in b.todo])
                for q, v in b.todo:
                    q.grad = v
                b.todo = []
            if self.no_comm:      # measurement knob: bucket plumbing without the collectives
                return
            if self._symm is not None:
                self._launch_symm(b)
            else:
                b.work = dist.all_reduce(b.flat, op=dist.ReduceOp.SUM, group=self.group,
                                         async_op=True)
            if self.sm_reserve:
                from . import ops
                ops.reserve_sms_for(self.reserve_launches, self.sm_reserve)

    # -- public API --------------------------------------------------------------------------
    def backward(self, loss: torch.Tensor) -> None:
        """``loss.backward()`` with the gradient exchange overlapped; on return every ``p.grad``
        holds the average over ranks."""
        if not self.enabled or self.world == 1:
            loss.backward()
            return
        in_place_ok = True
        for b in self.buckets:
            b.pending = len(b.params)
            b.work = None
            b.todo = []
            # After a step p.grad is a view of its all-reduce bucket and holds the AVERAGED gradient.
            # A second backward() without zero_grad(set_to_none=True) would make autograd accumulate
            # the new local gradient into that view and the whole bucket would be SUM-reduced again
            # (the old contribution multiplied by the world size) - refuse instead of training on
            # silently wrong gradients.  The reference loops call optimizer.zero_grad() before every
            # backward (others/realformer.py:305), whose default is set_to_none=True.
            if any(p.grad is not None for p in b.params):
                raise RuntimeError(
                    "GradReducer.backward(): parameters still hold gradients from the previous "
                    "step; call optimizer.zero_grad() / model.zero_grad(set_to_none=True) first "
                    "(gradient accumulation across backward() calls is not supported)")
        if self.zero_copy:
            from . import ops
            ops.grad_dest_enabled = in_place_ok
            ops.grad_dest_zeroed = False
            ops.begin_backward()
            if in_place_ok and self._built and self.buckets and self.buckets[0].flat.is_cuda:
                # one fill for all buckets (they are views of one symmetric buffer) instead of one
                # per weight gradient inside the split-K GEMM launches
                if self._flat_all is not None:
                    self._flat_all.zero_()
                else:
                    for b in self.buckets:
                        b.flat.zero_()
                ops.grad_dest_zeroed = True
        try:
            (loss / self.world).backward()
        finally:
            if self.zero_copy:
                ops.grad_dest_zeroed = False
        self.finish()

    def finish(self) -> None:
        if not self._built:
            # first step: discover which parameters get gradients and in which order, then reduce
            # everything bucket by bucket (no overlap this once)
            self._build()
            for b in self.buckets:
                for p, off in zip(b.params, b.offsets):
                    view = b.flat[off:off + p.numel()].view_as(p)
                    view.copy_(p.grad)
                    p.grad = view
                if self.no_comm:
                    continue
                if self._symm is not None:
                    self._launch_symm(b)
                else:
                    dist.all_reduce(b.flat, op=dist.ReduceOp.SUM, group=self.group)
            if self._symm is not None:
                torch.cuda.current_stream().wait_stream(self._symm[1])
            return
        if self.sm_reserve:
            from . import ops
            ops.release_sms()
        for b in self.buckets:
            if b.pending != 0:
                raise RuntimeError("a bucketed parameter received no gradient this step; the set of "
                                   "used parameters must not change between steps")
            if b.work is not None:
                b.work.wait()
                b.work = None
        if self._symm is not None and not self.no_comm:
            torch.cuda.current_stream().wait_stream(self._symm[1])

    def remove(self) -> None:
        for h in self._hooks:
            h.remove()
        self._hooks = []
        if self.buckets:      # the fused backward must stop writing into this reducer's buckets
            from . import ops
            ops.unregister_zbuf_dests([b.flat for b in self.buckets])
