"""Multi-GPU plumbing for the two paths that shard (SURVEY.md 8e).  One process per GPU,
torch.distributed (NCCL over NVLink 5 / NVSwitch) for the plumbing only.

* Reverse sampling shards the batch of generated slices / volumes across ranks with NO data-path
  collective: every sample's trajectory depends only on its own noise stream (per-sample
  GroupNorm, per-sample attention).  Rank r draws from seed `base_seed + r`; an optional final
  gather brings the volumes to rank 0 for saving (ddpm_3d_ldm/show_model.py:254-255).
* DDP training is pure data parallelism.  The drop-in UNets are ordinary nn.Modules whose
  gradients arrive through one autograd node, so torch's DistributedDataParallel (the wrapper
  the reference uses, ddpm_3d_ldm/train.py:232-233) works unchanged but can only reduce after
  the whole backward.  `DistributedDataParallel` here has the same constructor and `.module`,
  and all-reduces contiguous buckets of the gradient arena on a communication stream while the
  rest of the backward launch list executes (GradSync).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def shard_bounds(total: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous [lo, hi) share of `total` items for `rank`; the first total % world ranks get
    one extra item."""
    if total < 0 or world < 1 or not (0 <= rank < world):
        raise ValueError(f"bad shard request total={total} world={world} rank={rank}")
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def _world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def sample_sharded(diffusion, total_batch: int, *sample_args, base_seed: int = 1234,
                   gather: bool = True, per_sample_kwargs: Optional[dict] = None,
                   method: str = "sample", **sample_kwargs) -> Optional[torch.Tensor]:
    """Generate `total_batch` samples across all ranks: rank r runs
    getattr(diffusion, method)(its share, *sample_args, **sample_kwargs) under seed
    base_seed + r (method="sample_dpmpp", num_steps=20: the few-step sampler).

    per_sample_kwargs: tensors with a leading dim of total_batch (e.g. z_pos of the 155 slices of
    a pseudo-3D brain, slice_cond_2d_ddpm/show_model.py:179-185) that are sliced per rank.
    Returns the concatenated samples on rank 0 (None elsewhere) if gather, else the local share.
    """
    world, rank = _world()
    lo, hi = shard_bounds(total_batch, world, rank)
    kw = dict(sample_kwargs)
    for k, v in (per_sample_kwargs or {}).items():
        if v.shape[0] != total_batch:
            raise ValueError(f"{k} must have leading dim {total_batch}")
        kw[k] = v[lo:hi]
    local = None
    if hi > lo:
        torch.manual_seed(base_seed + rank)
        local = getattr(diffusion, method)(hi - lo, *sample_args, **kw)
    if not gather or world == 1:
        return local
    return gather_to_rank0(local, total_batch)


def gather_to_rank0(local: Optional[torch.Tensor], total: int) -> Optional[torch.Tensor]:
    """Concatenate ragged per-rank shares on rank 0 (control-plane collective, off the hot path)."""
    world, rank = _world()
    if world == 1:
        return local
    objs: List[Optional[torch.Tensor]] = [None] * world if rank == 0 else None
    payload = None if local is None else local.detach().cpu()
    dist.gather_object(payload, objs, dst=0)
    if rank != 0:
        return None
    parts = [o for o in objs if o is not None]
    out = torch.cat(parts, dim=0)
    assert out.shape[0] == total
    return out


class GradSync:
    """Bucketed gradient all-reduce (mean) that overlaps the backward launch list.

    The UNet programs keep all parameter gradients in one flat fp32 arena ordered by the time
    the backward pass finishes them (backward.py: plan_segments), so a bucket is a contiguous
    slice.  `bucket_ready(lo, hi)` is called right after the launches that complete
    arena[lo:hi] were enqueued: an event on the compute stream gates the communication stream,
    where NCCL reduces the slice in place over NVLink / NVSwitch while the compute stream keeps
    executing the next segment.  `finish()` makes the compute stream wait for every bucket.
    Works on CPU tensors / gloo as well (host-logic tests): there the reduction is synchronous.

    Reference: torch DDP's reducer as used by ddpm_3d_ldm/train.py:232-233 (bucketed mean
    all-reduce of all UNet gradients, issued in reverse order, overlapped with backward)."""

    def __init__(self, process_group=None, bucket_cap_mb: float = 48.0):
        import os
        env = os.environ.get("MRI_DDP_BUCKET_MB")     # tuning experiments only
        if env:
            bucket_cap_mb = float(env)
        self.group = process_group
        self.bucket_bytes = int(bucket_cap_mb * (1 << 20))
        self.enabled = True                 # False inside DistributedDataParallel.no_sync()
        self._armed = False                 # set by the wrapper's forward, consumed by the UNet's
        self._arena: Optional[torch.Tensor] = None
        self._works: list = []
        self._comm_stream = None
        self.buckets_last_step: List[Tuple[int, int]] = []
        self._pending_local = False         # a backward ran under no_sync(): .grad holds local sums
        self.bucket_events: list = []       # per bucket (ready, start, end) CUDA events when timing
        self.time_buckets = False

    def take(self) -> Optional["GradSync"]:
        """Called by the UNet's forward: the next backward synchronises only if the call came
        through the DistributedDataParallel wrapper (calling `.module` directly stays local,
        as with torch DDP)."""
        armed, self._armed = self._armed, False
        return self if armed else None

    def world(self) -> int:
        return dist.get_world_size(self.group) if dist.is_available() and dist.is_initialized() else 1

    def active(self) -> bool:
        return self.enabled and self.world() > 1

    def note_local_backward(self) -> None:
        """A backward pass ran with the all-reduce disabled (no_sync()): its gradients were
        accumulated into `.grad` rank-locally."""
        if self.world() > 1:
            self._pending_local = True

    def reduce_pending(self, params) -> None:
        """torch DDP semantics for gradient accumulation: the first synchronised backward after
        no_sync() steps reduces what those steps left in `.grad` as well (mean of the sums = sum of
        the means).  Called before autograd accumulates the new, already reduced gradients."""
        if not self._pending_local:
            return
        self._pending_local = False
        grads = [p.grad for p in params if p.grad is not None]
        if not grads:
            return
        flat = torch._utils._flatten_dense_tensors(grads)
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
        flat.mul_(1.0 / self.world())
        for g, f in zip(grads, torch._utils._unflatten_dense_tensors(flat, grads)):
            g.copy_(f)

    def begin(self, arena: torch.Tensor) -> None:
        self._arena = arena
        self._works = []
        self.buckets_last_step = []
        self.bucket_events = []
        if arena.is_cuda and self._comm_stream is None:
            self._comm_stream = torch.cuda.Stream(arena.device)

    def bucket_ready(self, lo: int, hi: int) -> None:
        if hi <= lo:
            return
        self.buckets_last_step.append((lo, hi))
        buf = self._arena[lo:hi]
        backend = dist.get_backend(self.group)
        if not buf.is_cuda:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.group)
            buf.mul_(1.0 / self.world())
            return
        cur = torch.cuda.current_stream(buf.device)
        timing = self.time_buckets
        ev = torch.cuda.Event(enable_timing=timing)
        ev.record(cur)
        with torch.cuda.stream(self._comm_stream):
            self._comm_stream.wait_event(ev)
            if timing:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(self._comm_stream)
            if backend == "nccl":
                w = dist.all_reduce(buf, op=dist.ReduceOp.AVG, group=self.group, async_op=True)
            else:
                w = dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            if timing:
                # NCCL runs the collective on its own stream: make the communication stream wait
                # for it, so that the second event fires when the bucket has really been reduced
                w.wait()
                e1.record(self._comm_stream)
                self.bucket_events.append((ev, e0, e1, (hi - lo) * buf.element_size()))
            self._works.append((w, buf, backend))

    def finish(self) -> None:
        """Compute stream waits for all buckets (no host synchronisation with NCCL)."""
        timing = self.time_buckets and self._works and self._works[0][1].is_cuda
        if timing:  # how long the compute stream stalls here = the exposed communication
            cur = torch.cuda.current_stream(self._works[0][1].device)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(cur)
        for w, buf, backend in self._works:
            w.wait()
            if backend != "nccl":
                buf.mul_(1.0 / self.world())
        if timing:
            b.record(cur)
            self.finish_events = (a, b)
        self._works = []

    def bucket_report(self) -> Optional[dict]:
        """After a step run with time_buckets = True (and a device synchronise): per-bucket
        queueing / transfer times, the time the compute stream stalled in finish() (exposed
        communication) and the bucket that ended last."""
        if not self.bucket_events or getattr(self, "finish_events", None) is None:
            return None
        a, b = self.finish_events
        rows = []
        for i, (ready, e0, e1, nbytes) in enumerate(self.bucket_events):
            rows.append({"bucket": i, "mbytes": round(nbytes / 1e6, 2),
                         "queue_ms": round(ready.elapsed_time(e0), 4),
                         "comm_ms": round(e0.elapsed_time(e1), 4),
                         # > 0: this bucket was still in flight when the backward launch list ended
                         "end_after_backward_ms": round(a.elapsed_time(e1), 4)})
        last = max(rows, key=lambda r: r["end_after_backward_ms"])
        return {"exposed_comm_ms": round(a.elapsed_time(b), 4), "limiting_bucket": last["bucket"],
                "buckets": rows}


class DistributedDataParallel(torch.nn.Module):
    """Drop-in for `torch.nn.parallel.DistributedDataParallel` around the drop-in UNets
    (`DDP(model, device_ids=[local_rank])`, ddpm_3d_ldm/train.py:232-233; `.module` unwrap,
    train.py:607): parameters and buffers are broadcast from rank 0 at construction, and every
    backward pass mean-all-reduces the gradients in buckets that overlap the remaining backward
    launches (GradSync).  torch's own DDP also works on these modules, but their gradients come
    out of ONE autograd node, so its reducer can only start after the whole backward."""

    def __init__(self, module: torch.nn.Module, device_ids=None, output_device=None, dim=0,
                 broadcast_buffers=True, process_group=None, bucket_cap_mb: float = 48.0,
                 find_unused_parameters=False, gradient_as_bucket_view=False, static_graph=False,
                 **_ignored):
        super().__init__()
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("DistributedDataParallel needs an initialised process group")
        from .modules import EngineModule
        if not isinstance(module, EngineModule):
            raise TypeError("mri_image_generation_b200.parallel.DistributedDataParallel wraps the "
                            "drop-in UNet classes; use torch's DDP for other modules")
        self.module = module
        self.process_group = process_group
        self.device_ids = device_ids
        self.broadcast_buffers = broadcast_buffers
        with torch.no_grad():
            for t in list(module.parameters()) + list(module.buffers()):
                dist.broadcast(t, src=dist.get_global_rank(process_group, 0) if process_group else 0,
                               group=process_group)
        self.grad_sync = GradSync(process_group, bucket_cap_mb)
        module.__dict__["_mri_grad_sync"] = self.grad_sync

    def forward(self, *args, **kwargs):
        self.grad_sync._armed = True
        try:
            return self.module(*args, **kwargs)
        finally:
            self.grad_sync._armed = False

    def no_sync(self):
        """Context manager: backward passes inside it skip the all-reduce (local gradients).

        As with torch DDP, the first synchronised backward afterwards also mean-all-reduces what
        the no_sync() steps accumulated in `.grad` (GradSync.reduce_pending), so gradient
        accumulation gives the same result as torch's wrapper.  The reference scripts never use
        no_sync()."""
        import contextlib

        @contextlib.contextmanager
        def ctx():
            old = self.grad_sync.enabled
            self.grad_sync.enabled = False
            try:
                yield
            finally:
                self.grad_sync.enabled = old
        return ctx()


def wrap_ddp(module: torch.nn.Module, device: torch.device, overlap: bool = True, **kw) -> torch.nn.Module:
    """Data-parallel wrapper of a drop-in UNet (train.py:232-233).  overlap=True: the bucketed
    all-reduce of this package, running under the backward launch list; overlap=False: torch's
    DistributedDataParallel, whose reducer fires after the (single-node) backward."""
    if overlap:
        return DistributedDataParallel(module, device_ids=[device.index], **kw)
    from torch.nn.parallel import DistributedDataParallel as DDP
    return DDP(module, device_ids=[device.index], output_device=device.index,
               find_unused_parameters=False, **kw)


def ddp_for_scripts(torch_ddp):
    """What `overlay.install(overlap_ddp=True)` binds `torch.nn.parallel.DistributedDataParallel`
    to: `DDP(unet, device_ids=[local_rank], ...)` (ddpm_3d_ldm/train.py:232-233) gives the
    overlapped wrapper for the drop-in UNets and torch's own wrapper for every other module (the
    VAE, train.py:232), with the reference's call signature."""
    from .modules import EngineModule

    def DDP(module, *args, **kwargs):
        if isinstance(module, EngineModule) and getattr(module, "SUPPORTS_GRAD_SYNC", False):
            return DistributedDataParallel(module, *args, **kwargs)
        return torch_ddp(module, *args, **kwargs)

    DDP.__wrapped__ = torch_ddp
    return DDP
