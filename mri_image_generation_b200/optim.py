"""Fused optimizer step for the training path (SURVEY.md 8f row 2).

`Adam` is a drop-in for `torch.optim.Adam(params, lr, betas, eps, weight_decay)` as the reference
constructs it (ddpm_3d_ldm/train.py:243, slice_cond_2d_ddpm/model.py:126): same constructor,
`state_dict()` layout (`step`, `exp_avg`, `exp_avg_sq` per parameter), and
`torch.amp.GradScaler` support through the fused-optimizer protocol (`grad_scale` /
`found_inf`, no host synchronisation).  The whole update is ONE launch of mri_adam_step over all
parameters instead of torch's ~8 multi-tensor kernels per chunk of tensors.

`EMA` keeps an exponential moving average of a model's weights (the copy DDPM, improved-diffusion
and diffusers' training scripts sample from) with ONE mri_ema_update launch per step; passed to
`Adam(..., ema=)` it runs inside the optimizer step under GradScaler's skip rule.

fp32 parameters on a B200 only; anything else raises (no fallback).
"""
from __future__ import annotations

import copy
import ctypes as C
from typing import Iterable, Optional

import torch

from . import _lib


def _bump_versions(tensors) -> None:
    """The kernel updated the parameters in place; advance their autograd version counters so
    that UNetProgram.params_changed() (engine.py) notices and re-packs the bf16 weight buffers."""
    inc = getattr(torch._C, "_increment_version", None)
    if inc is not None:
        try:
            inc(tensors)
            return
        except TypeError:
            for t in tensors:
                inc(t)
            return
    torch._foreach_add_(tensors, 0.0)


class Adam(torch.optim.Optimizer):
    """torch.optim.Adam's update in one launch.  With `ema=EMA(model)`, step() also updates that
    moving average: one more launch on the same stream, after every parameter update, skipped
    together with them when GradScaler found inf / nan gradients.  Do not call `ema.update()` as
    well: that would apply the average twice per step."""

    _step_supports_amp_scaling = True  # GradScaler hands over grad_scale / found_inf

    def __init__(self, params: Iterable, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0, ema: Optional["EMA"] = None):
        if lr < 0 or eps < 0 or not (0 <= betas[0] < 1) or not (0 <= betas[1] < 1) or weight_decay < 0:
            raise ValueError("invalid Adam hyper-parameters")
        super().__init__(params, dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay))
        if ema is not None:
            devs = {p.device for g in self.param_groups for p in g["params"]}
            if devs != {ema.device}:
                raise ValueError(f"Adam(ema=): the EMA tracks parameters on {ema.device}, the optimizer's "
                                 f"are on {sorted(str(d) for d in devs)}")
        self.ema = ema
        # grad_scale / found_inf are set (and deleted again) by torch.amp.GradScaler around step()
        self._tables = {}
        self._group_steps = {}

    def load_state_dict(self, state_dict):
        """Loaded moment tensors replace the ones the cached segment tables point at."""
        out = super().load_state_dict(state_dict)
        self._tables.clear()
        self._group_steps.clear()
        return out

    def add_param_group(self, param_group):
        out = super().add_param_group(param_group)
        if hasattr(self, "_tables"):
            self._tables.clear()
        return out

    def _group_step(self, gi: int, plist) -> torch.Tensor:
        """ONE device-resident step counter per param group (the kernel applies one bias
        correction per launch).  It starts from the LARGEST step any parameter of the group
        already has -- after load_state_dict, or when parameters that had no gradient before
        join -- never from whichever parameter happens to come first."""
        st = self._group_steps.get(gi)
        dev = plist[0].device
        if st is None:
            have = [self.state[p]["step"] for p in plist if "step" in self.state[p]]
            if have:
                st = torch.stack([h.detach().to(dev, torch.float32).reshape(()) for h in have]).max()
            else:
                st = torch.zeros((), dtype=torch.float32, device=dev)
            st = st.clone()
            self._group_steps[gi] = st
        return st

    def _table(self, gi: int, plist, grads):
        """Device segment table of one param group; rebuilt when a pointer changed (new .grad
        tensors appear after zero_grad(set_to_none=True))."""
        # the table bakes in all four pointers: parameter, gradient AND both moments
        key = tuple((p.data_ptr(), g.data_ptr(), self.state[p]["exp_avg"].data_ptr(),
                     self.state[p]["exp_avg_sq"].data_ptr()) for p, g in zip(plist, grads))
        hit = self._tables.get(gi)
        if hit is not None and hit[0] == key:
            return hit[1], hit[2], hit[3]
        segs, blocks = [], 0
        for p, g in zip(plist, grads):
            st = self.state[p]
            sg = _lib.MriAdamSeg()
            sg.p, sg.g = p.data_ptr(), g.data_ptr()
            sg.m, sg.v = st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr()
            sg.n, sg.block0 = p.numel(), blocks
            blocks += -(-p.numel() // 1024)
            segs.append(sg)
        arr = (_lib.MriAdamSeg * len(segs))(*segs)
        table = torch.frombuffer(bytearray(bytes(memoryview(arr))), dtype=torch.uint8).to(plist[0].device)
        self._tables[gi] = (key, table, len(segs), blocks)
        return table, len(segs), blocks

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _lib.load()
        for gi, group in enumerate(self.param_groups):
            plist, grads = [], []
            for p in group["params"]:
                if p.grad is None:
                    continue
                if not p.is_cuda or p.dtype != torch.float32 or p.grad.dtype != torch.float32:
                    raise _lib.MriError("mri Adam: fp32 CUDA parameters and gradients only (no fallback)")
                if p.grad.is_sparse or not p.is_contiguous() or not p.grad.is_contiguous():
                    raise _lib.MriError("mri Adam: dense contiguous parameters / gradients only")
                st = self.state[p]
                if len(st) == 0:
                    # device-resident step counter (as torch's fused Adam keeps it): it must not
                    # advance when GradScaler skips the update, and the host never syncs on that
                    st["step"] = torch.zeros((), dtype=torch.float32, device=p.device)
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                plist.append(p)
                grads.append(p.grad)
            if not plist:
                continue
            # one counter per group: every parameter's state["step"] aliases it
            step_t = self._group_step(gi, plist)
            for p in plist:
                self.state[p]["step"] = step_t
            table, n, blocks = self._table(gi, plist, grads)
            dev = plist[0].device
            gs, fi = getattr(self, "grad_scale", None), getattr(self, "found_inf", None)
            gs = gs.to(dev, torch.float32).reshape(-1) if gs is not None else None
            fi = fi.to(dev, torch.float32).reshape(-1) if fi is not None else None
            with torch.cuda.device(dev):
                rc = lib.mri_adam_step(table.data_ptr(), n, blocks, float(group["lr"]),
                                       float(group["betas"][0]), float(group["betas"][1]),
                                       float(group["eps"]), float(group["weight_decay"]),
                                       step_t.data_ptr(),
                                       gs.data_ptr() if gs is not None else None,
                                       fi.data_ptr() if fi is not None else None,
                                       torch.cuda.current_stream(dev).cuda_stream)
            _lib.check(rc, "mri_adam_step")
            _bump_versions(plist)  # parameters changed behind autograd's back: packed buffers re-gather
        if self.ema is not None:
            # the same found_inf as the parameter update: a skipped step leaves the average alone
            self.ema._launch(getattr(self, "found_inf", None))
        return loss


def ema_decay(k: int, decay: float, warmup: bool) -> float:
    """Decay d of the k-th EMA update (k >= 1), the rule ema_update_kernel evaluates in fp64:
    `decay`, or with warm-up 0 for k = 1 and min(decay, k / (9 + k)) after (diffusers' EMAModel with
    update_after_step = 0).  The shadow moves by e <- lerp(e, p, float32(1 - d))."""
    if not warmup:
        return decay
    return 0.0 if k <= 1 else min(decay, k / (9.0 + k))


def ema_segments(shadow, live, device):
    """Device table of mri_ema_update over the pairs (shadow[i] <- live[i]): (table, n_segs, blocks)."""
    segs, blocks = [], 0
    for e, p in zip(shadow, live):
        if (p.device != device or e.device != device or p.dtype != torch.float32 or e.dtype != torch.float32
                or p.shape != e.shape or not p.is_contiguous() or not e.is_contiguous()):
            raise _lib.MriError(f"mri EMA: contiguous fp32 tensors of equal shape on {device} only "
                                "(no fallback)")
        sg = _lib.MriEmaSeg()
        sg.e, sg.p, sg.n, sg.block0 = e.data_ptr(), p.data_ptr(), p.numel(), blocks
        blocks += -(-p.numel() // 1024)
        segs.append(sg)
    arr = (_lib.MriEmaSeg * len(segs))(*segs)
    table = torch.frombuffer(bytearray(bytes(memoryview(arr))), dtype=torch.uint8).to(device)
    return table, len(segs), blocks


class EMA:
    """Exponential moving average of a model's weights: e <- d * e + (1 - d) * p after every optimizer
    step, with d from `ema_decay`.  Bit-identical to torch.optim.swa_utils.AveragedModel(model,
    multi_avg_fn=get_ema_multi_avg_fn(decay)) after its first update_parameters call (which copies),
    without its two host synchronisations per update.

    `ema.module` is a deep copy of the model (unwrapped from either DistributedDataParallel) with
    `requires_grad` off: a complete drop-in UNet / VAE3D to pass to GaussianDiffusion* or sample
    from, in either precision, on programs of its own.  Its state_dict() has the live model's keys,
    so it saves as an ordinary model checkpoint.

    Call `update()` after each optimizer step, or pass the EMA to `Adam(..., ema=)`, which updates it
    inside step() and skips it on GradScaler's skipped steps -- not both.  Every parameter moves,
    including ones that had no gradient this step (toward their unchanged value).  The update
    counter lives on the device; from the second update on nothing synchronises with the host."""

    def __init__(self, model: torch.nn.Module, decay: float = 0.9999, warmup: bool = False):
        decay = float(decay)
        if not 0.0 <= decay < 1.0:  # NaN fails too
            raise ValueError(f"EMA decay must lie in [0, 1), got {decay}")
        from . import parallel
        if isinstance(model, (torch.nn.parallel.DistributedDataParallel, parallel.DistributedDataParallel)):
            model = model.module
        params = list(model.parameters())
        if not params:
            raise ValueError("EMA: the model has no parameters")
        dev = params[0].device
        for p in params:
            if not p.is_cuda or p.device != dev or p.dtype != torch.float32 or not p.is_contiguous():
                raise _lib.MriError("mri EMA: contiguous fp32 CUDA parameters on one device only "
                                    f"(no fallback), got {p.dtype} on {p.device}")
        self.decay, self.warmup = decay, bool(warmup)
        self._model = model
        self.module = copy.deepcopy(model)
        for p in self.module.parameters():
            p.requires_grad_(False)
        self.num_updates = torch.zeros((), dtype=torch.int64, device=dev)
        self._cached = None

    @property
    def device(self) -> torch.device:
        return self.num_updates.device

    def _table(self, shadow, live):
        """The segment table, rebuilt when a pointer changed (the live model was moved, or loaded
        with assign=True)."""
        key = tuple((e.data_ptr(), p.data_ptr()) for e, p in zip(shadow, live))
        if self._cached is None or self._cached[0] != key:
            if len(shadow) != len(live):
                raise _lib.MriError(f"mri EMA: the model has {len(live)} parameters, its average {len(shadow)}")
            self._cached = (key,) + ema_segments(shadow, live, self.device)
        return self._cached[1:]

    @torch.no_grad()
    def _launch(self, found_inf) -> None:
        shadow, live = list(self.module.parameters()), list(self._model.parameters())
        table, n, blocks = self._table(shadow, live)
        if found_inf is not None:
            found_inf = found_inf.to(self.device, torch.float32).reshape(-1)
        with torch.cuda.device(self.device):
            rc = _lib.load().mri_ema_update(table.data_ptr(), n, blocks, self.decay, int(self.warmup),
                                            self.num_updates.data_ptr(),
                                            found_inf.data_ptr() if found_inf is not None else None,
                                            torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(rc, "mri_ema_update")
        # the shadow's packed bf16 weights re-gather the next time it runs, not now
        _bump_versions(shadow)

    def update(self) -> None:
        """Move the average one step toward the model's current weights (one launch)."""
        self._launch(None)

    def state_dict(self) -> dict:
        return {"decay": self.decay, "warmup": self.warmup, "num_updates": self.num_updates.clone(),
                "module": self.module.state_dict()}

    def load_state_dict(self, state_dict: dict) -> None:
        decay = float(state_dict["decay"])
        if not 0.0 <= decay < 1.0:
            raise ValueError(f"EMA decay must lie in [0, 1), got {decay}")
        self.module.load_state_dict(state_dict["module"])
        self.decay, self.warmup = decay, bool(state_dict["warmup"])
        self.num_updates.copy_(torch.as_tensor(state_dict["num_updates"]).reshape(()))
        self._cached = None
