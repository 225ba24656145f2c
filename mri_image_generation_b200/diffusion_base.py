"""Shared implementation of the diffusion wrappers (q_sample / p_sample / loops) on the C ABI.

The three public classes (model_scripts/*/diffusion.py) differ only in schedule, the extra
model arguments (z_pos, context) and the loss; everything that touches the GPU is here:
  - q_sample / p_sample / DDIM arithmetic: one fused fp32 kernel each (mri_q_sample,
    mri_ddpm_step, mri_ddim_step), bit-exact w.r.t. the reference's eager association order;
    DPM-Solver++(2M) (not in the reference): mri_dpmpp_step over a host-built coefficient table;
    inpainting (not in the reference): mri_inpaint_merge after each update of either sampler;
    undersampled k-space reconstruction (not in the reference): mri_kspace_merge in the same slot;
    RePaint's resampling (not in the reference): mri_repaint_undo between the inpainting steps;
    measurement-guided sampling of the 3D LDM (not in the reference): mri_guided_x0, the VAE
    decoder forward, mri_dc_project3d / mri_dc_mask, the decoder's input gradient and
    mri_guided_eps before each unfused update;
    the variational bound in bits per dimension (not in the reference): mri_vb_terms after each
    evaluation step, on a step graph of its own;
  - the reverse loop: when the denoiser is one of this package's UNets, one CUDA graph holds a
    whole reverse step (time embedding, UNet, fused update with the noise drawn INSIDE the
    kernel, t -= 1) and is replayed T times.  The kernels draw Philox4x32-10 + Box-Muller
    normals with ATen's (seed, subsequence, offset) mapping (csrc/diffusion_ops.cu), seeded from
    torch's CUDA generator, and the host advances that generator by what the draws consumed: for
    a given torch.manual_seed the noise is bit-identical to what `torch.randn_like` would have
    produced at the reference's call sites, and no ATen kernel runs inside a replayed step.
"""
from __future__ import annotations

import math
import os
import weakref
from typing import Callable, Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib, ops, schedules
from .modules import EngineModule


def _require_cuda(x: torch.Tensor, what: str) -> None:
    if not x.is_cuda:
        raise _lib.MriError(f"{what}: tensors must live on a B200 GPU (got {x.device}); "
                            "this framework has no CPU fallback")


def kspace_completion(y: torch.Tensor, m: torch.Tensor,
                      dims: Tuple[int, ...] = (-2, -1)) -> Tuple[torch.Tensor, torch.Tensor]:
    """Hermitian completion of a measured k-space, on y's device: (x_zf, M) with M = m | m(-k),
    y(k) = conj(y(-k)) where k is measured only at its mirror, and x_zf = Re ifftn(M y) over `dims`
    in fp64 (orthonormal, unshifted).  y: complex (..., H, W), or (..., D, H, W) with
    dims = (-3, -2, -1); m: bool of y's shape.  Values of y outside m are never read."""
    mir = lambda a: torch.roll(torch.flip(a, dims), (1,) * len(dims), dims)   # a(-k)
    full = m | mir(m)
    y = y.to(torch.complex128)
    y = torch.where(m, y, torch.where(full, mir(y).conj(), torch.zeros_like(y)))
    return torch.fft.ifftn(y, dim=dims, norm="ortho").real, full


class _LossFn(torch.autograd.Function):
    """min-SNR / plain MSE loss with its gradient kernel (ddpm_3d_ldm/diffusion.py:91-99)."""

    @staticmethod
    def forward(ctx, pred, noise, t, snr, gamma):
        B = pred.shape[0]
        per = torch.empty(B, dtype=torch.float32, device=pred.device)
        loss = torch.empty(1, dtype=torch.float32, device=pred.device)
        ops.minsnr_loss(pred, noise, t, snr, gamma, per, loss)
        ctx.save_for_backward(pred, noise, t, snr)
        ctx.gamma = gamma
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        pred, noise, t, snr = ctx.saved_tensors
        dpred = torch.empty_like(pred)
        ops.minsnr_loss_bwd(pred, noise, t, snr, ctx.gamma, g.reshape(1).float().contiguous(), dpred)
        return dpred, None, None, None, None


class DiffusionBase(nn.Module):
    """Host logic common to GaussianDiffusion (2D, 2.5D) and GaussianDiffusionLatent3D."""

    model: nn.Module
    timesteps: int

    # ------------------------------------------------------------------ device-side generator state
    def _rng(self, dev) -> ops.DeviceRng:
        rngs = self.__dict__.setdefault("_mri_rng", {})
        key = torch.device(dev)
        if key not in rngs:
            rngs[key] = ops.DeviceRng(key)
        return rngs[key]

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop("_mri_rng", None)
        return state

    def _apply(self, fn, *args, **kwargs):
        self.__dict__.pop("_mri_rng", None)
        return super()._apply(fn, *args, **kwargs)

    def _randn(self, shape, device) -> torch.Tensor:
        """torch.randn(shape, device=device) drawn by mri_randn (bit-identical, generator advanced)."""
        out = torch.empty(shape, dtype=torch.float32, device=device)
        _require_cuda(out, "sample")
        if out.numel() == 0:
            return out
        with torch.cuda.device(out.device):
            rng = self._rng(out.device)
            off = rng.load()
            ops.randn(out, rng)
            rng.commit(off + ops.randn_offset_increment(out.numel()))
        return out

    # ------------------------------------------------------------------ fused arithmetic
    def _q_sample(self, x_start, t, noise):
        _require_cuda(x_start, "q_sample")
        x0 = x_start.float().contiguous()
        out = torch.empty_like(x0)
        with torch.cuda.device(x0.device):
            ops.q_sample(x0, noise.float().contiguous(), t.to(x0.device).long().contiguous(),
                         self.sqrt_alphas_cumprod, self.sqrt_one_minus_alphas_cumprod, out)
        return out

    def _q_sample_draw(self, x_start, t) -> Tuple[torch.Tensor, torch.Tensor]:
        """q_sample with `noise = torch.randn_like(x_start)` drawn inside the kernel
        (ddpm_3d_ldm/diffusion.py:75-82): returns (x_t, noise)."""
        _require_cuda(x_start, "q_sample")
        x0 = x_start.float().contiguous()
        out, noise = torch.empty_like(x0), torch.empty_like(x0)
        with torch.cuda.device(x0.device):
            rng = self._rng(x0.device)
            off = rng.load()
            ops.q_sample_rng(x0, rng, t.to(x0.device).long().contiguous(), self.sqrt_alphas_cumprod,
                             self.sqrt_one_minus_alphas_cumprod, out, noise)
            rng.commit(off + ops.randn_offset_increment(x0.numel()))
        return out, noise

    def _p_update(self, x, t, eps, noise=None):
        """x_{t-1} from (x_t, eps, z): ddpm_3d_ldm/diffusion.py:118-126.  noise=None: z =
        randn_like(x) is drawn inside the kernel."""
        _require_cuda(x, "p_sample")
        xc = x.float().contiguous()
        out = torch.empty_like(xc)
        tl = t.to(xc.device).long().contiguous()
        with torch.cuda.device(xc.device):
            if noise is None:
                rng = self._rng(xc.device)
                off = rng.load()
                ops.ddpm_step_rng(xc, eps.float().contiguous(), rng, tl, self.betas,
                                  self.sqrt_one_minus_alphas_cumprod, self.sqrt_recip_alphas,
                                  self.posterior_variance, out)
                rng.commit(off + ops.randn_offset_increment(xc.numel()))
            else:
                ops.ddpm_step(xc, eps.float().contiguous(), noise.float().contiguous(), tl, self.betas,
                              self.sqrt_one_minus_alphas_cumprod, self.sqrt_recip_alphas,
                              self.posterior_variance, out)
        return out

    def _ddim_update(self, x, t, t_prev, eps):
        _require_cuda(x, "p_sample_ddim")
        xc = x.float().contiguous()
        out = torch.empty_like(xc)
        with torch.cuda.device(xc.device):
            ops.ddim_step(xc, eps.float().contiguous(), t.to(xc.device).long().contiguous(),
                          t_prev.to(xc.device).long().contiguous(), self.alphas_cumprod, out)
        return out

    def _loss(self, pred, noise, t, gamma: float):
        """min-SNR weighted (gamma > 0) or plain (gamma <= 0) MSE, fused reduce."""
        _require_cuda(pred, "p_losses")
        snr = getattr(self, "snr", None)
        if gamma > 0 and snr is None:
            raise _lib.MriError("min-SNR loss needs the `snr` buffer")
        with torch.cuda.device(pred.device):
            return _LossFn.apply(pred.float().contiguous(), noise.float().contiguous(),
                                 t.to(pred.device).long().contiguous(),
                                 snr if snr is not None else self.betas, float(gamma))

    # ------------------------------------------------------------------ DPM-Solver++(2M)
    def _dpmpp_table(self, start_t, num_steps) -> Tuple[torch.Tensor, torch.Tensor]:
        """(ts, coef) of schedules.dpmpp_2m_table for num_steps UNet calls from start_t to sigma = 0."""
        T, s, M = self.timesteps, int(start_t), int(num_steps)
        if not 1 <= M <= s <= T - 1:
            raise ValueError(f"DPM-Solver++ needs 1 <= num_steps <= start_t <= {T - 1} "
                             f"(got num_steps={M}, start_t={s})")
        return schedules.dpmpp_2m_table(self.alphas_cumprod, schedules.dpmpp_timesteps(s, M))

    def _sample_dpmpp(self, img, table, prog, eps_fn: Callable, inpaint=None,
                      kspace: bool = False) -> torch.Tensor:
        """Run the solver over `table` from x = img.  prog: a UNetProgram whose conditioning inputs
        the caller has set (replayed step graph), or None: eager, eps = eps_fn(x, t) per step.
        inpaint: (known, mask) of _inpaint_inputs; after row i the kept region is replaced by
        q_sample(known, ts[i + 1], noise=img), and by known itself after the last row.  With
        kspace, (x_zf, mask) of _kspace_inputs, and the merge is the k-space one (_merge).
        Returns the fp32 x0 estimate."""
        _require_cuda(img, "sample_dpmpp")
        ts, coef = table
        if prog is not None:
            return self._reverse_loop(prog, img.float(), int(ts[0]), ts.numel(), "dpmpp", table=table,
                                      inpaint=inpaint, kspace=kspace)
        dev = img.device
        with torch.cuda.device(dev):
            coef = coef.to(dev)
            x = img.float().contiguous().clone()
            x_T = x.clone() if inpaint is not None else None
            x0_prev = torch.empty_like(x)
            tau = ts.tolist()[1:] + [-1]
            for i, t in enumerate(ts.tolist()):
                tt = torch.full((x.shape[0],), t, device=dev, dtype=torch.long)
                eps = eps_fn(x, tt)
                ops.dpmpp_step(x, eps.float().contiguous(), x0_prev, coef[i], None, x)
                if inpaint is not None:
                    tt.fill_(tau[i])
                    self._merge(x, inpaint, tt, 0, kspace, noise=x_T)
        return x

    # ------------------------------------------------------------------ inpainting
    def _inpaint_inputs(self, x_known, mask, rank: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """Check (x_known, mask) and return them as the kernel reads them: x_known fp32, mask one
        uint8 per element (1 = regenerate, 0 = keep), both contiguous on x_known's device.  Raises
        ValueError on a bad shape or mask; callers check before anything is drawn."""
        if not torch.is_tensor(x_known) or x_known.dim() != rank or x_known.shape[1] != self.channels:
            raise ValueError(f"x_known must be a (B, {self.channels}, ...) tensor of rank {rank} "
                             f"(got {tuple(x_known.shape) if torch.is_tensor(x_known) else type(x_known)})")
        if x_known.numel() == 0:
            raise ValueError("x_known is empty")
        mask = torch.as_tensor(mask)
        try:
            ok = torch.broadcast_shapes(mask.shape, x_known.shape) == x_known.shape
        except RuntimeError:
            ok = False
        if not ok:
            raise ValueError(f"mask of shape {tuple(mask.shape)} does not broadcast to x_known's "
                             f"{tuple(x_known.shape)}")
        if mask.dtype != torch.bool and not bool(((mask == 0) | (mask == 1)).all()):
            raise ValueError("mask must be bool or hold only 0 / 1 (1 = regenerate, 0 = keep)")
        known = x_known.float().contiguous()
        m = torch.empty(known.shape, dtype=torch.uint8, device=known.device)
        m.copy_(mask.to(known.device).expand(known.shape))
        return known, m

    def _inpaint_buffers(self, prog, with_noise: bool, kspace: bool = False) -> Dict[str, torch.Tensor]:
        """The program's inpainting inputs: known, mask and, for DPM-Solver++, the x_T copy the
        known region is noised with.  Each call copies into them, so one captured graph serves
        every x_known and mask.  The k-space merge reads x_zf and its mask from the same buffers
        and adds a work buffer of its own (mri_kspace_work_bytes)."""
        bufs = prog.__dict__.setdefault("_inpaint_bufs", {})
        if "known" not in bufs:
            bufs["known"] = torch.zeros_like(prog.x_in)
            bufs["mask"] = torch.zeros(prog.x_in.shape, dtype=torch.uint8, device=prog.x_in.device)
        if with_noise and "noise" not in bufs:
            bufs["noise"] = torch.zeros_like(prog.x_in)
        if kspace and "work" not in bufs:
            bufs["work"] = torch.zeros(ops.kspace_work_bytes(*prog.x_in.shape), dtype=torch.uint8,
                                       device=prog.x_in.device)
        return bufs

    def _merge(self, x, cond, t, t_delta: int, kspace: bool, work=None, **z) -> None:
        """The merge after a reverse update, in place on x: mri_inpaint_merge with cond = (known,
        mask), or with kspace mri_kspace_merge with cond = (x_zf, mask) and its work buffer (None:
        allocated per call).  z: noise= or rng= / rng_skip= as the ops take them."""
        if kspace:
            ops.kspace_merge(x, cond[0], cond[1], t, t_delta, self.sqrt_alphas_cumprod,
                             self.sqrt_one_minus_alphas_cumprod, work=work, **z)
        else:
            ops.inpaint_merge(x, cond[0], cond[1], t, t_delta, self.sqrt_alphas_cumprod,
                              self.sqrt_one_minus_alphas_cumprod, **z)

    # ------------------------------------------------------------------ k-space reconstruction
    def _kspace_inputs(self, kspace, kmask) -> Tuple[torch.Tensor, torch.Tensor]:
        """Check (kspace, kmask) and complete them once per call: M = m | m(-k), y(k) = conj(y(-k))
        where k is measured only at its mirror, x_zf = Re ifft2(M y) (orthonormal, in fp64).
        Returns (x_zf fp32, M as one uint8 per element) on the model's device, as mri_kspace_merge
        reads them.  ValueError on a bad kspace or mask, MriError on a CPU tensor or H, W over the
        kernel's limit; callers check before anything is drawn."""
        if not torch.is_tensor(kspace) or not kspace.is_complex() or kspace.dim() != 4 \
                or kspace.shape[1] != self.channels:
            got = (tuple(kspace.shape), kspace.dtype) if torch.is_tensor(kspace) else type(kspace)
            raise ValueError(f"kspace must be a complex (B, {self.channels}, H, W) tensor (got {got})")
        if kspace.numel() == 0:
            raise ValueError("kspace is empty")
        mask = torch.as_tensor(kmask)
        try:
            ok = torch.broadcast_shapes(mask.shape, kspace.shape) == kspace.shape
        except RuntimeError:
            ok = False
        if not ok:
            raise ValueError(f"kmask of shape {tuple(mask.shape)} does not broadcast to kspace's "
                             f"{tuple(kspace.shape)}")
        if mask.dtype != torch.bool and not bool(((mask == 0) | (mask == 1)).all()):
            raise ValueError("kmask must be bool or hold only 0 / 1 (1 = measured)")
        _require_cuda(kspace, "reconstruct")
        ops.kspace_work_bytes(*kspace.shape)      # MriError when H or W is over the kernel's limit
        dev = self.betas.device
        with torch.cuda.device(dev):
            x_zf, full = kspace_completion(kspace.to(dev), mask.to(dev).expand(kspace.shape).bool())
            return x_zf.float().contiguous(), full.to(torch.uint8).contiguous()

    def _repaint_levels(self, jump_length, jump_n_sample) -> Optional[list]:
        """schedules.repaint_levels for this schedule (ValueError on bad arguments), or None when
        it has no undo step (jump_n_sample = 1 or jump_length >= T): plain replacement."""
        levels = schedules.repaint_levels(self.timesteps, jump_length, jump_n_sample)
        return levels if len(levels) > self.timesteps + 1 else None

    def _inpaint_ddpm(self, img, inpaint, prog, eps_fn: Callable, levels=None,
                      kspace: bool = False) -> torch.Tensor:
        """Ancestral sampling from x_T = img over every timestep with the kept region replaced after
        each update by q_sample(known, i - 1, noise=randn_like(x)) (known itself after i = 0).
        prog / eps_fn / kspace as for _sample_dpmpp.  levels: RePaint's resampling
        (_inpaint_repaint; not with kspace)."""
        _require_cuda(img, "inpaint")
        if levels is not None:
            return self._inpaint_repaint(img, inpaint, prog, eps_fn, levels)
        T = self.timesteps
        if prog is not None:
            return self._reverse_loop(prog, img.float(), T - 1, T, "ddpm", inpaint=inpaint,
                                      kspace=kspace)
        dev = img.device
        x = img.float().contiguous()
        with torch.cuda.device(dev):
            rng = self._rng(dev)
            inc = ops.randn_offset_increment(x.numel())
            for i in reversed(range(T)):
                x = self._inpaint_step(x, i, inpaint, eps_fn, rng, inc, kspace)
        return x

    def _inpaint_step(self, x, i, inpaint, eps_fn, rng, inc, kspace: bool = False) -> torch.Tensor:
        """One eager DDPM inpainting step at t = i: update, then the kept region becomes
        q_sample(known, i - 1, noise=randn_like(x)) (known itself at i = 0); with kspace the
        k-space merge with the same z."""
        t = torch.full((x.shape[0],), i, device=x.device, dtype=torch.long)
        x = self._p_update(x, t, eps_fn(x, t))
        off = rng.load()
        self._merge(x, inpaint, t, -1, kspace, rng=rng)
        rng.commit(off + inc)
        return x

    def _inpaint_repaint(self, img, inpaint, prog, eps_fn: Callable, levels) -> torch.Tensor:
        """RePaint: _inpaint_ddpm's steps walked along `levels` (schedules.repaint_levels).  A move
        l -> l - 1 is the inpainting step at t = l; a move l -> l + 1 re-noises the merged state by
        one step, x = sqrt(alphas[l + 1]) x + sqrt(betas[l + 1]) z with z = randn_like(x), so that
        the next steps reconcile the regenerated region with the kept one.  The generator advances
        by (1 + 2 n_reverse + n_undo) draws, x_T included."""
        n_reverse = sum(1 for a, b in zip(levels, levels[1:]) if b < a)
        if prog is not None:
            return self._reverse_loop(prog, img.float(), levels[0], n_reverse, "ddpm",
                                      inpaint=inpaint, levels=levels)
        dev = img.device
        x = img.float().contiguous()
        with torch.cuda.device(dev):
            rng = self._rng(dev)
            inc = ops.randn_offset_increment(x.numel())
            for lv, nxt in zip(levels, levels[1:]):
                if nxt < lv:
                    x = self._inpaint_step(x, lv, inpaint, eps_fn, rng, inc)
                    continue
                t = torch.full((x.shape[0],), lv, device=dev, dtype=torch.long)
                off = rng.load()
                ops.repaint_undo(x, t, self.alphas, self.betas, rng=rng)
                rng.commit(off + inc)
        return x

    def _dpmpp_buffers(self, prog, rows: int) -> Dict[str, torch.Tensor]:
        """The program's solver state: table (>= T rows, so that one captured graph serves every
        num_steps and start_t), row index k and x0_prev."""
        bufs = prog.__dict__.get("_dpmpp_bufs")
        if bufs is None or bufs["ts"].numel() < rows:
            dev, n = prog.x_in.device, max(rows, self.timesteps)
            bufs = dict(coef=torch.zeros(n, 5, dtype=torch.float32, device=dev),
                        ts=torch.zeros(n, dtype=torch.int64, device=dev),
                        k=torch.zeros(1, dtype=torch.int64, device=dev),
                        x0_prev=torch.zeros_like(prog.x_in))
            prog.__dict__["_dpmpp_bufs"] = bufs
            graphs = prog.__dict__.get("_step_graphs", {})
            for key in [k for k in graphs if k.startswith("dpmpp")]:   # captured on the old buffers
                graphs.pop(key)
        return bufs

    # ------------------------------------------------------------------ measurement-guided sampling
    def _guided_buffers(self, owner, dec, kspace: bool) -> Dict[str, torch.Tensor]:
        """The guided step's state on `owner` (the UNet program, or a dict for the eager loop): the
        data-gradient-only decoder program `dec` and the buffers the step reads through device
        pointers -- zf (x_zf, or x_known for the image mask), mask, lam and inv_s (copied into on
        every call, so one captured graph serves every measurement), gg, the data term's work and
        eps (the guided eps, fp32 in the latent's layout).  A new decoder program drops the guided
        graphs captured on the old one."""
        d = owner if isinstance(owner, dict) else owner.__dict__
        bufs = d.setdefault("_guided_bufs", {})
        if bufs.get("dec") is not dec:
            bufs.clear()
            graphs = d.get("_step_graphs", {})
            for key in [k for k in graphs if "+guided" in k]:
                graphs.pop(key)
            dev, B = dec.device, dec.B
            img = dec.out
            bufs.update(dec=dec, zf=torch.zeros_like(img), mask=torch.zeros(img.shape, dtype=torch.uint8, device=dev),
                        gg=torch.zeros(B, dtype=torch.float32, device=dev),
                        lam=torch.zeros(1, dtype=torch.float32, device=dev),
                        inv_s=torch.ones(1, dtype=torch.float32, device=dev),
                        eps=torch.zeros_like(dec.x_in))
        key = "work_k" if kspace else "work_m"
        if key not in bufs:
            img = dec.out
            n = ops.kspace3d_work_bytes(*img.shape) if kspace else img.shape[0] * ops.DC_MASK_WORK_PER_SAMPLE
            bufs[key] = torch.zeros(n, dtype=torch.uint8, device=img.device)
        bufs["work"], bufs["kspace"] = bufs[key], kspace
        return bufs

    def _guided_stage(self, z, eps, ldc: int, C: int, t, b) -> None:
        """Steps 2-7 of the guided step (DESIGN.md §4) up to the guided eps, written to b['eps']:
        x0 / s into the decoder's input, u = D(x0 / s), g and ||g||^2 of the data term into the
        decoder's output gradient, dz = D^T g, then eps' = eps - (sac / s1m) * delta."""
        dec = b["dec"]
        sa, s1m = self.sqrt_alphas_cumprod, self.sqrt_one_minus_alphas_cumprod
        ops.guided_x0(z, eps, t, sa, s1m, b["inv_s"], dec.x_in, eps_nhwc_ldc=ldc, channels=C)
        dec.run()
        dec.finish_output()
        if b["kspace"]:
            ops.dc_project3d(dec.out, b["zf"], b["mask"], dec.dout_in, b["gg"], b["work"])
        else:
            ops.dc_mask(dec.out, b["zf"], b["mask"], dec.dout_in, b["gg"], b["work"])
        dec.run_input_backward()
        ops.guided_eps(eps, dec.dz_out, b["gg"], b["lam"], b["inv_s"], t, sa, s1m, b["eps"],
                       eps_nhwc_ldc=ldc, channels=C)

    def _guided_sample(self, img, table, prog, eps_fn: Callable, dec, data, kspace: bool,
                       lam: float, inv_s: float) -> torch.Tensor:
        """Measurement-guided sampling from the latent x_T = img: DDPM over every timestep (table
        None) or DPM-Solver++ over `table`, with the guided eps of _guided_stage in every update.
        data: (zf, mask) on the image grid; dec: the VAE's data-gradient-only decoder program.
        prog: the UNet program (step graphs 'ddpm+guided:kspace' etc.) or None: eager with
        eps = eps_fn(x, t).  Draws what sample() / sample_dpmpp() draw.  Returns the latent z_0."""
        _require_cuda(img, "guided sampling")
        if dec.params_changed():
            dec.do_refresh()
        b = self._guided_buffers(prog if prog is not None else self.__dict__.setdefault("_guided_eager", {}),
                                 dec, kspace)
        b["zf"].copy_(data[0])
        b["mask"].copy_(data[1])
        b["lam"].fill_(lam)
        b["inv_s"].fill_(inv_s)
        mode = "ddpm" if table is None else "dpmpp"
        T = self.timesteps
        if prog is not None:
            if table is None:
                return self._reverse_loop(prog, img.float(), T - 1, T, mode, guided=b)
            return self._reverse_loop(prog, img.float(), int(table[0][0]), table[0].numel(), mode,
                                      table=table, guided=b)
        dev = img.device
        x = img.float().contiguous().clone()
        with torch.cuda.device(dev):
            if table is None:
                for i in reversed(range(T)):
                    t = torch.full((x.shape[0],), i, device=dev, dtype=torch.long)
                    eps = eps_fn(x, t).float().contiguous()
                    self._guided_stage(x, eps, 0, 0, t, b)
                    x = self._p_update(x, t, b["eps"])
                return x
            ts, coef = table
            coef = coef.to(dev)
            x0_prev = torch.empty_like(x)
            for i, t in enumerate(ts.tolist()):
                tt = torch.full((x.shape[0],), t, device=dev, dtype=torch.long)
                eps = eps_fn(x, tt).float().contiguous()
                self._guided_stage(x, eps, 0, 0, tt, b)
                ops.dpmpp_step(x, b["eps"], x0_prev, coef[i], None, x)
        return x

    # ------------------------------------------------------------------ variational bound
    def _vb_input(self, x_start, rank: int) -> torch.Tensor:
        """x_start as the kernels read it (fp32, contiguous).  ValueError on a bad shape, MriError
        on a CPU tensor; callers check before anything is drawn."""
        if not torch.is_tensor(x_start) or x_start.dim() != rank or x_start.shape[1] != self.channels:
            raise ValueError(f"x_start must be a (B, {self.channels}, ...) tensor of rank {rank} "
                             f"(got {tuple(x_start.shape) if torch.is_tensor(x_start) else type(x_start)})")
        if x_start.numel() == 0:
            raise ValueError("x_start is empty")
        _require_cuda(x_start, "calc_bpd_loop")
        return x_start.float().contiguous()

    def _vb_buffers(self, prog) -> Dict[str, torch.Tensor]:
        """The program's evaluation inputs and sums: x0 (copied into on every call, so one captured
        graph serves every x_start), z, acc (B, T, 2) and prior (B,) in fp64."""
        bufs = prog.__dict__.setdefault("_vb_bufs", {})
        T = self.timesteps
        if "acc" not in bufs or bufs["acc"].shape[1] != T:
            B, dev = prog.x_in.shape[0], prog.x_in.device
            bufs.update(x0=torch.zeros_like(prog.x_in), z=torch.zeros_like(prog.x_in),
                        acc=torch.zeros(B, T, 2, dtype=torch.float64, device=dev),
                        prior=torch.zeros(B, dtype=torch.float64, device=dev))
            prog.__dict__.get("_step_graphs", {}).pop("vb", None)   # captured on the old buffers
        return bufs

    def _vb_loop(self, prog, x0: torch.Tensor, eps_fn: Callable, decoder: int) -> Dict[str, torch.Tensor]:
        """The variational bound on -log p(x0) in bits per dimension (improved-diffusion's
        calc_bpd_loop for the fixed-small-variance model).  For t = T - 1 ... 0: z = randn_like(x0),
        x_t = q_sample(x0, t, z), eps = model(x_t, t), then mri_vb_terms.  prog: a UNetProgram whose
        conditioning inputs the caller has set (one step graph 'vb' replayed T times), or None: the
        same sequence eagerly with eps = eps_fn(x_t, t).  The generator advances by T draws."""
        B, T, N = x0.shape[0], self.timesteps, x0[0].numel()
        dev = x0.device
        sched = (self.betas, self.sqrt_one_minus_alphas_cumprod, self.sqrt_recip_alphas,
                 self.posterior_variance, self.posterior_log_variance_clipped)
        with torch.cuda.device(dev):
            rng = self._rng(dev)
            inc = ops.randn_offset_increment(x0.numel())
            if prog is None:
                acc = torch.zeros(B, T, 2, dtype=torch.float64, device=dev)
                prior = torch.zeros(B, dtype=torch.float64, device=dev)
                for i in reversed(range(T)):
                    t = torch.full((B,), i, device=dev, dtype=torch.long)
                    x_t, z = self._q_sample_draw(x0, t)
                    ops.vb_terms(x0, x_t, eps_fn(x_t, t).float().contiguous(), z, t, *sched, acc, prior,
                                 decoder)
            else:
                if prog.params_changed():
                    prog.do_refresh()
                bufs = self._vb_buffers(prog)
                tprev = prog.__dict__.setdefault("_tprev_buf", torch.zeros(B, dtype=torch.int64, device=dev))

                def one_step():
                    ops.q_sample_rng(bufs["x0"], rng, prog.t_in, self.sqrt_alphas_cumprod,
                                     self.sqrt_one_minus_alphas_cumprod, prog.x_in, bufs["z"])
                    prog.run()
                    ops.vb_terms(bufs["x0"], prog.x_in, prog.eps_nhwc, bufs["z"], prog.t_in, *sched,
                                 bufs["acc"], bufs["prior"], decoder, eps_nhwc_ldc=prog.cout_pad,
                                 channels=prog.cout)
                    ops.step_advance(prog.t_in, -1, rng=rng, rng_increment=inc)

                graph = self._step_graph(prog, "vb", one_step, tprev)
                acc, prior = bufs["acc"], bufs["prior"]
                bufs["x0"].copy_(x0)
                acc.zero_()      # after the capture: its warm-up launch accumulated at t = 1
                prior.zero_()
                prog.t_in.fill_(T - 1)
                off = rng.load()
                for _ in range(T):
                    graph.replay()
                rng.commit(off + T * inc)
            c = schedules.vb_constants(self.betas)
            lam = c["lam"].to(dev)
            nats = acc[:, :, 0] * lam
            nats[:, 0] = acc[:, 0, 1]
            prior_nats = 0.5 * (N * c["prior_const"] + c["prior_coef"] * prior)
            scale = 1.0 / (N * math.log(2.0))
            return {"total_bpd": (prior_nats + nats.sum(1)) * scale, "prior_bpd": prior_nats * scale,
                    "vb": nats * scale, "mse": acc[:, :, 0] / N}

    # ------------------------------------------------------------------ graph-replayed loops
    def _engine_model(self) -> Optional[EngineModule]:
        m = self.model
        inner = getattr(m, "module", None)  # DataParallel / DDP wrappers
        if isinstance(inner, EngineModule):
            m = inner
        return m if isinstance(m, EngineModule) else None

    def _schedule_ptrs(self) -> Tuple[int, ...]:
        return tuple(getattr(self, n).data_ptr() for n in
                     ("betas", "sqrt_one_minus_alphas_cumprod", "sqrt_recip_alphas",
                      "posterior_variance", "alphas_cumprod", "sqrt_alphas_cumprod", "alphas",
                      "posterior_log_variance_clipped"))

    def _step_graph(self, prog, mode: str, one_step, tprev):
        """The CUDA graph of one reverse step on `prog`.  The graph lives ON the program (it
        replays launches into the program's buffers, so it must die with it: evicted or dropped
        programs take their graphs along) and remembers which diffusion object and which schedule
        buffers it was captured for; anything else re-captures."""
        dev = prog.x_in.device
        graphs = prog.__dict__.setdefault("_step_graphs", {})
        hit = graphs.get(mode)
        ptrs = self._schedule_ptrs()
        if hit is not None and hit[0]() is self and hit[1] == ptrs:
            return hit[2]
        prog.x_in.zero_()
        prog.t_in.fill_(1)
        tprev.fill_(0)
        self._rng(dev).load()           # a valid (seed, offset) for the warm-up / capture launches
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            one_step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        prog.t_in.fill_(1)
        with torch.cuda.graph(graph):
            one_step()
        torch.cuda.synchronize(dev)
        graphs[mode] = (weakref.ref(self), ptrs, graph)
        return graph

    def _p_sample_on(self, prog, x: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        """One ancestral step x_t -> x_{t-1} on `prog` (whose conditioning inputs the caller has
        set): eager the first time a program is used, a replay of the captured step afterwards
        (the same launches, so the same values and the same draws)."""
        calls = prog.__dict__.get("_p_sample_calls", 0)
        prog.__dict__["_p_sample_calls"] = calls + 1
        out = self._reverse_loop(prog, x.float(), 0, 1, "ddpm", use_graph=calls >= 1, t_vec=t)
        return out

    def _reverse_loop(self, prog, img: torch.Tensor, start_t: int, n_steps: int, mode: str,
                      use_graph: bool = True, t_vec: Optional[torch.Tensor] = None,
                      stride: int = 1, table=None, inpaint=None, levels=None,
                      kspace: bool = False, guided=None) -> torch.Tensor:
        """Run n_steps reverse steps (i = start_t, start_t - stride, ...) on `prog` (a UNetProgram
        whose x_in is the sampler state).  mode: 'ddpm' | 'ddim' (t_prev = max(t - stride, 0)) |
        'dpmpp' (table = (ts, coef) of schedules.dpmpp_2m_table, n_steps = its rows).
        inpaint: (known, mask) of _inpaint_inputs, 'ddpm' or 'dpmpp' only: mri_inpaint_merge
        after every update, on a step graph of its own ('ddpm+inpaint' / 'dpmpp+inpaint').
        kspace: inpaint holds (x_zf, mask) of _kspace_inputs and the merge is mri_kspace_merge with
        the same z, on 'ddpm+kspace' / 'dpmpp+kspace'.
        levels: RePaint's walk (schedules.repaint_levels), 'ddpm' with inpaint only: its n_steps
        reverse steps replay 'ddpm+inpaint', its undo steps a graph of their own
        ('repaint-undo': mri_repaint_undo at t, then t += 1), in the walk's order.
        guided: the buffers of _guided_buffers, 'ddpm' or 'dpmpp' only: the unfused step with the
        guided eps of _guided_stage in the update, on 'ddpm+guided:kspace' / 'dpmpp+guided:mask'
        etc."""
        dev = img.device
        with torch.cuda.device(dev):
            return self._reverse_loop_on(prog, img, start_t, n_steps, mode, use_graph, t_vec, stride,
                                         table, inpaint, levels, kspace, guided)

    def _reverse_loop_on(self, prog, img, start_t, n_steps, mode, use_graph, t_vec, stride,
                         table=None, inpaint=None, levels=None, kspace=False, guided=None):
        dev = img.device
        if prog.params_changed():
            prog.do_refresh()
        B = prog.B
        per_sample = img[0].numel()
        tprev = prog.__dict__.setdefault("_tprev_buf", torch.zeros(B, dtype=torch.int64, device=dev))
        C, ldc = prog.cout, prog.cout_pad
        rng = self._rng(dev)
        inc = ops.randn_offset_increment(prog.x_in.numel())
        if stride != 1 and mode != "ddim":
            raise _lib.MriError("strided timesteps need the DDIM update")
        # the graph bakes the stride in: one graph per (mode, stride)
        gkey = mode if stride == 1 else f"{mode}/{stride}"
        inp = None
        if inpaint is not None:
            if mode not in ("ddpm", "dpmpp") or stride != 1 or t_vec is not None:
                raise _lib.MriError("inpainting runs on the full DDPM or the DPM-Solver++ loop")
            inp = self._inpaint_buffers(prog, mode == "dpmpp", kspace)
            gkey += "+kspace" if kspace else "+inpaint"
        if levels is not None and (inp is None or mode != "ddpm" or kspace):
            raise _lib.MriError("RePaint resampling runs on the DDPM inpainting loop")
        if guided is not None:
            if mode not in ("ddpm", "dpmpp") or stride != 1 or t_vec is not None or inp is not None:
                raise _lib.MriError("guided sampling runs on the full DDPM or the DPM-Solver++ loop")
            gkey += "+guided:" + ("kspace" if guided["kspace"] else "mask")
        # DDPM inpainting draws a second randn_like(x) per step (the merge's noise)
        adv = 2 * inc if inp is not None else inc

        # the guided step needs eps in HBM: it runs unfused
        fused = (getattr(prog, "fused_head", None) is not None and not prog.training
                 and os.environ.get("MRI_FUSED_STEP", "1") != "0" and guided is None)
        if mode == "dpmpp":
            # the graph reads its row of the table through the device index k: it bakes in no
            # timestep, so changing num_steps or start_t only rewrites the table
            dpm = self._dpmpp_buffers(prog, n_steps)
            kbuf, xp, rows = dpm["k"], dpm["x0_prev"], dpm["ts"].numel()
            kbuf.zero_()   # a valid row for the warm-up launch of a capture

        def merge():
            cond, work = (inp["known"], inp["mask"]), inp.get("work")
            if mode == "ddpm":   # before step_advance: tau = t - 1, z drawn after the update's z
                self._merge(prog.x_in, cond, prog.t_in, -1, kspace, work, rng=rng, rng_skip=inc)
            else:                # after step_table_advance: t = ts[k], -1 past the last row
                self._merge(prog.x_in, cond, prog.t_in, 0, kspace, work, noise=inp["noise"])

        def one_step():
            if fused:  # out_conv's tap sum + the update in one kernel: eps never goes to HBM
                if mode == "ddpm":
                    prog.run_fused_step(0, rng=rng, t=prog.t_in, betas=self.betas,
                                        sqrt_1mac=self.sqrt_one_minus_alphas_cumprod,
                                        sqrt_recip_alphas=self.sqrt_recip_alphas,
                                        post_var=self.posterior_variance)
                    if inp is not None:
                        merge()
                    ops.step_advance(prog.t_in, -1, rng=rng, rng_increment=adv)
                elif mode == "dpmpp":
                    prog.run_fused_step(3, x0_prev=xp, coef=dpm["coef"], k=kbuf)
                    ops.step_table_advance(prog.t_in, kbuf, dpm["ts"], rows)
                    if inp is not None:
                        merge()
                else:
                    prog.run_fused_step(1, t=prog.t_in, t_prev=tprev, alphas_cumprod=self.alphas_cumprod)
                    ops.step_advance(prog.t_in, -stride, t_prev=tprev)
                return
            prog.run()
            eps, e_ldc, e_c = prog.eps_nhwc, ldc, C
            if guided is not None:
                self._guided_stage(prog.x_in, eps, ldc, C, prog.t_in, guided)
                eps, e_ldc, e_c = guided["eps"], 0, 0
            if mode == "ddpm":
                ops.ddpm_step_rng(prog.x_in, eps, rng, prog.t_in, self.betas,
                                  self.sqrt_one_minus_alphas_cumprod, self.sqrt_recip_alphas,
                                  self.posterior_variance, prog.x_in, eps_nhwc_ldc=e_ldc, channels=e_c)
                if inp is not None:
                    merge()
                ops.step_advance(prog.t_in, -1, rng=rng, rng_increment=adv)
            elif mode == "dpmpp":
                ops.dpmpp_step(prog.x_in, eps, xp, dpm["coef"], kbuf, prog.x_in,
                               eps_nhwc_ldc=e_ldc, channels=e_c)
                ops.step_table_advance(prog.t_in, kbuf, dpm["ts"], rows)
                if inp is not None:
                    merge()
            else:
                ops.ddim_step(prog.x_in, prog.eps_nhwc, prog.t_in, tprev, self.alphas_cumprod,
                              prog.x_in, eps_nhwc_ldc=ldc, channels=C)
                ops.step_advance(prog.t_in, -stride, t_prev=tprev)

        def undo_step():
            ops.repaint_undo(prog.x_in, prog.t_in, self.alphas, self.betas, rng=rng)
            ops.step_advance(prog.t_in, 1, rng=rng, rng_increment=inc)

        graph = undo = None
        # the capture's warm-up runs the undo at t = 1, which reads alphas[2]
        walk_ok = levels is None or self.timesteps >= 3
        if use_graph and (n_steps >= 3 or t_vec is not None) and walk_ok:
            graph = self._step_graph(prog, gkey, one_step, tprev)
            if levels is not None:   # both captured before x_in / t_in are loaded below
                undo = self._step_graph(prog, "repaint-undo", undo_step, tprev)
        prog.x_in.copy_(img)
        if t_vec is not None:  # per-sample timesteps (p_sample called directly)
            prog.t_in.copy_(t_vec.to(dev).long())
        else:
            prog.t_in.fill_(start_t)
        tprev.fill_(max(start_t - stride, 0))
        if mode == "dpmpp":   # undo the warm-up launches of a capture and load this call's table
            ts, coef = table
            M = ts.numel()
            dpm["coef"][:M].copy_(coef)
            dpm["ts"][:M].copy_(ts)
            # with inpainting, t after the last row's advance is -1: the merge then keeps x_known
            dpm["ts"][M:].fill_(-1 if inp is not None else int(ts[-1]))
            kbuf.zero_()
        if inp is not None:
            inp["known"].copy_(inpaint[0])
            inp["mask"].copy_(inpaint[1])
            if mode == "dpmpp":
                inp["noise"].copy_(img)
        off = rng.load() if mode == "ddpm" else 0
        n_undo = 0
        if levels is None:
            for _ in range(n_steps):
                if graph is not None:
                    graph.replay()
                else:
                    one_step()
        else:   # no host synchronisation inside the walk
            for a, b in zip(levels, levels[1:]):
                if b < a:
                    step, g = one_step, graph
                else:
                    step, g, n_undo = undo_step, undo, n_undo + 1
                if g is not None:
                    g.replay()
                else:
                    step()
        if mode == "ddpm":  # z = randn_like(x) is drawn at every step, t = 0 included
            rng.commit(off + n_steps * adv + n_undo * inc)
        assert per_sample == prog.x_in[0].numel()
        return prog.x_in.clone()
