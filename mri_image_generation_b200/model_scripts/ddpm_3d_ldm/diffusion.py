"""Drop-in for model_scripts/ddpm_3d_ldm/diffusion.py (GaussianDiffusionLatent3D).

Same constructor, buffers (names, order, bit-identical values), methods and signatures; the
arithmetic runs in fused sm_100a kernels and the reverse loop is a replayed CUDA graph when the
denoiser is one of this package's UNets.
"""
import math

import torch

from ... import _lib, ops, schedules
from ...diffusion_base import DiffusionBase, _require_cuda, kspace_completion
from .vae import VAE3D


class GaussianDiffusionLatent3D(DiffusionBase):
    """ddpm_3d_ldm/diffusion.py:5-48."""

    def __init__(self, model, channels, timesteps=1000):
        super().__init__()
        self.model = model
        self.channels = channels
        self.timesteps = timesteps
        print(f"Setting up Gaussian Diffusion (3D latent) with {timesteps} timesteps.")
        for k, v in schedules.make_buffers(self.cosine_beta_schedule(), with_snr=True).items():
            self.register_buffer(k, v)

    def cosine_beta_schedule(self, s=0.008):
        """ddpm_3d_ldm/diffusion.py:50-56."""
        return schedules.cosine_beta_schedule(self.timesteps, s)

    def _extract(self, a, t, x_shape):
        """ddpm_3d_ldm/diffusion.py:58-66 (kept for callers; the fused kernels gather inline)."""
        B = t.shape[0]
        out = a.gather(-1, t)
        return out.view(B, *((1,) * (len(x_shape) - 1)))

    def q_sample(self, x_start, t, noise=None):
        """ddpm_3d_ldm/diffusion.py:68-82."""
        if noise is None:  # noise = torch.randn_like(x_start), drawn inside the kernel
            return self._q_sample_draw(x_start, t)[0]
        return self._q_sample(x_start, t, noise)

    def p_losses(self, x_start, t, cond=None, noise=None, min_snr_gamma=5.0):
        """ddpm_3d_ldm/diffusion.py:84-100."""
        if noise is None:  # noise = torch.randn_like(x_start), drawn inside the q_sample kernel
            x_noisy, noise = self._q_sample_draw(x_start, t)
        else:
            x_noisy = self.q_sample(x_start=x_start, t=t, noise=noise)
        predicted_noise = self.model(x_noisy, t) if cond is None else self.model(x_noisy, t, cond)
        return self._loss(predicted_noise, noise, t, float(min_snr_gamma))

    @torch.no_grad()
    def p_sample(self, x, t, cond=None):
        """ddpm_3d_ldm/diffusion.py:103-126: eps = model(x, t); z = randn_like(x) is drawn for
        every t (masked at t == 0)."""
        _require_cuda(x, "p_sample")
        eng = self._engine_model()
        if eng is not None and cond is None:
            return self._p_sample_on(eng.program(x.shape[0], x.shape[2:]), x, t)
        eps_theta = self.model(x, t) if cond is None else self.model(x, t, cond)
        return self._p_update(x, t, eps_theta)  # z = randn_like(x) drawn inside the kernel

    @torch.no_grad()
    def p_sample_loop(self, shape, cond=None):
        """ddpm_3d_ldm/diffusion.py:128-141."""
        device = self.betas.device
        img = self._randn(shape, device)
        return self.sample_from(img, self.timesteps - 1, cond)

    @torch.no_grad()
    def sample(self, batch_size, spatial_size, cond=None):
        """ddpm_3d_ldm/diffusion.py:143-152."""
        if isinstance(spatial_size, int):
            spatial_size = (spatial_size,) * 3
        shape = (batch_size, self.channels, *spatial_size)
        return self.p_sample_loop(shape, cond=cond)

    @torch.no_grad()
    def sample_from(self, x_t: torch.Tensor, start_t: int, cond=None) -> torch.Tensor:
        """ddpm_3d_ldm/diffusion.py:154-165 (i = start_t ... 0 inclusive)."""
        _require_cuda(x_t, "sample_from")
        eng = self._engine_model()
        if eng is not None and cond is None:
            prog = eng.program(x_t.shape[0], x_t.shape[2:])
            return self._reverse_loop(prog, x_t.float(), int(start_t), int(start_t) + 1, "ddpm")
        B = x_t.shape[0]
        img = x_t
        for i in reversed(range(start_t + 1)):
            t = torch.full((B,), i, device=img.device, dtype=torch.long)
            img = self.p_sample(img, t, cond)
        return img

    @torch.no_grad()
    def p_sample_ddim(self, x, t, t_prev, cond=None):
        """ddpm_3d_ldm/diffusion.py:167-186 (deterministic DDIM, eta = 0)."""
        _require_cuda(x, "p_sample_ddim")
        eps = self.model(x, t) if cond is None else self.model(x, t, cond)
        return self._ddim_update(x, t, t_prev, eps)

    @torch.no_grad()
    def sample_from_ddim(self, x_t: torch.Tensor, start_t: int, cond=None, stride: int = 1) -> torch.Tensor:
        """ddpm_3d_ldm/diffusion.py:188-196 (i = start_t ... 1, t_prev = i - 1).  `stride` > 1 is the
        strided-timestep fast sampler (SURVEY.md 8f row 3; not in the reference): timesteps
        start_t, start_t - stride, ... with t_prev = max(t - stride, 0), i.e. ceil(start_t / stride)
        UNet calls instead of start_t."""
        _require_cuda(x_t, "sample_from_ddim")
        stride = int(stride)
        if stride < 1:
            raise ValueError("stride must be >= 1")
        steps = -(-int(start_t) // stride)
        eng = self._engine_model()
        if eng is not None and cond is None and start_t >= 1:
            prog = eng.program(x_t.shape[0], x_t.shape[2:])
            return self._reverse_loop(prog, x_t.float(), int(start_t), steps, "ddim", stride=stride)
        B = x_t.shape[0]
        img = x_t
        for k in range(steps):
            i = int(start_t) - k * stride
            t = torch.full((B,), i, device=img.device, dtype=torch.long)
            t_prev = torch.full((B,), max(i - stride, 0), device=img.device, dtype=torch.long)
            img = self.p_sample_ddim(img, t, t_prev, cond)
        return img

    @torch.no_grad()
    def sample_ddim(self, batch_size, spatial_size, num_steps=50, cond=None):
        """Fast sampler (not in the reference): x_T ~ N(0, I), then `num_steps` strided DDIM steps
        from t = T - 1 down to 0 on the replayed step graph."""
        if isinstance(spatial_size, int):
            spatial_size = (spatial_size,) * 3
        shape = (batch_size, self.channels, *spatial_size)
        img = self._randn(shape, self.betas.device)
        stride = max(1, -(-(self.timesteps - 1) // int(num_steps)))
        return self.sample_from_ddim(img, self.timesteps - 1, cond, stride=stride)

    @torch.no_grad()
    def sample_dpmpp(self, batch_size, spatial_size, num_steps=20, cond=None):
        """Few-step sampler (not in the reference): x_T drawn as sample() draws it, then
        DPM-Solver++(2M) with `num_steps` UNet calls from t = T - 1 to sigma = 0 (returns x0)."""
        if isinstance(spatial_size, int):
            spatial_size = (spatial_size,) * 3
        table = self._dpmpp_table(self.timesteps - 1, num_steps)
        img = self._randn((batch_size, self.channels, *spatial_size), self.betas.device)
        return self._dpmpp_from(img, table, cond)

    @torch.no_grad()
    def sample_from_dpmpp(self, x_t: torch.Tensor, start_t: int, num_steps=20, cond=None) -> torch.Tensor:
        """DPM-Solver++(2M) from x_t at timestep start_t to sigma = 0 in `num_steps` UNet calls
        (not in the reference); the result is the fp32 x0 estimate."""
        return self._dpmpp_from(x_t, self._dpmpp_table(start_t, num_steps), cond)

    def _dpmpp_from(self, x_t, table, cond, inpaint=None):
        _require_cuda(x_t, "sample_from_dpmpp")
        return self._sample_dpmpp(x_t, table, self._program_for(x_t, cond), self._eps_fn(cond),
                                  inpaint=inpaint)

    def _program_for(self, x, cond):
        eng = self._engine_model()
        return eng.program(x.shape[0], x.shape[2:]) if eng is not None and cond is None else None

    def _eps_fn(self, cond):
        return lambda x, t: self.model(x, t) if cond is None else self.model(x, t, cond)

    @torch.no_grad()
    def inpaint(self, x_known, mask, cond=None, jump_length=10, jump_n_sample=1):
        """Inpainting by replacement with the full DDPM sampler (not in the reference).  x_known:
        (B, channels, D, H, W) latents; mask broadcasts to it, True / 1 = regenerate, False / 0 =
        keep.  x_T is drawn as sample() draws it; after the update at every step i the kept region
        is set to q_sample(x_known, i - 1, noise=randn_like(x)) (x_known itself after i = 0).  The
        mask is at latent resolution; for a mask at image resolution use inpaint_image().

        jump_n_sample > 1 adds RePaint's resampling: after the step at every multiple j of
        jump_length below T - jump_length, the state is re-noised jump_length steps
        (x = sqrt(alphas[l + 1]) x + sqrt(betas[l + 1]) randn_like(x) per step) and denoised again,
        jump_n_sample - 1 times (schedules.repaint_levels).  That is
        T + (jump_n_sample - 1) * jump_length * len(range(0, T - jump_length, jump_length)) UNet
        calls, 1990 at T = 1000 with (10, 2), and a more coherent regenerated region.  The default
        jump_n_sample = 1 is plain replacement."""
        known, m = self._inpaint_inputs(x_known, mask, 5)
        levels = self._repaint_levels(jump_length, jump_n_sample)
        img = self._randn(known.shape, self.betas.device)
        return self._inpaint_ddpm(img, (known.to(img.device), m.to(img.device)),
                                  self._program_for(img, cond), self._eps_fn(cond), levels)

    @torch.no_grad()
    def calc_bpd_loop(self, x_start, cond=None):
        """The variational bound on -log p(x_start) in bits per dimension (not in the reference;
        improved-diffusion's calc_bpd_loop for this fixed-small-variance model).  One UNet call per
        timestep, with z = randn_like(x_start) drawn for t = T - 1 ... 0.  Returns float64 device
        tensors: total_bpd (B,), prior_bpd (B,), vb (B, T) (the KL terms for t >= 1, the decoder's
        -log p(x_start | x at t = 0) at t = 0) and mse (B, T) (the mean (eps - z)^2 at each t).
        Latents are continuous, so the decoder term is a Gaussian density: it can be negative and
        these numbers do not compare with the pixel-space classes' bits per dimension."""
        x0 = self._vb_input(x_start, 5)
        return self._vb_loop(self._program_for(x0, cond), x0, self._eps_fn(cond), ops.VB_GAUSSIAN)

    @torch.no_grad()
    def inpaint_dpmpp(self, x_known, mask, num_steps=20, cond=None):
        """inpaint() with DPM-Solver++(2M) in `num_steps` UNet calls (not in the reference): after
        each step the kept region is set to q_sample(x_known, next timestep, noise=x_T), and to
        x_known after the last.  Conditions less strongly than inpaint() (DESIGN.md §4)."""
        known, m = self._inpaint_inputs(x_known, mask, 5)
        table = self._dpmpp_table(self.timesteps - 1, num_steps)
        img = self._randn(known.shape, self.betas.device)
        return self._dpmpp_from(img, table, cond, inpaint=(known.to(img.device), m.to(img.device)))

    # ------------------------------------------------------------------ measurement-guided sampling
    @torch.no_grad()
    def reconstruct(self, kspace, kmask, vae, guidance_scale=1.0, latent_scale=1.0, cond=None):
        """Undersampled 3-D k-space reconstruction through the VAE decoder (not in the reference;
        DESIGN.md §4).  kspace: complex (B, C, D, H, W), torch.fft.fftn(x, dim=(-3, -2, -1),
        norm="ortho") of the image x; kmask broadcasts to it, True / 1 = measured (e.g. a
        phase-encode-plane mask (1, 1, D, H, 1), or one per modality with T1 / T2 fully sampled).
        The latent is (B, channels, D/f, H/f, W/f) with f = 2^(vae.encoder.num_down - 1).

        The full DDPM sampler, x_T drawn as sample() draws it.  At every step the clean estimate
        x0 = (z_t - s1m eps) / sac is decoded, u = D(x0 / s), and moved by
        delta = -guidance_scale * D^T g / (s ||g||), g = P u - x_zf with P u = Re F^-1(M F u)
        (M the Hermitian completion of kmask, x_zf = Re F^-1(M y)); the update then uses the eps
        that gives x0 + delta.  No gradient flows through the UNet (MPGD, He et al. ICLR 2024, with
        DPS's step normalisation).  latent_scale s: the factor the LDM's training latents were
        multiplied by, z_train = s * vae.encode_to_latent(x) (train.py:540-553).  Returns the fp32
        image vae.decode_from_latent(z_0 / s), (B, C, D, H, W).  guidance_scale = 1.0 is untuned,
        and the reconstruction quality on real volumes is unverified.

        ValueError (before anything is drawn): bad shapes or mask, guidance_scale < 0 or not finite,
        latent_scale <= 0.  MriError: vae not this package's VAE3D, 'split' precision of the VAE or
        the UNet, CPU tensors, D, H or W over 512."""
        return self._guided("kspace", kspace, kmask, vae, None, guidance_scale, latent_scale, cond)

    @torch.no_grad()
    def reconstruct_dpmpp(self, kspace, kmask, vae, num_steps=20, guidance_scale=1.0, latent_scale=1.0,
                          cond=None):
        """reconstruct() with DPM-Solver++(2M) in `num_steps` UNet calls (not in the reference): x_T
        drawn as sample_dpmpp() draws it, the same guided eps in every solver update."""
        return self._guided("kspace", kspace, kmask, vae, num_steps, guidance_scale, latent_scale, cond)

    @torch.no_grad()
    def inpaint_image(self, x_known, mask, vae, guidance_scale=1.0, latent_scale=1.0, cond=None):
        """Inpainting with an image-space mask through the VAE decoder (not in the reference):
        reconstruct() with the data term g = (1 - mask) (u - x_known).  x_known: (B, C, D, H, W)
        image; mask broadcasts to it, True / 1 = regenerate, False / 0 = keep, at image resolution:
        it can keep an acquired modality and regenerate a missing one inside the same latent
        voxel.  Returns the fp32 image; the kept region is pulled toward x_known, not replaced."""
        return self._guided("mask", x_known, mask, vae, None, guidance_scale, latent_scale, cond)

    @torch.no_grad()
    def inpaint_image_dpmpp(self, x_known, mask, vae, num_steps=20, guidance_scale=1.0, latent_scale=1.0,
                            cond=None):
        """inpaint_image() with DPM-Solver++(2M) in `num_steps` UNet calls (not in the reference)."""
        return self._guided("mask", x_known, mask, vae, num_steps, guidance_scale, latent_scale, cond)

    def _guided(self, kind, meas, mask, vae, num_steps, guidance_scale, latent_scale, cond):
        lam, s = float(guidance_scale), float(latent_scale)
        if not math.isfinite(lam) or lam < 0:
            raise ValueError(f"guidance_scale must be finite and >= 0 (got {guidance_scale})")
        if not math.isfinite(s) or s <= 0:
            raise ValueError(f"latent_scale must be finite and > 0 (got {latent_scale})")
        if not isinstance(vae, VAE3D):
            raise _lib.MriError(f"vae must be this package's VAE3D (got {type(vae).__name__})")
        name = "kspace" if kind == "kspace" else "x_known"
        cout = vae.decoder.out_conv.weight.shape[0]
        ok = torch.is_tensor(meas) and meas.dim() == 5 and meas.shape[1] == cout and meas.numel() > 0 \
            and meas.is_complex() == (kind == "kspace")
        if not ok:
            got = (tuple(meas.shape), meas.dtype) if torch.is_tensor(meas) else type(meas)
            want = "complex" if kind == "kspace" else "real"
            raise ValueError(f"{name} must be a non-empty {want} (B, {cout}, D, H, W) tensor (got {got})")
        if vae.decoder.from_latent.weight.shape[1] != self.channels:
            raise ValueError(f"the VAE's latent has {vae.decoder.from_latent.weight.shape[1]} channels, "
                             f"the diffusion model {self.channels}")
        f = 2 ** (vae.encoder.num_down - 1)
        if any(n % f for n in meas.shape[2:]):
            raise ValueError(f"volume size {tuple(meas.shape[2:])} must be divisible by {f}")
        m = torch.as_tensor(mask)
        try:
            ok = torch.broadcast_shapes(m.shape, meas.shape) == meas.shape
        except RuntimeError:
            ok = False
        if not ok:
            raise ValueError(f"mask of shape {tuple(m.shape)} does not broadcast to {name}'s {tuple(meas.shape)}")
        if m.dtype != torch.bool and not bool(((m == 0) | (m == 1)).all()):
            raise ValueError("mask must be bool or hold only 0 / 1")
        table = self._dpmpp_table(self.timesteps - 1, num_steps) if num_steps is not None else None
        _require_cuda(meas, "guided sampling")
        ops.kspace3d_work_bytes(*meas.shape)      # MriError when D, H or W is over 512
        eng = self._engine_model()
        if vae.precision == "split" or getattr(eng if eng is not None else self.model, "precision", "bf16") == "split":
            raise _lib.MriError("guided sampling runs in bf16 precision ('split' is not supported)")
        dev = self.betas.device
        B = meas.shape[0]
        with torch.cuda.device(dev):
            meas, m = meas.to(dev), m.to(dev).expand(meas.shape).bool()
            if kind == "kspace":
                zf, full = kspace_completion(meas, m, dims=(-3, -2, -1))
                data = (zf.float().contiguous(), full.to(torch.uint8).contiguous())
            else:
                data = (meas.float().contiguous(), m.to(torch.uint8).contiguous())
            lat = torch.empty(B, self.channels, *(n // f for n in meas.shape[2:]), device=dev)
            dec = vae._program("decode", lat, training=True, wgrad=False)
            img = self._randn(lat.shape, dev)
            z0 = self._guided_sample(img, table, self._program_for(img, cond), self._eps_fn(cond), dec, data,
                                     kind == "kspace", lam, 1.0 / s)
            return vae.decode_from_latent(z0 / latent_scale)
