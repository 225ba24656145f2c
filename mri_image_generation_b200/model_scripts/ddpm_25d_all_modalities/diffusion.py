"""Drop-in for model_scripts/ddpm_25d_all_modalities/diffusion.py (GaussianDiffusion with
`context` threaded through, plain MSE loss, no `snr` buffer)."""
import torch

from ... import ops, schedules
from ...diffusion_base import DiffusionBase, _require_cuda
from ..slice_cond_2d_ddpm.diffusion import GaussianDiffusion as _GD2


class GaussianDiffusion(_GD2):
    """ddpm_25d_all_modalities/diffusion.py:5-48 (same buffers minus `snr`)."""

    WITH_SNR = False

    def p_losses(self, x_start, t, z_pos, context=None, noise=None):
        """ddpm_25d_all_modalities/diffusion.py:76-89: F.mse_loss(model(x_t, t, z, context), noise)."""
        if noise is None:  # noise = torch.randn_like(x_start), drawn inside the q_sample kernel
            x_noisy, noise = self._q_sample_draw(x_start, t)
        else:
            x_noisy = self.q_sample(x_start=x_start, t=t, noise=noise)
        predicted_noise = self.model(x_noisy, t, z_pos, context=context)
        return self._loss(predicted_noise, noise, t, 0.0)

    @torch.no_grad()
    def p_sample(self, x, t, z_pos, context=None):
        """ddpm_25d_all_modalities/diffusion.py:91-112."""
        _require_cuda(x, "p_sample")
        eps_theta = self.model(x, t, z_pos, context=context)
        return self._p_update(x, t, eps_theta)  # z = randn_like(x) drawn inside the kernel

    @torch.no_grad()
    def p_sample_loop(self, shape, z_pos, context=None):
        """ddpm_25d_all_modalities/diffusion.py:114-137."""
        device = self.betas.device
        B = shape[0]
        img = self._randn(shape, device)
        z_pos = self._z_tensor(z_pos, B, device)
        if context is not None:
            context = context.to(device)
        eng = self._engine_model()
        if eng is not None:
            _require_cuda(img, "p_sample_loop")
            cc = 0 if context is None else context.shape[1]
            prog = eng.program(B, shape[2:], shape[1], cc)
            prog.z_in.copy_(z_pos.reshape(-1, 1))
            if context is not None:
                prog.ctx_in.copy_(context)
            return self._reverse_loop(prog, img, self.timesteps - 1, self.timesteps, "ddpm")
        for i in reversed(range(self.timesteps)):
            t = torch.full((B,), i, device=device, dtype=torch.long)
            img = self.p_sample(img, t, z_pos, context=context)
        return img

    @torch.no_grad()
    def sample(self, batch_size=16, z_pos=0.5, context=None):
        """ddpm_25d_all_modalities/diffusion.py:139-149."""
        return self.p_sample_loop(
            (batch_size, self.channels, self.image_size, self.image_size), z_pos=z_pos,
            context=context)

    @torch.no_grad()
    def sample_dpmpp(self, batch_size=16, z_pos=0.5, context=None, num_steps=20):
        """Few-step sampler (not in the reference): x_T drawn as sample() draws it, then
        DPM-Solver++(2M) with `num_steps` UNet calls from t = T - 1 to sigma = 0 (returns x0)."""
        table = self._dpmpp_table(self.timesteps - 1, num_steps)
        device = self.betas.device
        shape = (batch_size, self.channels, self.image_size, self.image_size)
        img = self._randn(shape, device)
        z_pos = self._z_tensor(z_pos, batch_size, device)
        if context is not None:
            context = context.to(device)
        eng = self._engine_model()
        prog = None
        if eng is not None:
            _require_cuda(img, "sample_dpmpp")
            cc = 0 if context is None else context.shape[1]
            prog = eng.program(batch_size, shape[2:], shape[1], cc)
            prog.z_in.copy_(z_pos.reshape(-1, 1))
            if context is not None:
                prog.ctx_in.copy_(context)
        return self._sample_dpmpp(img, table, prog,
                                  lambda x, t: self.model(x, t, z_pos, context=context))

    @torch.no_grad()
    def calc_bpd_loop(self, x_start, z_pos, context=None):
        """The variational bound on -log p(x_start) in bits per dimension, x_start (B, 4, H, W) in
        [-1, 1] (not in the reference): see the 2D class's calc_bpd_loop()."""
        x0 = self._vb_input(x_start, 4)
        z_pos = self._z_tensor(z_pos, x0.shape[0], x0.device)
        if context is not None:
            context = context.to(x0.device)
        return self._vb_loop(self._cond_program(x0, z_pos, context), x0,
                             lambda x, t: self.model(x, t, z_pos, context=context), ops.VB_DISCRETIZED)

    @torch.no_grad()
    def inpaint(self, x_known, mask, z_pos=0.5, context=None, jump_length=10, jump_n_sample=1):
        """Inpainting by replacement with the full DDPM sampler (not in the reference), e.g.
        missing-modality imputation: x_known (B, 4, H, W) holds t1, t1ce, t2, flair and a mask of
        shape (1, 4, 1, 1) set only at the missing channel regenerates that modality.  See the 2D
        class's inpaint() for the method and the 3D class's for RePaint's resampling
        (jump_length, jump_n_sample)."""
        known, m = self._inpaint_inputs(x_known, mask, 4)
        levels = self._repaint_levels(jump_length, jump_n_sample)
        device = self.betas.device
        if context is not None:
            context = context.to(device)
        img, prog = self._inpaint_start(known, z_pos, context)
        z_pos = self._z_tensor(z_pos, img.shape[0], device)
        return self._inpaint_ddpm(img, (known.to(device), m.to(device)), prog,
                                  lambda x, t: self.model(x, t, z_pos, context=context), levels)

    @torch.no_grad()
    def reconstruct(self, kspace, kmask, z_pos=0.5, context=None):
        """Reconstruction from undersampled k-space with the full DDPM sampler (not in the
        reference), e.g. multi-contrast: t1, t1ce and t2 fully sampled (kmask 1 on their channels)
        and an undersampled flair.  See the 2D class's reconstruct()."""
        zf, m = self._kspace_inputs(kspace, kmask)
        device = self.betas.device
        if context is not None:
            context = context.to(device)
        img, prog = self._inpaint_start(zf, z_pos, context)
        z_pos = self._z_tensor(z_pos, img.shape[0], device)
        return self._inpaint_ddpm(img, (zf, m), prog,
                                  lambda x, t: self.model(x, t, z_pos, context=context), kspace=True)

    @torch.no_grad()
    def reconstruct_dpmpp(self, kspace, kmask, z_pos=0.5, context=None, num_steps=20):
        """reconstruct() with DPM-Solver++(2M) in `num_steps` UNet calls (not in the reference);
        see the 2D class's reconstruct_dpmpp()."""
        table = self._dpmpp_table(self.timesteps - 1, num_steps)
        zf, m = self._kspace_inputs(kspace, kmask)
        device = self.betas.device
        if context is not None:
            context = context.to(device)
        img, prog = self._inpaint_start(zf, z_pos, context)
        z_pos = self._z_tensor(z_pos, img.shape[0], device)
        return self._sample_dpmpp(img, table, prog,
                                  lambda x, t: self.model(x, t, z_pos, context=context),
                                  inpaint=(zf, m), kspace=True)

    @torch.no_grad()
    def inpaint_dpmpp(self, x_known, mask, z_pos=0.5, context=None, num_steps=20):
        """inpaint() with DPM-Solver++(2M) in `num_steps` UNet calls (not in the reference); see
        the 2D class's inpaint_dpmpp()."""
        known, m = self._inpaint_inputs(x_known, mask, 4)
        table = self._dpmpp_table(self.timesteps - 1, num_steps)
        device = self.betas.device
        if context is not None:
            context = context.to(device)
        img, prog = self._inpaint_start(known, z_pos, context)
        z_pos = self._z_tensor(z_pos, img.shape[0], device)
        return self._sample_dpmpp(img, table, prog,
                                  lambda x, t: self.model(x, t, z_pos, context=context),
                                  inpaint=(known.to(device), m.to(device)))
