"""Drop-in for model_scripts/slice_cond_2d_ddpm/diffusion.py (GaussianDiffusion, linear betas)."""
import torch

from ... import _lib, schedules
from ...diffusion_base import DiffusionBase, _require_cuda


class GaussianDiffusion(DiffusionBase):
    """slice_cond_2d_ddpm/diffusion.py:5-49."""

    WITH_SNR = True

    def __init__(self, model, image_size, channels=1, timesteps=1000, beta_start=1e-4, beta_end=0.02):
        super().__init__()
        self.model = model
        self.image_size = image_size
        self.channels = channels
        self.timesteps = timesteps
        print(f"Setting up Gaussian Diffusion with {timesteps} timesteps.")
        betas = schedules.linear_beta_schedule(timesteps, beta_start, beta_end)
        for k, v in schedules.make_buffers(betas, with_snr=self.WITH_SNR).items():
            self.register_buffer(k, v)

    def _extract(self, a, t, x_shape):
        """diffusion.py:51-58."""
        B = t.shape[0]
        out = a.gather(-1, t)
        return out.view(B, 1, 1, 1).expand(x_shape)

    def q_sample(self, x_start, t, noise=None):
        """diffusion.py:60-75."""
        if noise is None:  # noise = torch.randn_like(x_start), drawn inside the kernel
            return self._q_sample_draw(x_start, t)[0]
        return self._q_sample(x_start, t, noise)

    def p_losses(self, x_start, t, cond=None, noise=None, min_snr_gamma=5.0):
        """The LIVE definition, diffusion.py:91-107 (the second `def p_losses` wins): min-SNR
        weighted per-sample MSE, `cond` passed as the model's third positional argument (the
        training script passes z_pos there, model.py:164).  The reference's hard-coded
        mean(dim=(1,2,3,4)) raises IndexError on 4-D slices (SURVEY.md 0); this computes the same
        quantity rank-generically instead of reproducing the crash."""
        if noise is None:  # noise = torch.randn_like(x_start), drawn inside the q_sample kernel
            x_noisy, noise = self._q_sample_draw(x_start, t)
        else:
            x_noisy = self.q_sample(x_start=x_start, t=t, noise=noise)
        predicted_noise = self.model(x_noisy, t) if cond is None else self.model(x_noisy, t, cond)
        return self._loss(predicted_noise, noise, t, float(min_snr_gamma))

    @torch.no_grad()
    def p_sample(self, x, t, z_pos):
        """diffusion.py:110-132."""
        _require_cuda(x, "p_sample")
        eng = self._engine_model()
        if eng is not None:
            prog = eng.program(x.shape[0], x.shape[2:], x.shape[1], 0)
            prog.z_in.copy_(self._z_tensor(z_pos, x.shape[0], x.device).reshape(-1, 1))
            return self._p_sample_on(prog, x, t)
        eps_theta = self.model(x, t, z_pos)
        return self._p_update(x, t, eps_theta)  # z = randn_like(x) drawn inside the kernel

    def _z_tensor(self, z_pos, B, device):
        if not torch.is_tensor(z_pos):
            return torch.full((B,), float(z_pos), device=device)
        return z_pos.to(device).float()

    @torch.no_grad()
    def p_sample_loop(self, shape, z_pos):
        """diffusion.py:134-155."""
        device = self.betas.device
        B = shape[0]
        img = self._randn(shape, device)
        z_pos = self._z_tensor(z_pos, B, device)
        eng = self._engine_model()
        if eng is not None:
            _require_cuda(img, "p_sample_loop")
            prog = eng.program(B, shape[2:], shape[1], 0)
            prog.z_in.copy_(z_pos.reshape(-1, 1))
            return self._reverse_loop(prog, img, self.timesteps - 1, self.timesteps, "ddpm")
        for i in reversed(range(self.timesteps)):
            t = torch.full((B,), i, device=device, dtype=torch.long)
            img = self.p_sample(img, t, z_pos)
        return img

    @torch.no_grad()
    def sample(self, batch_size=16, z_pos=0.5):
        """diffusion.py:157-166."""
        return self.p_sample_loop(
            (batch_size, self.channels, self.image_size, self.image_size), z_pos=z_pos)

    @torch.no_grad()
    def sample_dpmpp(self, batch_size=16, z_pos=0.5, num_steps=20):
        """Few-step sampler (not in the reference): x_T drawn as sample() draws it, then
        DPM-Solver++(2M) with `num_steps` UNet calls from t = T - 1 to sigma = 0 (returns x0)."""
        table = self._dpmpp_table(self.timesteps - 1, num_steps)
        device = self.betas.device
        shape = (batch_size, self.channels, self.image_size, self.image_size)
        img = self._randn(shape, device)
        z_pos = self._z_tensor(z_pos, batch_size, device)
        eng = self._engine_model()
        prog = None
        if eng is not None:
            _require_cuda(img, "sample_dpmpp")
            prog = eng.program(batch_size, shape[2:], shape[1], 0)
            prog.z_in.copy_(z_pos.reshape(-1, 1))
        return self._sample_dpmpp(img, table, prog, lambda x, t: self.model(x, t, z_pos))

    @torch.no_grad()
    def inpaint(self, x_known, mask, z_pos=0.5, jump_length=10, jump_n_sample=1):
        """Inpainting by replacement with the full DDPM sampler (not in the reference).  x_known:
        (B, channels, H, W); mask broadcasts to it, True / 1 = regenerate, False / 0 = keep.  x_T
        is drawn as sample() draws it; after the update at every step i the kept region is set to
        q_sample(x_known, i - 1, noise=randn_like(x)) (x_known itself after i = 0).
        jump_n_sample > 1 adds RePaint's resampling with jumps of jump_length steps: see the 3D
        class's inpaint()."""
        known, m = self._inpaint_inputs(x_known, mask, 4)
        levels = self._repaint_levels(jump_length, jump_n_sample)
        img, prog = self._inpaint_start(known, z_pos)
        inp = (known.to(img.device), m.to(img.device))
        z_pos = self._z_tensor(z_pos, img.shape[0], img.device)
        return self._inpaint_ddpm(img, inp, prog, lambda x, t: self.model(x, t, z_pos), levels)

    @torch.no_grad()
    def inpaint_dpmpp(self, x_known, mask, z_pos=0.5, num_steps=20):
        """inpaint() with DPM-Solver++(2M) in `num_steps` UNet calls (not in the reference): after
        each step the kept region is set to q_sample(x_known, next timestep, noise=x_T), and to
        x_known after the last.  Conditions less strongly than inpaint() (DESIGN.md §4)."""
        known, m = self._inpaint_inputs(x_known, mask, 4)
        table = self._dpmpp_table(self.timesteps - 1, num_steps)
        img, prog = self._inpaint_start(known, z_pos)
        inp = (known.to(img.device), m.to(img.device))
        z_pos = self._z_tensor(z_pos, img.shape[0], img.device)
        return self._sample_dpmpp(img, table, prog, lambda x, t: self.model(x, t, z_pos), inpaint=inp)

    def _inpaint_start(self, known, z_pos, context=None):
        """x_T drawn as sample() draws it, and the program with its conditioning inputs set (None
        for a model that is not one of this package's UNets)."""
        device = self.betas.device
        img = self._randn(known.shape, device)
        eng = self._engine_model()
        if eng is None:
            return img, None
        B = known.shape[0]
        prog = eng.program(B, known.shape[2:], known.shape[1], 0 if context is None else context.shape[1])
        prog.z_in.copy_(self._z_tensor(z_pos, B, device).reshape(-1, 1))
        if context is not None:
            prog.ctx_in.copy_(context)
        return img, prog
