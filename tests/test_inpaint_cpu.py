"""Inpainting host logic without a GPU: argument checks (ValueError before x_T is drawn), and an
fp64 torch restatement of both inpainting loops on correlated Gaussian data with the exact noise
prediction, which shows how strongly the replacement method conditions the regenerated region.

Data: per sample x = s*1 + d*delta with s ~ N(0, a^2) shared by the n elements and delta ~ N(0, I),
so x ~ N(0, Sigma), Sigma = a^2 11^T + d^2 I.  The exact eps(x, t) = sigma_t Sigma_t^-1 x with
Sigma_t = alpha_t^2 Sigma + sigma_t^2 I, inverted in closed form by Sherman-Morrison.  Half of each
sample is known; the posterior mean of s given it is a^2 sum(x_K) / (n_K a^2 + d^2).  The error is
the RMS over samples of mean(regenerated half) - that posterior mean.

Measured (cosine T = 1000, B = 32, n = 1024, a = 1, d = 0.1), unconditional / inpainted from the
same x_T:
  DDPM, T = 1000:              1.332 / 0.01459, ratio 91.3   (test: >= 50)
  DPM-Solver++(2M), 20 steps:  1.091 / 0.1092,  ratio 10.0   (test: >= 5)
"""
import contextlib
import io
import math

import pytest
import torch

from mri_image_generation_b200 import _lib, schedules

T, A_SCALE, D_NOISE = 1000, 1.0, 0.1


def corr_eps(x, ac_t, a=A_SCALE, d=D_NOISE):
    """Exact eps for the data above at alphas_cumprod value(s) ac_t; x: (B, n) fp64."""
    ac_t = torch.as_tensor(ac_t, dtype=torch.float64).reshape(-1, 1)
    alpha2, sigma = ac_t, (1 - ac_t).sqrt()
    c = alpha2 * d * d + sigma * sigma
    u2 = alpha2 * a * a
    n = x.shape[-1]
    return sigma * (x / c - u2 * x.sum(-1, keepdim=True) / (c * (c + n * u2)))


def gaussian_problem(B, n, seed, a=A_SCALE, d=D_NOISE):
    """(x_known, mask, posterior mean of s): the first half of each sample is kept."""
    g = torch.Generator().manual_seed(seed)
    s = a * torch.randn(B, 1, generator=g, dtype=torch.float64)
    known = s + d * torch.randn(B, n, generator=g, dtype=torch.float64)
    mask = torch.zeros(B, n, dtype=torch.bool)
    mask[:, n // 2:] = True
    nk = n // 2
    post = a * a * known[:, :nk].sum(-1) / (nk * a * a + d * d)
    return known, mask, post


def region_error(x, mask, post):
    """RMS over samples of mean(x where mask) - post."""
    m = mask.double()
    mean_u = (x.double() * m).sum(-1) / m.sum(-1)
    return (mean_u - post).pow(2).mean().sqrt().item()


def _buffers():
    return {k: v.double() for k, v in schedules.make_buffers(schedules.cosine_beta_schedule(T), True).items()}


def ddpm_loop(buf, x_T, g, known=None, mask=None):
    """Ancestral sampling in fp64; with known / mask, the replacement step after every update."""
    x = x_T.clone()
    for i in reversed(range(T)):
        eps = corr_eps(x, buf["alphas_cumprod"][i])
        z = torch.randn(x.shape, generator=g, dtype=torch.float64)
        w = math.sqrt(buf["posterior_variance"][i]) if i > 0 else 0.0
        x = buf["sqrt_recip_alphas"][i] * (x - buf["betas"][i] / buf["sqrt_one_minus_alphas_cumprod"][i] * eps) + w * z
        if known is not None:
            nz = torch.randn(x.shape, generator=g, dtype=torch.float64)
            kn = known if i == 0 else (buf["sqrt_alphas_cumprod"][i - 1] * known
                                       + buf["sqrt_one_minus_alphas_cumprod"][i - 1] * nz)
            x = torch.where(mask, x, kn)
    return x


def dpmpp_loop(buf, x_T, M, known=None, mask=None):
    """DPM-Solver++(2M) over the package's table in fp64; with known / mask, the kept region is
    q_sample(known, next timestep, noise=x_T) after every row and known after the last."""
    ac32 = buf["alphas_cumprod"].float()
    ts, coef = schedules.dpmpp_2m_table(ac32, schedules.dpmpp_timesteps(T - 1, M))
    coef = coef.double()
    taus = ts.tolist()[1:] + [-1]
    x, x0p = x_T.clone(), torch.zeros_like(x_T)
    for i, t in enumerate(ts.tolist()):
        s, r, A, B, C = coef[i].tolist()
        x0 = (x - s * corr_eps(x, buf["alphas_cumprod"][t])) * r
        x, x0p = A * x + B * x0 + C * (x0 - x0p), x0
        if known is not None:
            tau = taus[i]
            kn = known if tau < 0 else (buf["sqrt_alphas_cumprod"][tau] * known
                                        + buf["sqrt_one_minus_alphas_cumprod"][tau] * x_T)
            x = torch.where(mask, x, kn)
    return x


def test_ddpm_replacement_conditions_the_unknown_region():
    buf = _buffers()
    known, mask, post = gaussian_problem(32, 1024, 0)
    x_T = torch.randn(known.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    free = ddpm_loop(buf, x_T, torch.Generator().manual_seed(2))
    inp = ddpm_loop(buf, x_T, torch.Generator().manual_seed(2), known, mask)
    assert torch.equal(inp[~mask], known[~mask])
    e_free, e_inp = region_error(free, mask, post), region_error(inp, mask, post)
    print(f"DDPM: unconditional {e_free:.4g}, inpainted {e_inp:.4g}, ratio {e_free / e_inp:.1f}")
    assert e_free / e_inp >= 50


def test_dpmpp_replacement_conditions_the_unknown_region():
    buf = _buffers()
    known, mask, post = gaussian_problem(32, 1024, 0)
    x_T = torch.randn(known.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    free = dpmpp_loop(buf, x_T, 20)
    inp = dpmpp_loop(buf, x_T, 20, known, mask)
    assert torch.equal(inp[~mask], known[~mask])
    e_free, e_inp = region_error(free, mask, post), region_error(inp, mask, post)
    print(f"DPM-Solver++: unconditional {e_free:.4g}, inpainted {e_inp:.4g}, ratio {e_free / e_inp:.1f}")
    assert e_free / e_inp >= 5


def test_exact_eps_matches_dense_inverse():
    """Sherman-Morrison against a dense solve, so the conditioning checks rest on the exact eps."""
    g = torch.Generator().manual_seed(3)
    n = 16
    x = torch.randn(3, n, generator=g, dtype=torch.float64)
    for ac_t in (0.999, 0.5, 0.01):
        sig = A_SCALE ** 2 * torch.ones(n, n, dtype=torch.float64) + D_NOISE ** 2 * torch.eye(n, dtype=torch.float64)
        sig_t = ac_t * sig + (1 - ac_t) * torch.eye(n, dtype=torch.float64)
        want = math.sqrt(1 - ac_t) * torch.linalg.solve(sig_t, x.T).T
        torch.testing.assert_close(corr_eps(x, ac_t), want, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------ argument checks
def _diffusions():
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.diffusion import \
        GaussianDiffusion as G25
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion as G2
    with contextlib.redirect_stdout(io.StringIO()):
        return {"3d": GaussianDiffusionLatent3D(torch.nn.Identity(), 3, timesteps=50),
                "2d": G2(torch.nn.Identity(), 8, timesteps=50),
                "25d": G25(torch.nn.Identity(), 8, channels=4, timesteps=50)}


_SHAPE = {"3d": (2, 3, 4, 6, 4), "2d": (2, 1, 8, 8), "25d": (2, 4, 8, 8)}
_BAD = {
    "rank": lambda s: (torch.zeros(*s, 1), torch.ones(1, dtype=torch.bool)),
    "rank_low": lambda s: (torch.zeros(*s[:-1]), torch.ones(1, dtype=torch.bool)),
    "channels": lambda s: (torch.zeros(s[0], s[1] + 1, *s[2:]), torch.ones(1, dtype=torch.bool)),
    "mask_shape": lambda s: (torch.zeros(s), torch.ones(s[0] + 1, *s[1:], dtype=torch.bool)),
    "mask_rank": lambda s: (torch.zeros(s), torch.ones(2, *s, dtype=torch.bool)),
    "mask_values": lambda s: (torch.zeros(s), torch.full(s, 0.5)),
    "mask_int2": lambda s: (torch.zeros(s), torch.full(s, 2, dtype=torch.int64)),
    "mask_nan": lambda s: (torch.zeros(s), torch.full(s, float("nan"))),
}


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
@pytest.mark.parametrize("bad", sorted(_BAD))
@pytest.mark.parametrize("method", ["inpaint", "inpaint_dpmpp"])
def test_bad_arguments_raise_before_any_draw(kind, bad, method):
    """ValueError, not the MriError these CPU objects raise when they draw x_T: the check comes
    first.  tests/test_gpu_inpaint.py checks that the CUDA generator is left untouched."""
    d = _diffusions()[kind]
    x_known, mask = _BAD[bad](_SHAPE[kind])
    with pytest.raises(ValueError):
        getattr(d, method)(x_known, mask)


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
@pytest.mark.parametrize("num_steps", [0, -3, 50, 51])
def test_bad_num_steps_raise_before_any_draw(kind, num_steps):
    d = _diffusions()[kind]
    with pytest.raises(ValueError):
        d.inpaint_dpmpp(torch.zeros(_SHAPE[kind]), torch.ones(1, dtype=torch.bool), num_steps=num_steps)


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
@pytest.mark.parametrize("method", ["inpaint", "inpaint_dpmpp"])
def test_valid_arguments_on_cpu_raise_mri_error(kind, method):
    d = _diffusions()[kind]
    s = _SHAPE[kind]
    for mask in (torch.ones(1, dtype=torch.bool), torch.zeros(s[0], 1, *([1] * (len(s) - 2))),
                 torch.tensor(1, dtype=torch.int64)):
        with pytest.raises(_lib.MriError):
            getattr(d, method)(torch.zeros(s), mask)
