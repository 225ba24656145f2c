"""The variational bound without a GPU: schedules.vb_constants against improved-diffusion's
formulas in fp64 (the KL of two Gaussians in means form, the prior KL) on three schedules, and
the argument checks of calc_bpd_loop (ValueError on a bad shape, MriError on a CPU tensor).

The fp64 restatements here are also the oracle of tests/test_gpu_likelihood.py."""
import contextlib
import io
import math

import numpy as np
import pytest
import torch

from mri_image_generation_b200 import schedules


def sched64(betas):
    """alpha, alpha_bar, alpha_bar_prev and beta~ in fp64 from the fp32 betas."""
    b = betas.detach().cpu().double()
    a = 1.0 - b
    ac = torch.cumprod(a, 0)
    ac_prev = torch.cat([torch.ones(1, dtype=torch.float64), ac[:-1]])
    return {"b": b, "a": a, "ac": ac, "ac_prev": ac_prev, "post": b * (1.0 - ac_prev) / (1.0 - ac)}


def kl_means(s, t, x0, z, eps):
    """sum KL(q(x_{t-1} | x_t, x0) || N(mu_theta, beta~_t)) in nats, improved-diffusion's
    q_posterior_mean_variance / p_mean_variance / normal_kl, with x_t = q_sample(x0, t, z) in fp64.
    t >= 1; x0, z, eps fp64, summed over the last dimension."""
    b, a, ac, acp = s["b"][t], s["a"][t], s["ac"][t], s["ac_prev"][t]
    x_t = ac.sqrt() * x0 + (1.0 - ac).sqrt() * z
    coef1 = b * acp.sqrt() / (1.0 - ac)
    coef2 = (1.0 - acp) * a.sqrt() / (1.0 - ac)
    mu_q = coef1 * x0 + coef2 * x_t
    mu_p = (x_t - b / (1.0 - ac).sqrt() * eps) / a.sqrt()
    lv = s["post"][t].log()
    # normal_kl(mu_q, lv, mu_p, lv) = 0.5 (-1 + lv - lv + exp(lv - lv) + (mu_q - mu_p)^2 exp(-lv))
    return (0.5 * (mu_q - mu_p) ** 2 * torch.exp(-lv)).sum(-1)


def approx_cdf64(x):
    return 0.5 * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x ** 3)))


# improved-diffusion applies its Python-float constants to fp32 data, so torch rounds them to fp32:
# x0 = -0.999f is not below the edge
EDGE, HALF_BIN = float(np.float32(0.999)), float(np.float32(1.0 / 255.0))


def discretized_nll64(x0, mu, log_scale):
    """-log p of improved-diffusion's discretized_gaussian_log_likelihood, per element, fp64."""
    c = x0 - mu
    inv = math.exp(-log_scale)
    cdf_plus = approx_cdf64(inv * (c + HALF_BIN))
    cdf_min = approx_cdf64(inv * (c - HALF_BIN))
    lp = torch.where(x0 < -EDGE, cdf_plus.clamp(min=1e-12).log(),
                     torch.where(x0 > EDGE, (1.0 - cdf_min).clamp(min=1e-12).log(),
                                 (cdf_plus - cdf_min).clamp(min=1e-12).log()))
    return -lp


def gaussian_nll64(x0, mu, log_scale):
    """-log N(x0; mu, exp(log_scale)^2) per element, fp64."""
    y = (x0 - mu) * math.exp(-log_scale)
    return 0.5 * y * y + log_scale + 0.5 * math.log(2.0 * math.pi)


SCHEDULES = {
    "linear1000": lambda: schedules.linear_beta_schedule(1000, 1e-4, 0.02),
    "cosine1000": lambda: schedules.cosine_beta_schedule(1000),
    "linear12": lambda: schedules.linear_beta_schedule(12, 1e-4, 0.02),
    "cosine12": lambda: schedules.cosine_beta_schedule(12),
}


@pytest.mark.parametrize("name", sorted(SCHEDULES))
def test_lambda_form_equals_the_means_form_kl(name):
    betas = SCHEDULES[name]()
    T = betas.numel()
    lam = schedules.vb_constants(betas)["lam"]
    assert lam.dtype == torch.float64 and lam.shape == (T,) and lam[0] == 0
    s = sched64(betas)
    g = torch.Generator().manual_seed(T)
    n = 512
    ts = torch.arange(1, T)
    x0 = torch.rand(T - 1, n, generator=g, dtype=torch.float64) * 2 - 1
    z = torch.randn(T - 1, n, generator=g, dtype=torch.float64)
    eps = z + 0.3 * torch.randn(T - 1, n, generator=g, dtype=torch.float64)
    want = kl_means(s, ts.view(-1, 1), x0, z, eps).view(-1)
    got = lam[1:] * ((eps - z) ** 2).sum(-1)
    rel = ((got - want).abs() / want).max().item()
    assert rel <= 1e-6, rel


@pytest.mark.parametrize("name", sorted(SCHEDULES))
def test_prior_constants(name):
    betas = SCHEDULES[name]()
    c = schedules.vb_constants(betas)
    aT = torch.cumprod(1.0 - betas.double(), 0)[-1].item()
    assert c["prior_coef"] == pytest.approx(aT, rel=1e-15)
    x0 = torch.linspace(-3, 3, 101, dtype=torch.float64)
    # normal_kl(sqrt(a) x0, log(1 - a), 0, 0)
    m1, lv1 = math.sqrt(aT) * x0, math.log(1.0 - aT)
    want = 0.5 * (-1.0 + 0.0 - lv1 + math.exp(lv1 - 0.0) + m1 ** 2 * math.exp(-0.0))
    got = 0.5 * (c["prior_const"] + c["prior_coef"] * x0 ** 2)
    assert torch.allclose(got, want, rtol=1e-12, atol=1e-15)


def test_decoder_oracles_match_numpy_restatements():
    """The fp64 oracles above against numpy versions of the same formulas, at the bin edges."""
    x0 = torch.tensor([-1.0, -0.9995, -0.5, 0.0, 0.999, 0.9995, 1.0, 1.5], dtype=torch.float64)
    mu = x0 + torch.tensor([0.001, -0.004, 0.002, 0.01, -0.001, 0.0, 0.003, 0.3], dtype=torch.float64)
    ls = 0.5 * math.log(1e-4)
    xn, mn = x0.numpy(), mu.numpy()
    cdf = lambda v: 0.5 * (1.0 + np.tanh(np.sqrt(2.0 / np.pi) * (v + 0.044715 * v ** 3)))
    h, e = np.float32(1 / 255.0).item(), np.float32(0.999).item()
    cp = cdf(np.exp(-ls) * (xn - mn + h))
    cm = cdf(np.exp(-ls) * (xn - mn - h))
    lp = np.where(xn < -e, np.log(np.maximum(cp, 1e-12)),
                  np.where(xn > e, np.log(np.maximum(1 - cm, 1e-12)), np.log(np.maximum(cp - cm, 1e-12))))
    np.testing.assert_allclose(discretized_nll64(x0, mu, ls).numpy(), -lp, rtol=1e-14)
    var = math.exp(2 * ls)
    want = 0.5 * np.log(2 * np.pi * var) + (xn - mn) ** 2 / (2 * var)
    np.testing.assert_allclose(gaussian_nll64(x0, mu, ls).numpy(), want, rtol=1e-12)


# ------------------------------------------------------------------------------------------ arguments
def _diffusions():
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.diffusion import \
        GaussianDiffusion as G25
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion as G2
    with contextlib.redirect_stdout(io.StringIO()):
        return {"3d": (GaussianDiffusionLatent3D(torch.nn.Identity(), 3, timesteps=12), ()),
                "2d": (G2(torch.nn.Identity(), 8, timesteps=12), (0.5,)),
                "25d": (G25(torch.nn.Identity(), 8, channels=4, timesteps=12), (0.5,))}


_SHAPE = {"3d": (2, 3, 4, 6, 4), "2d": (2, 1, 8, 8), "25d": (2, 4, 8, 8)}
_BAD = {
    "rank": lambda s: torch.zeros(*s, 1),
    "rank_low": lambda s: torch.zeros(*s[:-1]),
    "channels": lambda s: torch.zeros(s[0], s[1] + 1, *s[2:]),
    "empty": lambda s: torch.zeros(0, *s[1:]),
    "not_a_tensor": lambda s: np.zeros(s, dtype=np.float32),
}


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
@pytest.mark.parametrize("bad", sorted(_BAD))
def test_bad_shapes_raise_value_error(kind, bad):
    d, extra = _diffusions()[kind]
    with pytest.raises(ValueError):
        d.calc_bpd_loop(_BAD[bad](_SHAPE[kind]), *extra)


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_cpu_tensors_raise_mri_error(kind):
    from mri_image_generation_b200 import _lib
    d, extra = _diffusions()[kind]
    with pytest.raises(_lib.MriError):
        d.calc_bpd_loop(torch.zeros(_SHAPE[kind]), *extra)
