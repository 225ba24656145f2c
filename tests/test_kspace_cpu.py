"""Undersampled k-space reconstruction without a GPU: argument checks (ValueError before x_T is
drawn), the algebra of the Hermitian completion and of the projector P u = Re ifft2(M fft2(u)),
and an fp64 torch restatement of both reconstruction loops on Gaussian data with the exact noise
prediction, which shows how strongly the Fourier merge conditions the unmeasured frequencies.

Data: per sample x = s*v + d*delta with v a centred Gaussian bump (width 1.5 pixels) on a 24 x 24
plane, s ~ N(0, a^2) and delta ~ N(0, I), so x ~ N(0, a^2 v v^T + d^2 I).  The exact
eps(x, t) = sigma_t Sigma_t^-1 x comes from Sherman-Morrison with v.  Given x_zf = P x, the
posterior mean of s is a^2 <Pv, x_zf> / (d^2 + a^2 |Pv|^2).  The error is the RMS over samples of
<(I - P)v, x_hat> / |(I - P)v|^2 minus that posterior mean: what the reconstruction put into the
unmeasured part of k-space, read as an estimate of s.  The bump is narrow enough that a third of
its norm lies in unmeasured frequencies; d is small enough that the estimate's own noise,
d / |(I - P)v| = 0.02, stays below what the merge achieves.

Measured (the 2D class's linear schedule, T = 1000, B = 32, a = 1, d = 0.02, every fourth
phase-encode row plus the four lowest), unconditional / reconstructed from the same x_T:
  DDPM, T = 1000:              1.065 / 0.02063, ratio 51.6   (test: >= 25)
  DPM-Solver++(2M), 20 steps:  1.505 / 0.09753, ratio 15.4   (test: >= 7)
"""
import contextlib
import io
import math

import pytest
import torch

from mri_image_generation_b200 import _lib, schedules
from mri_image_generation_b200.diffusion_base import kspace_completion

T, A_SCALE, D_NOISE, HW = 1000, 1.0, 0.02, 24


def mirror(a):
    """a(-k) for the unshifted DFT grid: index j -> (-j) mod N on the last two axes."""
    return torch.roll(torch.flip(a, (-2, -1)), (1, 1), (-2, -1))


def projector(M):
    """P u = Re ifft2(M fft2(u)), orthonormal, in fp64."""
    return lambda u: torch.fft.ifft2(M * torch.fft.fft2(u.double(), norm="ortho"), norm="ortho").real


def line_mask(H, W, step=4, centre=4, axis=-2):
    """Every step-th line along `axis` plus the `centre` lowest frequencies (DC at 0)."""
    n = H if axis == -2 else W
    keep = torch.zeros(n, dtype=torch.bool)
    keep[::step] = True
    for j in range(-(centre // 2), centre - centre // 2):
        keep[j % n] = True
    return (keep.view(n, 1).expand(H, W) if axis == -2 else keep.view(1, n).expand(H, W)).clone()


def bump(H, W, width):
    h = torch.arange(H, dtype=torch.float64) - (H - 1) / 2
    w = torch.arange(W, dtype=torch.float64) - (W - 1) / 2
    return torch.exp(-(h.view(-1, 1) ** 2 + w.view(1, -1) ** 2) / (2 * width * width))


# ------------------------------------------------------------------------------------ algebra
@pytest.mark.parametrize("H,W", [(1, 1), (7, 9), (8, 8), (33, 31), (36, 44)])
@pytest.mark.parametrize("kind", ["random", "rows", "cols"])
def test_completion_and_projector(H, W, kind):
    """M is Hermitian-symmetric and contains m; P is symmetric and idempotent; P x_true = x_zf;
    values of y outside m are never read (NaN there is harmless)."""
    g = torch.Generator().manual_seed(H * 100 + W)
    if kind == "random":
        m = torch.rand(2, 3, H, W, generator=g) < 0.3
    else:
        m = line_mask(H, W, axis=-2 if kind == "rows" else -1).expand(2, 3, H, W)
    x = torch.randn(2, 3, H, W, generator=g, dtype=torch.float64)
    y = torch.fft.fft2(x, norm="ortho")
    x_zf, M = kspace_completion(torch.where(m, y, torch.full_like(y, complex("nan"))), m)
    assert torch.equal(M, mirror(M)) and bool((M | ~m).all())
    P = projector(M)
    torch.testing.assert_close(P(x), x_zf, rtol=0, atol=1e-12)
    # the matrix of P on one plane: symmetric and idempotent
    Mp = M[0, 0]
    E = torch.eye(H * W, dtype=torch.float64).view(H * W, H, W)
    Pm = projector(Mp)(E).reshape(H * W, H * W)
    torch.testing.assert_close(Pm, Pm.T, rtol=0, atol=1e-12)
    torch.testing.assert_close(Pm @ Pm, Pm, rtol=0, atol=1e-12)
    assert abs(torch.trace(Pm).item() - Mp.sum().item()) < 1e-9   # rank = measured samples


def test_empty_and_full_masks():
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 1, 6, 7, generator=g, dtype=torch.float64)
    y = torch.fft.fft2(x, norm="ortho")
    zf0, M0 = kspace_completion(y, torch.zeros(y.shape, dtype=torch.bool))
    assert not M0.any() and torch.equal(zf0, torch.zeros_like(zf0))
    zf1, M1 = kspace_completion(y, torch.ones(y.shape, dtype=torch.bool))
    assert M1.all()
    torch.testing.assert_close(zf1, x, rtol=0, atol=1e-12)


# ------------------------------------------------------------------------------------ conditioning
def bump_eps(x, ac_t, v, a=A_SCALE, d=D_NOISE):
    """Exact eps for x = s v + d delta at alphas_cumprod value ac_t (Sherman-Morrison); x: (B, H, W)."""
    alpha2, sigma = ac_t, math.sqrt(1 - ac_t)
    c = alpha2 * d * d + sigma * sigma
    u2 = alpha2 * a * a
    vx = (x * v).sum((-2, -1), keepdim=True)
    return sigma * (x / c - u2 * v * vx / (c * (c + u2 * (v * v).sum())))


def bump_problem(B, seed, a=A_SCALE, d=D_NOISE):
    """(v, x_zf, M, P, posterior mean of s) for the line mask on HW x HW."""
    g = torch.Generator().manual_seed(seed)
    v = bump(HW, HW, 1.5)
    s = a * torch.randn(B, 1, 1, generator=g, dtype=torch.float64)
    x = s * v + d * torch.randn(B, HW, HW, generator=g, dtype=torch.float64)
    m = line_mask(HW, HW).expand(B, HW, HW)
    x_zf, M = kspace_completion(torch.fft.fft2(x, norm="ortho"), m)
    P = projector(M)
    Pv = P(v.expand(B, HW, HW))[0]
    post = a * a * (x_zf * Pv).sum((-2, -1)) / (d * d + a * a * (Pv * Pv).sum())
    return v, x_zf, P, post


def unmeasured_error(x_hat, v, P, post):
    r = v - P(v.unsqueeze(0))[0]
    est = (x_hat * r).sum((-2, -1)) / (r * r).sum()
    return (est - post).pow(2).mean().sqrt().item()


def _buffers():
    betas = schedules.linear_beta_schedule(T, 1e-4, 0.02)
    return {k: v.double() for k, v in schedules.make_buffers(betas, True).items()}


def ddpm_loop(buf, x_T, g, v, x_zf=None, P=None):
    """Ancestral sampling in fp64; with x_zf / P, the k-space merge after every update."""
    x = x_T.clone()
    for i in reversed(range(T)):
        eps = bump_eps(x, buf["alphas_cumprod"][i].item(), v)
        z = torch.randn(x.shape, generator=g, dtype=torch.float64)
        w = math.sqrt(buf["posterior_variance"][i]) if i > 0 else 0.0
        x = buf["sqrt_recip_alphas"][i] * (x - buf["betas"][i] / buf["sqrt_one_minus_alphas_cumprod"][i] * eps) + w * z
        if x_zf is not None:
            n = torch.randn(x.shape, generator=g, dtype=torch.float64)
            if i == 0:
                x = x - P(x) + x_zf
            else:
                x = x - P(x - buf["sqrt_one_minus_alphas_cumprod"][i - 1] * n) \
                    + buf["sqrt_alphas_cumprod"][i - 1] * x_zf
    return x


def dpmpp_loop(buf, x_T, steps, v, x_zf=None, P=None):
    """DPM-Solver++(2M) over the package's table in fp64; with x_zf / P, the k-space merge with
    noise x_T after every row (x - P x + x_zf after the last)."""
    ts, coef = schedules.dpmpp_2m_table(buf["alphas_cumprod"].float(), schedules.dpmpp_timesteps(T - 1, steps))
    coef = coef.double()
    taus = ts.tolist()[1:] + [-1]
    x, x0p = x_T.clone(), torch.zeros_like(x_T)
    for i, t in enumerate(ts.tolist()):
        s, r, A, B, C = coef[i].tolist()
        x0 = (x - s * bump_eps(x, buf["alphas_cumprod"][t].item(), v)) * r
        x, x0p = A * x + B * x0 + C * (x0 - x0p), x0
        if x_zf is not None:
            tau = taus[i]
            if tau < 0:
                x = x - P(x) + x_zf
            else:
                x = x - P(x - buf["sqrt_one_minus_alphas_cumprod"][tau] * x_T) + buf["sqrt_alphas_cumprod"][tau] * x_zf
    return x


def _consistency(x_hat, x_zf, P):
    """|P x_hat - x_zf| / |x_zf|: the measured part of k-space is the data's."""
    return ((P(x_hat) - x_zf).norm() / x_zf.norm()).item()


def test_ddpm_kspace_merge_conditions_the_unmeasured_frequencies():
    buf = _buffers()
    v, x_zf, P, post = bump_problem(32, 0)
    x_T = torch.randn(x_zf.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    free = ddpm_loop(buf, x_T, torch.Generator().manual_seed(2), v)
    rec = ddpm_loop(buf, x_T, torch.Generator().manual_seed(2), v, x_zf, P)
    assert _consistency(rec, x_zf, P) < 1e-12
    e_free, e_rec = unmeasured_error(free, v, P, post), unmeasured_error(rec, v, P, post)
    print(f"DDPM: unconditional {e_free:.4g}, reconstructed {e_rec:.4g}, ratio {e_free / e_rec:.1f}")
    assert e_free / e_rec >= 25


def test_dpmpp_kspace_merge_conditions_the_unmeasured_frequencies():
    buf = _buffers()
    v, x_zf, P, post = bump_problem(32, 0)
    x_T = torch.randn(x_zf.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    free = dpmpp_loop(buf, x_T, 20, v)
    rec = dpmpp_loop(buf, x_T, 20, v, x_zf, P)
    assert _consistency(rec, x_zf, P) < 1e-12
    e_free, e_rec = unmeasured_error(free, v, P, post), unmeasured_error(rec, v, P, post)
    print(f"DPM-Solver++: unconditional {e_free:.4g}, reconstructed {e_rec:.4g}, ratio {e_free / e_rec:.1f}")
    assert e_free / e_rec >= 7


def test_exact_eps_matches_dense_inverse():
    """Sherman-Morrison with v against a dense solve, so the conditioning checks rest on the exact eps."""
    g = torch.Generator().manual_seed(3)
    H = W = 4
    v = bump(H, W, 1.5)
    x = torch.randn(3, H, W, generator=g, dtype=torch.float64)
    vv = v.reshape(-1)
    for ac_t in (0.999, 0.5, 0.01):
        sig = A_SCALE ** 2 * torch.outer(vv, vv) + D_NOISE ** 2 * torch.eye(H * W, dtype=torch.float64)
        sig_t = ac_t * sig + (1 - ac_t) * torch.eye(H * W, dtype=torch.float64)
        want = math.sqrt(1 - ac_t) * torch.linalg.solve(sig_t, x.reshape(3, -1).T).T
        torch.testing.assert_close(bump_eps(x, ac_t, v).reshape(3, -1), want, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------ argument checks
def _diffusions():
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.diffusion import \
        GaussianDiffusion as G25
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion as G2
    with contextlib.redirect_stdout(io.StringIO()):
        return {"2d": G2(torch.nn.Identity(), 8, timesteps=50),
                "25d": G25(torch.nn.Identity(), 8, channels=4, timesteps=50)}


_SHAPE = {"2d": (2, 1, 8, 8), "25d": (2, 4, 8, 8)}
_C = torch.complex64
_BAD = {
    "real": lambda s: (torch.zeros(s), torch.ones(1, dtype=torch.bool)),
    "not_tensor": lambda s: ([[0j]], torch.ones(1, dtype=torch.bool)),
    "rank": lambda s: (torch.zeros(*s, 1, dtype=_C), torch.ones(1, dtype=torch.bool)),
    "rank_low": lambda s: (torch.zeros(*s[:-1], dtype=_C), torch.ones(1, dtype=torch.bool)),
    "channels": lambda s: (torch.zeros(s[0], s[1] + 1, *s[2:], dtype=_C), torch.ones(1, dtype=torch.bool)),
    "empty": lambda s: (torch.zeros(0, *s[1:], dtype=_C), torch.ones(1, dtype=torch.bool)),
    "mask_shape": lambda s: (torch.zeros(s, dtype=_C), torch.ones(s[0] + 1, *s[1:], dtype=torch.bool)),
    "mask_rank": lambda s: (torch.zeros(s, dtype=_C), torch.ones(2, *s, dtype=torch.bool)),
    "mask_values": lambda s: (torch.zeros(s, dtype=_C), torch.full(s, 0.5)),
    "mask_int2": lambda s: (torch.zeros(s, dtype=_C), torch.full(s, 2, dtype=torch.int64)),
    "mask_nan": lambda s: (torch.zeros(s, dtype=_C), torch.full(s, float("nan"))),
}


@pytest.mark.parametrize("kind", ["2d", "25d"])
@pytest.mark.parametrize("bad", sorted(_BAD))
@pytest.mark.parametrize("method", ["reconstruct", "reconstruct_dpmpp"])
def test_bad_arguments_raise_before_any_draw(kind, bad, method):
    """ValueError, not the MriError these CPU objects raise on a valid input: the check comes
    first.  tests/test_gpu_kspace.py checks that the CUDA generator is left untouched."""
    d = _diffusions()[kind]
    kspace, kmask = _BAD[bad](_SHAPE[kind])
    with pytest.raises(ValueError):
        getattr(d, method)(kspace, kmask)


@pytest.mark.parametrize("kind", ["2d", "25d"])
@pytest.mark.parametrize("num_steps", [0, -3, 50, 51])
def test_bad_num_steps_raise_before_any_draw(kind, num_steps):
    d = _diffusions()[kind]
    with pytest.raises(ValueError):
        d.reconstruct_dpmpp(torch.zeros(_SHAPE[kind], dtype=_C), torch.ones(1, dtype=torch.bool),
                            num_steps=num_steps)


@pytest.mark.parametrize("kind", ["2d", "25d"])
@pytest.mark.parametrize("method", ["reconstruct", "reconstruct_dpmpp"])
def test_valid_arguments_on_cpu_raise_mri_error(kind, method):
    d = _diffusions()[kind]
    s = _SHAPE[kind]
    for mask in (torch.ones(1, dtype=torch.bool), torch.zeros(s[0], 1, 1, 1),
                 torch.tensor(1, dtype=torch.int64), torch.zeros(s[-2], s[-1], dtype=torch.uint8)):
        with pytest.raises(_lib.MriError):
            getattr(d, method)(torch.zeros(s, dtype=_C), mask)
