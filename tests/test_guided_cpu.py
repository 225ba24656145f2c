"""Measurement-guided sampling of the 3D LDM through the VAE decoder, on the CPU: the argument
checks and their order (nothing is drawn on a bad call), the 3-D Hermitian completion against fp64
torch.fft (2-D results bit-identical to the 2-D formula), and an fp64 restatement of one guided
step, which tests/test_gpu_guided.py compares the kernels against stage by stage."""
import contextlib
import io
import math

import pytest
import torch

from mri_image_generation_b200 import _lib
from mri_image_generation_b200.diffusion_base import kspace_completion

DIMS3 = (-3, -2, -1)


# ------------------------------------------------------------------------------ fp64 restatement
def x0_ref(z, eps, t, sa, s1m, inv_s):
    """Step 2 divided by the latent scale: (z - s1m[t] eps) / sa[t] * inv_s, fp64."""
    B = z.shape[0]
    a = sa.double()[t].view(B, *([1] * (z.dim() - 1)))
    b = s1m.double()[t].view(B, *([1] * (z.dim() - 1)))
    return (z.double() - b * eps.double()) / a * float(inv_s)


def project3d_ref(u, zf, M):
    """Step 4, k-space: g = Re ifftn(M fftn(u)) - x_zf over (D, H, W), and ||g||^2 per sample."""
    Pu = torch.fft.ifftn(M.to(torch.complex128) * torch.fft.fftn(u.double(), dim=DIMS3, norm="ortho"),
                         dim=DIMS3, norm="ortho").real
    g = Pu - zf.double()
    return g, g.pow(2).flatten(1).sum(1)


def mask_term_ref(u, known, mask):
    """Step 4, image mask (1 = regenerate): g = (1 - mask)(u - x_known), and ||g||^2 per sample."""
    g = torch.where(mask.bool(), 0.0, u.double() - known.double())
    return g, g.pow(2).flatten(1).sum(1)


def guided_eps_ref(eps, dz, gg, lam, inv_s, t, sa, s1m):
    """Steps 5-7: g_z = dz * inv_s, delta = -lam g_z / ||g|| (0 where ||g|| = 0),
    eps' = eps - (sa[t] / s1m[t]) delta; also returns delta."""
    B = eps.shape[0]
    shp = (B,) + (1,) * (eps.dim() - 1)
    nrm = gg.double().clamp(min=0).sqrt().view(shp)
    c = torch.where(nrm > 0, float(lam) / torch.where(nrm > 0, nrm, 1.0), 0.0)
    delta = -c * (dz.double() * float(inv_s))
    r = (sa.double()[t] / s1m.double()[t]).view(shp)
    return eps.double() - r * delta, delta


def hermitian_mask(shape, gen, p=0.3):
    return torch.rand(shape, generator=gen) < p


def plane_mask(D, H, gen, frac=0.3):
    """Phase-encode plane mask (1, 1, D, H, 1): random (D, H) lines plus the centre."""
    m = torch.rand(D, H, generator=gen) < frac
    m[0, 0] = True
    return m.view(1, 1, D, H, 1)


# ------------------------------------------------------------------------------ completion
def test_completion_2d_bit_identical_to_the_2d_formula():
    g = torch.Generator().manual_seed(0)
    for shape in [(2, 3, 7, 9), (1, 1, 8, 6), (2, 1, 1, 1)]:
        y = torch.randn(shape, generator=g, dtype=torch.complex128)
        m = torch.rand(shape, generator=g) < 0.4
        mir = lambda a: torch.roll(torch.flip(a, (-2, -1)), (1, 1), (-2, -1))
        full = m | mir(m)
        yy = torch.where(m, y, torch.where(full, mir(y).conj(), torch.zeros_like(y)))
        want = torch.fft.ifft2(yy, norm="ortho").real
        zf, M = kspace_completion(y, m)
        assert torch.equal(M, full) and torch.equal(zf, want)


@pytest.mark.parametrize("shape", [(1, 1, 1, 1, 1), (2, 4, 9, 7, 11), (1, 2, 8, 6, 10)])
def test_completion_3d_against_fp64_fft(shape):
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(shape, generator=g, dtype=torch.float64)
    y = torch.fft.fftn(x, dim=DIMS3, norm="ortho")
    m = hermitian_mask(shape, g)
    zf, M = kspace_completion(y, m, dims=DIMS3)
    # M is m completed by its mirror k -> -k over (D, H, W)
    neg = lambda a: torch.roll(torch.flip(a, DIMS3), (1, 1, 1), DIMS3)
    assert torch.equal(M, m | neg(m)) and torch.equal(M, neg(M))
    # y of a real image is Hermitian, so the completion is M y and x_zf = P x
    want = torch.fft.ifftn(M * y, dim=DIMS3, norm="ortho")
    assert want.imag.abs().max() < 1e-12
    assert (zf - want.real).abs().max() < 1e-12
    # P is the orthogonal projector with x_zf in its range, and P x_true = x_zf
    P = lambda u: project3d_ref(u, torch.zeros_like(u), M)[0]
    assert (P(zf) - zf).abs().max() < 1e-12
    v = torch.randn(shape, generator=g, dtype=torch.float64)
    assert abs((P(x) * v).sum() - (x * P(v)).sum()) < 1e-10


# ------------------------------------------------------------------------------ one guided step
def test_data_terms_are_the_gradients_of_the_residuals():
    g = torch.Generator().manual_seed(1)
    shape = (2, 3, 6, 5, 8)
    x = torch.randn(shape, generator=g, dtype=torch.float64)
    y = torch.fft.fftn(x, dim=DIMS3, norm="ortho")
    zf, M = kspace_completion(y, hermitian_mask(shape, g), dims=DIMS3)
    u = torch.randn(shape, generator=g, dtype=torch.float64, requires_grad=True)
    res = M * (torch.fft.fftn(u, dim=DIMS3, norm="ortho") - y)
    (0.5 * res.abs().pow(2).sum()).backward()
    gk, ggk = project3d_ref(u.detach(), zf, M)
    assert (gk - u.grad).abs().max() < 1e-10
    assert torch.allclose(ggk, res.detach().abs().pow(2).flatten(1).sum(1), rtol=1e-10)
    # image mask: g = grad of 1/2 ||(1 - mask)(u - x_known)||^2
    mask = torch.rand(shape, generator=g) < 0.5
    known = torch.randn(shape, generator=g, dtype=torch.float64)
    u.grad = None
    (0.5 * ((~mask) * (u - known)).pow(2).sum()).backward()
    gm, ggm = mask_term_ref(u.detach(), known, mask)
    assert torch.equal(gm, u.grad) and torch.allclose(ggm, gm.pow(2).flatten(1).sum(1))


def test_guided_eps_moves_the_clean_estimate_by_delta():
    from mri_image_generation_b200 import schedules
    b = schedules.make_buffers(schedules.cosine_beta_schedule(100, 0.008), with_snr=True)
    sa, s1m = b["sqrt_alphas_cumprod"], b["sqrt_one_minus_alphas_cumprod"]
    g = torch.Generator().manual_seed(2)
    shape = (3, 3, 4, 5, 6)
    z, eps, dz = (torch.randn(shape, generator=g, dtype=torch.float64) for _ in range(3))
    t = torch.tensor([99, 40, 0])
    gg = torch.tensor([4.0, 0.0, 0.25], dtype=torch.float64)
    inv_s = 1 / 0.7
    eps2, delta = guided_eps_ref(eps, dz, gg, 1.5, inv_s, t, sa, s1m)
    x0 = x0_ref(z, eps, t, sa, s1m, 1.0)
    x0_new = x0_ref(z, eps2, t, sa, s1m, 1.0)
    assert (x0_new - (x0 + delta)).abs().max() < 1e-10
    assert torch.equal(eps2[1], eps[1])                       # ||g|| = 0: no move
    n0 = delta[0].norm() / (dz[0].norm() * inv_s)
    assert abs(n0 - 1.5 / 2.0) < 1e-12                        # DPS normalisation: lam / ||g||
    assert torch.equal(guided_eps_ref(eps, dz, gg, 0.0, inv_s, t, sa, s1m)[0], eps.double())


# ------------------------------------------------------------------------------ argument checks
def _objects(T=20):
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.vae import VAE3D
    torch.manual_seed(0)
    unet = UNet3DModelWithAttention(3, base_channels=32, time_emb_dim=32)
    with contextlib.redirect_stdout(io.StringIO()):
        diff = GaussianDiffusionLatent3D(unet, 3, timesteps=T)
    return diff, VAE3D(4, 32, 3, 3)


def test_argument_errors_in_order_before_any_draw():
    diff, vae = _objects()
    ks = torch.zeros(1, 4, 8, 8, 8, dtype=torch.complex64)
    xk = torch.zeros(1, 4, 8, 8, 8)
    m = torch.ones(1, 1, 8, 8, 1, dtype=torch.bool)
    lin = torch.nn.Linear(2, 2)
    state = torch.get_rng_state()
    cases = [
        # guidance / scale first, whatever else is wrong
        (ValueError, "guidance_scale", lambda: diff.reconstruct(None, None, None, guidance_scale=-1.0)),
        (ValueError, "guidance_scale", lambda: diff.inpaint_image(xk, m, vae, guidance_scale=math.nan)),
        (ValueError, "latent_scale", lambda: diff.reconstruct(ks, m, None, latent_scale=0.0)),
        (ValueError, "latent_scale", lambda: diff.reconstruct_dpmpp(ks, m, vae, latent_scale=math.inf)),
        # then the VAE
        (_lib.MriError, "VAE3D", lambda: diff.reconstruct(ks, m, object())),
        (_lib.MriError, "VAE3D", lambda: diff.inpaint_image(None, m, lin)),
        # then shapes and masks
        (ValueError, "kspace", lambda: diff.reconstruct(xk, m, vae)),                   # not complex
        (ValueError, "x_known", lambda: diff.inpaint_image(ks, m, vae)),                # complex
        (ValueError, "kspace", lambda: diff.reconstruct(ks[:, :3], m, vae)),            # channels
        (ValueError, "kspace", lambda: diff.reconstruct(ks[0], m, vae)),                # rank
        (ValueError, "divisible", lambda: diff.reconstruct(ks[..., :6], m[..., :6, :], vae)),
        (ValueError, "broadcast", lambda: diff.reconstruct(ks, torch.ones(2, 1, 8, 8, 1), vae)),
        (ValueError, "0 / 1", lambda: diff.inpaint_image(xk, torch.full((1, 1, 8, 8, 8), 2.0), vae)),
        (ValueError, "num_steps", lambda: diff.reconstruct_dpmpp(ks, m, vae, num_steps=0)),
        (ValueError, "num_steps", lambda: diff.inpaint_image_dpmpp(xk, m, vae, num_steps=20)),
        # then the device
        (_lib.MriError, "B200", lambda: diff.reconstruct(ks, m, vae)),
        (_lib.MriError, "B200", lambda: diff.inpaint_image_dpmpp(xk, m, vae, num_steps=5)),
    ]
    for exc, text, call in cases:
        with pytest.raises(exc, match=text):
            call()
    assert torch.equal(torch.get_rng_state(), state)


def test_work_size_limit():
    from mri_image_generation_b200 import ops
    try:
        _lib.load()
    except Exception:
        pytest.skip("library not built")
    assert ops.kspace3d_work_bytes(1, 1, 1, 1, 1) > 0
    for shp in [(1, 1, 513, 8, 8), (1, 1, 8, 513, 8), (1, 1, 8, 8, 513)]:
        with pytest.raises(_lib.MriError, match="512"):
            ops.kspace3d_work_bytes(*shp)
