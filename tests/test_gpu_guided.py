"""Measurement-guided sampling of the 3D LDM on the GPU: the 3-D projector and the image-mask data
term against fp64, the data-gradient-only decoder against the training program and fp32 autograd,
one guided step stage by stage against the fp64 restatement of test_guided_cpu.py, the
guidance_scale = 0 identities with sample() / sample_dpmpp(), replay against the eager loop, data
consistency with random weights, and graph reuse."""
import contextlib
import io

import pytest
import torch

from helpers import rel_l2
from test_guided_cpu import (DIMS3, guided_eps_ref, mask_term_ref, plane_mask, project3d_ref,
                             x0_ref)

pytestmark = pytest.mark.gpu

KERNEL_TOL = 2e-5       # rel-L2 of g against fp64; measured worst 5.15e-7 (DESIGN.md §4)
F32 = 2.0 ** -24


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _gen_offset():
    return torch.cuda.default_generators[torch.cuda.current_device()].get_offset()


def _complete(y, m):
    from mri_image_generation_b200.diffusion_base import kspace_completion
    zf, M = kspace_completion(y, m.expand(y.shape).bool(), dims=DIMS3)
    return zf.float().contiguous(), M.to(torch.uint8).contiguous()


# ------------------------------------------------------------------------------ data-term kernels
def _masks(shape, g):
    B, C, D, H, W = shape
    return {"plane": plane_mask(D, H, g),
            "random": torch.rand(shape, generator=g) < 0.3,
            "per_sample": torch.rand(B, 1, D, H, W, generator=g) < 0.25,
            "per_channel": torch.rand(1, C, D, H, W, generator=g) < torch.linspace(0.1, 0.9, C).view(1, C, 1, 1, 1),
            "zeros": torch.zeros(1, 1, 1, 1, 1, dtype=torch.bool),
            "ones": torch.ones(1, 1, 1, 1, 1, dtype=torch.bool)}


PROJ_SHAPES = [(1, 1, 1, 1, 1), (2, 4, 9, 7, 11), (1, 4, 40, 48, 40), (1, 4, 160, 192, 160)]
_worst = {}


@pytest.mark.parametrize("shape", PROJ_SHAPES)
def test_projector_against_fp64(shape):
    from mri_image_generation_b200 import ops
    g = torch.Generator().manual_seed(sum(shape))
    x_true = torch.randn(shape, generator=g, dtype=torch.float64).cuda()
    u = torch.randn(shape, generator=g).cuda()
    y = torch.fft.fftn(x_true, dim=DIMS3, norm="ortho")
    work = torch.empty(ops.kspace3d_work_bytes(*shape), dtype=torch.uint8, device="cuda")
    for name, m in _masks(shape, g).items():
        zf, M = _complete(y, m.cuda())
        gk = torch.empty_like(u)
        gg = torch.empty(shape[0], device="cuda")
        ops.dc_project3d(u, zf, M, gk, gg, work)
        want, want_gg = project3d_ref(u, zf, M)
        err = rel_l2(gk.double(), want) if want.norm() > 0 else gk.abs().max().item()
        err_gg = ((gg.double() - want_gg).abs() / want_gg.clamp(min=1e-30)).max().item()
        _worst[(shape, name)] = err
        print(f"{shape} {name}: g rel-L2 {err:.2e}, ||g||^2 rel {err_gg:.2e}")
        assert err < KERNEL_TOL, (name, err)
        assert err_gg < 10 * KERNEL_TOL, (name, err_gg)
        g2 = torch.empty_like(u)
        gg2 = torch.empty_like(gg)
        ops.dc_project3d(u, zf, M, g2, gg2, work)
        assert torch.equal(g2, gk) and torch.equal(gg2, gg)          # bit-reproducible
    print(f"worst so far: {max(_worst.values()):.2e}")


def test_image_mask_term_is_exact():
    from mri_image_generation_b200 import ops
    g = torch.Generator().manual_seed(5)
    for shape in [(1, 1, 1, 1, 1), (2, 4, 9, 7, 11), (2, 4, 40, 48, 40)]:
        u, known = torch.randn(shape, generator=g).cuda(), torch.randn(shape, generator=g).cuda()
        for name, m in _masks(shape, g).items():
            mk = m.expand(shape).to(torch.uint8).contiguous().cuda()
            known_nan = torch.where(mk.bool(), torch.nan, known)      # never read where regenerated
            gk, gg = torch.empty_like(u), torch.empty(shape[0], device="cuda")
            ops.dc_mask(u, known_nan, mk, gk, gg)
            assert torch.equal(gk, torch.where(mk.bool(), 0.0, u - known)), name
            want_gg = mask_term_ref(u, known, mk)[1]
            assert ((gg.double() - want_gg).abs() <= 2 * F32 * want_gg).all(), name
            g2, gg2 = torch.empty_like(u), torch.empty_like(gg)
            ops.dc_mask(u, known_nan, mk, g2, gg2)
            assert torch.equal(g2, gk) and torch.equal(gg2, gg)


# ------------------------------------------------------------------------------ dgrad-only decoder
def _vae(seed=0):
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.vae import VAE3D
    torch.manual_seed(seed)
    vae = VAE3D(4, 32, 3, 3)
    with torch.no_grad():
        for p in vae.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    return vae


def test_dgrad_only_decoder():
    from oracle import reference_oracle as O
    vae = _vae()
    sd = {k: v.detach().clone() for k, v in vae.state_dict().items()}
    vae = vae.cuda()
    z = torch.randn(2, 3, 6, 8, 4).cuda()
    full = vae._program("decode", z, training=True)
    dg = vae._program("decode", z, training=True, wgrad=False)
    assert dg is not full and dg.garena is None
    assert len(dg.bwd_ops) < len(full.bwd_ops)
    out_full = full.forward(z).clone()
    dout = torch.randn_like(out_full)
    full.backward(dout)
    dz_full = full.dz_out.clone()
    for _ in range(3):   # eager, then replays of the decoder's own forward graph
        dg.x_in.copy_(z)
        dg.run()
        dg.finish_output()
        dg.dout_in.copy_(dout)
        dg.run_input_backward()
        assert torch.equal(dg.out, out_full) and torch.equal(dg.dz_out, dz_full)
    assert dg.garena is None and all(p.grad is None for p in vae.parameters())
    zr = z.cpu().requires_grad_(True)
    (O.vae3d_decode(sd, zr) * dout.cpu()).sum().backward()
    e = rel_l2(dg.dz_out.cpu(), zr.grad)
    print(f"dgrad-only decoder: dz rel-L2 vs fp32 autograd {e:.3e}")
    assert e < 5e-2


# ------------------------------------------------------------------------------ the guided step
T = 50
LAT = (8, 8, 8)
IMG = (32, 32, 32)


def _setup(B=2, unet_seed=0, eager=False):
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    torch.manual_seed(unet_seed)
    unet = UNet3DModelWithAttention(3, base_channels=64, time_emb_dim=64).cuda().eval()
    model = unet
    if eager:
        class Eager(torch.nn.Module):   # not one of this package's UNets: the eager loop
            def __init__(self):
                super().__init__()
                self.m = unet

            def forward(self, x, t):
                return self.m(x, t)
        model = Eager()
    diff = quiet(GaussianDiffusionLatent3D, model, 3, timesteps=T).cuda()
    return diff, unet


def _measurement(vae, B, seed=3, s=0.8):
    g = torch.Generator().manual_seed(seed)
    z_star = torch.randn(B, 3, *LAT, generator=g).cuda()
    x_star = vae.decode_from_latent(z_star / s)
    y = torch.fft.fftn(x_star.double(), dim=DIMS3, norm="ortho")
    m = plane_mask(IMG[0], IMG[1], g).cuda()
    known_mask = torch.zeros(1, 4, *IMG, dtype=torch.bool)
    known_mask[:, 3] = True                       # FLAIR missing: regenerate it, keep the others
    known_mask[:, :, :, :8] = True                # and a slab of every channel
    return y, m, x_star, known_mask.cuda()


@pytest.mark.parametrize("mode", ["ddpm", "dpmpp"])
def test_one_guided_step_stage_by_stage(mode):
    from mri_image_generation_b200 import ops
    diff, unet = _setup()
    vae = _vae().cuda()
    B, s, lam = 2, 0.8, 1.3
    y, m, _, _ = _measurement(vae, B, s=s)
    zf, M = _complete(y, m)
    dec = vae._program("decode", torch.empty(B, 3, *LAT, device="cuda"), training=True, wgrad=False)
    prog = unet.program(B, LAT)
    b = diff._guided_buffers(prog, dec, True)
    b["zf"].copy_(zf)
    b["mask"].copy_(M)
    b["lam"].fill_(lam)
    b["inv_s"].fill_(1.0 / s)
    inv_s = b["inv_s"].item()
    sa, s1m = diff.sqrt_alphas_cumprod, diff.sqrt_one_minus_alphas_cumprod
    z = torch.randn(B, 3, *LAT, device="cuda")
    t = torch.tensor([37, 12], device="cuda")
    prog.x_in.copy_(z)
    prog.t_in.copy_(t)
    prog.run()
    eps = torch.empty_like(z)
    ops.nhwc_to_nchw(prog.eps_nhwc, eps, B, 512, 3, prog.cout_pad)
    diff._guided_stage(prog.x_in, prog.eps_nhwc, prog.cout_pad, 3, prog.t_in, b)
    # x0 / s: a few fp32 roundings of the operands
    want = x0_ref(z, eps, t, sa, s1m, inv_s)
    bound = 6 * F32 * (z.double().abs() + s1m.double()[t].view(B, 1, 1, 1, 1) * eps.double().abs()) \
        / sa.double()[t].view(B, 1, 1, 1, 1) * inv_s
    err = (dec.x_in.double() - want).abs()
    print(f"x0: max err / bound {(err / bound).max().item():.3f}")
    assert (err <= bound).all()
    # data term on the GPU's decoder output
    g_ref, gg_ref = project3d_ref(dec.out, zf, M)
    print(f"g rel-L2 {rel_l2(dec.dout_in.double(), g_ref):.2e}")
    assert rel_l2(dec.dout_in.double(), g_ref) < KERNEL_TOL
    assert ((b["gg"].double() - gg_ref).abs() / gg_ref).max() < 10 * KERNEL_TOL
    # eps' from the GPU's eps, dz and ||g||^2
    eps2_ref, delta = guided_eps_ref(eps, dec.dz_out, b["gg"], lam, inv_s, t, sa, s1m)
    r = (sa.double()[t] / s1m.double()[t]).view(B, 1, 1, 1, 1)
    bound = 8 * F32 * (eps.double().abs() + (r * delta).abs()) + 1e-30
    err = (b["eps"].double() - eps2_ref).abs()
    print(f"eps': max err / bound {(err / bound).max().item():.3f}, |delta| {delta.abs().max().item():.3e}")
    assert (err <= bound).all() and delta.abs().max() > 0
    # the update reads eps' unchanged: DDPM with explicit noise / DPM-Solver++ row 0
    x = z.clone()
    if mode == "ddpm":
        noise = torch.randn_like(z)
        out = torch.empty_like(z)
        ops.ddpm_step(x, b["eps"], noise, t, diff.betas, s1m, diff.sqrt_recip_alphas,
                      diff.posterior_variance, out)
        tt = t.view(B, 1, 1, 1, 1)
        q = diff.betas.double()[tt] / s1m.double()[tt]
        c1 = diff.sqrt_recip_alphas.double()[tt]
        w = (t != 0).double().view(B, 1, 1, 1, 1) * diff.posterior_variance.double()[tt].sqrt()
        e2 = b["eps"].double()
        want = c1 * (x.double() - q * e2) + w * noise.double()
        bound = 8 * F32 * (c1 * (x.double().abs() + (q * e2).abs()) + (w * noise.double()).abs())
    else:
        ts, coef = diff._dpmpp_table(T - 1, 10)
        c = coef[0].cuda()
        out = torch.empty_like(z)
        ops.dpmpp_step(x, b["eps"], torch.zeros_like(z), c, None, out)
        sc, rc, A, Bc = (c[i].double() for i in range(4))
        x0 = (x.double() - sc * b["eps"].double()) * rc
        want = A * x.double() + Bc * x0
        bound = 8 * F32 * ((A * x.double()).abs() + (Bc * rc).abs() * (x.double().abs() + (sc * b["eps"].double()).abs()))
    err = (out.double() - want).abs()
    print(f"update: max err / bound {(err / bound).max().item():.3f}")
    assert (err <= bound + 1e-30).all()


def _run(diff, kind, dpm, vae, y, m, known, mask, lam, s, seed=11):
    torch.manual_seed(seed)
    if kind == "kspace":
        if dpm:
            return diff.reconstruct_dpmpp(y, m, vae, num_steps=10, guidance_scale=lam, latent_scale=s)
        return diff.reconstruct(y, m, vae, guidance_scale=lam, latent_scale=s)
    if dpm:
        return diff.inpaint_image_dpmpp(known, mask, vae, num_steps=10, guidance_scale=lam, latent_scale=s)
    return diff.inpaint_image(known, mask, vae, guidance_scale=lam, latent_scale=s)


@pytest.mark.parametrize("kind", ["kspace", "mask"])
@pytest.mark.parametrize("dpm", [False, True])
def test_zero_guidance_is_the_plain_sampler(kind, dpm):
    diff, _ = _setup()
    vae = _vae().cuda()
    B, s = 2, 0.8
    y, m, x_star, mask = _measurement(vae, B, s=s)
    got = _run(diff, kind, dpm, vae, y.to(torch.complex64), m, x_star, mask, 0.0, s)
    off_got = _gen_offset()
    torch.manual_seed(11)
    z = diff.sample_dpmpp(B, LAT, num_steps=10) if dpm else diff.sample(B, LAT)
    want = vae.decode_from_latent(z / s)
    assert _gen_offset() == off_got
    assert torch.equal(got, want)


@pytest.mark.parametrize("kind", ["kspace", "mask"])
@pytest.mark.parametrize("dpm", [False, True])
def test_replay_equals_eager(kind, dpm):
    vae = _vae().cuda()
    B, s, lam = 2, 0.8, 0.7
    y, m, x_star, mask = _measurement(vae, B, s=s)
    diff, _ = _setup()
    got = _run(diff, kind, dpm, vae, y, m, x_star, mask, lam, s)
    off = _gen_offset()
    diff_e, _ = _setup(eager=True)
    want = _run(diff_e, kind, dpm, vae, y, m, x_star, mask, lam, s)
    assert _gen_offset() == off
    assert torch.equal(got, want)


def test_guidance_reduces_the_data_residual():
    """With random weights the sampled volume has nothing to do with x*; the guided run must still
    end closer to the measurement.  DPS's normalisation makes each step move the clean latent by
    guidance_scale * ||D^T g|| / (s ||g||), so a visible effect in 10 steps needs a scale of the
    order of the latent's norm (about 40 per sample here), not the default of 1."""
    vae = _vae().cuda()
    B, s, lam = 2, 0.8, 20.0
    y, m, x_star, mask = _measurement(vae, B, s=s)
    diff, _ = _setup()
    _, M = _complete(y, m)

    def kres(x):
        return (M.bool() * (torch.fft.fftn(x.double(), dim=DIMS3, norm="ortho") - y)).abs().norm().item()

    r = {v: kres(_run(diff, "kspace", True, vae, y, m, None, None, v, s)) for v in (0.0, 1.0, lam, 80.0)}
    print("reconstruct_dpmpp: ||M(F x - y)|| by guidance_scale: "
          + ", ".join(f"{k:g}: {v:.4e}" for k, v in r.items()))
    assert r[lam] < r[0.0]

    keep = ~mask.expand(x_star.shape)

    def ires(x):
        return (x - x_star)[keep].double().norm().item()

    i = {v: ires(_run(diff, "mask", False, vae, None, None, x_star, mask, v, s)) for v in (0.0, 1.0, lam, 80.0)}
    print("inpaint_image: kept-region error by guidance_scale: " + ", ".join(f"{k:g}: {v:.4e}" for k, v in i.items()))
    assert i[lam] < i[0.0]


def test_second_call_reuses_the_graph_and_matches_a_fresh_object():
    vae = _vae().cuda()
    B, s, lam = 2, 0.8, 0.9
    y1, m1, _, _ = _measurement(vae, B, seed=3, s=s)
    y2, m2, _, _ = _measurement(vae, B, seed=4, s=s)
    diff, unet = _setup()
    _run(diff, "kspace", True, vae, y1, m1, None, None, lam, s)
    prog = unet.program(B, LAT)
    graph = prog._step_graphs["dpmpp+guided:kspace"][2]
    got = _run(diff, "kspace", True, vae, y2, m2, None, None, lam, s, seed=5)
    assert prog._step_graphs["dpmpp+guided:kspace"][2] is graph
    fresh, _ = _setup()          # the same weights in a new UNet: new programs, a new capture
    want = _run(fresh, "kspace", True, vae, y2, m2, None, None, lam, s, seed=5)
    assert torch.equal(got, want)
