"""Inpainting on the GPU: mri_inpaint_merge against torch.where over mri_q_sample, the replayed
inpainting loops (fused and unfused, bf16 and split precision) against eager sequences of the
public ops, bit for bit, the invariants of the method, graph reuse, and the conditioning check of
test_inpaint_cpu.py through the eager path on the real kernels."""
import contextlib
import io
import math

import pytest
import torch

from helpers import shapes_of, synthetic_state_dict
from test_inpaint_cpu import corr_eps, gaussian_problem, region_error

pytestmark = pytest.mark.gpu


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _gen_offset():
    return torch.cuda.default_generators[torch.cuda.current_device()].get_offset()


# ------------------------------------------------------------------------------------------ kernel
def _sched():
    from mri_image_generation_b200 import schedules
    b = schedules.make_buffers(schedules.cosine_beta_schedule(1000), True)
    return b["sqrt_alphas_cumprod"].cuda(), b["sqrt_one_minus_alphas_cumprod"].cuda()


def _ref_merge(x, known, keep_mask, tau, noise, sac, s1m):
    """torch.where(mask, x, kn), kn = known (tau < 0) or mri_q_sample(known, tau, noise), per sample."""
    from mri_image_generation_b200 import ops
    qs = torch.empty_like(known)
    ops.q_sample(known.contiguous(), noise.contiguous(), tau.clamp(min=0), sac, s1m, qs)
    neg = (tau < 0).view(-1, *([1] * (x.dim() - 1)))
    kn = torch.where(neg, known, qs)
    return torch.where(keep_mask.bool(), x, kn)


def _masks(shape, g):
    B, C = shape[0], shape[1]
    sp = shape[2:]
    chan = torch.zeros(1, C, *([1] * len(sp)), dtype=torch.bool)
    chan[0, C - 1] = True
    box = torch.zeros(1, 1, *sp, dtype=torch.bool)
    box[(0, 0) + tuple(slice(s // 4, max(s // 4 + 1, 3 * s // 4)) for s in sp)] = True
    per_sample = torch.zeros(B, *([1] * (len(shape) - 1)), dtype=torch.bool)
    per_sample[::2] = True
    rand = torch.rand(shape, generator=g) < 0.5
    return {"channel": chan, "box": box, "per_sample": per_sample, "random": rand}


SHAPES = [(3, 1, 7, 9), (2, 4, 33, 31), (2, 3, 5, 6, 7), (1, 3, 8, 12, 8), (5, 1, 1, 1),
          (2, 2, 240, 241), (4, 3, 16, 16, 16)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("source", ["philox", "tensor"])
def test_merge_kernel_bit_exact(shape, source):
    from mri_image_generation_b200 import ops
    sac, s1m = _sched()
    g = torch.Generator().manual_seed(sum(shape) + len(source))
    B = shape[0]
    known = torch.randn(shape, generator=g).cuda()
    x0 = torch.randn(shape, generator=g).cuda()
    inc = ops.randn_offset_increment(x0.numel())
    taus = [torch.tensor([(7 * b + 3) % 1000 for b in range(B)]),   # mixed timesteps
            torch.tensor([0] + [999] * (B - 1)),                     # t = 0 with t_delta = -1: tau = -1
            torch.full((B,), -1)]
    for name, mask in _masks(shape, g).items():
        for ti, tv in enumerate(taus):
            for delta in (0, -1):
                t = tv.cuda()
                tau = t + delta
                keep = mask.expand(shape).cuda()          # True = regenerate: x is kept there
                # NaN where the merge must not read: known under the mask, x outside it
                kn_in = torch.where(keep, torch.full_like(known, float("nan")), known)
                x_in = torch.where(keep, x0, torch.full_like(x0, float("nan")))
                m8 = keep.to(torch.uint8).contiguous()
                if source == "philox":
                    seed = 1000 * ti + 7
                    torch.manual_seed(seed)
                    torch.randn_like(x0)                  # the update's own draw, skipped
                    noise = torch.randn_like(x0)
                    rng = ops.DeviceRng(x0.device)
                    torch.manual_seed(seed)
                    rng.load()
                    got = x_in.clone()
                    ops.inpaint_merge(got, kn_in, m8, t, delta, sac, s1m, rng=rng, rng_skip=inc)
                else:
                    noise = torch.randn(shape, generator=g).cuda()
                    got = x_in.clone()
                    ops.inpaint_merge(got, kn_in, m8, t, delta, sac, s1m, noise=noise)
                want = _ref_merge(x_in, known, keep, tau, noise, sac, s1m)
                assert torch.isfinite(got).all(), (name, ti, delta)
                assert torch.equal(got, want), (name, ti, delta, (got - want).abs().max().item())
                if (tau < 0).all():
                    assert torch.equal(got, torch.where(keep, x0, known))


def test_merge_kernel_philox_draw_is_randn_like_after_the_skip():
    """With known = 0, sqrt_ac = 0 and sqrt_1mac = 1 the merge writes its noise itself."""
    from mri_image_generation_b200 import ops
    x = torch.zeros(3, 3, 10, 11, 12, device="cuda")
    ones, zeros = torch.ones(1000, device="cuda"), torch.zeros(1000, device="cuda")
    t = torch.full((3,), 5, dtype=torch.int64, device="cuda")
    m8 = torch.zeros(x.shape, dtype=torch.uint8, device="cuda")
    inc = ops.randn_offset_increment(x.numel())
    rng = ops.DeviceRng(x.device)
    for skip in (0, inc, 3 * inc):
        torch.manual_seed(11)
        for _ in range(skip // inc):
            torch.randn_like(x)
        want = torch.randn_like(x)
        torch.manual_seed(11)
        rng.load()
        got = torch.empty_like(x)
        ops.inpaint_merge(got, torch.zeros_like(x), m8, t, 0, zeros, ones, rng=rng, rng_skip=skip)
        assert torch.equal(got, want), skip


def test_merge_kernel_unaligned_views():
    """Views off a 16-byte (x, known) or 4-byte (mask) boundary take the scalar path."""
    from mri_image_generation_b200 import ops
    sac, s1m = _sched()
    g = torch.Generator().manual_seed(5)
    shape = (4, 1, 7, 143)
    n = math.prod(shape)
    x = torch.randn(n + 1, generator=g).cuda()[1:].view(shape)
    known = torch.randn(n + 3, generator=g).cuda()[3:].view(shape)
    keep = (torch.rand(shape, generator=g) < 0.3).cuda()
    m8 = torch.zeros(n + 1, dtype=torch.uint8, device="cuda")[1:].view(shape)
    m8.copy_(keep)
    noise = torch.randn(n + 2, generator=g).cuda()[2:].view(shape)
    t = torch.tensor([10, 500, 0, 999], device="cuda")
    want = _ref_merge(x, known, keep, t - 1, noise, sac, s1m)
    ops.inpaint_merge(x, known, m8, t, -1, sac, s1m, noise=noise)
    assert torch.equal(x, want)


# ------------------------------------------------------------------------------------------ models
def _unet3d(seed, attn=False):
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet import UNet3DModel
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    m = (UNet3DModelWithAttention if attn else UNet3DModel)(3, base_channels=64, time_emb_dim=64)
    m.load_state_dict(synthetic_state_dict(shapes_of(m), seed=seed))
    return m.cuda().eval()


def _diff3d(m, T):
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    return quiet(GaussianDiffusionLatent3D, m, 3, timesteps=T).cuda()


def _model2d(kind, seed):
    if kind == "2d":
        from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion
        from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet
        m = quiet(UNet, img_channels=1, base_channels=64, time_emb_dim=64)
        mk = lambda mm, T: quiet(GaussianDiffusion, mm, 40, channels=1, timesteps=T).cuda()
    else:
        from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.diffusion import GaussianDiffusion
        from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.unet import UNet
        m = quiet(UNet, in_channels=20, out_channels=4, base_channels=64, time_emb_dim=64)
        mk = lambda mm, T: quiet(GaussianDiffusion, mm, 24, channels=4, timesteps=T).cuda()
    m.load_state_dict(synthetic_state_dict(shapes_of(m), seed=seed))
    return m.cuda().eval(), mk


def _case(kind, T, seed=91):
    """(model, diffusion, x_known, mask, eps_fn, inpaint(method, **kw), sample(method, **kw))."""
    g = torch.Generator().manual_seed(seed)
    if kind in ("3d", "3d_attn", "3d_split"):
        m = _unet3d(seed, attn=kind == "3d_attn")
        if kind == "3d_split":
            m.precision = "split"
        diff = _diff3d(m, T)
        shape = (2, 3, 8, 12, 8)
        mask = torch.zeros(1, 1, 8, 12, 8, dtype=torch.bool)
        mask[..., 2:6, 3:9, 2:6] = True                      # regenerate a box
        eps_fn = lambda a, t: m(a, t)
        inp = lambda meth, xk, mk, **kw: getattr(diff, meth)(xk, mk, **kw)
        smp = lambda meth, **kw: getattr(diff, meth)(shape[0], shape[2:], **kw)
    else:
        m, mk = _model2d(kind, seed)
        diff = mk(m, T)
        z = torch.tensor([0.2, 0.7], device="cuda")
        if kind == "2d":
            shape = (2, 1, 40, 40)
            mask = torch.zeros(1, 1, 40, 40, dtype=torch.bool)
            mask[..., 10:30, 5:25] = True
            eps_fn = lambda a, t: m(a, t, z)
            inp = lambda meth, xk, mk, **kw: getattr(diff, meth)(xk, mk, z_pos=z, **kw)
            smp = lambda meth, **kw: getattr(diff, meth)(shape[0], z_pos=z, **kw)
        else:
            shape = (2, 4, 24, 24)
            mask = torch.tensor([False, False, False, True]).view(1, 4, 1, 1)   # impute flair
            ctx = torch.randn(2, 16, 24, 24, generator=g).cuda()
            eps_fn = lambda a, t: m(a, t, z, context=ctx)
            inp = lambda meth, xk, mk, **kw: getattr(diff, meth)(xk, mk, z_pos=z, context=ctx, **kw)
            smp = lambda meth, **kw: getattr(diff, meth)(shape[0], z_pos=z, context=ctx, **kw)
    x_known = torch.randn(shape, generator=g).cuda()
    return m, diff, x_known, mask.cuda(), eps_fn, inp, smp


def _ref_ddpm(diff, eps_fn, x_known, mask, seed):
    """The DDPM inpainting sequence with the public ops, torch.randn_like and torch.where."""
    from mri_image_generation_b200 import ops
    B, T = x_known.shape[0], diff.timesteps
    torch.manual_seed(seed)
    x = torch.randn(x_known.shape, device="cuda")
    with torch.no_grad():
        for i in reversed(range(T)):
            t = torch.full((B,), i, device="cuda", dtype=torch.long)
            eps = eps_fn(x, t).float().contiguous()
            z = torch.randn_like(x)
            out = torch.empty_like(x)
            ops.ddpm_step(x, eps, z, t, diff.betas, diff.sqrt_one_minus_alphas_cumprod,
                          diff.sqrt_recip_alphas, diff.posterior_variance, out)
            n = torch.randn_like(out)
            kn = x_known if i == 0 else diff.q_sample(x_known, t - 1, noise=n)
            x = torch.where(mask, out, kn)
    return x


def _ref_dpmpp(diff, eps_fn, x_known, mask, seed, M):
    from mri_image_generation_b200 import ops, schedules
    B, T = x_known.shape[0], diff.timesteps
    ts, coef = schedules.dpmpp_2m_table(diff.alphas_cumprod, schedules.dpmpp_timesteps(T - 1, M))
    coef = coef.cuda()
    torch.manual_seed(seed)
    x_T = torch.randn(x_known.shape, device="cuda")
    x, x0p = x_T.clone(), torch.full_like(x_T, float("nan"))
    taus = ts.tolist()[1:] + [-1]
    with torch.no_grad():
        for i, t in enumerate(ts.tolist()):
            tt = torch.full((B,), t, device="cuda", dtype=torch.long)
            eps = eps_fn(x, tt).float().contiguous()
            ops.dpmpp_step(x, eps, x0p, coef, torch.tensor([i], device="cuda"), x)
            tau = taus[i]
            kn = x_known if tau < 0 else diff.q_sample(
                x_known, torch.full((B,), tau, device="cuda", dtype=torch.long), noise=x_T)
            x = torch.where(mask, x, kn)
    return x


def _check(got, want, x_known, mask):
    assert torch.isfinite(got).all()
    assert torch.equal(got, want), (got - want).abs().max().item()
    keep = ~mask.expand(x_known.shape)
    assert torch.equal(got[keep], x_known[keep])


@pytest.mark.parametrize("kind", ["3d", "3d_attn", "2d", "25d", "3d_split"])
@pytest.mark.parametrize("fused", ["1", "0"])
def test_replayed_loops_equal_eager_sequences(kind, fused, monkeypatch):
    monkeypatch.setenv("MRI_FUSED_STEP", fused)
    m, diff, x_known, mask, eps_fn, inp, _ = _case(kind, 12)
    torch.manual_seed(31)
    got = inp("inpaint", x_known, mask)
    off = _gen_offset()
    prog = next(iter(m._programs().values()))
    assert "ddpm+inpaint" in prog._step_graphs
    assert (prog.fused_head is not None) == (kind != "3d_split")
    want = _ref_ddpm(diff, eps_fn, x_known, mask, 31)
    _check(got, want, x_known, mask)
    assert _gen_offset() == off

    torch.manual_seed(32)
    got = inp("inpaint_dpmpp", x_known, mask, num_steps=6)
    off = _gen_offset()
    prog = next(iter(m._programs().values()))
    assert "dpmpp+inpaint" in prog._step_graphs
    want = _ref_dpmpp(diff, eps_fn, x_known, mask, 32, 6)
    _check(got, want, x_known, mask)
    assert _gen_offset() == off


def test_cfg4_shape_loops_equal_eager():
    """The benchmarked model and latent shape (attention UNet, base 128, 3x40x48x40) at B = 2."""
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    torch.manual_seed(0)
    m = UNet3DModelWithAttention(in_channels=3, base_channels=128, channel_mults=(1, 2, 4),
                                 time_emb_dim=256, groups=8, num_heads=4).cuda().eval()
    g = torch.Generator().manual_seed(6)
    x_known = torch.randn(2, 3, 40, 48, 40, generator=g).cuda()
    mask = torch.zeros(2, 1, 40, 48, 40, dtype=torch.bool)
    mask[0, :, 10:30, 12:36, 10:30] = True       # a box in sample 0
    mask[1, :, :, :, 20:] = True                 # a half volume in sample 1
    mask = mask.cuda()
    eps_fn = lambda a, t: m(a, t)
    diff = _diff3d(m, 4)
    torch.manual_seed(5)
    got = diff.inpaint(x_known, mask)
    _check(got, _ref_ddpm(diff, eps_fn, x_known, mask, 5), x_known, mask)
    diff = _diff3d(m, 1000)
    torch.manual_seed(5)
    got = diff.inpaint_dpmpp(x_known, mask, num_steps=3)
    _check(got, _ref_dpmpp(diff, eps_fn, x_known, mask, 5, 3), x_known, mask)


# ------------------------------------------------------------------------------------------ invariants
@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_all_false_mask_returns_x_known(kind):
    m, diff, x_known, mask, _, inp, _ = _case(kind, 12)
    none = torch.zeros_like(mask)
    assert torch.equal(inp("inpaint", x_known, none), x_known)
    assert torch.equal(inp("inpaint_dpmpp", x_known, none, num_steps=5), x_known)


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_all_true_mask_dpmpp_equals_sample_dpmpp(kind):
    m, diff, x_known, mask, _, inp, smp = _case(kind, 30)
    torch.manual_seed(77)
    want = smp("sample_dpmpp", num_steps=7)
    off = _gen_offset()
    torch.manual_seed(77)
    got = inp("inpaint_dpmpp", torch.full_like(x_known, float("nan")), torch.ones_like(mask),
              num_steps=7)
    assert torch.equal(got, want), (got - want).abs().max().item()
    assert _gen_offset() == off


@pytest.mark.parametrize("kind", ["3d", "2d"])
def test_generator_offsets(kind):
    from mri_image_generation_b200 import ops
    m, diff, x_known, mask, _, inp, _ = _case(kind, 9)
    inc = ops.randn_offset_increment(x_known.numel())
    for _ in range(2):            # first call captures the graph, the second replays it
        torch.manual_seed(3)
        o0 = _gen_offset()
        inp("inpaint", x_known, mask)
        assert _gen_offset() - o0 == (1 + 2 * 9) * inc
        torch.manual_seed(3)
        inp("inpaint_dpmpp", x_known, mask, num_steps=4)
        assert _gen_offset() - o0 == inc


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_bad_arguments_leave_the_cuda_generator_untouched(kind):
    m, diff, x_known, mask, _, inp, _ = _case(kind, 12)
    B, C = x_known.shape[:2]
    bad = [(x_known[:, :1] if C > 1 else torch.cat([x_known, x_known], 1), mask),   # channels
           (x_known[0], mask),                                                      # rank
           (x_known, torch.ones(B + 1, *x_known.shape[1:], dtype=torch.bool, device="cuda")),
           (x_known, torch.full_like(x_known, 0.5)),                                # not 0 / 1
           (x_known, torch.full(x_known.shape, 2, dtype=torch.int64, device="cuda"))]
    torch.manual_seed(5)
    off = _gen_offset()
    for xk, mk in bad:
        for method in ("inpaint", "inpaint_dpmpp"):
            with pytest.raises(ValueError):
                inp(method, xk, mk)
    for num_steps in (0, 12):
        with pytest.raises(ValueError):
            inp("inpaint_dpmpp", x_known, mask, num_steps=num_steps)
    assert _gen_offset() == off


# ------------------------------------------------------------------------------------------ graph reuse
def test_one_graph_serves_every_input_and_leaves_the_plain_samplers_alone():
    m, diff, x_known, mask, eps_fn, _, _ = _case("3d", 20, seed=84)
    shape = x_known.shape
    # the plain samplers alone, on a fresh program
    torch.manual_seed(1)
    plain = diff.sample(2, shape[2:])
    torch.manual_seed(2)
    plain_dpm = diff.sample_dpmpp(2, shape[2:], num_steps=8)
    m.__dict__.pop("_mri_programs", None)

    g = torch.Generator().manual_seed(9)
    xk2 = torch.randn(shape, generator=g).cuda()
    mask2 = (torch.rand(shape[0], 1, *shape[2:], generator=g) < 0.5).cuda()
    graphs = {}
    for i, (xk, mk, M) in enumerate([(x_known, mask, 5), (xk2, mask2, 9), (x_known, mask, 5)]):
        torch.manual_seed(10 + i)
        got = diff.inpaint(xk, mk)
        _check(got, _ref_ddpm(diff, eps_fn, xk, mk, 10 + i), xk, mk)
        torch.manual_seed(20 + i)
        got = diff.inpaint_dpmpp(xk, mk, num_steps=M)
        _check(got, _ref_dpmpp(diff, eps_fn, xk, mk, 20 + i, M), xk, mk)
        prog = next(iter(m._programs().values()))
        for key in ("ddpm+inpaint", "dpmpp+inpaint"):
            graphs.setdefault(key, []).append(prog._step_graphs[key][2])
    for key, gs in graphs.items():
        assert gs[0] is gs[1] is gs[2], key
    # the plain samplers after inpainting, on the same program
    torch.manual_seed(1)
    assert torch.equal(diff.sample(2, shape[2:]), plain)
    torch.manual_seed(2)
    assert torch.equal(diff.sample_dpmpp(2, shape[2:], num_steps=8), plain_dpm)


# ------------------------------------------------------------------------------------------ conditioning
class _CorrEps(torch.nn.Module):
    """The exact eps of test_inpaint_cpu.py's correlated Gaussian data, for (B, 1, D, H, W) states."""

    def __init__(self, ac):
        super().__init__()
        self.register_buffer("ac", ac.double())

    def forward(self, x, t):
        B = x.shape[0]
        return corr_eps(x.double().reshape(B, -1), self.ac[t]).float().reshape(x.shape)


def test_conditioning_through_the_eager_path():
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    B, vol = 32, (16, 8, 8)
    diff = quiet(GaussianDiffusionLatent3D, torch.nn.Identity(), 1, timesteps=1000).cuda()
    diff.model = _CorrEps(diff.alphas_cumprod).cuda()
    known, mask, post = gaussian_problem(B, math.prod(vol), 0)
    xk = known.float().reshape(B, 1, *vol).cuda()
    mk = mask.reshape(B, 1, *vol).cuda()
    res = {}
    for name, free, inp in [("ddpm", lambda: diff.sample(B, vol), lambda: diff.inpaint(xk, mk)),
                            ("dpmpp", lambda: diff.sample_dpmpp(B, vol, num_steps=20),
                             lambda: diff.inpaint_dpmpp(xk, mk, num_steps=20))]:
        torch.manual_seed(4)
        x_free = free()
        torch.manual_seed(4)
        x_inp = inp()
        assert torch.equal(x_inp[~mk], xk[~mk])
        e_free = region_error(x_free.reshape(B, -1).cpu(), mask, post)
        e_inp = region_error(x_inp.reshape(B, -1).cpu(), mask, post)
        res[name] = e_free / e_inp
        print(f"{name}: unconditional {e_free:.4g}, inpainted {e_inp:.4g}, ratio {res[name]:.1f}")
    assert res["ddpm"] >= 50 and res["dpmpp"] >= 5
