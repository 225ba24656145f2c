"""RePaint resampling on the GPU: mri_repaint_undo against the torch expression, the replayed
RePaint loops (fused and unfused, bf16 and split precision) and the eager loop against eager
sequences of public ops, bit for bit, generator bookkeeping, graph reuse, and the conditioning
check of test_repaint_cpu.py through the eager path on the real kernels."""
import math

import pytest
import torch

from test_gpu_inpaint import SHAPES, _case, _check, _CorrEps, _diff3d, _gen_offset, _unet3d, quiet
from test_inpaint_cpu import gaussian_problem, region_error

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------ kernel
def _tables():
    from mri_image_generation_b200 import schedules
    b = schedules.make_buffers(schedules.cosine_beta_schedule(1000), True)
    return b["alphas"].cuda(), b["betas"].cuda()


def _ref_undo(x, t, alphas, betas, z):
    """alphas[l + 1].sqrt() * x + betas[l + 1].sqrt() * z per sample, eager torch."""
    view = (-1,) + (1,) * (x.dim() - 1)
    return alphas[t + 1].sqrt().view(view) * x + betas[t + 1].sqrt().view(view) * z


def _levels(B):
    """mixed per-sample levels with both ends of the range, -1 and T - 2"""
    return torch.tensor([[-1, 998, (37 * b) % 998][b % 3] for b in range(B)], device="cuda")


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("source", ["philox", "tensor"])
def test_undo_kernel_bit_exact(shape, source):
    from mri_image_generation_b200 import ops
    alphas, betas = _tables()
    g = torch.Generator().manual_seed(sum(shape) + len(source))
    x0 = torch.randn(shape, generator=g).cuda()
    inc = ops.randn_offset_increment(x0.numel())
    for t in (_levels(shape[0]), torch.full((shape[0],), -1, device="cuda"),
              torch.full((shape[0],), 998, device="cuda")):
        for skip in ((0, inc, 2 * inc) if source == "philox" else (0,)):
            if source == "philox":
                torch.manual_seed(21)
                for _ in range(skip // inc):
                    torch.randn_like(x0)
                z = torch.randn_like(x0)
                rng = ops.DeviceRng(x0.device)
                torch.manual_seed(21)
                rng.load()
                got = x0.clone()
                ops.repaint_undo(got, t, alphas, betas, rng=rng, rng_skip=skip)
            else:
                z = torch.randn(shape, generator=g).cuda()
                got = x0.clone()
                ops.repaint_undo(got, t, alphas, betas, noise=z)
            want = _ref_undo(x0, t, alphas, betas, z)
            assert torch.equal(got, want), (t.tolist(), skip, (got - want).abs().max().item())


def test_undo_kernel_philox_draw_is_randn_like_after_the_skip():
    """With alphas = 0 and betas = 1 the undo writes its noise itself."""
    from mri_image_generation_b200 import ops
    x = torch.randn(3, 3, 10, 11, 12, device="cuda")
    zeros, ones = torch.zeros(1000, device="cuda"), torch.ones(1000, device="cuda")
    t = torch.tensor([-1, 4, 998], device="cuda")
    inc = ops.randn_offset_increment(x.numel())
    rng = ops.DeviceRng(x.device)
    for skip in (0, inc, 3 * inc):
        torch.manual_seed(11)
        for _ in range(skip // inc):
            torch.randn_like(x)
        want = torch.randn_like(x)
        torch.manual_seed(11)
        rng.load()
        got = x.clone()
        ops.repaint_undo(got, t, zeros, ones, rng=rng, rng_skip=skip)
        assert torch.equal(got, want), skip


def test_undo_kernel_unaligned_views():
    """Views off a 16-byte boundary take the scalar path."""
    from mri_image_generation_b200 import ops
    alphas, betas = _tables()
    g = torch.Generator().manual_seed(5)
    shape = (4, 1, 7, 143)
    n = math.prod(shape)
    x = torch.randn(n + 1, generator=g).cuda()[1:].view(shape)
    noise = torch.randn(n + 2, generator=g).cuda()[2:].view(shape)
    t = torch.tensor([10, 500, -1, 998], device="cuda")
    want = _ref_undo(x, t, alphas, betas, noise)
    ops.repaint_undo(x, t, alphas, betas, noise=noise)
    assert torch.equal(x, want)
    torch.manual_seed(8)
    z = torch.randn_like(x)
    want = _ref_undo(x, t, alphas, betas, z)
    rng = ops.DeviceRng(x.device)
    torch.manual_seed(8)
    rng.load()
    ops.repaint_undo(x, t, alphas, betas, rng=rng)
    assert torch.equal(x, want)


def test_undo_kernel_argument_checks():
    from mri_image_generation_b200 import _lib, ops
    alphas, betas = _tables()
    x = torch.zeros(2, 8, device="cuda")
    t = torch.zeros(2, dtype=torch.int64, device="cuda")
    rng = ops.DeviceRng(x.device)
    with pytest.raises(_lib.MriError):      # neither source
        ops.repaint_undo(x, t, alphas, betas)
    with pytest.raises(_lib.MriError):      # both
        ops.repaint_undo(x, t, alphas, betas, noise=torch.zeros_like(x), rng=rng)
    with pytest.raises(_lib.MriError):
        ops.repaint_undo(x, t, alphas, betas, rng=rng, rng_skip=2)


# ------------------------------------------------------------------------------------------ loops
def _ref_repaint(diff, eps_fn, x_known, mask, seed, levels):
    """The RePaint walk with the public ops, torch.randn_like and torch.where."""
    from mri_image_generation_b200 import ops
    B = x_known.shape[0]
    torch.manual_seed(seed)
    x = torch.randn(x_known.shape, device="cuda")
    with torch.no_grad():
        for lv, nxt in zip(levels, levels[1:]):
            t = torch.full((B,), lv, device="cuda", dtype=torch.long)
            if nxt < lv:
                eps = eps_fn(x, t).float().contiguous()
                z = torch.randn_like(x)
                out = torch.empty_like(x)
                ops.ddpm_step(x, eps, z, t, diff.betas, diff.sqrt_one_minus_alphas_cumprod,
                              diff.sqrt_recip_alphas, diff.posterior_variance, out)
                n = torch.randn_like(out)
                kn = x_known if lv == 0 else diff.q_sample(x_known, t - 1, noise=n)
                x = torch.where(mask, out, kn)
            else:
                z = torch.randn_like(x)
                x = diff.alphas[lv + 1].sqrt() * x + diff.betas[lv + 1].sqrt() * z
    return x


def _draws(levels):
    """x_T, two draws per reverse step and one per undo step"""
    n_rev = sum(b < a for a, b in zip(levels, levels[1:]))
    return 1 + 2 * n_rev + (len(levels) - 1 - n_rev)


@pytest.mark.parametrize("kind", ["3d", "3d_attn", "2d", "25d", "3d_split"])
@pytest.mark.parametrize("fused", ["1", "0"])
def test_replayed_repaint_equals_eager_sequence(kind, fused, monkeypatch):
    from mri_image_generation_b200 import ops, schedules
    monkeypatch.setenv("MRI_FUSED_STEP", fused)
    m, diff, x_known, mask, eps_fn, inp, _ = _case(kind, 12)
    inc = ops.randn_offset_increment(x_known.numel())
    graphs = []
    for seed, (L, r) in ((41, (3, 3)), (42, (1, 2))):   # the first call captures, the second replays
        levels = schedules.repaint_levels(12, L, r)
        torch.manual_seed(seed)
        o0 = _gen_offset()
        got = inp("inpaint", x_known, mask, jump_length=L, jump_n_sample=r)
        assert _gen_offset() - o0 == _draws(levels) * inc
        prog = next(iter(m._programs().values()))
        assert (prog.fused_head is not None) == (kind != "3d_split")
        graphs.append((prog._step_graphs["ddpm+inpaint"][2], prog._step_graphs["repaint-undo"][2]))
        _check(got, _ref_repaint(diff, eps_fn, x_known, mask, seed, levels), x_known, mask)
    assert graphs[0][0] is graphs[1][0] and graphs[0][1] is graphs[1][1]


class _Plain(torch.nn.Module):
    """The same UNet behind a module that is not one of this package's: the eager loop."""

    def __init__(self, m):
        super().__init__()
        self.inner = m

    def forward(self, x, t):
        return self.inner(x, t)


def test_eager_repaint_equals_eager_sequence():
    from mri_image_generation_b200 import ops, schedules
    m = _unet3d(93)
    diff = _diff3d(_Plain(m), 12)
    g = torch.Generator().manual_seed(3)
    x_known = torch.randn(2, 3, 8, 12, 8, generator=g).cuda()
    mask = (torch.rand(2, 1, 8, 12, 8, generator=g) < 0.5).cuda()
    inc = ops.randn_offset_increment(x_known.numel())
    for L, r in ((3, 3), (1, 2)):
        levels = schedules.repaint_levels(12, L, r)
        torch.manual_seed(17)
        o0 = _gen_offset()
        got = diff.inpaint(x_known, mask, jump_length=L, jump_n_sample=r)
        assert _gen_offset() - o0 == _draws(levels) * inc
        for prog in m._programs().values():                 # no step graph: the eager loop ran
            assert not prog.__dict__.get("_step_graphs")
        _check(got, _ref_repaint(diff, lambda a, t: m(a, t), x_known, mask, 17, levels), x_known, mask)


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_no_jumps_is_plain_inpaint(kind):
    m, diff, x_known, mask, _, inp, _ = _case(kind, 12)
    torch.manual_seed(61)
    want = inp("inpaint", x_known, mask)
    off = _gen_offset()
    for kw in (dict(jump_n_sample=1), dict(jump_length=3, jump_n_sample=1),
               dict(jump_length=12, jump_n_sample=3), dict(jump_length=50, jump_n_sample=2)):
        torch.manual_seed(61)
        got = inp("inpaint", x_known, mask, **kw)
        assert torch.equal(got, want), kw
        assert _gen_offset() == off, kw
    prog = next(iter(m._programs().values()))
    assert "repaint-undo" not in prog._step_graphs


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_bad_jump_arguments_leave_the_cuda_generator_untouched(kind):
    m, diff, x_known, mask, _, inp, _ = _case(kind, 12)
    torch.manual_seed(5)
    off = _gen_offset()
    for kw in (dict(jump_length=0, jump_n_sample=2), dict(jump_length=2.5, jump_n_sample=2),
               dict(jump_length=3, jump_n_sample=0), dict(jump_length=3, jump_n_sample=None)):
        with pytest.raises(ValueError):
            inp("inpaint", x_known, mask, **kw)
    assert _gen_offset() == off


def test_graphs_serve_every_input_and_leave_the_other_samplers_alone():
    from mri_image_generation_b200 import schedules
    m, diff, x_known, mask, eps_fn, _, _ = _case("3d", 20, seed=84)
    shape = x_known.shape
    # the plain samplers and plain inpainting alone, on a fresh program
    torch.manual_seed(1)
    plain = diff.sample(2, shape[2:])
    torch.manual_seed(2)
    plain_dpm = diff.sample_dpmpp(2, shape[2:], num_steps=8)
    torch.manual_seed(3)
    plain_inp = diff.inpaint(x_known, mask)
    m.__dict__.pop("_mri_programs", None)

    g = torch.Generator().manual_seed(9)
    xk2 = torch.randn(shape, generator=g).cuda()
    mask2 = (torch.rand(shape[0], 1, *shape[2:], generator=g) < 0.5).cuda()
    graphs = []
    for i, (xk, mk, L, r) in enumerate([(x_known, mask, 4, 2), (xk2, mask2, 1, 3), (x_known, mask, 7, 2)]):
        torch.manual_seed(10 + i)
        got = diff.inpaint(xk, mk, jump_length=L, jump_n_sample=r)
        _check(got, _ref_repaint(diff, eps_fn, xk, mk, 10 + i, schedules.repaint_levels(20, L, r)), xk, mk)
        prog = next(iter(m._programs().values()))
        graphs.append(tuple(prog._step_graphs[k][2] for k in ("ddpm+inpaint", "repaint-undo")))
    assert all(gs[0] is graphs[0][0] and gs[1] is graphs[0][1] for gs in graphs)
    # the other samplers after RePaint, on the same program
    torch.manual_seed(1)
    assert torch.equal(diff.sample(2, shape[2:]), plain)
    torch.manual_seed(2)
    assert torch.equal(diff.sample_dpmpp(2, shape[2:], num_steps=8), plain_dpm)
    torch.manual_seed(3)
    assert torch.equal(diff.inpaint(x_known, mask), plain_inp)
    assert next(iter(m._programs().values()))._step_graphs["ddpm+inpaint"][2] is graphs[0][0]


def test_cfg4_shape_repaint_equals_eager():
    """The benchmarked model and latent shape (attention UNet, base 128, 3x40x48x40) at B = 2."""
    from mri_image_generation_b200 import schedules
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
    diff = _diff3d(m, 4)
    torch.manual_seed(5)
    got = diff.inpaint(x_known, mask, jump_length=1, jump_n_sample=2)
    want = _ref_repaint(diff, lambda a, t: m(a, t), x_known, mask, 5, schedules.repaint_levels(4, 1, 2))
    _check(got, want, x_known, mask)


# ------------------------------------------------------------------------------------------ conditioning
def test_conditioning_through_the_eager_path():
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    B, vol = 32, (16, 8, 8)
    diff = quiet(GaussianDiffusionLatent3D, torch.nn.Identity(), 1, timesteps=1000).cuda()
    diff.model = _CorrEps(diff.alphas_cumprod).cuda()
    known, mask, post = gaussian_problem(B, math.prod(vol), 0)
    xk = known.float().reshape(B, 1, *vol).cuda()
    mk = mask.reshape(B, 1, *vol).cuda()
    torch.manual_seed(4)
    e_free = region_error(diff.sample(B, vol).reshape(B, -1).cpu(), mask, post)
    ratio = {}
    for name, kw in (("replacement", {}), ("repaint", dict(jump_length=10, jump_n_sample=2))):
        torch.manual_seed(4)
        x = diff.inpaint(xk, mk, **kw)
        assert torch.equal(x[~mk], xk[~mk])
        e = region_error(x.reshape(B, -1).cpu(), mask, post)
        ratio[name] = e_free / e
        print(f"{name}: unconditional {e_free:.4g}, inpainted {e:.4g}, ratio {ratio[name]:.1f}")
    assert ratio["repaint"] >= 100 and ratio["repaint"] > ratio["replacement"]
