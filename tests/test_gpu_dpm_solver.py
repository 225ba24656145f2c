"""DPM-Solver++(2M) on the GPU: mri_dpmpp_step / mri_step_table_advance against a torch fp32
restatement, the solver's order on Gaussian data with the exact noise prediction, and the
replayed step graph (fused and unfused, bf16 and split precision) against the step-by-step loop,
bit for bit."""
import contextlib
import io
import math

import pytest
import torch

from helpers import shapes_of, synthetic_state_dict

pytestmark = pytest.mark.gpu


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _table(T=1000, M=10, kind="cosine"):
    from mri_image_generation_b200 import schedules
    betas = (schedules.cosine_beta_schedule(T) if kind == "cosine"
             else schedules.linear_beta_schedule(T, 1e-4, 0.02))
    ac = schedules.make_buffers(betas, True)["alphas_cumprod"]
    return schedules.dpmpp_2m_table(ac, schedules.dpmpp_timesteps(T - 1, M))


def _ref_step(x, e, x0p, row):
    """The step in torch fp32, one rounding per operation (eager kernels never contract)."""
    s, r, A, B, C = (row[i] for i in range(5))
    x0 = (x - s * e) * r
    out = A * x + B * x0
    if C.item() != 0.0:
        out = out + C * (x0 - x0p)
    return out, x0


# ------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("shape", [(3, 1, 7, 9), (2, 4, 33, 31), (2, 3, 5, 6, 7), (1, 3, 8, 12, 8),
                                   (5, 1, 1, 1), (2, 2, 240, 241)])
@pytest.mark.parametrize("layout", ["f32", "nhwc"])
@pytest.mark.parametrize("inplace", [False, True])
def test_dpmpp_step_kernel_bit_exact(shape, layout, inplace):
    from mri_image_generation_b200 import ops
    g = torch.Generator().manual_seed(sum(shape) + len(layout) + inplace)
    _, coef_cpu = _table(M=10)
    coef = coef_cpu.cuda()
    B, C = shape[0], shape[1]
    S = math.prod(shape[2:])
    x = torch.randn(shape, generator=g).cuda()
    if layout == "f32":
        eps, ldc = torch.randn(shape, generator=g).cuda(), 0
        e = eps
    else:
        ldc = 16 if C < 16 else C + 8
        eps = torch.randn(B, S, ldc, generator=g).to(torch.bfloat16).cuda()
        e = eps[..., :C].float().permute(0, 2, 1).reshape(shape).contiguous()
    for row in (0, 3, 9):          # first order (C = 0), second order, the step to sigma = 0
        x0p = torch.randn(shape, generator=g).cuda()
        if row == 0:
            x0p.fill_(float("nan"))   # must not be read on a C = 0 row
        want, want_x0 = _ref_step(x, e, x0p, coef[row])
        k = torch.tensor([row], dtype=torch.int64, device="cuda")
        xin = x.clone()
        out = xin if inplace else torch.full_like(x, float("nan"))
        xp = x0p.clone()
        ops.dpmpp_step(xin, eps, xp, coef, k, out, eps_nhwc_ldc=ldc, channels=C if ldc else 0)
        assert torch.isfinite(out).all(), row
        assert torch.equal(out, want), (row, (out - want).abs().max().item())
        assert torch.equal(xp, want_x0), row
        if not inplace:
            assert torch.equal(xin, x)
        if row == 9:   # the last row returns the data prediction exactly
            assert torch.equal(out, want_x0)
        # k = None is row 0
        if row == 0:
            out2, xp2 = torch.empty_like(x), torch.full_like(x, float("nan"))
            ops.dpmpp_step(x, eps, xp2, coef, None, out2, eps_nhwc_ldc=ldc, channels=C if ldc else 0)
            assert torch.equal(out2, want)


def test_dpmpp_step_unaligned_views():
    """Views that start off a 16-byte boundary take the scalar path and stay exact."""
    from mri_image_generation_b200 import ops
    _, coef = _table(M=10)
    coef = coef.cuda()
    g = torch.Generator().manual_seed(5)
    base = torch.randn(4 * 1001 + 1, generator=g).cuda()
    x = base[1:].view(4, 1, 7, 143)
    e = torch.randn(4, 1, 7, 143, generator=g).cuda()
    x0p = torch.randn(4 * 1001 + 3, generator=g).cuda()[3:].view(4, 1, 7, 143)
    want, want_x0 = _ref_step(x, e, x0p, coef[4])
    k = torch.tensor([4], device="cuda")
    out = torch.empty_like(x)
    ops.dpmpp_step(x, e, x0p, coef, k, out)
    assert torch.equal(out, want) and torch.equal(x0p, want_x0)


@pytest.mark.parametrize("n", [1, 3, 255, 256, 257, 1000])
def test_step_table_advance_clamps_at_the_last_row(n):
    from mri_image_generation_b200 import ops
    ts = torch.tensor([900, 700, 400, 123, 55], dtype=torch.int64, device="cuda")
    t = torch.full((n,), -5, dtype=torch.int64, device="cuda")
    k = torch.zeros(1, dtype=torch.int64, device="cuda")
    for step in range(1, 8):
        ops.step_table_advance(t, k, ts, 4)          # rows = 4: entry 4 is never used
        assert k.item() == step
        assert (t == ts[min(step, 3)]).all(), (step, t.unique().tolist())


# ------------------------------------------------------------------------------------------ order
class _GaussEps(torch.nn.Module):
    """The exact noise prediction for data ~ N(mu, sd^2) elementwise:
    eps(x, t) = sigma (x - alpha mu) / (alpha^2 sd^2 + sigma^2), computed in fp64."""

    def __init__(self, ac, mu, sd):
        super().__init__()
        self.register_buffer("ac", ac.double())
        self.mu, self.sd = mu, sd

    def forward(self, x, t):
        a2 = self.ac[t].view(-1, *([1] * (x.dim() - 1)))
        a, s = a2.sqrt(), (1 - a2).sqrt()
        return (s * (x.double() - a * self.mu) / (a2 * self.sd ** 2 + s * s)).float()


def _exact(ac, x_T, t0, t1, mu, sd):
    """Probability-flow ODE endpoint at t1 (-1: sigma = 0) from x_T at t0."""
    a0 = float(ac[t0])
    z = (x_T.double() - math.sqrt(a0) * mu) / math.sqrt(a0 * sd ** 2 + 1 - a0)
    if t1 < 0:
        return mu + sd * z
    a1 = float(ac[t1])
    return math.sqrt(a1) * mu + math.sqrt(a1 * sd ** 2 + 1 - a1) * z


def _rel(a, b):
    return ((a.double() - b).norm() / b.norm()).item()


def test_second_order_convergence_on_gaussian_data():
    from mri_image_generation_b200 import schedules
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    mu, sd, T = 0.3, 0.5, 1000
    diff = quiet(GaussianDiffusionLatent3D, torch.nn.Identity(), 4, timesteps=T).cuda()
    ac = diff.alphas_cumprod
    diff.model = _GaussEps(ac, mu, sd).cuda()
    x_T = torch.randn(4, 4, 64, 64, 16, generator=torch.Generator().manual_seed(0)).cuda()   # 2^20
    exact = _exact(ac.double().cpu(), x_T, 999, 100, mu, sd)

    def err(M, first_order=False):
        ts_list = [int(v) for v in torch.linspace(999, 100, M + 1, dtype=torch.float64).round()]
        ts, coef = schedules.dpmpp_2m_table(ac, ts_list)
        if first_order:
            coef = coef.clone()
            coef[:, 4] = 0
        out = diff._sample_dpmpp(x_T, (ts, coef), None, lambda x, t: diff.model(x, t))
        return _rel(out, exact)

    e40, e80 = err(40), err(80)
    f40, f80 = err(40, True), err(80, True)
    print(f"2M: e40 {e40:.3e} e80 {e80:.3e} ratio {e40 / e80:.2f}; "
          f"first order: {f40:.3e} {f80:.3e} ratio {f40 / f80:.2f}")
    assert e40 / e80 >= 3.0 and e80 <= 3e-4
    assert 1.8 <= f40 / f80 <= 2.2
    # the public sampler: 20 calls from t = 999 to sigma = 0
    got = diff.sample_from_dpmpp(x_T, 999, 20)
    e = _rel(got, _exact(ac.double().cpu(), x_T, 999, -1, mu, sd))
    print(f"sample_from_dpmpp(x_T, 999, 20): {e:.3e}")
    assert e <= 1e-2


# ------------------------------------------------------------------------------------------ loops
def _eager_loop(diff, x, start_t, M, eps_fn):
    """The step-by-step loop: model call, then ops.dpmpp_step with that step's row."""
    from mri_image_generation_b200 import ops, schedules
    ts, coef = schedules.dpmpp_2m_table(diff.alphas_cumprod, schedules.dpmpp_timesteps(start_t, M))
    coef = coef.cuda()
    img = x.clone()
    x0p = torch.full_like(img, float("nan"))
    with torch.no_grad():
        for i, t in enumerate(ts.tolist()):
            tt = torch.full((img.shape[0],), t, device="cuda", dtype=torch.long)
            eps = eps_fn(img, tt)
            ops.dpmpp_step(img, eps.float().contiguous(), x0p, coef, torch.tensor([i], device="cuda"), img)
    return img


def _unet3d(seed, attn=False):
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet import UNet3DModel
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    m = (UNet3DModelWithAttention if attn else UNet3DModel)(3, base_channels=64, time_emb_dim=64)
    m.load_state_dict(synthetic_state_dict(shapes_of(m), seed=seed))
    return m.cuda().eval()


def _diff3d(m, T):
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    return quiet(GaussianDiffusionLatent3D, m, 3, timesteps=T).cuda()


def test_graph_loop_equals_eager_3d():
    m = _unet3d(81)
    T = 50
    diff = _diff3d(m, T)
    x = torch.randn(2, 3, 8, 12, 8, generator=torch.Generator().manual_seed(3)).cuda()
    for start_t in (T - 1, 23):
        for M in (1, 5, 7):
            got = diff.sample_from_dpmpp(x, start_t, M)
            want = _eager_loop(diff, x, start_t, M, lambda a, t: m(a, t))
            assert torch.isfinite(got).all()
            assert torch.equal(got, want), (start_t, M, (got - want).abs().max().item())
    prog = next(iter(m._programs().values()))
    assert "dpmpp" in prog._step_graphs


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


@pytest.mark.parametrize("kind", ["2d", "25d"])
def test_graph_loop_equals_eager_2d(kind):
    m, mk = _model2d(kind, 82)
    T, B, M = 40, 3, 6
    diff = mk(m, T)
    z = torch.tensor([0.1, 0.5, 0.9], device="cuda")
    if kind == "2d":
        shape = (B, 1, 40, 40)
        run = lambda: diff.sample_dpmpp(B, z_pos=z, num_steps=M)
        eps_fn = lambda a, t: m(a, t, z)
    else:
        shape = (B, 4, 24, 24)
        ctx = torch.randn(B, 16, 24, 24, generator=torch.Generator().manual_seed(1)).cuda()
        run = lambda: diff.sample_dpmpp(B, z_pos=z, context=ctx, num_steps=M)
        eps_fn = lambda a, t: m(a, t, z, context=ctx)
    torch.manual_seed(21)
    got = run()
    torch.manual_seed(21)
    x_T = torch.randn(shape, device="cuda")
    want = _eager_loop(diff, x_T, T - 1, M, eps_fn)
    assert got.shape == shape and torch.isfinite(got).all()
    assert torch.equal(got, want), (got - want).abs().max().item()


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_fused_dpmpp_step_equals_unfused_bit_exactly(kind, monkeypatch):
    """mri_tap_gather_step mode 3 (out_conv finished inside the update) against the forward's own
    tap gather followed by mri_dpmpp_step on the bf16 channels-last eps."""
    if kind == "3d":
        m = _unet3d(91)
        mk = lambda mm: _diff3d(mm, 12)
        run = lambda d: d.sample_dpmpp(2, (8, 12, 8), num_steps=6)
    else:
        m, mk2 = _model2d(kind, 91)
        mk = lambda mm: mk2(mm, 12)
        if kind == "2d":
            run = lambda d: d.sample_dpmpp(3, z_pos=0.3, num_steps=6)
        else:
            ctx = torch.randn(2, 16, 24, 24, generator=torch.Generator().manual_seed(1)).cuda()
            run = lambda d: d.sample_dpmpp(2, z_pos=0.6, context=ctx, num_steps=6)
    outs = []
    for fused in ("1", "0"):
        monkeypatch.setenv("MRI_FUSED_STEP", fused)
        m.__dict__.pop("_mri_programs", None)      # fresh program: fresh step graph
        torch.manual_seed(17)
        outs.append(run(mk(m)).clone())
        prog = next(iter(m._programs().values()))
        assert prog.fused_head is not None and "dpmpp" in prog._step_graphs
    assert torch.isfinite(outs[0]).all()
    assert torch.equal(outs[0], outs[1]), (outs[0] - outs[1]).abs().max().item()


def test_split_precision_graph_equals_eager():
    m = _unet3d(62)
    m.precision = "split"
    diff = _diff3d(m, 30)
    x = torch.randn(2, 3, 8, 8, 8, generator=torch.Generator().manual_seed(8)).cuda()
    got = diff.sample_from_dpmpp(x, 29, 5)
    prog = next(iter(m._programs().values()))
    assert prog.fused_head is None and prog.cout_pad == 0 and "dpmpp" in prog._step_graphs
    want = _eager_loop(diff, x, 29, 5, lambda a, t: m(a, t))
    assert torch.isfinite(got).all()
    assert torch.equal(got, want), (got - want).abs().max().item()


def test_generator_draws_only_x_T():
    m = _unet3d(83)
    diff = _diff3d(m, 20)
    torch.manual_seed(99)
    got = diff.sample_dpmpp(2, (8, 8, 8), num_steps=4)
    after = torch.randn(7, device="cuda")
    torch.manual_seed(99)
    x_T = torch.randn(2, 3, 8, 8, 8, device="cuda")
    assert torch.equal(after, torch.randn(7, device="cuda"))
    assert torch.equal(got, diff.sample_from_dpmpp(x_T, 19, 4))
    assert torch.equal(got, _eager_loop(diff, x_T, 19, 4, lambda a, t: m(a, t)))


def test_one_graph_serves_every_num_steps_and_follows_new_weights():
    m = _unet3d(84)
    T = 40
    diff = _diff3d(m, T)
    x = torch.randn(2, 3, 8, 8, 8, generator=torch.Generator().manual_seed(4)).cuda()
    res, graphs = {}, []
    for M in (10, 20, 10):
        res.setdefault(M, []).append(diff.sample_from_dpmpp(x, T - 1, M))
        prog = next(iter(m._programs().values()))
        graphs.append(prog._step_graphs["dpmpp"][2])
    assert graphs[0] is graphs[1] is graphs[2]
    assert torch.equal(res[10][0], res[10][1])
    for M in (10, 20):
        m.__dict__.pop("_mri_programs", None)
        assert torch.equal(diff.sample_from_dpmpp(x, T - 1, M), res[M][0]), M
    # new weights: the program refreshes its packed weights, the replayed graph follows
    m.load_state_dict(synthetic_state_dict(shapes_of(m), seed=85))
    got = diff.sample_from_dpmpp(x, T - 1, 10)
    assert not torch.equal(got, res[10][0])
    m.__dict__.pop("_mri_programs", None)
    assert torch.equal(got, diff.sample_from_dpmpp(x, T - 1, 10))
    assert torch.equal(got, _eager_loop(diff, x, T - 1, 10, lambda a, t: m(a, t)))


def test_cfg4_shape_graph_equals_eager():
    """The benchmarked model and latent shape (attention UNet, base 128, 3x40x48x40) at B = 2."""
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    torch.manual_seed(0)
    m = UNet3DModelWithAttention(in_channels=3, base_channels=128, channel_mults=(1, 2, 4),
                                 time_emb_dim=256, groups=8, num_heads=4).cuda().eval()
    diff = _diff3d(m, 1000)
    torch.manual_seed(5)
    got = diff.sample_dpmpp(2, (40, 48, 40), num_steps=3)
    torch.manual_seed(5)
    x_T = torch.randn(2, 3, 40, 48, 40, device="cuda")
    want = _eager_loop(diff, x_T, 999, 3, lambda a, t: m(a, t))
    assert torch.isfinite(got).all()
    assert torch.equal(got, want), (got - want).abs().max().item()
