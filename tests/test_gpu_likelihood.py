"""The variational bound on the GPU: mri_vb_terms against an fp64 oracle with injected z and eps,
the replayed 'vb' loop against an eager fp64 restatement of improved-diffusion's formulas (means
form) with the same torch.randn_like draws, the eager path against the replayed path, the
alignment of t and the noise, the benchmarked cfg4 shape, and graph reuse."""
import math

import pytest
import torch

from test_gpu_inpaint import _diff3d, _gen_offset, _model2d, _ref_ddpm, _unet3d, quiet
from test_likelihood_cpu import discretized_nll64, gaussian_nll64, kl_means, sched64

pytestmark = pytest.mark.gpu


def _bufs(T=1000, cosine=True):
    from mri_image_generation_b200 import schedules
    betas = schedules.cosine_beta_schedule(T) if cosine else schedules.linear_beta_schedule(T, 1e-4, 0.02)
    return {k: v.cuda() for k, v in schedules.make_buffers(betas, True).items()}


def _sched_args(b):
    return (b["betas"], b["sqrt_one_minus_alphas_cumprod"], b["sqrt_recip_alphas"],
            b["posterior_variance"], b["posterior_log_variance_clipped"])


def _mu0(b, x_t, eps):
    """The t = 0 mean as mri_ddpm_step computes it (w = 0 there), fp32."""
    from mri_image_generation_b200 import ops
    t = torch.zeros(x_t.shape[0], dtype=torch.int64, device="cuda")
    out = torch.empty_like(x_t)
    ops.ddpm_step(x_t.contiguous(), eps.contiguous(), torch.zeros_like(x_t), t, b["betas"],
                  b["sqrt_one_minus_alphas_cumprod"], b["sqrt_recip_alphas"], b["posterior_variance"], out)
    return out


def _nll(decoder, x0, mu, b):
    ls = float(0.5 * b["posterior_log_variance_clipped"][0].item())   # 0.5 * fp32 is exact
    f = discretized_nll64 if decoder == 0 else gaussian_nll64
    return f(x0.double(), mu.double(), ls)


def _unaligned(t):
    """A contiguous copy of t whose data pointer is 4 bytes off a 16-byte boundary."""
    flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)[1:]
    flat.copy_(t.reshape(-1))
    return flat.view(t.shape)


# ------------------------------------------------------------------------------------------ kernel
SHAPES = [(3, 1, 7, 9), (2, 3, 5, 6, 7), (4, 4, 16, 16), (2, 3, 8, 12, 8), (5, 1, 1, 1)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("decoder", [0, 1])
@pytest.mark.parametrize("layout", ["fp32", "fp32_unaligned", "bf16_nhwc"])
def test_vb_terms_kernel_against_fp64(shape, decoder, layout):
    from mri_image_generation_b200 import ops
    b = _bufs()
    B, C, T = shape[0], shape[1], 1000
    g = torch.Generator().manual_seed(sum(shape) + 7 * decoder + len(layout))
    x0 = torch.rand(shape, generator=g) * 2.4 - 1.2               # beyond [-1, 1] too
    flat = x0.view(-1)
    edge = torch.tensor([-1.0, 1.0, -0.9995, 0.9995, -1.2, 1.2, -0.999, 0.999])
    k = min(flat.numel(), edge.numel())
    flat[:k] = edge[:k]                                           # exactly +-1, the edges and beyond
    flat[-k:] = edge[:k]
    x0 = x0.cuda()
    z = torch.randn(shape, generator=g).cuda()
    eps = (z.cpu() + torch.randn(shape, generator=g)).cuda()     # mu - x0 straddles the bin half-width
    t = torch.tensor([[0, 5, 0, T - 1, 1][n % 5] for n in range(B)], device="cuda")
    x_t = torch.empty_like(x0)
    ops.q_sample(x0, z, t, b["sqrt_alphas_cumprod"], b["sqrt_one_minus_alphas_cumprod"], x_t)
    kw = {}
    if layout == "bf16_nhwc":
        ldc = 8
        nhwc = torch.full((B, *shape[2:], ldc), float("nan"), dtype=torch.bfloat16, device="cuda")
        nhwc[..., :C] = eps.movedim(1, -1).to(torch.bfloat16)
        eps = nhwc[..., :C].movedim(-1, 1).float().contiguous()  # the values the kernel reads
        eps_in, kw = nhwc, dict(eps_nhwc_ldc=ldc, channels=C)
    elif layout == "fp32_unaligned":
        eps_in = _unaligned(eps)
        x0, x_t, z = _unaligned(x0), _unaligned(x_t), _unaligned(z)
    else:
        eps_in = eps
    acc0 = torch.randn(B, T, 2, dtype=torch.float64, generator=g).cuda()
    prior0 = torch.randn(B, dtype=torch.float64, generator=g).cuda()
    acc, prior = acc0.clone(), prior0.clone()
    ops.vb_terms(x0, x_t, eps_in, z, t, *_sched_args(b), acc, prior, decoder, **kw)

    want, want_p = acc0.clone(), prior0.clone()
    mu = _mu0(b, x_t, eps)
    nll = _nll(decoder, x0, mu, b)
    for n in range(B):
        tn = int(t[n])
        want[n, tn, 0] += ((eps[n].double() - z[n].double()) ** 2).sum()
        if tn == 0:
            want[n, 0, 1] += nll[n].sum()
            want_p[n] += (x0[n].double() ** 2).sum()
    diff = (acc - want).abs()
    bound = 1e-6 * (want - acc0).abs() + 1e-12
    assert (diff <= bound).all(), (diff / (want - acc0).abs().clamp(min=1e-300)).max().item()
    assert ((prior - want_p).abs() <= 1e-6 * (want_p - prior0).abs() + 1e-12).all()
    sel = nll[t == 0]
    if decoder == 0 and sel.numel() >= 64:   # elements inside and outside their bin were summed
        assert (sel < 1e-6).any() and (sel > 27).any()
    # without prior: acc is the same
    acc2 = acc0.clone()
    ops.vb_terms(x0, x_t, eps_in, z, t, *_sched_args(b), acc2, None, decoder, **kw)
    assert ((acc2 - want).abs() <= bound).all()


def test_vb_terms_ignores_out_of_range_timesteps():
    from mri_image_generation_b200 import ops
    b = _bufs(12)
    x = torch.randn(3, 2, 4, 4, device="cuda")
    acc = torch.zeros(3, 12, 2, dtype=torch.float64, device="cuda")
    t = torch.tensor([-1, 12, 3], device="cuda")
    ops.vb_terms(x, x, torch.ones_like(x), torch.zeros_like(x), t, *_sched_args(b), acc, None, 0)
    want = torch.zeros_like(acc)
    want[2, 3, 0] = x[2].numel()
    assert torch.equal(acc, want)


# ------------------------------------------------------------------------------------------ loops
def _case(kind, T, seed=91):
    """(model, diffusion, x_start, eps_fn, bpd(x_start, model=None) -> dict, decoder)."""
    g = torch.Generator().manual_seed(seed)
    if kind in ("3d", "3d_attn", "3d_split"):
        m = _unet3d(seed, attn=kind == "3d_attn")
        if kind == "3d_split":
            m.precision = "split"
        diff = _diff3d(m, T)
        x0 = torch.randn(2, 3, 8, 12, 8, generator=g).cuda()
        eps_fn = lambda a, t: m(a, t)
        bpd = lambda x: diff.calc_bpd_loop(x)
        return m, diff, x0, eps_fn, bpd, 1
    m, mk = _model2d(kind, seed)
    diff = mk(m, T)
    z = torch.tensor([0.2, 0.7], device="cuda")
    shape = (2, 1, 40, 40) if kind == "2d" else (2, 4, 24, 24)
    x0 = (torch.rand(shape, generator=g) * 2 - 1).cuda()
    x0.view(-1)[:4] = torch.tensor([-1.0, 1.0, -1.0, 1.0])
    if kind == "2d":
        eps_fn = lambda a, t: m(a, t, z)
        bpd = lambda x: diff.calc_bpd_loop(x, z)
    else:
        ctx = torch.randn(2, 16, 24, 24, generator=g).cuda()
        eps_fn = lambda a, t: m(a, t, z, context=ctx)
        bpd = lambda x: diff.calc_bpd_loop(x, z, context=ctx)
    return m, diff, x0, eps_fn, bpd, 0


def _ref_bpd(diff, eps_fn, x0, seed, decoder):
    """improved-diffusion's calc_bpd_loop restated in fp64, means form, for t = T - 1 ... 0 with
    z = torch.randn_like(x0) and eps = eps_fn(q_sample(x0, t, z), t) on the fp32 x_t the model
    sees.  The KL's x_t is formed in fp64 from the same x0 and z, so that fp32 rounding of x_t does
    not swamp the difference of the two means."""
    B, T, N = x0.shape[0], diff.timesteps, x0[0].numel()
    s = {k: v.cuda() for k, v in sched64(diff.betas).items()}
    b = {k: getattr(diff, k) for k in ("betas", "sqrt_one_minus_alphas_cumprod", "sqrt_recip_alphas",
                                       "posterior_variance", "posterior_log_variance_clipped")}
    vb = torch.zeros(B, T, dtype=torch.float64, device="cuda")
    mse = torch.zeros_like(vb)
    torch.manual_seed(seed)
    with torch.no_grad():
        for i in reversed(range(T)):
            t = torch.full((B,), i, device="cuda", dtype=torch.long)
            z = torch.randn_like(x0)
            x_t = diff.q_sample(x0, t, noise=z)
            eps = eps_fn(x_t, t).float().contiguous()
            d = lambda v: v.double().reshape(B, -1)
            mse[:, i] = ((d(eps) - d(z)) ** 2).sum(1) / N
            if i >= 1:
                vb[:, i] = kl_means(s, i, d(x0), d(z), d(eps))
            else:
                vb[:, 0] = _nll(decoder, x0, _mu0(b, x_t, eps), b).reshape(B, -1).sum(1)
    a = s["ac"][T - 1]
    prior = 0.5 * (-1.0 - torch.log1p(-a) + (1.0 - a) + a * x0.double().reshape(B, -1) ** 2).sum(1)
    scale = 1.0 / (N * math.log(2.0))
    return {"total_bpd": (prior + vb.sum(1)) * scale, "prior_bpd": prior * scale, "vb": vb * scale,
            "mse": mse}


def _close(got, want, rel):
    for k in ("total_bpd", "prior_bpd", "vb", "mse"):
        g, w = got[k], want[k]
        assert g.dtype == torch.float64 and g.is_cuda and g.shape == w.shape, k
        err = ((g - w).abs() / w.abs().clamp(min=1e-300)).max().item()
        assert err <= rel, (k, err)


@pytest.mark.parametrize("kind", ["3d", "3d_attn", "2d", "25d", "3d_split"])
def test_replayed_loop_equals_the_fp64_restatement(kind):
    from mri_image_generation_b200 import ops
    m, diff, x0, eps_fn, bpd, dec = _case(kind, 12)
    torch.manual_seed(31)
    o0 = _gen_offset()
    got = bpd(x0)
    off = _gen_offset()
    assert off - o0 == 12 * ops.randn_offset_increment(x0.numel())
    prog = next(iter(m._programs().values()))
    assert "vb" in prog._step_graphs
    assert (prog.fused_head is not None) == (kind != "3d_split")
    want = _ref_bpd(diff, eps_fn, x0, 31, dec)
    assert _gen_offset() == off
    _close(got, want, 1e-5)
    assert torch.isfinite(got["total_bpd"]).all()


class _Wrap(torch.nn.Module):
    """Not an EngineModule: the diffusion classes run the eager path around it."""

    def __init__(self, m):
        super().__init__()
        self.m = m

    def forward(self, x, t, *a, **k):
        return self.m(x, t, *a, **k)


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_eager_path_equals_replayed_path(kind):
    m, diff, x0, eps_fn, bpd, _ = _case(kind, 12)
    torch.manual_seed(7)
    replayed = bpd(x0)
    off = _gen_offset()
    diff.model = _Wrap(m)
    torch.manual_seed(7)
    eager = bpd(x0)
    assert _gen_offset() == off
    _close(eager, replayed, 1e-12)


class _TrueNoise(torch.nn.Module):
    """eps = (x_t - sqrt(ac[t + shift]) x0) / sqrt(1 - ac[t + shift]): the exact noise at shift 0."""

    def __init__(self, diff, x0, shift):
        super().__init__()
        self.diff, self.x0, self.shift = diff, x0, shift

    def forward(self, x, t):
        T = self.diff.timesteps
        ts = (t + self.shift).clamp(0, T - 1)
        sh = (-1,) + (1,) * (x.dim() - 1)
        a = self.diff.sqrt_alphas_cumprod[ts].double().view(sh)
        s = self.diff.sqrt_one_minus_alphas_cumprod[ts].double().view(sh)
        return ((x.double() - a * self.x0.double()) / s).float()


def test_true_noise_gives_zero_mse_and_a_shifted_one_does_not():
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    g = torch.Generator().manual_seed(3)
    x0 = torch.randn(3, 2, 6, 5, 7, generator=g).cuda()
    diff = quiet(GaussianDiffusionLatent3D, torch.nn.Identity(), 2, timesteps=50).cuda()
    diff.model = _TrueNoise(diff, x0, 0)
    torch.manual_seed(1)
    r = diff.calc_bpd_loop(x0)
    assert (r["mse"] < 1e-8).all(), r["mse"].max().item()
    assert (r["vb"][:, 1:] < 1e-5).all()
    for shift in (1, -1):   # clamped at 0 and T - 1: those ends are exact again
        diff.model = _TrueNoise(diff, x0, shift)
        torch.manual_seed(1)
        r = diff.calc_bpd_loop(x0)
        assert (r["mse"][:, 1:-1] > 1e-5).all(), (shift, r["mse"][:, 1:-1].min().item())


def test_cfg4_shape_equals_the_restatement():
    """The benchmarked model and latent shape (attention UNet, base 128, 3x40x48x40) at B = 2."""
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    torch.manual_seed(0)
    m = UNet3DModelWithAttention(in_channels=3, base_channels=128, channel_mults=(1, 2, 4),
                                 time_emb_dim=256, groups=8, num_heads=4).cuda().eval()
    x0 = torch.randn(2, 3, 40, 48, 40, generator=torch.Generator().manual_seed(6)).cuda()
    diff = _diff3d(m, 4)
    torch.manual_seed(5)
    got = diff.calc_bpd_loop(x0)
    _close(got, _ref_bpd(diff, lambda a, t: m(a, t), x0, 5, 1), 1e-5)


def test_one_graph_serves_every_input_and_leaves_the_samplers_alone():
    m, diff, x0, eps_fn, bpd, dec = _case("3d", 20, seed=84)
    shape = x0.shape
    mask = torch.zeros(1, 1, *shape[2:], dtype=torch.bool, device="cuda")
    mask[..., 2:6, 3:9, 2:6] = True
    torch.manual_seed(1)
    plain = diff.sample(2, shape[2:])
    m.__dict__.pop("_mri_programs", None)

    x2 = torch.randn(shape, generator=torch.Generator().manual_seed(9)).cuda()
    graphs = []
    for i, x in enumerate([x0, x2, x0]):
        torch.manual_seed(10 + i)
        got = bpd(x)
        _close(got, _ref_bpd(diff, eps_fn, x, 10 + i, dec), 1e-5)
        graphs.append(next(iter(m._programs().values()))._step_graphs["vb"][2])
    assert graphs[0] is graphs[1] is graphs[2]
    torch.manual_seed(1)
    assert torch.equal(diff.sample(2, shape[2:]), plain)
    torch.manual_seed(2)
    got = diff.inpaint(x0, mask)
    want = _ref_ddpm(diff, eps_fn, x0, mask, 2)
    assert torch.equal(got, want), (got - want).abs().max().item()


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_bad_shapes_leave_the_cuda_generator_untouched(kind):
    m, diff, x0, eps_fn, bpd, _ = _case(kind, 12)
    B, C = x0.shape[:2]
    torch.manual_seed(5)
    off = _gen_offset()
    for bad in (x0[0], x0[:, :1] if C > 1 else torch.cat([x0, x0], 1), x0[:0]):
        with pytest.raises(ValueError):
            bpd(bad)
    assert _gen_offset() == off
