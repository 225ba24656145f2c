"""Undersampled k-space reconstruction on the GPU: mri_kspace_merge against an fp64 torch.fft
restatement, its edge cases, the replayed reconstruction loops (fused and unfused, bf16 and split
precision) against eager sequences of the public ops, bit for bit, data consistency and the
invariants of the method with random weights, graph reuse, and the conditioning check of
test_kspace_cpu.py through the eager path on the real kernels."""
import contextlib
import io

import pytest
import torch

from helpers import shapes_of, synthetic_state_dict
from test_kspace_cpu import (A_SCALE, D_NOISE, HW, bump, bump_eps, line_mask, projector,
                             unmeasured_error)

pytestmark = pytest.mark.gpu

KERNEL_TOL = 2e-5       # rel-L2 of mri_kspace_merge against fp64 (measured: see DESIGN.md §4)


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _gen_offset():
    return torch.cuda.default_generators[torch.cuda.current_device()].get_offset()


def _complete(y, m):
    from mri_image_generation_b200.diffusion_base import kspace_completion
    zf, M = kspace_completion(y, m.expand(y.shape).bool())
    return zf.float().contiguous(), M.to(torch.uint8).contiguous()


# ------------------------------------------------------------------------------------------ kernel
def _sched():
    from mri_image_generation_b200 import schedules
    b = schedules.make_buffers(schedules.linear_beta_schedule(1000, 1e-4, 0.02), True)
    return b["sqrt_alphas_cumprod"].cuda(), b["sqrt_one_minus_alphas_cumprod"].cuda()


def _ref_merge(x, zf, M, tau, z, sac, s1m):
    """fp64: x - P(x - s1m z) + sac zf per sample, x - P x + zf where tau < 0."""
    B = x.shape[0]
    neg = (tau < 0).view(B, 1, 1, 1)
    tc = tau.clamp(min=0)
    s1 = torch.where(neg, 0.0, s1m.double()[tc].view(B, 1, 1, 1))
    sa = torch.where(neg, 1.0, sac.double()[tc].view(B, 1, 1, 1))
    u = x.double() - s1 * z.double()
    Pu = projector(M.bool())(u)
    return x.double() - Pu + sa * zf.double()


def _kernel_masks(shape, g):
    B, C, H, W = shape
    return {"rows": line_mask(H, W, axis=-2).view(1, 1, H, W),
            "cols": line_mask(H, W, axis=-1).view(1, 1, H, W),
            "random": torch.rand(shape, generator=g) < 0.3,
            "per_sample": torch.rand(B, 1, H, W, generator=g) < 0.25,
            "per_channel": torch.rand(1, C, H, W, generator=g) < torch.linspace(0.1, 0.9, C).view(1, C, 1, 1),
            "zeros": torch.zeros(1, 1, 1, 1, dtype=torch.bool),
            "ones": torch.ones(1, 1, 1, 1, dtype=torch.bool)}


KERNEL_SHAPES = [(1, 1, 1, 1), (3, 1, 7, 9), (2, 4, 33, 31), (2, 1, 36, 44), (2, 1, 240, 240),
                 (4, 4, 192, 192)]
_worst = {}


@pytest.mark.parametrize("shape", KERNEL_SHAPES)
@pytest.mark.parametrize("source", ["philox", "tensor"])
def test_merge_kernel_against_fp64(shape, source):
    from mri_image_generation_b200 import ops
    g = torch.Generator().manual_seed(sum(shape))
    sac, s1m = _sched()
    B = shape[0]
    x = torch.randn(shape, generator=g).cuda()
    x_true = torch.randn(shape, generator=g, dtype=torch.float64).cuda()
    t = torch.tensor([0, 500, 999, 1, 250][:B] + [7] * max(0, B - 5), dtype=torch.int64).cuda()
    rng = ops.DeviceRng(torch.device("cuda"))
    inc = ops.randn_offset_increment(x.numel())
    for name, m in _kernel_masks(shape, g).items():
        zf, M = _complete(torch.fft.fft2(x_true, norm="ortho"), m.cuda())
        torch.manual_seed(7)
        off = _gen_offset()
        torch.randn(shape, device="cuda")                 # the skipped draw (the update's z)
        z = torch.randn(shape, device="cuda")
        got = x.clone()
        if source == "philox":
            torch.cuda.default_generators[torch.cuda.current_device()].set_offset(off)
            rng.load()
            ops.kspace_merge(got, zf, M, t, -1, sac, s1m, rng=rng, rng_skip=inc)
        else:
            ops.kspace_merge(got, zf, M, t, -1, sac, s1m, noise=z)
        want = _ref_merge(x, zf, M, t - 1, z, sac, s1m)
        err = ((got.double() - want).norm() / want.norm()).item()
        _worst[name] = max(_worst.get(name, 0.0), err)
        print(f"{shape} {source} {name}: rel-L2 {err:.3e}")
        assert err <= KERNEL_TOL, (name, err)


def test_merge_kernel_worst_case_report():
    """The largest error per mask over the shapes above (printed for DESIGN.md §4)."""
    print("worst rel-L2 per mask:", {k: f"{v:.2e}" for k, v in sorted(_worst.items())})


def test_empty_mask_returns_x_bit_for_bit():
    from mri_image_generation_b200 import ops
    sac, s1m = _sched()
    for shape in ((3, 1, 7, 9), (2, 4, 33, 31), (2, 1, 240, 240)):
        x = torch.randn(shape, device="cuda")
        zf, M = _complete(torch.fft.fft2(torch.randn(shape, device="cuda").double()),
                          torch.zeros(1, 1, 1, 1, dtype=torch.bool, device="cuda"))
        assert torch.equal(zf, torch.zeros_like(zf))
        got = x.clone()
        ops.kspace_merge(got, zf, M, torch.arange(shape[0], device="cuda") * 300, -1, sac, s1m,
                         noise=torch.randn(shape, device="cuda"))
        assert torch.equal(got, x)


def test_full_mask_writes_the_kernels_own_draw():
    """x = 0, M = 1, s1m = 1, sac = 0: x = P z = z, and z is randn_like after the skip."""
    from mri_image_generation_b200 import ops
    shape = (2, 3, 40, 36)
    ones, zeros = torch.ones(1000, device="cuda"), torch.zeros(1000, device="cuda")
    M = torch.ones(shape, dtype=torch.uint8, device="cuda")
    t = torch.tensor([10, 500], device="cuda")
    rng = ops.DeviceRng(torch.device("cuda"))
    inc = ops.randn_offset_increment(M.numel())
    torch.manual_seed(12)
    off = _gen_offset()
    torch.randn(shape, device="cuda")
    want = torch.randn(shape, device="cuda")
    torch.cuda.default_generators[torch.cuda.current_device()].set_offset(off)
    rng.load()
    got = torch.zeros(shape, device="cuda")
    ops.kspace_merge(got, torch.zeros_like(got), M, t, 0, zeros, ones, rng=rng, rng_skip=inc)
    err = ((got - want).norm() / want.norm()).item()
    print(f"own draw: rel-L2 {err:.3e}")
    assert err <= 1e-5


def test_size_limit_and_work_buffer_checks():
    from mri_image_generation_b200 import _lib, ops
    with pytest.raises(_lib.MriError):
        ops.kspace_work_bytes(1, 1, 513, 8)
    assert ops.kspace_work_bytes(2, 3, 512, 512) == 2 * 3 * 512 * 257 * 8
    sac, s1m = _sched()
    x = torch.zeros(1, 1, 8, 8, device="cuda")
    small = torch.zeros(ops.kspace_work_bytes(1, 1, 8, 8) - 8, dtype=torch.uint8, device="cuda")
    with pytest.raises(_lib.MriError):
        ops.kspace_merge(x, x, torch.zeros(x.shape, dtype=torch.uint8, device="cuda"),
                         torch.zeros(1, dtype=torch.int64, device="cuda"), 0, sac, s1m, work=small,
                         noise=x)


# ------------------------------------------------------------------------------------------ loops
def _model2d(kind, seed):
    if kind.startswith("2d"):
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
    m = m.cuda().eval()
    if kind.endswith("_split"):
        m.precision = "split"
    return m, mk


def _case(kind, T, seed=91):
    """(model, diffusion, x_true, kspace, kmask, eps_fn, call(method, *a, **kw))."""
    g = torch.Generator().manual_seed(seed)
    m, mk = _model2d(kind, seed)
    diff = mk(m, T)
    z = torch.tensor([0.2, 0.7], device="cuda")
    if kind.startswith("2d"):
        shape = (2, 1, 40, 40)
        kmask = line_mask(40, 40).view(1, 1, 40, 40)
        kw = dict(z_pos=z)
        eps_fn = lambda a, t: m(a, t, z)
    else:   # multi-contrast: t1, t1ce, t2 fully sampled, flair along every fourth row
        shape = (2, 4, 24, 24)
        kmask = torch.ones(1, 4, 24, 24, dtype=torch.bool)
        kmask[0, 3] = line_mask(24, 24)
        ctx = torch.randn(2, 16, 24, 24, generator=g).cuda()
        kw = dict(z_pos=z, context=ctx)
        eps_fn = lambda a, t: m(a, t, z, context=ctx)
    x_true = torch.randn(shape, generator=g).cuda()
    kspace = torch.fft.fft2(x_true.double(), norm="ortho").to(torch.complex64)
    call = lambda meth, *a, **k: getattr(diff, meth)(*a, **kw, **k)
    return m, diff, x_true, kspace, kmask.cuda(), eps_fn, call


def _ref_ddpm(diff, eps_fn, kspace, kmask, seed):
    """The DDPM reconstruction sequence with the public ops and torch.randn_like."""
    from mri_image_generation_b200 import ops
    zf, M = _complete(kspace, kmask)
    B, T = zf.shape[0], diff.timesteps
    torch.manual_seed(seed)
    x = torch.randn(zf.shape, device="cuda")
    with torch.no_grad():
        for i in reversed(range(T)):
            t = torch.full((B,), i, device="cuda", dtype=torch.long)
            eps = eps_fn(x, t).float().contiguous()
            z = torch.randn_like(x)
            out = torch.empty_like(x)
            ops.ddpm_step(x, eps, z, t, diff.betas, diff.sqrt_one_minus_alphas_cumprod,
                          diff.sqrt_recip_alphas, diff.posterior_variance, out)
            n = torch.randn_like(out)
            ops.kspace_merge(out, zf, M, t, -1, diff.sqrt_alphas_cumprod,
                             diff.sqrt_one_minus_alphas_cumprod, noise=n)
            x = out
    return x


def _ref_dpmpp(diff, eps_fn, kspace, kmask, seed, steps):
    from mri_image_generation_b200 import ops, schedules
    zf, M = _complete(kspace, kmask)
    B, T = zf.shape[0], diff.timesteps
    ts, coef = schedules.dpmpp_2m_table(diff.alphas_cumprod, schedules.dpmpp_timesteps(T - 1, steps))
    coef = coef.cuda()
    torch.manual_seed(seed)
    x_T = torch.randn(zf.shape, device="cuda")
    x, x0p = x_T.clone(), torch.full_like(x_T, float("nan"))
    taus = ts.tolist()[1:] + [-1]
    with torch.no_grad():
        for i, t in enumerate(ts.tolist()):
            tt = torch.full((B,), t, device="cuda", dtype=torch.long)
            eps = eps_fn(x, tt).float().contiguous()
            ops.dpmpp_step(x, eps, x0p, coef, torch.tensor([i], device="cuda"), x)
            ops.kspace_merge(x, zf, M, torch.full((B,), taus[i], device="cuda", dtype=torch.long), 0,
                             diff.sqrt_alphas_cumprod, diff.sqrt_one_minus_alphas_cumprod, noise=x_T)
    return x


def _consistency(x_hat, kspace, kmask):
    """|M (fft2(x_hat) - y)| / |M y| on the completed mask."""
    _, M = _complete(kspace, kmask)
    M = M.bool()
    y = kspace.to(torch.complex128) * M
    y = torch.fft.fft2(torch.fft.ifft2(y, norm="ortho").real, norm="ortho")   # its Hermitian part
    d = torch.fft.fft2(x_hat.double(), norm="ortho") - y
    return ((d * M).abs().norm() / (y * M).abs().norm()).item()


@pytest.mark.parametrize("kind", ["2d", "25d", "2d_split", "25d_split"])
@pytest.mark.parametrize("fused", ["1", "0"])
def test_replayed_loops_equal_eager_sequences(kind, fused, monkeypatch):
    from mri_image_generation_b200 import ops
    monkeypatch.setenv("MRI_FUSED_STEP", fused)
    T = 12
    m, diff, x_true, kspace, kmask, eps_fn, call = _case(kind, T)
    inc = ops.randn_offset_increment(x_true.numel())
    torch.manual_seed(31)
    o0 = _gen_offset()
    got = call("reconstruct", kspace, kmask)
    assert _gen_offset() - o0 == (1 + 2 * T) * inc
    off = _gen_offset()
    prog = next(iter(m._programs().values()))
    assert "ddpm+kspace" in prog._step_graphs
    if not kind.endswith("_split"):
        assert prog.fused_head is not None
    want = _ref_ddpm(diff, eps_fn, kspace, kmask, 31)
    assert torch.isfinite(got).all()
    assert torch.equal(got, want), (got - want).abs().max().item()
    assert _gen_offset() == off

    torch.manual_seed(32)
    o0 = _gen_offset()
    got = call("reconstruct_dpmpp", kspace, kmask, num_steps=6)
    assert _gen_offset() - o0 == inc
    assert "dpmpp+kspace" in prog._step_graphs
    want = _ref_dpmpp(diff, eps_fn, kspace, kmask, 32, 6)
    assert torch.isfinite(got).all()
    assert torch.equal(got, want), (got - want).abs().max().item()


@pytest.mark.parametrize("kind", ["2d", "25d"])
def test_data_consistency_and_fully_sampled_channels(kind):
    m, diff, x_true, kspace, kmask, _, call = _case(kind, 50)
    for meth, kw in (("reconstruct", {}), ("reconstruct_dpmpp", {"num_steps": 10})):
        torch.manual_seed(8)
        x_hat = call(meth, kspace, kmask, **kw)
        assert torch.isfinite(x_hat).all()
        c = _consistency(x_hat, kspace, kmask)
        print(f"{kind} {meth}: consistency {c:.3e}")
        assert c <= 1e-4
        if kind == "25d":     # t1, t1ce and t2 are fully sampled
            err = ((x_hat[:, :3] - x_true[:, :3]).norm() / x_true[:, :3].norm()).item()
            print(f"{kind} {meth}: fully sampled channels rel-L2 {err:.3e}")
            assert err <= 1e-5


@pytest.mark.parametrize("kind", ["2d", "25d"])
def test_empty_mask_is_the_unconditioned_sampler(kind):
    """kmask all zero: P = 0 and x_zf = 0, so every merge leaves x bit for bit.  The DDPM loop then
    is inpaint() with nothing kept (the same two draws per step); the DPM-Solver++ loop, which draws
    nothing after x_T, is sample_dpmpp()."""
    m, diff, x_true, kspace, kmask, _, call = _case(kind, 20)
    none = torch.zeros_like(kmask)
    torch.manual_seed(77)
    want = call("inpaint", torch.full_like(x_true, float("nan")), torch.ones_like(kmask))
    torch.manual_seed(77)
    got = call("reconstruct", kspace, none)
    assert torch.equal(got, want), (got - want).abs().max().item()
    torch.manual_seed(78)
    want = call("sample_dpmpp", 2, num_steps=7)
    torch.manual_seed(78)
    got = call("reconstruct_dpmpp", kspace, none, num_steps=7)
    assert torch.equal(got, want), (got - want).abs().max().item()


def test_bad_arguments_leave_the_cuda_generator_untouched():
    m, diff, x_true, kspace, kmask, _, call = _case("2d", 12)
    B = kspace.shape[0]
    bad = [(kspace.real.contiguous(), kmask),                                      # not complex
           (torch.cat([kspace, kspace], 1), kmask),                                # channels
           (kspace[0], kmask),                                                     # rank
           (kspace, torch.ones(B + 1, 1, 40, 40, dtype=torch.bool, device="cuda")),
           (kspace, torch.full(kspace.shape, 0.5, device="cuda")),                 # not 0 / 1
           (kspace, torch.full(kspace.shape, 2, dtype=torch.int64, device="cuda"))]
    torch.manual_seed(5)
    off = _gen_offset()
    for k, mk in bad:
        for method in ("reconstruct", "reconstruct_dpmpp"):
            with pytest.raises(ValueError):
                call(method, k, mk)
    for num_steps in (0, 12):
        with pytest.raises(ValueError):
            call("reconstruct_dpmpp", kspace, kmask, num_steps=num_steps)
    assert _gen_offset() == off


def test_one_graph_serves_every_input_and_leaves_the_other_loops_alone():
    m, diff, x_true, kspace, kmask, eps_fn, call = _case("2d", 20, seed=84)
    z = torch.tensor([0.2, 0.7], device="cuda")
    torch.manual_seed(1)
    plain = diff.sample(2, z_pos=z)
    torch.manual_seed(2)
    plain_dpm = diff.sample_dpmpp(2, z_pos=z, num_steps=8)
    g = torch.Generator().manual_seed(9)
    k2 = torch.fft.fft2(torch.randn(x_true.shape, generator=g).cuda().double(), norm="ortho")
    m2 = (torch.rand(2, 1, 40, 40, generator=g) < 0.2).cuda()
    graphs = {}
    for i, (k, mk, M) in enumerate([(kspace, kmask, 5), (k2, m2, 9), (kspace, kmask, 5)]):
        torch.manual_seed(10 + i)
        got = call("reconstruct", k, mk)
        assert torch.equal(got, _ref_ddpm(diff, eps_fn, k, mk, 10 + i))
        torch.manual_seed(20 + i)
        got = call("reconstruct_dpmpp", k, mk, num_steps=M)
        assert torch.equal(got, _ref_dpmpp(diff, eps_fn, k, mk, 20 + i, M))
        prog = next(iter(m._programs().values()))
        for key in ("ddpm+kspace", "dpmpp+kspace"):
            graphs.setdefault(key, []).append(prog._step_graphs[key][2])
    for key, gs in graphs.items():
        assert gs[0] is gs[1] is gs[2], key
    torch.manual_seed(1)
    assert torch.equal(diff.sample(2, z_pos=z), plain)
    torch.manual_seed(2)
    assert torch.equal(diff.sample_dpmpp(2, z_pos=z, num_steps=8), plain_dpm)


# ------------------------------------------------------------------------------------------ conditioning
class _BumpEps(torch.nn.Module):
    """The exact eps of test_kspace_cpu.py's bump data, for (B, 1, H, W) states."""

    def __init__(self, ac):
        super().__init__()
        self.register_buffer("ac", ac.double())
        self.register_buffer("v", bump(HW, HW, 1.5).cuda())

    def forward(self, x, t, z_pos=None):
        ac = self.ac[t]
        assert bool((ac == ac[0]).all())      # the samplers step every sample together
        return bump_eps(x[:, 0].double(), ac[0].item(), self.v).unsqueeze(1).float()


def test_conditioning_through_the_eager_path():
    from mri_image_generation_b200.diffusion_base import kspace_completion
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion
    B = 32
    diff = quiet(GaussianDiffusion, torch.nn.Identity(), HW, channels=1, timesteps=1000).cuda()
    diff.model = _BumpEps(diff.alphas_cumprod).cuda()
    g = torch.Generator().manual_seed(0)
    v = bump(HW, HW, 1.5)
    s = A_SCALE * torch.randn(B, 1, 1, generator=g, dtype=torch.float64)
    x = s * v + D_NOISE * torch.randn(B, HW, HW, generator=g, dtype=torch.float64)
    y = torch.fft.fft2(x, norm="ortho")
    m = line_mask(HW, HW).expand(B, HW, HW)
    x_zf, M = kspace_completion(y, m)
    P = projector(M)
    Pv = P(v.expand(B, HW, HW))[0]
    post = A_SCALE ** 2 * (x_zf * Pv).sum((-2, -1)) / (D_NOISE ** 2 + A_SCALE ** 2 * (Pv * Pv).sum())
    yk, mk = y.unsqueeze(1).cuda(), m.unsqueeze(1).cuda()
    res = {}
    for name, free, rec in [("ddpm", lambda: diff.sample(B), lambda: diff.reconstruct(yk, mk)),
                            ("dpmpp", lambda: diff.sample_dpmpp(B, num_steps=20),
                             lambda: diff.reconstruct_dpmpp(yk, mk, num_steps=20))]:
        torch.manual_seed(4)
        x_free = free()[:, 0].double().cpu()
        torch.manual_seed(4)
        x_rec = rec()[:, 0].double().cpu()
        assert ((P(x_rec) - x_zf).norm() / x_zf.norm()).item() < 1e-5
        e_free, e_rec = unmeasured_error(x_free, v, P, post), unmeasured_error(x_rec, v, P, post)
        res[name] = e_free / e_rec
        print(f"{name}: unconditional {e_free:.4g}, reconstructed {e_rec:.4g}, ratio {res[name]:.1f}")
    assert res["ddpm"] >= 25 and res["dpmpp"] >= 7
