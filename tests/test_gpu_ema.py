"""optim.EMA on the GPU: mri_ema_update against torch._foreach_lerp_ (what torch.optim.swa_utils'
get_ema_multi_avg_fn runs) bit for bit, the warm-up rule against fp64, Adam(ema=) against plain
Adam + ema.update() and against AveragedModel, GradScaler's skip, resume, no host sync, sampling
from the shadow (its packed weights follow every update), and DDP unwrapping."""
import contextlib
import copy
import io

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _launch(e_list, p_list, decay, warmup, count, found_inf=None):
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.optim import ema_segments
    table, n, blocks = ema_segments(e_list, p_list, e_list[0].device)
    rc = _lib.load().mri_ema_update(table.data_ptr(), n, blocks, decay, int(warmup), count.data_ptr(),
                                    found_inf.data_ptr() if found_inf is not None else None,
                                    torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "mri_ema_update")


def _offset(t):
    """A contiguous copy of t whose data pointer is 4 bytes off a 16-byte boundary."""
    flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)[1:]
    flat.copy_(t.reshape(-1))
    return flat.view(t.shape)


# ------------------------------------------------------------------------------------------ kernel
NUMELS = [1, 7, 255, 1023, 1024, 1025, 2048, 3000, 4099, 65536 + 13]


@pytest.mark.parametrize("decay", [0.9999, 0.9, 0.5, 0.3, 0.0])
@pytest.mark.parametrize("unaligned", [False, True])
def test_kernel_equals_foreach_lerp(decay, unaligned):
    """Odd sizes, whole and partial 1024-element blocks in one launch, both of ATen's lerp branches
    (w = 1 - d below 0.5, and at or above it), 16-byte-aligned and offset-by-one-float tensors."""
    g = torch.Generator().manual_seed(int(decay * 1e4) + unaligned)
    place = _offset if unaligned else (lambda t: t)
    e = [place(torch.randn(n, generator=g).cuda()) for n in NUMELS]
    want = [t.clone() for t in e]
    count = torch.zeros((), dtype=torch.int64, device="cuda")
    for step in range(3):
        p = [place(torch.randn(n, generator=g).cuda() * 3) for n in NUMELS]
        assert all((t.data_ptr() % 16 != 0) == unaligned for t in e + p)
        torch._foreach_lerp_(want, p, 1 - decay)
        _launch(e, p, decay, False, count)
        for a, b in zip(e, want):
            assert torch.equal(a, b), (step, a.numel(), (a - b).abs().max().item())
    assert int(count) == 3


def test_kernel_skips_on_found_inf_and_the_counter_stays():
    e = [torch.randn(5000, device="cuda")]
    p = [torch.randn(5000, device="cuda")]
    before = e[0].clone()
    count = torch.full((), 7, dtype=torch.int64, device="cuda")
    _launch(e, p, 0.9, True, count, torch.ones(1, device="cuda"))
    assert torch.equal(e[0], before) and int(count) == 7
    _launch(e, p, 0.9, True, count, torch.zeros(1, device="cuda"))
    assert not torch.equal(e[0], before) and int(count) == 8


def _cfg5_unet():
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    torch.manual_seed(0)
    return UNet3DModelWithAttention(in_channels=3, base_channels=128, channel_mults=(1, 2, 4),
                                    time_emb_dim=256, groups=8, num_heads=4).cuda().train()


def test_cfg5_unet_parameter_list_equals_foreach_lerp():
    """Every parameter of the benchmarked training model (136.4 M, 170 tensors) in one launch."""
    from mri_image_generation_b200.optim import EMA
    m = _cfg5_unet()
    ema = EMA(m, 0.9999)
    live = list(m.parameters())
    shadow = list(ema.module.parameters())
    assert len(live) == 170 and sum(p.numel() for p in live) > 136e6
    want = [p.detach().clone() for p in live]
    g = torch.Generator(device="cuda").manual_seed(3)
    for _ in range(2):
        with torch.no_grad():
            for p in live:
                p.add_(torch.randn(p.shape, device="cuda", generator=g), alpha=1e-2)
        ema.update()
        torch._foreach_lerp_(want, [p.detach() for p in live], 1 - 0.9999)
        for a, b in zip(shadow, want):
            assert torch.equal(a, b)


def test_warmup_first_update_copies_then_follows_fp64():
    from mri_image_generation_b200.optim import ema_decay
    g = torch.Generator().manual_seed(5)
    n = 4096
    p = torch.rand(n, generator=g).cuda() + 1          # values in [1, 2): p - e is exact
    e = torch.rand(n, generator=g).cuda() + 1
    count = torch.zeros((), dtype=torch.int64, device="cuda")
    _launch([e], [p], 0.9999, True, count)
    assert torch.equal(e, p), "the first warm-up update has d = 0"
    ref = e.double()
    for k in range(2, 201):
        p = torch.rand(n, generator=g).cuda() + 1
        w = float(np.float32(1.0 - ema_decay(k, 0.9999, True)))   # the kernel's fp32 weight
        _launch([e], [p], 0.9999, True, count)
        ref = ref + w * (p.double() - ref)
    err = ((e.double() - ref).abs() / ref.abs()).max().item()
    assert err <= 1e-6, err
    assert int(count) == 200


# ------------------------------------------------------------------------------------------ Adam(ema=)
def _params(seed, shapes=((128, 64, 3, 3, 3), (128,), (7, 5), (1,), (300, 33))):
    g = torch.Generator().manual_seed(seed)
    return torch.nn.ParameterList([torch.nn.Parameter(torch.randn(*s, generator=g).cuda()) for s in shapes])


def _grads(mods, g):
    for ps in zip(*[list(m.parameters()) for m in mods]):
        gr = torch.randn(*ps[0].shape, generator=g).cuda()
        for p in ps:
            p.grad = gr.clone()


def _moments(opt, params):
    return [t for p in params for t in (opt.state[p]["exp_avg"], opt.state[p]["exp_avg_sq"])]


@pytest.mark.parametrize("decay", [0.9999, 0.3])
def test_adam_with_ema_matches_adam_then_update_and_averaged_model(decay):
    from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn
    from mri_image_generation_b200.optim import EMA, Adam
    ma, mb, mc, md = _params(1), _params(1), _params(1), _params(1)
    ema_a = EMA(ma, decay)
    oa = Adam(ma.parameters(), lr=1e-3, ema=ema_a)
    ob, ema_b = Adam(mb.parameters(), lr=1e-3), EMA(mb, decay)
    oc = Adam(mc.parameters(), lr=1e-3)                        # plain, no EMA
    od = Adam(md.parameters(), lr=1e-3)
    avg = AveragedModel(md, multi_avg_fn=get_ema_multi_avg_fn(decay))
    avg.update_parameters(md)                                 # n_averaged == 0: copies only
    g = torch.Generator().manual_seed(2)
    for step in range(10):
        _grads([ma, mb, mc, md], g)
        oa.step()
        ob.step()
        ema_b.update()
        oc.step()
        od.step()
        avg.update_parameters(md)
        for a, b, c in zip(ma.parameters(), mb.parameters(), mc.parameters()):
            assert torch.equal(a, b) and torch.equal(a, c), step
        for a, c in zip(_moments(oa, list(ma.parameters())), _moments(oc, list(mc.parameters()))):
            assert torch.equal(a, c), step
        for a, b, c in zip(ema_a.module.parameters(), ema_b.module.parameters(), avg.module.parameters()):
            assert torch.equal(a, b) and torch.equal(a, c), (step, (a - c).abs().max().item())
    assert int(ema_a.num_updates) == int(ema_b.num_updates) == 10


def test_grad_scaler_skip_leaves_everything_and_the_next_step_goes_on():
    from mri_image_generation_b200.optim import EMA, Adam
    ma, mc = _params(3), _params(3)
    ema = EMA(ma, 0.9, warmup=True)
    oa = Adam(ma.parameters(), lr=1e-3, ema=ema)
    oc, ema_c = Adam(mc.parameters(), lr=1e-3), EMA(mc, 0.9, warmup=True)
    sa = torch.amp.GradScaler("cuda", init_scale=1024.0)
    sc = torch.amp.GradScaler("cuda", init_scale=1024.0)
    pa = list(ma.parameters())
    for it in range(4):
        for m, o, s in ((ma, oa, sa), (mc, oc, sc)):
            o.zero_grad(set_to_none=True)
            s.scale(sum((p * p).sum() for p in m.parameters())).backward()
        if it == 1:
            pa[0].grad[0, 0, 0, 0, 0] = float("inf")
            list(mc.parameters())[0].grad[0, 0, 0, 0, 0] = float("inf")
        snap = [t.clone() for t in pa + _moments(oa, pa) + list(ema.module.parameters())] if it else None
        counters = (float(oa.state[pa[0]]["step"]), int(ema.num_updates)) if it else None
        sa.step(oa)
        sa.update()
        # the reference: the same Adam, then ema.update() only when the scaler did not skip
        before_c = float(oc.state[list(mc.parameters())[0]]["step"]) if it else 0.0
        sc.step(oc)
        sc.update()
        if float(oc.state[list(mc.parameters())[0]]["step"]) != before_c:
            ema_c.update()
        now = pa + _moments(oa, pa) + list(ema.module.parameters())
        if it == 1:
            # AveragedModel.update_parameters would have moved e on this step: it cannot see found_inf
            assert all(torch.equal(a, b) for a, b in zip(snap, now))
            assert (float(oa.state[pa[0]]["step"]), int(ema.num_updates)) == counters
        elif it >= 2:
            assert not any(torch.equal(a, b) for a, b in zip(snap[-len(pa):], now[-len(pa):]))
            assert (float(oa.state[pa[0]]["step"]), int(ema.num_updates)) == (counters[0] + 1, counters[1] + 1)
        for a, b in zip(ema.module.parameters(), ema_c.module.parameters()):
            assert torch.equal(a, b), it
    assert int(ema.num_updates) == 3


def test_parameters_without_a_gradient_are_still_averaged():
    from mri_image_generation_b200.optim import EMA, Adam
    m = _params(4)
    ema = EMA(m, 0.8)
    opt = Adam(m.parameters(), lr=1e-2, ema=ema)
    ps = list(m.parameters())
    want = [p.detach().clone() for p in ps]
    g = torch.Generator().manual_seed(9)
    for step in range(3):
        for i, p in enumerate(ps):   # from the second step on, parameter 2 gets no gradient
            p.grad = torch.randn(*p.shape, generator=g).cuda() if (i != 2 or step == 0) else None
        frozen = ps[2].detach().clone()
        opt.step()
        if step:
            assert torch.equal(ps[2], frozen)
        torch._foreach_lerp_(want, [p.detach() for p in ps], 1 - 0.8)
        for a, b in zip(ema.module.parameters(), want):
            assert torch.equal(a, b), step
    # the shadow of the frozen parameter moved toward it on every step
    assert not torch.equal(list(ema.module.parameters())[2], ps[2])


def test_no_host_sync_from_the_second_step_on():
    from mri_image_generation_b200.optim import EMA, Adam
    m = _params(6)
    ema = EMA(m, 0.999, warmup=True)
    opt = Adam(m.parameters(), lr=1e-3, ema=ema)
    scaler = torch.amp.GradScaler("cuda", init_scale=256.0)

    def step():
        opt.zero_grad(set_to_none=False)
        scaler.scale(sum((p * p).sum() for p in m.parameters())).backward()
        scaler.step(opt)
        scaler.update()

    step()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            step()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert int(ema.num_updates) == 4


def test_resume_equals_an_uninterrupted_run():
    from mri_image_generation_b200.optim import EMA, Adam

    def run(m, opt, g, n):
        for _ in range(n):
            _grads([m], g)
            opt.step()

    m0 = _params(8)
    ema0 = EMA(m0, 0.999, warmup=True)           # warm-up: the restored counter sets d
    opt0 = Adam(m0.parameters(), lr=1e-3, ema=ema0)
    g0 = torch.Generator().manual_seed(10)
    run(m0, opt0, g0, 6)

    m1 = _params(8)
    ema1 = EMA(m1, 0.999, warmup=True)
    opt1 = Adam(m1.parameters(), lr=1e-3, ema=ema1)
    g1 = torch.Generator().manual_seed(10)
    run(m1, opt1, g1, 3)
    saved = copy.deepcopy({"model": m1.state_dict(), "opt": opt1.state_dict(), "ema": ema1.state_dict()})
    assert set(saved["ema"]) == {"decay", "warmup", "num_updates", "module"}
    del m1, ema1, opt1

    m2 = _params(99)
    m2.load_state_dict(saved["model"])
    ema2 = EMA(m2, 0.5)
    ema2.load_state_dict(saved["ema"])
    assert (ema2.decay, ema2.warmup, int(ema2.num_updates)) == (0.999, True, 3)
    opt2 = Adam(m2.parameters(), lr=1e-3, ema=ema2)
    opt2.load_state_dict(saved["opt"])
    run(m2, opt2, g1, 3)
    for a, b in zip(list(m0.parameters()) + list(ema0.module.parameters()),
                    list(m2.parameters()) + list(ema2.module.parameters())):
        assert torch.equal(a, b)
    assert int(ema2.num_updates) == 6


def test_argument_checks_on_the_gpu():
    from mri_image_generation_b200._lib import MriError
    from mri_image_generation_b200.optim import EMA, Adam
    ema = EMA(_params(1), 0.99)
    with pytest.raises(ValueError):
        Adam([torch.nn.Parameter(torch.zeros(3))], lr=1e-3, ema=ema)
    with pytest.raises(MriError):
        EMA(torch.nn.Linear(3, 2).cuda().half())


# ------------------------------------------------------------------------------------------ models
def _models(kind):
    """(fresh model factory, sample(model, method) -> tensor) for one model family, small sizes."""
    from helpers import shapes_of, synthetic_state_dict
    z = torch.tensor([0.2, 0.7], device="cuda")
    if kind in ("3d_attn", "3d_split"):
        from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
        from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import \
            UNet3DModelWithAttention
        make = lambda: UNet3DModelWithAttention(3, base_channels=64, time_emb_dim=64)

        def sample(m, method):
            d = quiet(GaussianDiffusionLatent3D, m, 3, timesteps=12).cuda()
            return d.sample(2, (8, 12, 8)) if method == "ddpm" else d.sample_dpmpp(2, (8, 12, 8), num_steps=4)
    elif kind == "2d":
        from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion
        from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet
        make = lambda: quiet(UNet, img_channels=1, base_channels=64, time_emb_dim=64)

        def sample(m, method):
            d = quiet(GaussianDiffusion, m, 40, channels=1, timesteps=12).cuda()
            return d.sample(2, z) if method == "ddpm" else d.sample_dpmpp(2, z, num_steps=4)
    else:
        from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.diffusion import GaussianDiffusion
        from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.unet import UNet
        make = lambda: quiet(UNet, in_channels=20, out_channels=4, base_channels=64, time_emb_dim=64)
        ctx = torch.randn(2, 16, 24, 24, generator=torch.Generator().manual_seed(4)).cuda()

        def sample(m, method):
            d = quiet(GaussianDiffusion, m, 24, channels=4, timesteps=12).cuda()
            return (d.sample(2, z, context=ctx) if method == "ddpm"
                    else d.sample_dpmpp(2, z, context=ctx, num_steps=4))

    def fresh(sd=None):
        m = make()
        m.load_state_dict(sd if sd is not None else synthetic_state_dict(shapes_of(m), seed=17))
        m = m.cuda()
        if kind == "3d_split":
            m.precision = "split"
        return m
    return fresh, sample


def _train(m, opt, g, n):
    for _ in range(n):
        for p in m.parameters():
            p.grad = torch.randn(*p.shape, generator=g).cuda()
        opt.step()


@pytest.mark.parametrize("kind", ["3d_attn", "2d", "25d", "3d_split"])
def test_sampling_from_the_shadow_equals_a_fresh_model_and_follows_updates(kind):
    from mri_image_generation_b200.optim import EMA, Adam
    fresh, sample = _models(kind)
    m = fresh()
    m.precision = "bf16"             # the live model trains; only the shadow samples
    ema = EMA(m, 0.7)
    if kind == "3d_split":
        ema.module.precision = "split"
    opt = Adam(m.parameters(), lr=1e-2, ema=ema)
    g = torch.Generator().manual_seed(21)
    _train(m, opt, g, 3)
    first = {}
    for method in ("ddpm", "dpmpp"):
        torch.manual_seed(5)
        first[method] = sample(ema.module, method)
        torch.manual_seed(5)
        ref = sample(fresh(ema.module.state_dict()), method)
        assert torch.isfinite(first[method]).all()
        assert torch.equal(first[method], ref), (kind, method)
    _train(m, opt, g, 3)             # the shadow's cached programs must re-pack its new weights
    for method in ("ddpm", "dpmpp"):
        torch.manual_seed(5)
        again = sample(ema.module, method)
        assert not torch.equal(again, first[method]), (kind, method)
        torch.manual_seed(5)
        assert torch.equal(again, sample(fresh(ema.module.state_dict()), method)), (kind, method)


def test_vae_decode_from_the_shadow():
    from helpers import shapes_of, synthetic_state_dict
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.vae import VAE3D
    from mri_image_generation_b200.optim import EMA, Adam

    def fresh(sd=None):
        v = VAE3D(4, 32, 3, 3)
        v.load_state_dict(sd if sd is not None else synthetic_state_dict(shapes_of(v), seed=23))
        return v.cuda()

    vae = fresh()
    ema = EMA(vae, 0.7)
    opt = Adam(vae.parameters(), lr=1e-2, ema=ema)
    g = torch.Generator().manual_seed(24)
    zl = torch.randn(2, 3, 4, 4, 4, generator=g).cuda()
    _train(vae, opt, g, 2)
    first = ema.module.decode_from_latent(zl)
    assert torch.equal(first, fresh(ema.module.state_dict()).decode_from_latent(zl))
    _train(vae, opt, g, 2)
    again = ema.module.decode_from_latent(zl)
    assert not torch.equal(again, first)
    assert torch.equal(again, fresh(ema.module.state_dict()).decode_from_latent(zl))


def test_state_dict_keys_equal_the_live_models():
    """ema.module.state_dict() saves as the UNet checkpoint the reference's scripts load."""
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.unet import UNet as UNet25
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet
    from mri_image_generation_b200.optim import EMA
    cases = [(_cfg5_unet(), 170), (quiet(UNet).cuda(), 178), (quiet(UNet25, in_channels=20, out_channels=4).cuda(), 178)]
    for m, n_keys in cases:
        sd = EMA(m, 0.9999).state_dict()
        assert set(sd) == {"decay", "warmup", "num_updates", "module"}
        assert sd["decay"] == 0.9999 and sd["warmup"] is False and int(sd["num_updates"]) == 0
        assert list(sd["module"]) == list(m.state_dict()) and len(sd["module"]) == n_keys
        for k, v in m.state_dict().items():
            assert torch.equal(sd["module"][k], v), k
        del m


def test_ddp_wrappers_are_unwrapped(tmp_path):
    import torch.distributed as dist
    from mri_image_generation_b200 import parallel
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    from mri_image_generation_b200.optim import EMA
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/pg", rank=0, world_size=1)
    try:
        for wrap in (lambda m: torch.nn.parallel.DistributedDataParallel(m),
                     lambda m: parallel.DistributedDataParallel(m)):
            m = UNet3DModelWithAttention(3, base_channels=64, time_emb_dim=64).cuda()
            ema = EMA(wrap(m), 0.99)
            assert type(ema.module) is UNet3DModelWithAttention
            assert list(ema.module.state_dict()) == list(m.state_dict())
            assert "_mri_grad_sync" not in ema.module.__dict__
            assert not any(p.requires_grad for p in ema.module.parameters())
            with torch.no_grad():
                for p in m.parameters():
                    p.add_(1.0)
            ema.update()
            for e, p in zip(ema.module.parameters(), m.parameters()):
                assert not torch.equal(e, p)
    finally:
        dist.destroy_process_group()
