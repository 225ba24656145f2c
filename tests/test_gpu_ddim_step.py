"""mri_ddim_step against the reference's DDIM update (oracle.reference_oracle.ddim_update) computed
by torch in fp32 on the same GPU, bit for bit: both eps layouts, in place and out of place, at
shapes whose per-sample or per-channel length is odd (groups of four elements that straddle a
sample or channel boundary) and on views that start off a 16-byte boundary."""
import math

import pytest
import torch

from oracle import reference_oracle as O

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape", [(3, 1, 7, 9), (2, 4, 33, 31), (2, 3, 5, 7, 9), (5, 1, 1, 1),
                                   (2, 2, 240, 241)])
@pytest.mark.parametrize("layout", ["f32", "nhwc"])
@pytest.mark.parametrize("offset", [0, 1])     # fp32 elements between a 16-byte boundary and the views
@pytest.mark.parametrize("inplace", [False, True])
def test_ddim_step_bit_exact(shape, layout, offset, inplace):
    from mri_image_generation_b200 import ops
    g = torch.Generator().manual_seed(sum(shape) + len(layout) + 2 * offset + inplace)
    ac = O.schedule_buffers(O.cosine_betas(1000))["alphas_cumprod"].float().cuda()
    B, C = shape[0], shape[1]
    S = math.prod(shape[2:])
    n = B * C * S

    def view(v):   # v's values in a fresh buffer, `offset` floats past its 16-byte-aligned start
        buf = torch.full((n + offset,), float("nan"), device="cuda")
        buf[offset:] = v.reshape(-1).cuda()
        return buf[offset:].view(shape)

    x = view(torch.randn(shape, generator=g))
    if layout == "f32":
        eps, ldc = view(torch.randn(shape, generator=g)), 0
        e = eps
    else:
        ldc = 16 if C < 16 else C + 8
        eps = torch.randn(B, S, ldc, generator=g).to(torch.bfloat16).cuda()
        e = eps[..., :C].float().permute(0, 2, 1).reshape(shape).contiguous()
    # t = 999 (sqrt(a_t) at its smallest), t_prev = 0 (the last step), and strided steps between
    t = torch.tensor([999, 500, 60, 1, 999][:B], device="cuda")
    t_prev = torch.tensor([949, 0, 10, 0, 0][:B], device="cuda")
    want = O.ddim_update({"alphas_cumprod": ac}, x, t, t_prev, e)
    x_before = x.clone()
    out = x if inplace else view(torch.full(shape, float("nan")))
    ops.ddim_step(x, eps, t, t_prev, ac, out, eps_nhwc_ldc=ldc, channels=C if ldc else 0)
    assert torch.isfinite(out).all()
    assert torch.equal(out, want), (out - want).abs().max().item()
    if not inplace:
        assert torch.equal(x, x_before)
