"""Thin torch-tensor wrappers over the C ABI (include/mri_b200.h).

Each function takes CUDA tensors, passes raw device pointers and the current CUDA stream to
libmri_b200.so and returns nothing (outputs are caller-allocated).  No wrapper has a fallback:
a CPU tensor or a missing library raises.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.MriError("mri_image_generation_b200 ops need CUDA tensors (no CPU path)")
    return t.data_ptr()


def _s() -> int:
    return _lib.current_stream_ptr()


def _chk_contig(*ts):
    for t in ts:
        if t is not None and not t.is_contiguous():
            raise _lib.MriError("non-contiguous tensor passed to a libmri_b200 op")


def gn_stats(x: torch.Tensor, stats: torch.Tensor, samples: int, spatial: int, C: int,
             stats_cpg: int, stats_g0: int = 0) -> None:
    _chk_contig(x, stats)
    _lib.check(_lib.load().mri_gn_stats(_p(x), _p(stats), samples, spatial, C, stats.shape[1],
                                        stats_g0, stats_cpg, _s()), "mri_gn_stats")


def gn_apply(x, y, stats, gamma, beta, samples: int, spatial: int, C: int, groups: int,
             stats_cpg: int, eps: float, silu: bool, rowbias=None, rowbias_ld: int = 0,
             residual=None, stats_g0: int = 0) -> None:
    _chk_contig(x, y, stats, residual)
    _lib.check(_lib.load().mri_gn_apply(_p(x), _p(y), _p(stats), _p(gamma), _p(beta), _p(rowbias),
                                        rowbias_ld, _p(residual), samples, spatial, C, groups,
                                        stats.shape[1], stats_g0, stats_cpg, eps, 1 if silu else 0,
                                        _s()), "mri_gn_apply")


def sinusoidal_freqs(dim: int, device) -> torch.Tensor:
    """Frequency table of SinusoidalPosEmb, built on the host with the reference's own fp32
    expression (slice_cond_2d_ddpm/unet.py:18-20) so that t * f is bit-identical."""
    import math
    half = dim // 2
    f = math.log(10000) / (half - 1)
    return torch.exp(torch.arange(half) * -f).to(device)


def sinusoidal(t: torch.Tensor, freqs: torch.Tensor, out: torch.Tensor) -> None:
    assert t.dtype == torch.int64 and out.dtype == torch.float32 and freqs.dtype == torch.float32
    _lib.check(_lib.load().mri_sinusoidal(_p(t), _p(freqs), _p(out), out.shape[0], out.shape[1],
                                          _s()), "mri_sinusoidal")


def linear(x, W, bias, y, act: int = 0, addend=None) -> None:
    _chk_contig(x, W, y, addend)
    assert x.dtype == W.dtype == y.dtype == torch.float32
    _lib.check(_lib.load().mri_linear(_p(x), _p(W), _p(bias), _p(addend), _p(y), x.shape[0],
                                      W.shape[1], W.shape[0], act, _s()), "mri_linear")


def im2col(src, dst, samples, cin, D, H, W, ksize, ndim, kpad, src2=None, cin2: int = 0) -> None:
    _chk_contig(src, src2, dst)
    _lib.check(_lib.load().mri_im2col(_p(src), _p(src2), _p(dst), samples, cin, cin2, D, H, W,
                                      ksize, ndim, kpad, _s()), "mri_im2col")


def im2col4(src, dst, samples, cp, D, H, W, ksize, ndim, kpad) -> None:
    _chk_contig(src, dst)
    _lib.check(_lib.load().mri_im2col4(_p(src), _p(dst), samples, cp, D, H, W, ksize, ndim, kpad, _s()),
               "mri_im2col4")


def thin_in_conv(x, w_packed, bias, y, stats, samples, cin, D, H, W, ndim, cout) -> None:
    """in_conv / init_conv (<= 4 input channels) in one tcgen05 launch: patch matrix built in smem."""
    _chk_contig(x, w_packed, y, stats)
    _lib.check(_lib.load().mri_thin_in_conv(_p(x), _p(w_packed), _p(bias), _p(y), _p(stats),
                                            stats.shape[1] if stats is not None else 0, samples, cin,
                                            D, H, W, ndim, cout, _s()), "mri_thin_in_conv")


def tap_gather(y, out, bias, samples, D, H, W, ksize, ndim, cout, ldy, ldo) -> None:
    _chk_contig(y, out, bias)
    _lib.check(_lib.load().mri_tap_gather(_p(y), _p(out), _p(bias), samples, D, H, W, ksize, ndim,
                                          cout, ldy, ldo, _s()), "mri_tap_gather")


def nhwc_to_nchw(src, dst, samples, spatial, C, ldc) -> None:
    _chk_contig(src, dst)
    _lib.check(_lib.load().mri_nhwc_to_nchw(_p(src), _p(dst), samples, spatial, C, ldc, _s()),
               "mri_nhwc_to_nchw")


def nchw_to_nhwc(src, dst, samples, spatial, C, ldc) -> None:
    _chk_contig(src, dst)
    _lib.check(_lib.load().mri_nchw_to_nhwc(_p(src), _p(dst), samples, spatial, C, ldc, _s()),
               "mri_nchw_to_nhwc")


def softmax_rows(S, P, rows, cols, ld_s, ld_p, scale) -> None:
    _lib.check(_lib.load().mri_softmax_rows(_p(S), _p(P), rows, cols, ld_s, ld_p, scale, _s()),
               "mri_softmax_rows")


def q_sample(x0, noise, t, sqrt_ac, sqrt_1mac, out) -> None:
    _chk_contig(x0, noise, out)
    n = x0.shape[0]
    _lib.check(_lib.load().mri_q_sample(_p(x0), _p(noise), _p(t), _p(sqrt_ac), _p(sqrt_1mac),
                                        _p(out), n, x0.numel() // n, _s()), "mri_q_sample")


def ddpm_step(x, eps, noise, t, betas, sqrt_1mac, sqrt_recip_alphas, post_var, out,
              eps_nhwc_ldc: int = 0, channels: int = 0) -> None:
    _chk_contig(x, eps, noise, out)
    n = x.shape[0]
    _lib.check(_lib.load().mri_ddpm_step(_p(x), _p(eps), eps_nhwc_ldc, channels, _p(noise), _p(t),
                                         _p(betas), _p(sqrt_1mac), _p(sqrt_recip_alphas),
                                         _p(post_var), _p(out), n, x.numel() // n, _s()),
               "mri_ddpm_step")


def ddim_step(x, eps, t, t_prev, alphas_cumprod, out, eps_nhwc_ldc: int = 0,
              channels: int = 0) -> None:
    _chk_contig(x, eps, out)
    n = x.shape[0]
    _lib.check(_lib.load().mri_ddim_step(_p(x), _p(eps), eps_nhwc_ldc, channels, _p(t), _p(t_prev),
                                         _p(alphas_cumprod), _p(out), n, x.numel() // n, _s()),
               "mri_ddim_step")


def dpmpp_step(x, eps, x0_prev, coef, k, out, eps_nhwc_ldc: int = 0, channels: int = 0) -> None:
    """One DPM-Solver++(2M) step with row k (device int64 tensor, or None for row 0) of the fp32
    [rows][5] table of schedules.dpmpp_2m_table; x0_prev (x's shape, fp32) is read on
    second-order rows and overwritten with this step's x0.  x and out may alias."""
    _chk_contig(x, eps, x0_prev, coef, out)
    assert x0_prev.dtype == coef.dtype == torch.float32 and x0_prev.numel() == x.numel()
    assert k is None or k.dtype == torch.int64
    n = x.shape[0]
    _lib.check(_lib.load().mri_dpmpp_step(_p(x), _p(eps), eps_nhwc_ldc, channels, _p(x0_prev),
                                          _p(coef), _p(k), _p(out), n, x.numel() // n, _s()),
               "mri_dpmpp_step")


def step_table_advance(t: torch.Tensor, k: torch.Tensor, ts: torch.Tensor, rows: int) -> None:
    """k += 1, then t[:] = ts[min(k, rows - 1)] (one launch, stream-ordered)."""
    assert t.dtype == k.dtype == ts.dtype == torch.int64 and 1 <= rows <= ts.numel()
    _lib.check(_lib.load().mri_step_table_advance(_p(t), t.numel(), _p(k), _p(ts), int(rows), _s()),
               "mri_step_table_advance")


def minsnr_loss(pred, noise, t, snr, gamma: float, per_sample_out, loss_out) -> None:
    _chk_contig(pred, noise)
    n = pred.shape[0]
    _lib.check(_lib.load().mri_minsnr_loss(_p(pred), _p(noise), _p(t), _p(snr), gamma,
                                           _p(per_sample_out), _p(loss_out), n, pred.numel() // n,
                                           _s()), "mri_minsnr_loss")


def add_i64(t: torch.Tensor, delta: int) -> None:
    _lib.check(_lib.load().mri_add_i64(_p(t), t.numel(), delta, _s()), "mri_add_i64")


# ------------------------------------------------------------------------------ in-kernel RNG
def randn_offset_increment(numel: int) -> int:
    """Philox offset consumed by one draw of `numel` normals (what torch.randn advances its CUDA
    generator by for a tensor of that size on this device)."""
    import ctypes as C
    inc = C.c_uint64(0)
    _lib.check(_lib.load().mri_randn_offset_increment(int(numel), C.byref(inc)),
               "mri_randn_offset_increment")
    return int(inc.value)


class DeviceRng:
    """Bridge between torch's CUDA generator and the kernels that draw their own noise.

    The kernels read (seed, philox offset) from a small device tensor and reproduce ATen's
    element mapping, so a draw through them equals torch.randn / randn_like under the same
    torch.manual_seed; the host then advances torch's generator by the offset the draw consumed,
    which keeps every LATER torch draw identical to the reference's as well."""

    def __init__(self, device: torch.device):
        self.device = torch.device(device)
        self.state = torch.zeros(2, dtype=torch.int64, device=self.device)  # {seed, offset} bits

    def generator(self) -> torch.Generator:
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        return torch.cuda.default_generators[idx]

    def load(self) -> int:
        """Copy torch's current (seed, offset) into the device state; returns the offset."""
        g = self.generator()
        seed, off = int(g.initial_seed()), int(g.get_offset())
        if off % 4:
            raise _lib.MriError("CUDA generator offset must be a multiple of 4")
        # stream-ordered 1-thread launch: no host synchronisation, no pinned staging buffer
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().mri_rng_seed(_p(self.state), seed & ((1 << 64) - 1), off, _s()),
                       "mri_rng_seed")
        return off

    def commit(self, offset: int) -> None:
        self.generator().set_offset(int(offset))


def randn(out: torch.Tensor, rng: DeviceRng) -> None:
    _chk_contig(out)
    assert out.dtype == torch.float32
    _lib.check(_lib.load().mri_randn(_p(out), out.numel(), _p(rng.state), _s()), "mri_randn")


def q_sample_rng(x0, rng: DeviceRng, t, sqrt_ac, sqrt_1mac, out, noise_out=None) -> None:
    _chk_contig(x0, out, noise_out)
    n = x0.shape[0]
    _lib.check(_lib.load().mri_q_sample_rng(_p(x0), _p(rng.state), _p(t), _p(sqrt_ac), _p(sqrt_1mac),
                                            _p(out), _p(noise_out), n, x0.numel() // n, _s()),
               "mri_q_sample_rng")


def ddpm_step_rng(x, eps, rng: DeviceRng, t, betas, sqrt_1mac, sqrt_recip_alphas, post_var, out,
                  eps_nhwc_ldc: int = 0, channels: int = 0) -> None:
    _chk_contig(x, eps, out)
    n = x.shape[0]
    _lib.check(_lib.load().mri_ddpm_step_rng(_p(x), _p(eps), eps_nhwc_ldc, channels, _p(rng.state),
                                             _p(t), _p(betas), _p(sqrt_1mac), _p(sqrt_recip_alphas),
                                             _p(post_var), _p(out), n, x.numel() // n, _s()),
               "mri_ddpm_step_rng")


def tap_gather_step(y, bias, samples, D, H, W, ndim, cout, ldy, x, mode: int, rng=None, t=None,
                    t_prev=None, betas=None, sqrt_1mac=None, sqrt_recip_alphas=None, post_var=None,
                    alphas_cumprod=None, eps_out=None, ldo: int = 0, x0_prev=None, coef=None,
                    k=None) -> None:
    """Finish the thin out_conv (sum of shifted tap products) and apply the reverse-step update to
    the sampler state x in place: mode 0 DDPM (noise drawn in-kernel), 1 DDIM, 2 eps only,
    3 DPM-Solver++(2M) (x0_prev, coef row k: see dpmpp_step)."""
    _chk_contig(y, x, eps_out, x0_prev, coef)
    _lib.check(_lib.load().mri_tap_gather_step(
        _p(y), _p(bias), samples, D, H, W, ndim, cout, ldy, _p(x), _p(eps_out), ldo, mode,
        _p(rng.state) if rng is not None else None, _p(t), _p(t_prev), _p(betas), _p(sqrt_1mac),
        _p(sqrt_recip_alphas), _p(post_var), _p(alphas_cumprod), _p(x0_prev), _p(coef), _p(k),
        _s()), "mri_tap_gather_step")


def inpaint_merge(x, known, mask, t, t_delta: int, sqrt_ac, sqrt_1mac, noise=None,
                  rng: Optional[DeviceRng] = None, rng_skip: int = 0) -> None:
    """x = where(mask, x, kn) in place, kn = known if tau < 0 else q_sample(known, tau, z) with
    tau = t + t_delta per sample (t: device int64 [samples]).  mask: uint8, one byte per element
    of x.  z: `noise`, or with rng the torch.randn_like drawn rng_skip past the generator offset."""
    _chk_contig(x, known, mask, noise)
    assert x.dtype == known.dtype == torch.float32 and mask.dtype == torch.uint8
    assert known.numel() == mask.numel() == x.numel() and t.dtype == torch.int64
    assert noise is None or (noise.dtype == torch.float32 and noise.numel() == x.numel())
    n = x.shape[0]
    _lib.check(_lib.load().mri_inpaint_merge(_p(x), _p(known), _p(mask), _p(noise),
                                             _p(rng.state) if rng is not None else None,
                                             int(rng_skip), _p(t), int(t_delta), _p(sqrt_ac),
                                             _p(sqrt_1mac), n, x.numel() // n, _s()),
               "mri_inpaint_merge")


def repaint_undo(x, t, alphas, betas, noise=None, rng: Optional[DeviceRng] = None,
                 rng_skip: int = 0) -> None:
    """RePaint's undo step in place: x = sqrt(alphas[l + 1]) * x + sqrt(betas[l + 1]) * z with
    l = t per sample (device int64 [samples], -1 <= l <= T - 2).  z: `noise`, or with rng the
    torch.randn_like drawn rng_skip past the generator offset."""
    _chk_contig(x, noise)
    assert x.dtype == alphas.dtype == betas.dtype == torch.float32 and t.dtype == torch.int64
    assert noise is None or (noise.dtype == torch.float32 and noise.numel() == x.numel())
    n = x.shape[0]
    _lib.check(_lib.load().mri_repaint_undo(_p(x), _p(noise),
                                            _p(rng.state) if rng is not None else None,
                                            int(rng_skip), _p(t), _p(alphas), _p(betas), n,
                                            x.numel() // n, _s()),
               "mri_repaint_undo")


def step_advance(t: torch.Tensor, delta: int, t_prev=None, rng: Optional[DeviceRng] = None,
                 rng_increment: int = 0) -> None:
    _lib.check(_lib.load().mri_step_advance(_p(t), _p(t_prev), t.numel(), delta,
                                            _p(rng.state) if rng is not None else None,
                                            rng_increment, _s()), "mri_step_advance")


# ------------------------------------------------------------------------------ backward
def gn_bwd_reduce(x, dy, stats, gamma, beta, sums, samples, spatial, C, groups, stats_cpg, eps,
                  silu: bool) -> None:
    _chk_contig(x, dy, sums)
    _lib.check(_lib.load().mri_gn_bwd_reduce(_p(x), _p(dy), _p(stats), _p(gamma), _p(beta), _p(sums),
                                             samples, spatial, C, groups,
                                             stats.shape[1] if stats is not None else 0, stats_cpg,
                                             eps, 1 if silu else 0, _s()), "mri_gn_bwd_reduce")


def colsum(dy, sums, samples, spatial, C) -> None:
    """sums[0][n][c] += sum_s dy[n, s, c]"""
    _chk_contig(dy, sums)
    _lib.check(_lib.load().mri_gn_bwd_reduce(None, _p(dy), None, None, None, _p(sums), samples,
                                             spatial, C, 1, 0, 8, 0.0, 0, _s()), "mri_gn_bwd_reduce")


def gn_bwd_apply(x, dy, add, dx, stats, gamma, beta, sums, samples, spatial, C, groups, stats_cpg,
                 eps, silu: bool, colsum=None) -> None:
    _chk_contig(x, dy, add, dx, sums, colsum)
    _lib.check(_lib.load().mri_gn_bwd_apply(_p(x), _p(dy), _p(add), _p(dx), _p(stats), _p(gamma),
                                            _p(beta), _p(sums), samples, spatial, C, groups,
                                            stats.shape[1], stats_cpg, eps, 1 if silu else 0,
                                            _p(colsum), _s()),
               "mri_gn_bwd_apply")


def add_bf16(a, b, out) -> None:
    _chk_contig(a, b, out)
    _lib.check(_lib.load().mri_add_bf16(_p(a), _p(b), _p(out), a.numel(), _s()), "mri_add_bf16")


# ---- split precision mode (csrc/split_precision.cu) ----------------------------------------------
def gn_split(x, y, stats, gamma, beta, samples, spatial, C, groups, stats_cpg, eps, silu, rowbias=None,
             rowbias_ld=0, residual=None, y32=None) -> None:
    """v = act(GroupNorm(x)) (+ rowbias) (+ residual fp32) of x fp32 [samples, spatial, C]; stats None:
    v = x (+ ...).  y: bf16 [samples, spatial, 3C] = [hi | lo | hi] of v, y32: fp32 v (either may be None)."""
    _chk_contig(x, y, y32, residual)
    _lib.check(_lib.load().mri_gn_split(_p(x), _p(y), _p(y32), _p(stats), _p(gamma), _p(beta), _p(rowbias),
                                        rowbias_ld, _p(residual), samples, spatial, C, groups,
                                        stats.shape[1] if stats is not None else 0, stats_cpg, eps,
                                        1 if silu else 0, _s()), "mri_gn_split")


def stats_f32(x, stats, samples, spatial, C, groups) -> None:
    _chk_contig(x, stats)
    _lib.check(_lib.load().mri_stats_f32(_p(x), _p(stats), samples, spatial, C, groups, _s()), "mri_stats_f32")


def split3(src, dst, outer, inner, width, src_outer_ld, src_inner_ld, dst_outer_ld, dst_inner_ld, seg,
           pattern, src_off=0, dst_off=0) -> None:
    lib = _lib.load()
    _lib.check(lib.mri_split3(src.data_ptr() + 4 * src_off, dst.data_ptr() + 2 * dst_off, outer, inner, width,
                              src_outer_ld, src_inner_ld, dst_outer_ld, dst_inner_ld, seg, pattern, _s()),
               "mri_split3")


def softmax_rows_split(S, P, rows, cols, ld_s, ld_p, seg, scale) -> None:
    _lib.check(_lib.load().mri_softmax_rows_split(_p(S), _p(P), rows, cols, ld_s, ld_p, seg, scale, _s()),
               "mri_softmax_rows_split")


def bf16_residual_nchw(x, out, samples, per_sample, out_sample_stride=0, out_off=0) -> None:
    """out[b, out_off : out_off + 2 * per_sample] = [x - bf16(x) | x] (flat channel-major samples)."""
    _chk_contig(x)
    _lib.check(_lib.load().mri_bf16_residual_nchw(_p(x), out.data_ptr() + 4 * out_off, samples, per_sample,
                                                  out_sample_stride or 2 * per_sample, _s()),
               "mri_bf16_residual_nchw")


def copy_window(src, dst, src_off, dst_off, size, add=None) -> None:
    """dst[:, dh0:dh0+nH, dw0:dw0+nW] = src[:, sh0:sh0+nH, sw0:sw0+nW] (+ add), [B, H, W, C] bf16."""
    _chk_contig(src, dst)
    B, sH, sW, C = src.shape
    _lib.check(_lib.load().mri_copy_window_nhwc(_p(src), _p(dst), _p(add) if add is not None else None,
                                                B, sH, sW, dst.shape[1], dst.shape[2], C, src_off[0],
                                                src_off[1], dst_off[0], dst_off[1], size[0], size[1],
                                                _s()), "mri_copy_window_nhwc")


def resize_bilinear(src, dst) -> None:
    _chk_contig(src, dst)
    B, sH, sW, C = src.shape
    _lib.check(_lib.load().mri_resize_bilinear_nhwc(_p(src), _p(dst), B, sH, sW, dst.shape[1],
                                                    dst.shape[2], C, _s()), "mri_resize_bilinear_nhwc")


def resize_bilinear_bwd(dy, dx, add=None) -> None:
    _chk_contig(dy, dx)
    B, sH, sW, C = dx.shape
    _lib.check(_lib.load().mri_resize_bilinear_nhwc_bwd(_p(dy), _p(dx), _p(add) if add is not None else None,
                                                        B, sH, sW, dy.shape[1], dy.shape[2], C, _s()),
               "mri_resize_bilinear_nhwc_bwd")


def softmax_bwd(P, dP, dS, rows, cols, ld_p, ld_dp, scale) -> None:
    _lib.check(_lib.load().mri_softmax_bwd(_p(P), _p(dP), _p(dS), rows, cols, ld_p, ld_dp, scale,
                                           _s()), "mri_softmax_bwd")


def linear_bwd(dZ, X, W, dX=None, dW=None, db=None) -> None:
    _chk_contig(dZ, X, W, dX, dW, db)
    _lib.check(_lib.load().mri_linear_bwd(_p(dZ), _p(X), _p(W), _p(dX), _p(dW), _p(db), dZ.shape[0],
                                          W.shape[1], W.shape[0], _s()), "mri_linear_bwd")


def silu(z, y) -> None:
    _lib.check(_lib.load().mri_silu(_p(z), _p(y), z.numel(), _s()), "mri_silu")


def silu_bwd(z, dy, dz) -> None:
    _lib.check(_lib.load().mri_silu_bwd(_p(z), _p(dy), _p(dz), z.numel(), _s()), "mri_silu_bwd")


def minsnr_loss_bwd(pred, noise, t, snr, gamma, upstream, dpred) -> None:
    _chk_contig(pred, noise, dpred)
    n = pred.shape[0]
    _lib.check(_lib.load().mri_minsnr_loss_bwd(_p(pred), _p(noise), _p(t), _p(snr), gamma,
                                               _p(upstream), _p(dpred), n, pred.numel() // n, _s()),
               "mri_minsnr_loss_bwd")



_DT = {torch.bfloat16: 0, torch.float32: 1, torch.float64: 2}


def copy_cast(src: torch.Tensor, dst: torch.Tensor) -> None:
    """dst <- src (same shape, any strides, up to 4 dims after merging; bf16/f32/f64 -> bf16/f32):
    what `dst.copy_(src)` does, through mri_copy_cast."""
    import ctypes as C
    if tuple(src.shape) != tuple(dst.shape) or src.dim() > 4:
        raise _lib.MriError(f"copy_cast: shapes {tuple(src.shape)} -> {tuple(dst.shape)} unsupported")
    pad = 4 - src.dim()
    shape = (C.c_int64 * 4)(*([1] * pad + list(src.shape)))
    ss = (C.c_int64 * 4)(*([0] * pad + list(src.stride())))
    ds = (C.c_int64 * 4)(*([0] * pad + list(dst.stride())))
    _lib.check(_lib.load().mri_copy_cast(_p(src), _DT[src.dtype], ss, _p(dst), _DT[dst.dtype], ds,
                                         shape, _s()), "mri_copy_cast")


def memset_zero(t: torch.Tensor, nbytes: Optional[int] = None) -> None:
    """Zero the first `nbytes` bytes of t's storage view (cudaMemsetAsync on the current stream)."""
    _chk_contig(t)
    n = t.numel() * t.element_size() if nbytes is None else int(nbytes)
    _lib.check(_lib.load().mri_memset_zero(_p(t), n, _s()), "mri_memset_zero")


# ---- data path (csrc/data_path.cu) ---------------------------------------------------------------
def _f32_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise _lib.MriError(f"{what}: needs a CUDA tensor (no CPU path)")
    if t.dtype != torch.float32:
        raise _lib.MriError(f"{what}: needs float32, got {t.dtype}")


def masked_stats(x: torch.Tensor, item_dim: Optional[int] = None, eps: float = 0.0) -> torch.Tensor:
    """fp32 [items, 2] = (mean, std) over the non-zero elements of each item of x (any strides).
    x is 2-D (one item) / 3-D with the item axis `item_dim`; or any contiguous tensor with
    item_dim=None (one item: the whole tensor).  Rules for std: see mri_masked_stats."""
    _f32_cuda(x, "masked_stats")
    if item_dim is None:
        if not x.is_contiguous():
            raise _lib.MriError("masked_stats: a whole-tensor item must be contiguous")
        items, ist, rows, cols, rs, cs = 1, 0, 1, x.numel(), 0, 1
    else:
        if x.dim() != 3:
            raise _lib.MriError("masked_stats: item_dim needs a 3-D tensor")
        item_dim %= 3
        r, c = [d for d in range(3) if d != item_dim]
        items, ist = x.shape[item_dim], x.stride(item_dim)
        rows, cols, rs, cs = x.shape[r], x.shape[c], x.stride(r), x.stride(c)
        if cs != 1 and rs == 1:          # statistics do not care which axis is called "row"
            rows, cols, rs, cs = cols, rows, cs, rs
        if items == 1 and cs != 1:       # a single strided slice: the item-major kernel, one lane
            ist = 1
    with torch.cuda.device(x.device):
        acc = torch.empty(items, 3, dtype=torch.float64, device=x.device)
        out = torch.empty(items, 2, dtype=torch.float32, device=x.device)
        _lib.check(_lib.load().mri_masked_stats(_p(x), items, ist, rows, cols, rs, cs,
                                                float(eps), _p(acc), _p(out), _s()),
                   "mri_masked_stats")
    return out


def slice_normalize_resize(x: torch.Tensor, item_dim: int, mean_std: torch.Tensor,
                           out: torch.Tensor) -> None:
    """out[i] (a contiguous [S_h, S_w] block per item; out is [items, S_h, S_w] or any view whose
    last two dims are contiguous, e.g. batch[:, c0:c0+items] of a [B, C, S, S] tensor with B == 1,
    or batch[:, c] with one item per sample) <- normalised, bilinearly resized slice i of the 3-D
    tensor x, mapped to [-1, 1]."""
    _f32_cuda(x, "slice_normalize_resize")
    _f32_cuda(out, "slice_normalize_resize")
    if x.dim() != 3 or out.dim() != 3:
        raise _lib.MriError("slice_normalize_resize: x and out must be 3-D (items on one axis)")
    item_dim %= 3
    r, c = [d for d in range(3) if d != item_dim]
    items = x.shape[item_dim]
    if out.shape[0] != items or out.stride(2) != 1 or out.stride(1) != out.shape[2]:
        raise _lib.MriError("slice_normalize_resize: out must be [items, S_h, S_w] with contiguous "
                            "slices")
    if tuple(mean_std.shape) != (items, 2) or not mean_std.is_contiguous():
        raise _lib.MriError("slice_normalize_resize: mean_std must be contiguous [items, 2]")
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().mri_slice_normalize_resize(
            _p(x), items, x.stride(item_dim), x.shape[r], x.shape[c], x.stride(r), x.stride(c),
            _p(mean_std), out.shape[1], out.shape[2], _p(out), out.stride(0), _s()),
            "mri_slice_normalize_resize")


def volume_normalize_patch(vol_dhw: torch.Tensor, mean_std: torch.Tensor, origin, out: torch.Tensor,
                           clip: float = 5.0) -> None:
    """out (contiguous [pd, ph, pw]) <- normalised patch of the (D, H, W)-indexed view vol_dhw (any
    strides, e.g. nib_array.permute(2, 0, 1)) whose first voxel is vol_dhw[origin]; positions
    outside the volume are the zero padding."""
    _f32_cuda(vol_dhw, "volume_normalize_patch")
    _f32_cuda(out, "volume_normalize_patch")
    if vol_dhw.dim() != 3 or out.dim() != 3 or not out.is_contiguous():
        raise _lib.MriError("volume_normalize_patch: vol must be 3-D, out contiguous 3-D")
    D, H, W = vol_dhw.shape
    sd, sh, sw = vol_dhw.stride()
    od, oh, ow = (int(v) for v in origin)
    with torch.cuda.device(vol_dhw.device):
        _lib.check(_lib.load().mri_volume_normalize_patch(
            _p(vol_dhw), D, H, W, sd, sh, sw, _p(mean_std), float(clip), od, oh, ow, out.shape[0],
            out.shape[1], out.shape[2], _p(out), _s()), "mri_volume_normalize_patch")
