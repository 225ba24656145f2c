"""Static-shape inference programs for the 3D VAE of the latent-diffusion package
(ddpm_3d_ldm/vae.py): the step either side of the diffusion hot path -- `encode_to_latent`
before every LDM training step (ddpm_3d_ldm/train.py:386-388) and `decode_from_latent` after
sampling (ddpm_3d_ldm/show_model.py:255).

Same kernels as the UNets (engine.py): tcgen05 implicit-GEMM convolutions with fused bias /
residual / GroupNorm partial sums, one fused GroupNorm-apply + SiLU pass per norm, 1x1 skip
convolutions folded into conv2's K loop, im2col'd thin input convolutions and the
GEMM-over-taps + gather head for the thin output convolutions.

Channel counts below 64 (the VAE's 32-channel full-resolution level) are zero-padded to 64 so
that every K slab is 64 channels wide; the padding channels stay exactly zero through
GroupNorm (gamma = beta = 0 there), SiLU and the convolutions (zero weight rows / columns), and
GroupNorm(8, 32) runs as 16 groups of 4 channels over the padded tensor.

Training (stage 1 of ddpm_3d_ldm/train.py:258-300, `recon, mu, logvar = vae(x)` under autocast +
GradScaler + DDP): `training=True` programs record the same tape as the UNets and replay it in
reverse (backward.py) -- data gradients on the tensor-core kernel through adjoint plans, weight
gradients on the MN-major kernel, GroupNorm+SiLU backward as two bf16 passes.  What is specific
to the VAE is the channel padding: every record carries how to read the parameter gradient out of
the padded wgrad matrix (`unpack`) and the zero-padded weights the adjoint plans are packed from
(`wfull`); GroupNorm(8, 32) over the padded tensor is 16 groups of 4 channels (the `kFine`
instantiation of the GroupNorm backward kernels).  The encoder and the decoder are two programs
joined by the reparameterisation in between (three tiny element-wise torch ops on the latent); the
decoder program returns the gradient of its input latent.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import _lib, ops
from . import plan as P
from .backward import ConvRec
from .engine import Act, UNetProgram, _pad_vec, _rup


def _pad_cin(w: torch.Tensor, cin_pad: int) -> torch.Tensor:
    """Zero-pad dim 1 (input channels of a Conv weight / output channels of a ConvTranspose)."""
    if w.shape[1] == cin_pad:
        return w
    out = torch.zeros(w.shape[0], cin_pad, *w.shape[2:], dtype=w.dtype, device=w.device)
    out[:, :w.shape[1]] = w
    return out


def _pad_c0(w: torch.Tensor, c0_pad: int) -> torch.Tensor:
    if w.shape[0] == c0_pad:
        return w
    out = torch.zeros(c0_pad, *w.shape[1:], dtype=w.dtype, device=w.device)
    out[:w.shape[0]] = w
    return out


class VAE3DProgram(UNetProgram):
    """mode 'encode': x (B, Cin, D, H, W) fp32 -> [mu | logvar] (B, 2*latent, d, h, w) fp32
    (Encoder3D.forward, vae.py:49-55);
    mode 'decode': z (B, latent, d, h, w) fp32 -> reconstruction (B, Cout, D, H, W) fp32
    (Decoder3D.forward, vae.py:82-87).

    wgrad=False (training programs only): the backward computes data gradients alone -- for the
    decoder, dz_out = D^T dout without any parameter gradient, as measurement-guided sampling needs
    (diffusion_base._guided_loop).  Its forward and dz_out are the training program's, bit for bit."""

    def __init__(self, vae, mode: str, batch: int, spatial: Sequence[int], training: bool = False,
                 wgrad: bool = True):
        dev = next(vae.parameters()).device
        enc, dec = vae.encoder, vae.decoder
        first_block = enc.downs[0] if mode == "encode" else dec.ups[0]
        self.gn_groups = first_block.norm1.num_groups
        super().__init__(dev, batch, spatial, groups=self.gn_groups, training=training)
        if not wgrad and not training:
            raise _lib.MriError("VAE3DProgram: wgrad=False applies to training programs")
        self.wgrad = wgrad
        self.dz_out: Optional[torch.Tensor] = None
        self.mode = mode
        if len(self.sp) != 3:
            raise _lib.MriError("VAE3D expects 3 spatial dims")
        self.eps_gn = first_block.norm1.eps
        B = batch
        if mode == "encode":
            n_down = enc.num_down
            for s in self.sp:
                if s % (2 ** (n_down - 1)) != 0:
                    raise _lib.MriError(f"volume size {self.sp} must be divisible by {2 ** (n_down - 1)}")
            cin = enc.in_conv.weight.shape[1]
            self.x_in = torch.zeros(B, cin, *self.sp, device=dev)
            h = self.thin_in_conv(self.x_in, enc.in_conv, self.sp, "encoder.in_conv")
            for i, layer in enumerate(enc.downs):
                h = self.layer(h, layer, f"encoder.downs.{i}")
            self.head(h, enc.to_mu_logvar, "encoder.to_mu_logvar")
        elif mode == "decode":
            lat = dec.from_latent.weight.shape[1]
            self.x_in = torch.zeros(B, lat, *self.sp, device=dev)
            if training:
                h = self.latent_in_conv(self.x_in, dec.from_latent, self.sp, "decoder.from_latent")
            else:
                h = self.thin_in_conv(self.x_in, dec.from_latent, self.sp, "decoder.from_latent")
            for i, layer in enumerate(dec.ups):
                h = self.layer(h, layer, f"decoder.ups.{i}")
            self.head(h, dec.out_conv, "decoder.out_conv")
        else:
            raise ValueError(mode)
        self.params_changed()
        if training:
            self.dout_in = torch.zeros_like(self.out)
            self.deps16 = torch.zeros_like(self.eps_nhwc)
            self.build_backward({id(self.eps_nhwc): self.deps16})
            if mode == "decode":
                self.dz64 = self.grads[id(self.z64)]
                self.dz_out = torch.zeros_like(self.x_in)

    # ------------------------------------------------------------------ helpers
    def cpad(self, c: int) -> int:
        return _rup(c, 64)

    def groups_of(self, c_real: int) -> int:
        """Normalisation groups over the padded tensor (real groups + all-zero padding groups)."""
        cpg = c_real // self.gn_groups
        if c_real % self.gn_groups or cpg % 4:
            raise _lib.MriError(f"GroupNorm({self.gn_groups}, {c_real}): channels per group must be a "
                                "multiple of 4 on the B200 path")
        return self.cpad(c_real) // cpg

    def new_vact(self, sp: Sequence[int], c_real: int) -> Act:
        """Activation [B, *sp, cpad(c)] whose producer convolution can emit GroupNorm partial
        sums (swap-mode epilogue: any power-of-two group width)."""
        cp = self.cpad(c_real)
        t = self.pool.get((self.B, *sp, cp))
        g = self.groups_of(c_real)
        return Act(t, self.new_stats(g), cp // g)

    def ensure_stats(self, x: Act, c_real: int, name: str) -> None:
        if x.stats is not None:
            return
        g = self.groups_of(c_real)
        x.stats = self.new_stats(g)
        x.cpg = x.C // g
        B, S, C, xs, st, cpg = self.B, x.spatial, x.C, x.t, x.stats, x.cpg
        self._add(f"{name}.stats", lambda: ops.gn_stats(xs, st, B, S, C, cpg), [st])

    def norm_silu(self, x: Act, norm, c_real: int, name: str) -> torch.Tensor:
        self.ensure_stats(x, c_real, name)
        cp = x.C
        self.track(norm.weight, norm.bias)
        gm = self.packed(lambda: _pad_vec(norm.weight.detach(), cp))
        bt = self.packed(lambda: _pad_vec(norm.bias.detach(), cp))
        return self.gn(x, gm, bt, self.groups_of(c_real), norm.eps, True, name=name,
                       gparam=norm.weight, bparam=norm.bias)

    # ---- what the backward pass needs to know about a channel-padded convolution ------------
    @staticmethod
    def _conv_rec_pads(conv, cop: int, cip: int, extra=None, ecip: int = 0) -> dict:
        """nn.Conv3d weight [Cout, Cin, k, k, k] run as [cop, cip, ...]: `unpack` reads the real
        block out of the packed wgrad matrix [1, rows, taps * cip (+ ecip)], `wfull` is the padded
        weight the adjoint (dgrad) plans are packed from; `extra` = the folded 1x1 skip."""
        cout, cin = conv.weight.shape[0], conv.weight.shape[1]
        kshape = tuple(conv.weight.shape[2:])
        eshape = [(cout, ecip)] if extra is not None else []

        def unpack(d):
            return P.unpack_conv_wgrad(d[0], (cout, cip) + kshape, [cip], eshape)[0][:, :cin]

        rec = dict(unpack=unpack, wfull=lambda: _pad_c0(_pad_cin(conv.weight.detach(), cip), cop))
        if extra is not None:
            ecin = extra.weight.shape[1]
            rec["unpack_extra"] = lambda d: P.unpack_conv_wgrad(
                d[0], (cout, cip) + kshape, [cip], eshape)[1][0][:, :ecin].reshape(extra.weight.shape)
            rec["efull"] = lambda: _pad_c0(_pad_cin(extra.weight.detach().reshape(cout, ecin), ecip), cop)
        return rec

    def latent_in_conv(self, x_in: torch.Tensor, conv, sp, name: str) -> Act:
        """Training: from_latent (vae.py:67) over a channels-last bf16 copy of z padded to 64
        channels -- an ordinary 3x3x3 convolution whose adjoint gives the gradient of z.  The
        latent volume is 1/64 (num_down = 3) of the image: the padding costs nothing."""
        B, S = self.B, sp[0] * sp[1] * sp[2]
        cout, lat = conv.weight.shape[0], conv.weight.shape[1]
        if lat > 64:
            raise _lib.MriError("VAE3D training: more than 64 latent channels are not supported")
        cop = self.cpad(cout)
        self.track(conv.weight, conv.bias)
        z64 = torch.zeros(B, *sp, 64, dtype=torch.bfloat16, device=self.device)
        self._add(f"{name}.nhwc", lambda: ops.nchw_to_nhwc(x_in, z64, B, S, lat, 64), [z64])
        w = self.packed(lambda: P.pack_conv_weight(_pad_cin(conv.weight.detach(), 64), cout_pad=cop))
        b = self.packed(lambda: _pad_vec(conv.bias.detach(), cop))
        h = self.new_vact(sp, cout)
        pl = P.conv_plan([P.ConvSource(z64)], w, h.t, 3, bias=b, stats=h.stats, stats_cpg=h.cpg, name=name)
        self._conv_or_stats(pl, h)
        self.tape.append(ConvRec(kind="conv", plan=pl, y=h.t, ksize=3, sources=[(z64, True)],
                                 weight=conv.weight, splits=[64], bias_params=[conv.bias], cout=cout,
                                 name=name, **self._conv_rec_pads(conv, cop, 64)))
        self.z64 = z64
        return h

    def thin_in_conv(self, x_in: torch.Tensor, conv, sp, name: str) -> Act:
        """Conv3d with 1..8 input channels: patch matrix + GEMM (vae.py:31,67)."""
        B, S = self.B, sp[0] * sp[1] * sp[2]
        cout, cin = conv.weight.shape[0], conv.weight.shape[1]
        self.track(conv.weight, conv.bias)
        cp = self.cpad(cout)
        col, w0, kpad = self.thin_patch_matrix(x_in, conv, sp, name)
        w = w0 if cp == cout else self.packed(lambda: _pad_c0(w0, cp))
        b = self.packed(lambda: _pad_vec(conv.bias.detach(), cp))
        h = self.new_vact(sp, cout)
        a = P.TView(col, (kpad, S, B, 1, 1), (1, kpad, S * kpad, B * S * kpad, B * S * kpad))
        bv = P.TView(w, (kpad, cp, 1, 1), (1, kpad, kpad * cp, kpad * cp))
        o = P.TView(h.t, (cp, S, B, 1, 1), (1, cp, S * cp, B * S * cp, B * S * cp))
        pl = P.matrix_plan(a, (128, 1, 1, 1), bv, o, K=kpad, n_total=cp, block_n=P.pick_block_n(cp),
                           ext=(S, B, 1, 1), tiles=(-(-S // 128), B, 1, 1), sample_dim=2, bias=b,
                           stats=h.stats, stats_cpg=h.cpg, name=name, flops=2 * B * S * cp * kpad)
        self.gemm(pl)
        if self.training:   # the image needs no gradient: weight / bias gradients only
            c4, kk = _rup(cin, 4), tuple(conv.weight.shape[2:])
            taps = kk[0] * kk[1] * kk[2]
            self.tape.append(ConvRec(
                kind="matrix", plan=pl, y=h.t, ksize=kk[0], sources=[(col, True)], weight=conv.weight,
                splits=[cin], bias_params=[conv.bias], cout=cout, need_dgrad=False, kpad=kpad, name=name,
                unpack=lambda d: P.unpack_conv_wgrad(d[0][:, :taps * c4], (cout, c4) + kk)[0][:, :cin]))
        return h

    def layer(self, h: Act, layer, name: str) -> Act:
        if isinstance(layer, torch.nn.ConvTranspose3d):
            return self.up(h, layer, name)
        if isinstance(layer, torch.nn.Conv3d):
            return self.down(h, layer, name)
        return self.resblock(h, layer, name)

    def resblock(self, x: Act, blk, name: str) -> Act:
        """ResidualBlock3DNoTime.forward (vae.py:19-22): conv2(silu(gn2(conv1(silu(gn1(x)))))) + skip(x)."""
        c1, c2 = blk.conv1, blk.conv2
        cin, cout = c1.weight.shape[1], c1.weight.shape[0]
        cip, cop = self.cpad(cin), self.cpad(cout)
        sp = tuple(x.t.shape[1:-1])
        self.track(c1.weight, c1.bias, c2.weight, c2.bias)
        a1 = self.norm_silu(x, blk.norm1, cin, f"{name}.norm1")
        w1 = self.packed(lambda: P.pack_conv_weight(_pad_cin(c1.weight.detach(), cip), cout_pad=cop))
        b1 = self.packed(lambda: _pad_vec(c1.bias.detach(), cop))
        h = self.new_vact(sp, cout)
        pl = P.conv_plan([P.ConvSource(a1)], w1, h.t, 3, bias=b1, stats=h.stats, stats_cpg=h.cpg,
                         name=f"{name}.conv1")
        self._conv_or_stats(pl, h)
        if self.training:
            self.tape.append(ConvRec(kind="conv", plan=pl, y=h.t, ksize=3, sources=[(a1, True)],
                                     weight=c1.weight, splits=[cip], bias_params=[c1.bias], cout=cout,
                                     name=f"{name}.conv1", **self._conv_rec_pads(c1, cop, cip)))
        self.pool.release(a1)
        a2 = self.norm_silu(h, blk.norm2, cout, f"{name}.norm2")
        self.pool.release(h.t)
        out = self.new_vact(sp, cout)
        if isinstance(blk.skip, torch.nn.Identity):
            w2 = self.packed(lambda: P.pack_conv_weight(_pad_cin(c2.weight.detach(), cop), cout_pad=cop))
            b2 = self.packed(lambda: _pad_vec(c2.bias.detach(), cop))
            pl = P.conv_plan([P.ConvSource(a2)], w2, out.t, 3, bias=b2, residual=x.t, stats=out.stats,
                             stats_cpg=out.cpg, name=f"{name}.conv2")
            rec = ConvRec(kind="conv", plan=pl, y=out.t, ksize=3, sources=[(a2, True)], weight=c2.weight,
                          splits=[cop], bias_params=[c2.bias], residual=x.t, cout=cout,
                          name=f"{name}.conv2", **self._conv_rec_pads(c2, cop, cop))
        else:
            sk = blk.skip
            self.track(sk.weight, sk.bias)
            w2 = self.packed(lambda: P.pack_conv_weight(
                _pad_cin(c2.weight.detach(), cop), cout_pad=cop,
                extra=[_pad_cin(sk.weight.detach().reshape(cout, cin), cip)]))
            b2 = self.packed(lambda: _pad_vec(c2.bias.detach() + sk.bias.detach(), cop))
            pl = P.conv_plan([P.ConvSource(a2), P.ConvSource(x.t, taps=False)], w2, out.t, 3, bias=b2,
                             stats=out.stats, stats_cpg=out.cpg, name=f"{name}.conv2+skip")
            rec = ConvRec(kind="conv", plan=pl, y=out.t, ksize=3, sources=[(a2, True), (x.t, False)],
                          weight=c2.weight, splits=[cop], extra_weight=sk.weight,
                          bias_params=[c2.bias, sk.bias], cout=cout, name=f"{name}.conv2+skip",
                          **self._conv_rec_pads(c2, cop, cop, extra=sk, ecip=cip))
        self._conv_or_stats(pl, out)
        if self.training:
            self.tape.append(rec)
        self.pool.release(a2)
        self.pool.release(x.t)
        return out

    def _conv_or_stats(self, pl: P.GemmPlan, y: Act) -> None:
        """Emit the convolution; if its epilogue cannot produce statistics at this group width
        (normal mode needs groups of >= 8 channels) leave them to a standalone pass."""
        if not pl.pick_swap() and y.cpg % 8 != 0:
            pl.stats, pl.stats_ld, pl.stats_cpg = None, 0, 0
            y.stats = None
        self.gemm(pl)

    def down(self, x: Act, conv, name: str) -> Act:
        """Conv3d k=4 s=2 p=1 (vae.py:41-43)."""
        c = conv.weight.shape[0]
        cp = self.cpad(c)
        self.track(conv.weight, conv.bias)
        w = self.packed(lambda: P.pack_conv_weight(_pad_cin(conv.weight.detach(), cp), cout_pad=cp))
        b = self.packed(lambda: _pad_vec(conv.bias.detach(), cp))
        y = self.new_vact([s // 2 for s in x.t.shape[1:-1]], c)
        pl = P.down_conv_plan(x.t, w, y.t, bias=b, stats=y.stats, stats_cpg=y.cpg, name=name)
        self._conv_or_stats(pl, y)
        if self.training:
            self.tape.append(ConvRec(kind="down", plan=pl, y=y.t, ksize=4, sources=[(x.t, True)],
                                     weight=conv.weight, splits=[cp], bias_params=[conv.bias], cout=c,
                                     name=name, **self._conv_rec_pads(conv, cp, cp)))
        self.pool.release(x.t)
        return y

    def up(self, x: Act, conv, name: str) -> Act:
        """ConvTranspose3d k=4 s=2 p=1 (vae.py:75-79); weight layout [Cin, Cout, 4, 4, 4]."""
        c = conv.weight.shape[1]
        cp = self.cpad(c)
        cip = self.cpad(conv.weight.shape[0])
        self.track(conv.weight, conv.bias)
        w = self.packed(lambda: P.pack_convT_weight(_pad_c0(_pad_cin(conv.weight.detach(), cp), cip),
                                                    cout_pad=cp))
        b = self.packed(lambda: _pad_vec(conv.bias.detach(), cp))
        y = self.new_vact([s * 2 for s in x.t.shape[1:-1]], c)
        pl = P.up_conv_plan(x.t, w, y.t, bias=b, stats=y.stats, stats_cpg=y.cpg, name=name)
        self._conv_or_stats(pl, y)
        if self.training:
            cin_r, wshape = conv.weight.shape[0], tuple(conv.weight.shape)
            self.tape.append(ConvRec(
                kind="up", plan=pl, y=y.t, ksize=4, sources=[(x.t, True)], weight=conv.weight,
                splits=[cip], bias_params=[conv.bias], cout=c, name=name,
                unpack=lambda d: P.unpack_convT_wgrad(d, (cip, c) + wshape[2:])[:cin_r],
                wfull=lambda: _pad_c0(_pad_cin(conv.weight.detach(), cp), cip)))
        self.pool.release(x.t)
        return y

    def head(self, h: Act, conv, name: str) -> None:
        """Thin-Cout 3x3x3 convolution WITHOUT a preceding norm (to_mu_logvar vae.py:47,
        out_conv vae.py:81): GEMM over taps + gather."""
        self.sp_out = tuple(h.t.shape[1:-1])
        if not self.training:
            self.thin_out_conv(h.t, conv, name=name, cin_pad=h.C)
        else:
            cout, cin = conv.weight.shape[0], conv.weight.shape[1]
            if cout > 64:
                raise _lib.MriError("VAE3D training: more than 32 latent channels are not supported")
            self.cout, self.cout_pad = cout, _rup(cout, 16)
            cip, cop = h.C, self.cout_pad
            self.track(conv.weight, conv.bias)
            w_out = self.packed(lambda: P.pack_conv_weight(_pad_cin(conv.weight.detach(), cip), cout_pad=cop))
            b_out = self.packed(lambda: _pad_vec(conv.bias.detach(), cop))
            # the adjoint convolution reads a 64-channel copy of dY (K slabs are 64 channels wide)
            self.deps64 = torch.zeros(self.B, *self.sp_out, 64, dtype=torch.bfloat16, device=self.device)
            rec = self._conv_rec_pads(conv, cop, cip)
            rec["wfull"] = lambda: _pad_cin(conv.weight.detach(), cip)   # rows padded to dY's 64 later
            y = self.conv([P.ConvSource(h.t)], w_out, cop, 3, b_out, with_stats=False, name=name,
                          rec=dict(weight=conv.weight, splits=[cip], bias_params=[conv.bias], cout=cout,
                                   dgrad_dy=self.deps64, **rec))
            self.eps_nhwc = y.t
        self.out = torch.zeros(self.B, self.cout, *self.sp_out, device=self.device)

    # ------------------------------------------------------------------ entry
    def backward(self, dout: torch.Tensor, sync=None) -> None:
        """Gradient of the loss w.r.t. the fp32 NCDHW output -> parameter gradients in the arena
        (and, for the decoder, the gradient of the input latent in self.dz_out)."""
        self._backward(dout, self.sp_out[0] * self.sp_out[1] * self.sp_out[2], sync)

    def _bwd_tail(self) -> None:
        if self.dz_out is not None:
            S = self.sp[0] * self.sp[1] * self.sp[2]
            ops.nhwc_to_nchw(self.dz64, self.dz_out, self.B, S, self.dz_out.shape[1], 64)

    def finish_output(self) -> None:
        """self.out (fp32 NCDHW) from the last run()'s channels-last output."""
        S = self.sp_out[0] * self.sp_out[1] * self.sp_out[2]
        ops.nhwc_to_nchw(self.eps_nhwc, self.out, self.B, S, self.cout, self.cout_pad)

    def run_input_backward(self) -> None:
        """The backward launches on what dout_in holds, enqueued without a graph of their own (a
        caller's step graph captures them): dz_out = D^T dout_in after the last run()."""
        self._bwd_head(self.sp_out[0] * self.sp_out[1] * self.sp_out[2])
        self.run_backward()
        self._bwd_tail()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if self.params_changed():
            self.do_refresh()
        self.x_in.copy_(x)
        self.run()
        self.finish_output()
        return self.out
