"""Backward program of the UNet engines (training).

The forward builder (engine.py) records one tape entry per op; `build_backward()` walks the tape
in reverse and emits the launch list that computes what autograd computes for the reference
modules: data gradients on the forward tensor-core kernel through adjoint plans (flipped /
transposed packed weights; stride-2 <-> parity-decomposed transposed convolution), weight
gradients on the MN-major tcgen05 kernel (mri_wgrad_launch) over the forward k-tables,
GroupNorm(+SiLU) backward as two bf16 passes, the attention backward as GEMMs + a fused
softmax-backward, and the tiny fp32 linears of the time embedding.

Gradient buffers are bf16 channels-last like the activations; parameter gradients are fp32 in
the reference parameter layout (what `.grad` must hold).
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, ops
from . import plan as P


@dataclass
class ConvRec:
    kind: str                      # 'conv' | 'down' | 'up' | 'matrix'
    plan: P.GemmPlan
    y: torch.Tensor                # forward output tensor (channels-last bf16)
    ksize: int
    sources: List[Tuple[torch.Tensor, bool]]    # (tensor, has_taps)
    weight: Optional[torch.Tensor]              # nn.Parameter in the reference layout
    splits: List[int]
    extra_weight: Optional[torch.Tensor] = None  # folded 1x1 skip weight [Cout, sum(centre srcs)]
    bias_params: List[torch.Tensor] = field(default_factory=list)
    residual: Optional[torch.Tensor] = None
    tproj_off: Optional[int] = None
    cout: int = 0
    need_dgrad: bool = True
    w_rows: Optional[Tuple[int, int]] = None     # use only weight rows [a, b) (qkv slices)
    kpad: int = 0                                # 'matrix': padded K of the im2col'd weight
    dgrad_dy: Optional[torch.Tensor] = None      # 64-channel copy of dY when Cout is thin (out_conv)
    # channel-padded layers (the VAE's 32-channel level runs zero-padded to 64, vae_engine.py):
    # how to read the parameter gradients out of the packed wgrad matrix, and the zero-padded
    # reference-layout weights the adjoint plans are packed from
    unpack: Optional[Callable[[torch.Tensor], torch.Tensor]] = None
    unpack_extra: Optional[Callable[[torch.Tensor], torch.Tensor]] = None
    wfull: Optional[Callable[[], torch.Tensor]] = None
    efull: Optional[Callable[[], torch.Tensor]] = None
    name: str = ""


@dataclass
class GnRec:
    x: object                      # engine.Act (tensor + statistics)
    y: torch.Tensor
    gamma: torch.Tensor            # parameter
    beta: torch.Tensor
    c_off: int
    groups: int
    eps: float
    silu: bool
    tproj_off: Optional[int] = None
    residual: Optional[torch.Tensor] = None
    name: str = ""
    gparam: Optional[torch.Tensor] = None   # the nn.Parameters when gamma / beta are zero-padded
    bparam: Optional[torch.Tensor] = None   # packed copies (vae_engine.py)


@dataclass
class WindowRec:
    """dst[:, d0:d0+n] = src[:, s0:s0+n] over (H, W) of channels-last tensors (zero padding an odd
    level in front of the stride-2 convolution / cropping its output)."""
    src: torch.Tensor
    dst: torch.Tensor
    src_off: Tuple[int, int]
    dst_off: Tuple[int, int]
    size: Tuple[int, int]
    name: str = ""


@dataclass
class ResizeRec:
    """dst = bilinear resize of src (slice_cond_2d_ddpm/unet.py:98-99)."""
    src: torch.Tensor
    dst: torch.Tensor
    name: str = ""


@dataclass
class AttnRec:
    x: object
    hn: torch.Tensor
    qkv: torch.Tensor
    kvT: torch.Tensor
    Pm: torch.Tensor
    O: torch.Tensor
    out: torch.Tensor
    blk: object
    qkv_plan: P.GemmPlan
    proj_plan: P.GemmPlan
    heads: int
    n: int
    npad: int
    name: str = ""


@dataclass
class TimeRec:
    """time_mlp (+ slice_mlp) + concatenated per-block projections."""
    sin: torch.Tensor
    z1: torch.Tensor
    h1: torch.Tensor
    temb: torch.Tensor
    l1: object
    l2: object
    cond: torch.Tensor             # input of the block projections (temb, or temb + z_emb in 2D)
    W_all: torch.Tensor
    zproj: torch.Tensor            # pre-activation of the projections
    act: int
    blocks: Sequence
    offs: List[int]
    slice: Optional[dict] = None   # 2D: {"z_in", "zz", "zh", "s0", "s2"}


def _noop() -> None:
    return None


class BackwardMixin:
    """Mixed into engine.UNetProgram."""

    # ------------------------------------------------------------------ bookkeeping
    def _binit(self):
        self.tape: List[object] = []
        self.grads: Dict[int, torch.Tensor] = {}
        self.pgrad: Dict[int, torch.Tensor] = {}
        self.bwd_ops: List[Callable[[], None]] = []
        self.bwd_names: List[str] = []
        self._zero_each_bwd: List[list] = []   # [uint8 chunk, bytes used]
        self.dtproj: Optional[torch.Tensor] = None
        self.bwd_flops = 0
        # id(gradient tensor) -> [colsum buffer or None] when its LAST writer is a gn_bwd_apply
        # launch (which can then emit the tensor's per-(sample, channel) sums for free)
        self._gn_writer: Dict[int, Optional[list]] = {}
        # parameter gradients live in ONE flat fp32 arena, allocated in the order the backward
        # pass first touches them, so that "everything ready after op k" is a prefix of the
        # arena: DDP buckets are contiguous slices (parallel.GradSync)
        self.garena: Optional[torch.Tensor] = None
        self._garena_used = 0
        self._g_off: Dict[int, Tuple[int, int]] = {}      # id(param) -> (offset, numel)
        self._g_last_op: Dict[int, int] = {}              # id(param) -> index of the last op of
        self._g_touched: List[int] = []                   # ... the last tape record touching it
        self.bwd_segments: List[Tuple[int, int, int, int]] = []  # (op_lo, op_hi, arena_lo, arena_hi)
        self.bwd_ranges: List[Tuple[int, int]] = []   # ops [lo, hi) of each tape record, in tape order
        # deferred parameter-gradient finalisers: (op index, dst, src, idx or None, batch, ld);
        # all finalisers of a launch range run as ONE mri_grad_finalize launch at its end
        self._final: List[Tuple[int, torch.Tensor, torch.Tensor, Optional[torch.Tensor], int, int]] = []
        self._final_tables: Dict[Tuple[int, int], Optional[tuple]] = {}
        self._fuse_final = os.environ.get("MRI_NO_FINAL_FUSION") != "1"
        # False: data gradients only -- no weight-gradient launches, bias / norm-parameter sums or
        # final gathers, and no gradient arena (a decoder differentiated w.r.t. its input alone)
        self.wgrad = True

    def badd(self, name: str, fn: Callable[[], None]) -> None:
        self.bwd_names.append(name)
        self.bwd_ops.append(fn)

    def bfinal_gather(self, dst: torch.Tensor, src: torch.Tensor, fn: Callable[[torch.Tensor], torch.Tensor],
                      name: str = "unpack") -> None:
        """dst <- fn(src) where fn only re-orders elements (reshape / permute / cat / slicing).
        The element map is read off by running fn on element indices once; at run time it is a
        segment of the range's single mri_grad_finalize launch."""
        assert dst.is_contiguous() and src.is_contiguous() and dst.dtype == src.dtype == torch.float32
        if not self._fuse_final:
            self.badd(name, lambda: dst.copy_(fn(src).reshape(dst.shape)))
            return
        probe = torch.arange(1, src.numel() + 1, dtype=torch.int32, device=src.device).view(src.shape)
        idx = (fn(probe).reshape(-1) - 1).to(torch.int32).contiguous()
        assert idx.numel() == dst.numel(), (name, idx.numel(), dst.numel())
        self._final.append((len(self.bwd_ops), dst, src, idx, 0, 0))
        self.badd(name, _noop)

    def bfinal_bsum(self, dst: torch.Tensor, src: torch.Tensor, name: str) -> None:
        """dst[i] <- sum_b src[b, i] (src fp64 [batch, ld], dst fp32 [n <= ld])."""
        assert dst.is_contiguous() and src.is_contiguous() and src.dim() == 2
        assert dst.dtype == torch.float32 and src.dtype == torch.float64 and dst.numel() <= src.shape[1]
        if not self._fuse_final:
            n = dst.numel()
            self.badd(name, lambda: dst.copy_(src.sum(0)[:n]))
            return
        self._final.append((len(self.bwd_ops), dst, src, None, src.shape[0], src.shape[1]))
        self.badd(name, _noop)

    def _final_table(self, lo: int, hi: int):
        key = (lo, hi)
        if key not in self._final_tables:
            import ctypes as C
            segs, blocks = [], 0
            for (k, dst, src, idx, batch, ld) in self._final:
                if lo <= k < hi:
                    sg = _lib.MriFinalSeg()
                    sg.dst, sg.src = dst.data_ptr(), src.data_ptr()
                    sg.idx = idx.data_ptr() if idx is not None else None
                    sg.n, sg.block0, sg.batch, sg.ld = dst.numel(), blocks, batch, ld
                    blocks += -(-dst.numel() // 2048)
                    segs.append(sg)
            if not segs:
                self._final_tables[key] = None
            else:
                arr = (_lib.MriFinalSeg * len(segs))(*segs)
                table = torch.frombuffer(bytearray(bytes(memoryview(arr))), dtype=torch.uint8).to(self.device)
                self._final_tables[key] = (table, len(segs), blocks)
        return self._final_tables[key]

    def bgemm(self, pl, name=None) -> None:
        pl.materialize(self.device)
        self.bwd_flops += pl.flops
        self.badd(f"gemm:{name or pl.name}", pl.launch)

    ZERO_CHUNK = 256 << 20

    def zeros_each_bwd(self, *shape, dtype=torch.float32) -> torch.Tensor:
        """A buffer that is zero at the start of every backward pass.  All of them are carved out
        of a few large chunks, so that zeroing is one cudaMemsetAsync per chunk."""
        n = 1
        for e in shape:
            n *= int(e)
        nbytes = -(-n * torch.empty((), dtype=dtype).element_size() // 256) * 256
        if not self._zero_each_bwd or self._zero_each_bwd[-1][1] + nbytes > self._zero_each_bwd[-1][0].numel():
            chunk = torch.zeros(max(nbytes, self.ZERO_CHUNK), dtype=torch.uint8, device=self.device)
            self._zero_each_bwd.append([chunk, 0])
        chunk, used = self._zero_each_bwd[-1]
        self._zero_each_bwd[-1][1] = used + nbytes
        return chunk[used:used + n * torch.empty((), dtype=dtype).element_size()].view(dtype).view(*shape)

    def _galloc(self, n: int) -> Tuple[int, torch.Tensor]:
        if self.garena is None:
            seen, total = set(), 0
            for p_ in self._params:
                if id(p_) not in seen:
                    seen.add(id(p_))
                    total += -(-p_.numel() // 64) * 64
            self.garena = torch.zeros(total + 4096, dtype=torch.float32, device=self.device)
        off = self._garena_used
        if off + n > self.garena.numel():
            raise _lib.MriError("backward: gradient arena overflow (untracked parameter?)")
        self._garena_used = off + -(-n // 64) * 64   # 256-byte aligned slices
        return off, self.garena[off:off + n]

    def pg(self, p: torch.Tensor) -> torch.Tensor:
        """fp32 gradient buffer of parameter p (reference layout), a view of the arena."""
        g = self.pgrad.get(id(p))
        if g is None:
            off, flat = self._galloc(p.numel())
            g = flat.view(p.shape)
            self.pgrad[id(p)] = g
            self._g_off[id(p)] = (off, p.numel())
        self._g_touched.append(id(p))
        return g

    def pg_block(self, params: Sequence[torch.Tensor], width: int) -> torch.Tensor:
        """One contiguous [sum rows, width] gradient block for parameters that are row-slices of
        a concatenated matrix (the per-block time projections); registers every slice."""
        rows = [p.shape[0] for p in params]
        off, flat = self._galloc(sum(rows) * width)
        blk = flat.view(sum(rows), width) if width > 1 else flat
        o = 0
        for p, n in zip(params, rows):
            self.pgrad[id(p)] = blk[o:o + n]
            self._g_off[id(p)] = (off + o * width, n * width)
            self._g_touched.append(id(p))
            o += n
        return blk

    def emit_grad(self, t: torch.Tensor, produce: Callable[[torch.Tensor, Optional[torch.Tensor]], None]):
        """grad[t] (+)= contribution; produce(out, add) must emit ops writing contribution + add."""
        g = self.grads.get(id(t))
        if g is None:
            g = torch.zeros(tuple(t.shape), dtype=torch.bfloat16, device=self.device)
            self.grads[id(t)] = g
            produce(g, None)
        else:
            produce(g, g)
        self._gn_writer[id(g)] = None

    def pass_grad(self, t: torch.Tensor, dy: torch.Tensor) -> None:
        """grad[t] += dy for an identity edge (residual); aliases dy when it is the first."""
        g = self.grads.get(id(t))
        if g is None:
            self.grads[id(t)] = dy
        else:
            self.badd("add", lambda: ops.add_bf16(g, dy, g))
            self._gn_writer[id(g)] = None

    # ------------------------------------------------------------------ per-op backward
    def _bwd_bias_and_tproj(self, dy: torch.Tensor, C: int, bias_params, tproj_off, name):
        if not bias_params and tproj_off is None:
            return
        B = self.B
        S = dy.numel() // (B * C)
        cs = self.zeros_each_bwd(1, B, C, dtype=torch.float64)
        holder = self._gn_writer.get(id(dy))
        if holder is not None and holder[0] is None and os.environ.get("MRI_NO_COLSUM_FUSION") != "1":
            holder[0] = cs[0]  # the gn_bwd_apply launch that writes dy also accumulates its column sums
        else:
            self.badd(f"colsum:{name}", lambda: ops.colsum(dy, cs, B, S, C))
        for bp in bias_params:
            g = self.pg(bp)
            n = bp.numel()
            self.bfinal_bsum(g.view(-1)[:n], cs[0], "bias_grad")
        if tproj_off is not None:
            dst = self.dtproj[:, tproj_off:tproj_off + C]
            self.badd("dtproj", lambda: ops.copy_cast(cs[0], dst))

    def bwd_conv(self, r: ConvRec) -> None:
        dy = self.grads.get(id(r.y))
        if dy is None:
            raise _lib.MriError(f"backward: no gradient reached {r.name}")
        nd = self.ndim
        C = r.y.shape[-1]
        if r.residual is not None:
            self.pass_grad(r.residual, dy)
        if self.wgrad:
            self._bwd_bias_and_tproj(dy, C, r.bias_params, r.tproj_off, r.name)
        # ---- weight gradient over the forward k-table ------------------------------------
        if r.weight is not None and self.wgrad:
            pl = r.plan
            K = pl.n_kb * P.BLOCK_K
            dw = self.zeros_each_bwd(pl.n_class, max(r.cout, 8), K)
            wg = P.WgradPlan(pl, dy, dw, r.cout, name=r.name)
            wg.materialize(self.device)
            self.bwd_flops += pl.flops
            self.badd(f"wgrad:{r.name}", wg.launch)
            gw = self.pg(r.weight)
            wshape = tuple(r.weight.shape)
            if r.unpack is not None:
                self.bfinal_gather(gw, dw, r.unpack)
                if r.unpack_extra is not None:
                    self.bfinal_gather(self.pg(r.extra_weight), dw, r.unpack_extra)
            elif r.kind == "up":
                self.bfinal_gather(gw, dw, lambda d: P.unpack_convT_wgrad(d, wshape))
            else:
                taps_splits = r.splits
                extra_shapes = []
                if r.extra_weight is not None:
                    cin_e = r.extra_weight.shape[1]
                    for (t, has_taps) in r.sources:
                        if not has_taps:
                            extra_shapes.append((r.cout, t.shape[-1]))
                    assert sum(s[1] for s in extra_shapes) == cin_e
                ge = self.pg(r.extra_weight) if r.extra_weight is not None else None
                rows = r.w_rows
                shp = wshape if rows is None else (rows[1] - rows[0],) + wshape[1:]

                def unpack(d):
                    if r.kind == "matrix":
                        return P.unpack_conv_wgrad(d[0][:, :int(np.prod(shp[1:]))], shp)[0], []
                    return P.unpack_conv_wgrad(d[0], shp, taps_splits, extra_shapes)

                self.bfinal_gather(gw if rows is None else gw[rows[0]:rows[1]], dw, lambda d: unpack(d)[0])
                if ge is not None:
                    self.bfinal_gather(ge, dw, lambda d: torch.cat(unpack(d)[1], dim=1))
        # ---- data gradients through the adjoint plans ---------------------------------------
        if not r.need_dgrad:
            return
        w = r.weight
        wfull = r.wfull if r.wfull is not None else (lambda: w.detach())
        if r.kind == "down":
            (src, _), = r.sources
            wT = self.packed(lambda: P.pack_convT_weight(wfull()))
            self.emit_grad(src, lambda out, add: self.bgemm(
                P.up_conv_plan(dy, wT, out, residual=add, name=f"dgrad:{r.name}")))
            return
        if r.kind == "up":
            (src, _), = r.sources
            wT = self.packed(lambda: P.pack_conv_weight(wfull()))
            self.emit_grad(src, lambda out, add: self.bgemm(
                P.down_conv_plan(dy, wT, out, residual=add, name=f"dgrad:{r.name}")))
            return
        assert r.kind == "conv"
        c0 = 0
        e0 = 0
        dyd = r.dgrad_dy if r.dgrad_dy is not None else dy
        cy = dyd.shape[-1]
        for (src, has_taps) in r.sources:
            Ci = src.shape[-1]
            if has_taps:
                a, b = c0, c0 + Ci
                rows = r.w_rows

                def make(a=a, b=b, rows=rows):
                    ww = wfull() if rows is None else wfull()[rows[0]:rows[1]]
                    wt = ww[:, a:b].transpose(0, 1).flip(*range(2, 2 + nd))  # [Ci, Co, *k]
                    if wt.shape[1] < cy:  # thin Cout padded to the 64-channel dY copy
                        pad = torch.zeros(wt.shape[0], cy - wt.shape[1], *wt.shape[2:],
                                          dtype=wt.dtype, device=wt.device)
                        wt = torch.cat([wt, pad], dim=1)
                    return P.pack_conv_weight(wt)

                wT = self.packed(make)
                self.emit_grad(src, lambda out, add, wT=wT: self.bgemm(
                    P.conv_plan([P.ConvSource(dyd)], wT, out, r.ksize, residual=add,
                                name=f"dgrad:{r.name}")))
                c0 += Ci
            else:
                a, b = e0, e0 + Ci
                efull = r.efull if r.efull is not None else (lambda: r.extra_weight.detach())

                def make_e(a=a, b=b):
                    ew = efull()
                    wt = ew.reshape(ew.shape[0], -1)[:, a:b].t().contiguous()
                    return P.pack_conv_weight(wt.reshape(b - a, ew.shape[0], *([1] * nd)))

                wTe = self.packed(make_e)
                self.emit_grad(src, lambda out, add, wTe=wTe: self.bgemm(
                    P.conv_plan([P.ConvSource(dy)], wTe, out, 1, residual=add,
                                name=f"dgrad_skip:{r.name}")))
                e0 += Ci

    def bwd_gn(self, r: GnRec) -> None:
        dy = self.grads.get(id(r.y))
        if dy is None:
            raise _lib.MriError(f"backward: no gradient reached {r.name}")
        x = r.x
        B, S, C = self.B, x.spatial, x.C
        if r.residual is not None:
            self.pass_grad(r.residual, dy)
        sums = self.zeros_each_bwd(3, B, C, dtype=torch.float64)
        gamma = r.gamma[r.c_off:r.c_off + C]
        beta = r.beta[r.c_off:r.c_off + C]
        xs, st, cpg = x.t, x.stats, x.cpg
        self.badd(f"gn_bwd_reduce:{r.name}", lambda: ops.gn_bwd_reduce(
            xs, dy, st, gamma, beta, sums, B, S, C, r.groups, cpg, r.eps, r.silu))
        if self.wgrad:
            if r.gparam is not None:   # padded copies feed the kernels; the real channels come first
                gg, gb = self.pg(r.gparam), self.pg(r.bparam)
            else:
                gg = self.pg(r.gamma)[r.c_off:r.c_off + C]
                gb = self.pg(r.beta)[r.c_off:r.c_off + C]
            self.bfinal_bsum(gg, sums[2], "gn_param_grad")
            self.bfinal_bsum(gb, sums[1], "gn_param_grad")
        if r.tproj_off is not None:
            dst = self.dtproj[:, r.tproj_off:r.tproj_off + C]
            self.badd("dtproj", lambda: ops.copy_cast(sums[0], dst))
        holder = [None]
        self.emit_grad(xs, lambda out, add: self.badd(f"gn_bwd_apply:{r.name}", lambda: ops.gn_bwd_apply(
            xs, dy, add, out, st, gamma, beta, sums, B, S, C, r.groups, cpg, r.eps, r.silu,
            colsum=holder[0])))
        self._gn_writer[id(self.grads[id(xs)])] = holder

    def bwd_window(self, r: "WindowRec") -> None:
        dy = self.grads.get(id(r.dst))
        if dy is None:
            raise _lib.MriError(f"backward: no gradient reached {r.name}")
        # the adjoint of a window copy is the window copied back; outside the window the gradient
        # buffer keeps what it held (zeros when this is its only producer)
        self.emit_grad(r.src, lambda out, add: self.badd(
            f"window_bwd:{r.name}", lambda: ops.copy_window(dy, out, r.dst_off, r.src_off, r.size, add=add)))

    def bwd_resize(self, r: "ResizeRec") -> None:
        dy = self.grads.get(id(r.dst))
        if dy is None:
            raise _lib.MriError(f"backward: no gradient reached {r.name}")
        self.emit_grad(r.src, lambda out, add: self.badd(
            f"resize_bwd:{r.name}", lambda: ops.resize_bilinear_bwd(dy, out, add=add)))

    def bwd_attention(self, r: AttnRec) -> None:
        dev, B = self.device, self.B
        blk = r.blk
        C = r.x.C
        heads, n, npad = r.heads, r.n, r.npad
        d = C // heads
        dout = self.grads.get(id(r.out))
        if dout is None:
            raise _lib.MriError(f"backward: no gradient reached {r.name}")
        bf = torch.bfloat16
        sp = tuple(r.out.shape[1:-1])
        # residual + proj (1x1 conv) -------------------------------------------------------------
        self.pass_grad(r.x.t, dout)
        self._bwd_bias_and_tproj(dout, C, [blk.proj.bias], None, f"{r.name}.proj")
        dwp = self.zeros_each_bwd(1, C, C)
        wg = P.WgradPlan(r.proj_plan, dout, dwp, C, name=f"{r.name}.proj")
        wg.materialize(dev)
        self.badd(f"wgrad:{r.name}.proj", wg.launch)
        gwp = self.pg(blk.proj.weight)
        self.bfinal_gather(gwp, dwp, lambda d: d[0])
        dO = torch.zeros(B, *sp, C, dtype=bf, device=dev)
        wpT = self.packed(lambda: P.pack_conv_weight(
            blk.proj.weight.detach().reshape(C, C).t().reshape(C, C, *([1] * self.ndim))))
        self.bgemm(P.conv_plan([P.ConvSource(dout)], wpT, dO, 1, name=f"dgrad:{r.name}.proj"))
        # dP = dO v^T (fp32) -------------------------------------------------------------------------
        dP = torch.zeros(B, heads, n, npad, dtype=torch.float32, device=dev)
        C3 = 3 * C
        doa = P.TView(dO, (d, n, heads, B, 1), (1, C, d, n * C, B * n * C))
        vb = P.TView(r.qkv, (d, n, heads, B), (1, C3, d, n * C3), offset=2 * C)
        dpo = P.TView(dP, (npad, n, heads, B, 1),
                      (1, npad, n * npad, heads * n * npad, B * heads * n * npad))
        tiles = (-(-n // 128), heads, B, 1)
        self.bgemm(P.matrix_plan(doa, (128, 1, 1, 1), vb, dpo, K=d, n_total=npad, block_n=128,
                                 ext=(n, heads, B, 1), tiles=tiles, bz_sel=(3, 4), out_f32=True,
                                 name=f"{r.name}.dP", flops=2 * B * heads * n * n * d))
        # dS = softmax backward ------------------------------------------------------------------------
        dS = torch.zeros(B, heads, n, npad, dtype=bf, device=dev)
        scale = float(d) ** -0.5
        Pm = r.Pm
        self.badd(f"{r.name}.softmax_bwd",
                  lambda: ops.softmax_bwd(Pm, dP, dS, B * heads * n, n, npad, npad, scale))
        # dqkv assembled token-major [B, n, 3C] ------------------------------------------------------------
        dqkv = torch.zeros(B, *sp, C3, dtype=bf, device=dev)
        # dq = dS k  (B operand = k^T rows from kvT)
        dsa = P.TView(dS, (npad, n, heads, B, 1),
                      (1, npad, n * npad, heads * n * npad, B * heads * n * npad))
        ktb = P.TView(r.kvT, (npad, d, heads, B), (1, npad, d * npad, 2 * C * npad))
        dqo = P.TView(dqkv, (d, n, heads, B, 1), (1, C3, d, n * C3, B * n * C3))
        self.bgemm(P.matrix_plan(dsa, (128, 1, 1, 1), ktb, dqo, K=npad, n_total=d, block_n=min(d, 128),
                                 ext=(n, heads, B, 1), tiles=tiles, bz_sel=(3, 4),
                                 name=f"{r.name}.dq", flops=2 * B * heads * n * n * d))
        # dk = dS^T q and dv = P^T dO: reductions over the query rows -> MN-major kernel
        n_tiles = -(-n // 128)
        mpad = n_tiles * 128

        def rowsum_product(lhs: torch.Tensor, rhs_base: torch.Tensor, rhs_off: int, rhs_ld: int,
                           dst_slot: int, nm: str):
            """dst[b, m, slot, h, :] = sum_n lhs[b, h, n, m] * rhs[b, n, h, :]"""
            ncls = B * heads
            a_maps, dy_views, kts = [], [], []
            for b in range(B):
                for h in range(heads):
                    cls = b * heads + h
                    av = P.TView(rhs_base, (d, n, 1, 1, 1), (1, rhs_ld, n * rhs_ld, n * rhs_ld, n * rhs_ld),
                                 offset=b * n * rhs_ld + rhs_off + h * d)
                    a_maps.append(P.MapSpec(av, (P.BLOCK_K, 128, 1, 1, 1), 3))
                    dv_ = P.TView(lhs, (npad, n, 1, 1, 1), (1, npad, n * npad, n * npad, n * npad),
                                  offset=cls * n * npad)
                    dy_views.append(dv_)
                    kts.append([[cls, c0, 0, 0, 0, 0, c0, 0] for c0 in range(0, d, P.BLOCK_K)])
            fake = P.GemmPlan(a_maps=a_maps, b_map=None, o_maps=[], ktable=np.asarray(kts, dtype=np.int32),
                              tiles=(n_tiles, 1, 1, 1), box=(128, 1, 1, 1), ext=(n, 1, 1, 1),
                              block_n=128, n_total=d, name=nm)
            dwb = self.zeros_each_bwd(ncls, mpad, d)
            wgp = P.WgradPlan(fake, lhs, dwb, n, name=nm, dy_views=dy_views)
            wgp.materialize(dev)
            self.bwd_flops += 2 * B * heads * n * n * d
            self.badd(f"wgrad:{nm}", wgp.launch)
            dst = dqkv.view(B, n, 3, heads, d)[:, :, dst_slot]

            src = dwb.view(B, heads, mpad, d)[:, :, :n].permute(0, 2, 1, 3)

            def scatter():
                ops.copy_cast(src, dst)

            self.badd(f"scatter:{nm}", scatter)

        rowsum_product(dS, r.qkv, 0, C3, 1, f"{r.name}.dk")
        rowsum_product(Pm, dO, 0, C, 2, f"{r.name}.dv")
        # qkv 1x1 conv backward --------------------------------------------------------------------------
        self._bwd_bias_and_tproj(dqkv, C3, [blk.qkv.bias], None, f"{r.name}.qkv")
        dwq = self.zeros_each_bwd(1, C3, C)
        wg2 = P.WgradPlan(r.qkv_plan, dqkv, dwq, C3, name=f"{r.name}.qkv")
        wg2.materialize(dev)
        self.badd(f"wgrad:{r.name}.qkv", wg2.launch)
        gwq = self.pg(blk.qkv.weight)
        self.bfinal_gather(gwq, dwq, lambda d: d[0])
        wqT = self.packed(lambda: P.pack_conv_weight(
            blk.qkv.weight.detach().reshape(C3, C).t().reshape(C, C3, *([1] * self.ndim))))
        hn = r.hn
        self.emit_grad(hn, lambda out, add: self.bgemm(
            P.conv_plan([P.ConvSource(dqkv)], wqT, out, 1, residual=add, name=f"dgrad:{r.name}.qkv")))
        r.dO, r.dP, r.dS, r.dqkv = dO, dP, dS, dqkv   # kept for stage-by-stage checks

    def bwd_time(self, r: TimeRec) -> None:
        B = self.B
        dev = self.device
        dz = self.dtproj
        if r.act == 1:
            dzz = torch.zeros_like(self.dtproj)
            self.badd("silu_bwd:tproj", lambda: ops.silu_bwd(r.zproj, self.dtproj, dzz))
            dz = dzz
        total, tdim = r.W_all.shape
        o_chk = 0
        for blk, o in zip(r.blocks, r.offs):   # W_all is the row-wise concatenation, in order
            assert o == o_chk, "block projections are not contiguous"
            o_chk += blk.time_mlp.weight.shape[0]
        assert o_chk == total
        dW_all = self.pg_block([blk.time_mlp.weight for blk in r.blocks], tdim)
        db_all = self.pg_block([blk.time_mlp.bias for blk in r.blocks], 1)
        dcond = torch.zeros(B, tdim, device=dev)
        self.badd("linear_bwd:tproj", lambda: ops.linear_bwd(dz, r.cond, r.W_all, dcond, dW_all, db_all))

        def mlp_bwd(dout, lin_a, lin_b, x_in, z_mid, h_mid, tag):
            """out = lin_b(silu(lin_a(x_in)))"""
            dh = torch.zeros_like(h_mid)
            gWb, gbb = self.pg(lin_b.weight), self.pg(lin_b.bias)
            self.badd(f"linear_bwd:{tag}.b", lambda: ops.linear_bwd(dout, h_mid, lin_b.weight, dh, gWb, gbb))
            dzm = torch.zeros_like(z_mid)
            self.badd(f"silu_bwd:{tag}", lambda: ops.silu_bwd(z_mid, dh, dzm))
            gWa, gba = self.pg(lin_a.weight), self.pg(lin_a.bias)
            self.badd(f"linear_bwd:{tag}.a", lambda: ops.linear_bwd(dzm, x_in, lin_a.weight, None, gWa, gba))

        mlp_bwd(dcond, r.l1, r.l2, r.sin, r.z1, r.h1, "time_mlp")
        if r.slice is not None:
            s = r.slice
            mlp_bwd(dcond, s["s0"], s["s2"], s["z_in"], s["zz"], s["zh"], "slice_mlp")

    # ------------------------------------------------------------------ driver
    def build_backward(self, dy_seed: Dict[int, torch.Tensor]) -> None:
        """dy_seed: id(forward tensor) -> gradient buffer filled before the backward ops run."""
        self.grads.update(dy_seed)
        for rec in reversed(self.tape):
            self._g_touched = []
            lo = len(self.bwd_ops)
            if isinstance(rec, ConvRec):
                self.bwd_conv(rec)
            elif isinstance(rec, GnRec):
                self.bwd_gn(rec)
            elif isinstance(rec, AttnRec):
                self.bwd_attention(rec)
            elif isinstance(rec, TimeRec):
                self.bwd_time(rec)
            elif isinstance(rec, WindowRec):
                self.bwd_window(rec)
            elif isinstance(rec, ResizeRec):
                self.bwd_resize(rec)
            else:  # pragma: no cover
                raise _lib.MriError(f"unknown tape record {type(rec)}")
            self._close_record()
            self.bwd_ranges.insert(0, (lo, len(self.bwd_ops)))
        self.bwd_segments = []

    def _close_record(self) -> None:
        """Gradients touched by the record just emitted are final once all its ops have run."""
        for pid in self._g_touched:
            self._g_last_op[pid] = len(self.bwd_ops)
        self._g_touched = []

    def plan_segments(self, bucket_bytes: int) -> List[Tuple[int, int, int, int]]:
        """Cut the backward launch list into segments (op_lo, op_hi, arena_lo, arena_hi): after
        ops[:op_hi] have run, arena[:arena_hi] holds final parameter gradients.  Cuts are placed
        where at least `bucket_bytes` of new gradients became final; the last segment takes the
        rest.  The gradient all-reduce of segment i overlaps the launches of segment i + 1."""
        order = sorted(self._g_off.items(), key=lambda kv: kv[1][0])   # by arena offset
        segs, op_lo, a_lo, i = [], 0, 0, 0
        n_ops = len(self.bwd_ops)
        ready_at = 0   # ops needed for arena[:a_hi]
        a_hi = 0
        while i < len(order):
            pid, (off, n) = order[i]
            ready_at = max(ready_at, self._g_last_op[pid])
            a_hi = -(-(off + n) // 64) * 64
            i += 1
            # the prefix is final only if no later-placed parameter finishes earlier... it is a
            # prefix property: ready_at is the max over the prefix, which is what we need.
            # The LAST bucket cannot overlap anything (the backward list has ended when it is
            # ready), so its size is the exposed communication: 29 MB took 0.8 ms on 8 GPUs
            # (profiles/r03d).  Near the end the cap therefore shrinks to a sixth, which leaves
            # only the gradients of the very last records (time embedding, first layers) exposed.
            remaining = (self._garena_used - a_lo) * 4
            cap = bucket_bytes if remaining > 2 * bucket_bytes else max(bucket_bytes // 6, 1 << 10)
            if (a_hi - a_lo) * 4 >= cap and ready_at < n_ops and ready_at > op_lo:
                segs.append((op_lo, ready_at, a_lo, a_hi))
                op_lo, a_lo = ready_at, a_hi
        segs.append((op_lo, n_ops, a_lo, self._garena_used))
        self.bwd_segments = segs
        return segs

    def run_backward(self, lo: int = 0, hi: Optional[int] = None) -> None:
        """Enqueue backward ops [lo, hi) (all by default)."""
        if lo == 0:
            for chunk, used in self._zero_each_bwd:
                ops.memset_zero(chunk, used)
        hi = len(self.bwd_ops) if hi is None else hi
        for fn in self.bwd_ops[lo:hi]:
            fn()
        if self._final:
            tab = self._final_table(lo, hi)
            if tab is not None:
                _lib.check(_lib.load().mri_grad_finalize(tab[0].data_ptr(), tab[1], tab[2],
                                                         _lib.current_stream_ptr()), "mri_grad_finalize")

    def _bwd_head(self, S: int) -> None:
        """fp32 NC[D]HW loss gradient -> the bf16 channels-last seeds of the backward list."""
        ops.nchw_to_nhwc(self.dout_in, self.deps16, self.B, S, self.cout, self.cout_pad)
        ops.nchw_to_nhwc(self.dout_in, self.deps64, self.B, S, self.cout, 64)

    def _bwd_tail(self) -> None:
        """After the last backward op (programs that return an input gradient override this)."""

    def _backward(self, dout: torch.Tensor, S: int, sync) -> None:
        self.dout_in.copy_(dout)
        if sync is None or not sync.active():
            if sync is not None and not sync.enabled:
                sync.note_local_backward()

            def body():
                self._bwd_head(S)
                self.run_backward()
                self._bwd_tail()
            self._replay("bwd", body)
            return
        # segmented: one replayed graph per segment; after each, its (contiguous) slice of the
        # gradient arena is handed to the all-reduce, which runs on the communication stream
        # while the next segment's launches execute
        segs = self.bwd_segments or self.plan_segments(sync.bucket_bytes)
        sync.begin(self.garena)
        for i, (lo, hi, a_lo, a_hi) in enumerate(segs):
            def body(lo=lo, hi=hi):
                if lo == 0:
                    self._bwd_head(S)
                self.run_backward(lo, hi)
                if hi == len(self.bwd_ops):
                    self._bwd_tail()
            self._replay(f"bwd_seg{i}/{len(segs)}", body)
            sync.bucket_ready(a_lo, a_hi)
        sync.finish()
