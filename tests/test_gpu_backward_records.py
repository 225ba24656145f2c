"""The training backward pass (backward.py) record by record against float64 vector-Jacobian
products on the engine's own activations.

The whole-model tests (test_gpu_train2d.py, test_gpu_train3d.py, test_gpu_vae_train.py, ...) hold
every parameter gradient to rel-L2 <= 5e-2 against the fp32 oracle, a tolerance wide enough for
bf16 rounding compounded through the network, and wide enough for wiring errors too: a gradient
path lost or counted twice that carries a few percent, a time-projection slice written to the
neighbouring block, a column sum taken before the last contribution was added.  Here each tape
record's backward is checked by itself (teacher forcing): a training program keeps every forward
tensor and every data-gradient buffer, so after the forward and the loss-gradient head, the test
walks the records in backward order and for each one

1. snapshots every data-gradient buffer, the time-projection gradient `dtproj` and the parameter
   gradient arena,
2. runs exactly the record's launches, `run_backward(lo, hi)` over `bwd_ranges[i]` (the production
   entry point, with the range's fused gradient finalisation),
3. restates the record's forward in fp64 from the record's fields and inputs and requires it to
   reproduce the recorded output (this proves the reference reads `sources`, `splits`,
   `extra_weight`, `residual`, `tproj_off`, `c_off` and the channel padding as the forward used
   them),
4. computes the record's VJP in fp64 from the same bf16 forward tensors, the bf16-rounded weights
   (what the kernels are packed from), the engine's GroupNorm statistics and the snapshotted
   incoming gradient, and compares element by element,
5. requires every buffer the record has no business writing to be bit-identical.

Error model.  r is the fp64 value of the same operation on the same inputs plus what the buffer
held before (a first contribution replaces the buffer, later ones add to it), A the same sum over
absolute values, so A bounds the fp32 accumulation error whatever the cancellation:

* bf16 data gradients:        |g - r| <= 2^-8 |r| + beta A   (one rounding to bf16 of the fp32 result)
* fp32 parameter gradients:   |g - r| <= 2^-23 |r| + beta A   (also dtproj slices and column sums)

beta per operation class: BETA (outputs, also the attention products written by the forward
kernel) and BETA_W (weight gradients and the MN-major row-sum products dk, dv) are the GEMM
kernel constants of test_gpu_gemm_kernels.py; ADD_BETA = 2^-24 is the exact fp32 sum of two bf16
values before its one rounding (pass_grad, the window adjoint).  The others were measured on the
program records below on one B200 at its 1000 W power limit and set to 4x the worst value (0
where the worst is negative: the rounding term alone holds):

    GN_DX_BETA     GroupNorm(+SiLU) dx             worst 5.50e-06
    GN_SUM_BETA    gamma / beta sums               worst 1.81e-05
    COLSUM_BETA    bias / dtproj column sums       worst 7.81e-10
    TIME_BETA      the fp32 time-embedding chain   worst 1.76e-07
    SM_BETA        softmax backward dS             worst -1.84e-06
    RESIZE_BETA    bilinear adjoint and forward    worst 2.54e-07
    FWD_GN_BETA    GroupNorm forward (self-check)  worst 2.94e-06
    FWD_SM_BETA    softmax forward P (self-check)  worst -1.65e-04

Across the whole program the test also checks completeness (every gradient a record sends goes to
another record's output or to a gradient target of the program; every tracked parameter, and
every column of dtproj, is written by exactly one record per element; channel padding of data
gradients stays exactly 0), finality (the record recorded in `_g_last_op` is the last one that
writes the parameter, so `plan_segments()` may hand its arena slice to the all-reduce), the DDP
segments of `plan_segments()` on the real launch list (a segment's arena slice is bit-identical at
the end of the pass), and both finalisation / column-sum paths (MRI_NO_FINAL_FUSION=1 +
MRI_NO_COLSUM_FUSION=1).  Run with -s for the worst measured beta and err / bound per program and
record kind.
"""
import contextlib
import io
import math

import pytest
import torch
import torch.nn.functional as F

from helpers import shapes_of, synthetic_state_dict
from test_gpu_gemm_kernels import BETA, BETA_W

pytestmark = pytest.mark.gpu

U16 = 2.0 ** -8
U32 = 2.0 ** -23
ADD_BETA = 2.0 ** -24
GN_DX_BETA = 2.2e-5
GN_SUM_BETA = 7.3e-5
COLSUM_BETA = 3.2e-9
TIME_BETA = 7.1e-7
SM_BETA = 0.0
RESIZE_BETA = 1.0e-6
FWD_GN_BETA = 1.2e-5
FWD_SM_BETA = 0.0

BOUNDS = {   # class -> (rounding unit of the stored type, beta)
    "gemm": (U16, BETA), "gemm_f32": (U32, BETA), "wgrad": (U32, BETA_W), "rowsum": (U16, BETA_W),
    "add": (U16, ADD_BETA), "gn_dx": (U16, GN_DX_BETA), "gn_sum": (U32, GN_SUM_BETA),
    "colsum": (U32, COLSUM_BETA), "time": (U32, TIME_BETA), "softmax": (U16, SM_BETA),
    "resize": (U16, RESIZE_BETA), "fwd_gn": (U16, FWD_GN_BETA), "fwd_softmax": (U16, FWD_SM_BETA),
}

WORST = {}   # (program, record kind, class) -> [worst beta, worst err / bound]


@pytest.fixture(scope="module", autouse=True)
def _print_worst():
    yield
    if WORST:
        print("\n[backward records] worst measured beta and err / bound")
        per_cls = {}
        for (prog, kind, cls), (b, q) in sorted(WORST.items()):
            print(f"  {prog:12s} {kind:10s} {cls:12s} beta {b: .3e}  err/bound {q:.3f}")
            per_cls[cls] = max(per_cls.get(cls, -math.inf), b)
        for cls, b in sorted(per_cls.items()):
            print(f"  all programs {cls:12s} worst beta {b: .3e} (bound uses {BOUNDS[cls][1]:.3g})")


def _quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


# ------------------------------------------------------------------------------------ programs
B = 2
PROGRAMS = ["unet3d", "unet3d_attn", "unet2d", "unet25d", "vae_enc", "vae_dec"]
FUSIONS = ["fused", "unfused"]


def _build(name):
    """(training program, callable that loads seeded inputs and runs the forward)."""
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.engine import UNet2DProgram, UNet3DProgram
    from mri_image_generation_b200.vae_engine import VAE3DProgram
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm import unet, unet_attention, vae
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm import unet as unet2d
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities import unet as unet25d
    _lib.require_device()
    g = torch.Generator().manual_seed(PROGRAMS.index(name) + 5)
    if name in ("unet3d", "unet3d_attn"):
        cls = unet.UNet3DModel if name == "unet3d" else unet_attention.UNet3DModelWithAttention
        m = _quiet(cls, 3, base_channels=64, time_emb_dim=64)
        sp, cin = (8, 12, 8), 3
    elif name == "unet2d":
        m = _quiet(unet2d.UNet, img_channels=1, base_channels=64, time_emb_dim=64)
        sp, cin, ctx = (36, 44), 1, 0
    elif name == "unet25d":
        m = _quiet(unet25d.UNet, in_channels=20, out_channels=4, base_channels=64, time_emb_dim=64)
        sp, cin, ctx = (24, 24), 4, 16
    else:
        m = vae.VAE3D(4, 32, 3, 3)
        sp, cin = ((24, 16, 32), 4) if name == "vae_enc" else ((6, 4, 8), 3)
    m.load_state_dict(synthetic_state_dict(shapes_of(m), seed=31 + PROGRAMS.index(name)))
    m = m.cuda()
    x = torch.randn(B, cin, *sp, generator=g).cuda()
    t = torch.randint(1, 1000, (B,), generator=g).cuda()
    if name.startswith("unet3d"):
        prog = UNet3DProgram(m, B, sp, training=True)
        return prog, m, lambda: prog.forward(x, t)
    if name.startswith("unet2"):
        prog = UNet2DProgram(m, B, sp, cin, ctx, training=True)
        z = torch.rand(B, generator=g).cuda()
        c = torch.randn(B, ctx, *sp, generator=g).cuda() if ctx else None
        return prog, m, lambda: prog.forward(x, t, z, c)
    prog = VAE3DProgram(m, "encode" if name == "vae_enc" else "decode", B, sp, training=True)
    return prog, m, lambda: prog.forward(x)


_CACHE = {}


def program(name, fusion):
    key = (name, fusion)
    if key not in _CACHE:
        with pytest.MonkeyPatch.context() as mp:
            if fusion == "unfused":
                mp.setenv("MRI_NO_FINAL_FUSION", "1")
                mp.setenv("MRI_NO_COLSUM_FUSION", "1")
            else:
                mp.delenv("MRI_NO_FINAL_FUSION", raising=False)
                mp.delenv("MRI_NO_COLSUM_FUSION", raising=False)
            _CACHE[key] = _build(name)
    return _CACHE[key]


# ------------------------------------------------------------------------------------ helpers
def f64(t):
    return t.detach().double()


def nc(t):
    """channels-last [B, *sp, C] -> fp64 [B, C, *sp]"""
    return f64(t).movedim(-1, 1)


def cl(t):
    return t.movedim(1, -1)


def wbf(p):
    """A weight as the kernels see it: rounded to bf16 when packed."""
    return p.detach().to(torch.bfloat16).double()


def padded(w, shape):
    out = torch.zeros(shape, dtype=torch.float64, device=w.device)
    out[tuple(slice(0, s) for s in w.shape)] = w
    return out


def dsilu(z):
    s = torch.sigmoid(z)
    return s * (1 + z * (1 - s))


def conv_fn(kind, nd, k):
    conv = F.conv2d if nd == 2 else F.conv3d
    convT = F.conv_transpose2d if nd == 2 else F.conv_transpose3d
    if kind == "down":
        return lambda x, w: conv(x, w, stride=2, padding=1)
    if kind == "up":
        return lambda x, w: convT(x, w, stride=2, padding=1)
    return lambda x, w: conv(x, w, padding=k // 2)


def kind_of(rec):
    return getattr(rec, "kind", None) or type(rec).__name__


class Walk:
    """One backward pass record by record, with the snapshots and bookkeeping of the checks."""

    def __init__(self, prog, name):
        self.prog, self.name = prog, name
        seen, self.bufs = set(), []
        for g in prog.grads.values():
            if g.data_ptr() not in seen:
                seen.add(g.data_ptr())
                self.bufs.append(g)
        self.slot = {g.data_ptr(): i for i, g in enumerate(self.bufs)}
        self.touched = {id(prog.eps_nhwc)}           # forward tensors holding a gradient so far
        self.outputs = {id(prog.eps_nhwc)}
        for rec in prog.tape:
            for t in (getattr(rec, "y", None), getattr(rec, "out", None), getattr(rec, "dst", None)):
                if isinstance(t, torch.Tensor):
                    self.outputs.add(id(t))
        if getattr(prog, "z64", None) is not None:   # the decoder returns the gradient of z
            self.outputs.add(id(prog.z64))
        self.written = {}     # id(param) -> [(lo, hi, record index)]
        self.cols = []        # (lo, hi) columns of dtproj written
        self.params = {}
        for p in prog._params:
            self.params[id(p)] = p
        tp = [v for v in getattr(prog, "_tproj", {}).values() if v[2] == 0]
        self.tproj = tp[0][0] if tp else None       # the block-projection output [B, total]

    def snap(self):
        out = [b.clone() for b in self.bufs]
        out.append(self.prog.dtproj.clone() if self.prog.dtproj is not None else None)
        out.append(self.prog.garena.clone() if self.prog.garena is not None else None)
        return out

    # ---- access to the snapshots
    def grad(self, s, t):
        return s[self.slot[self.prog.grads[id(t)].data_ptr()]]

    def pgrad(self, s, p):
        off, n = self.prog._g_off[id(p)]
        return s[-1][off:off + n].view(p.shape)

    # ---- checks
    def check(self, what, cls, got, r, A):
        rnd, beta = BOUNDS[cls]
        g = got.double()
        assert g.shape == r.shape == A.shape, (what, g.shape, r.shape, A.shape)
        assert bool(torch.isfinite(g).all()), f"{self.where}: {what}: non-finite values"
        err = (g - r).abs()
        meas = float(((err - rnd * r.abs()) / A.clamp_min(1e-300)).max()) if g.numel() else 0.0
        ratio = err / (rnd * r.abs() + beta * A).clamp_min(1e-300)
        q = float(ratio.max()) if g.numel() else 0.0
        key = (self.name, self.kind, cls)
        w = WORST.setdefault(key, [-math.inf, 0.0])
        w[0], w[1] = max(w[0], meas), max(w[1], q)
        if q > 1.0:
            i = int(ratio.reshape(-1).argmax())
            idx = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), tuple(g.shape)))
            raise AssertionError(
                f"{self.where}: {what}: {int((ratio > 1).sum())} of {g.numel()} elements outside the "
                f"bound; worst {q:.3g}x at {idx}: got {float(g.reshape(-1)[i]):.6g}, "
                f"ref {float(r.reshape(-1)[i]):.6g}, A {float(A.reshape(-1)[i]):.3g}")

    def emit(self, t, contrib, A, cls, what):
        """grad[t] (+)= contrib: the first contribution replaces the buffer, later ones add."""
        assert id(t) in self.outputs, f"{self.where}: {what}: gradient sent to a tensor no record produced"
        gb = self.prog.grads[id(t)]
        self.bufs_written.add(gb.data_ptr())
        first = id(t) not in self.touched
        before = torch.zeros_like(contrib) if first else self.grad(self.before, t).double()
        self.check(what, cls, self.grad(self.after, t), before + contrib, before.abs() + A)
        self.touched.add(id(t))

    def pass_through(self, t, dy_owner, dy):
        """Identity edge: grad[t] aliases dy when it is the first, else grad[t] += dy."""
        assert id(t) in self.outputs, f"{self.where}: residual gradient sent to a tensor no record produced"
        if id(t) not in self.touched:
            assert self.prog.grads[id(t)].data_ptr() == self.prog.grads[id(dy_owner)].data_ptr(), \
                f"{self.where}: the first gradient of the residual must alias dy"
            self.touched.add(id(t))
            return
        d = dy.double()
        self.emit(t, d, d.abs(), "add", "residual")

    def param(self, p, lo, hi, got_view, r, A, cls, what):
        self.written.setdefault(id(p), []).append((lo, hi, self.rec_index))
        self.check(what, cls, got_view, r, A)

    def dtproj(self, off, r, A, what):
        C = r.shape[1]
        self.cols.append((off, off + C))
        self.check(what, "colsum", self.after[-2][:, off:off + C], r, A)

    def untouched(self):
        """Everything the record declares no write to is bit-identical."""
        for i, b in enumerate(self.bufs):
            if b.data_ptr() not in self.bufs_written:
                assert torch.equal(self.before[i].view(torch.int16), self.after[i].view(torch.int16)), \
                    f"{self.where}: wrote a data-gradient buffer it sends no gradient to (buffer {i})"
        if self.before[-2] is not None:
            m = torch.ones(self.before[-2].shape[1], dtype=torch.bool, device=self.before[-2].device)
            for (a, b) in self.cols[self.cols_at:]:
                m[a:b] = False
            assert torch.equal(self.before[-2][:, m].view(torch.int32), self.after[-2][:, m].view(torch.int32)), \
                f"{self.where}: wrote dtproj columns outside its own block"
        if self.before[-1] is not None:
            m = torch.ones(self.before[-1].numel(), dtype=torch.bool, device=self.before[-1].device)
            for pid, lst in self.written.items():
                off, n = self.prog._g_off[pid]
                for (a, b, k) in lst:
                    if k == self.rec_index:
                        m[off + a:off + b] = False
            assert torch.equal(self.before[-1][m].view(torch.int32), self.after[-1][m].view(torch.int32)), \
                f"{self.where}: wrote parameter gradients outside its own parameters"


# ------------------------------------------------------------------------------------ records
def check_conv(w, r):
    prog = w.prog
    nd = prog.ndim
    Cy = r.y.shape[-1]
    dy_b = w.grad(w.before, r.y)
    dy = nc(dy_b)
    cout = r.cout or Cy
    if cout < Cy:   # padded output channels (thin out_conv, the VAE's 32-channel level)
        assert not bool(dy_b[..., cout:].any()), f"{w.where}: gradient in the padding channels of dY"
    if r.dgrad_dy is not None:
        d = r.dgrad_dy
        assert torch.equal(d[..., :cout], dy_b[..., :cout]) and not bool(d[..., cout:].any()), \
            f"{w.where}: the 64-channel copy of dY differs from dY"
    if r.kind == "matrix":   # the patch matrix of the network input: conv over the bf16 input
        xin = prog.x_in if getattr(prog, "ctx_in", None) is None else torch.cat([prog.x_in, prog.ctx_in], 1)
        tapped, untapped = [xin.to(torch.bfloat16).double()], []
        fn = conv_fn("conv", nd, r.ksize)
    else:
        tapped = [nc(t) for t, tp in r.sources if tp]
        untapped = [nc(t) for t, tp in r.sources if not tp]
        fn = conv_fn(r.kind, nd, r.ksize)
    Ct = sum(t.shape[1] for t in tapped)
    wt = wbf(r.weight)
    W = padded(wt, ((Ct, Cy) if r.kind == "up" else (Cy, Ct)) + tuple(wt.shape[2:]))
    E = None
    if r.extra_weight is not None:
        e = wbf(r.extra_weight).reshape(r.extra_weight.shape[0], -1)
        E = padded(e, (Cy, sum(t.shape[1] for t in untapped))).view(Cy, -1, *([1] * nd))
    one = (1, Cy) + (1,) * nd
    bias = sum(padded(b.detach().double(), (Cy,)) for b in r.bias_params) if r.bias_params else \
        torch.zeros(Cy, dtype=torch.float64, device=dy.device)
    rb = torch.zeros((B, Cy) + (1,) * nd, dtype=torch.float64, device=dy.device)
    if r.tproj_off is not None:
        rb = f64(w.tproj[:, r.tproj_off:r.tproj_off + Cy]).view(B, Cy, *([1] * nd))
    res = nc(r.residual) if r.residual is not None else torch.zeros_like(dy)

    def lin(xs, W_, xu, E_):
        y = fn(torch.cat(xs, 1), W_)
        if E_ is not None:
            y = y + fn1(torch.cat(xu, 1), E_)
        return y

    fn1 = conv_fn("conv", nd, 1)
    with torch.no_grad():
        yr = lin(tapped, W, untapped, E) + bias.view(one) + rb + res
        Ay = lin([t.abs() for t in tapped], W.abs(), [t.abs() for t in untapped],
                 E.abs() if E is not None else None) + bias.abs().view(one) + rb.abs() + res.abs()
    w.check("forward restated from the record", "gemm", r.y, cl(yr), cl(Ay))

    def vjp(xs, W_, xu, E_, g):
        xs = [t.clone().requires_grad_() for t in xs]
        xu = [t.clone().requires_grad_() for t in xu]
        W_ = W_.clone().requires_grad_()
        E_ = E_.clone().requires_grad_() if E_ is not None else None
        with torch.enable_grad():
            lin(xs, W_, xu, E_).backward(g)
        return [t.grad for t in xs], W_.grad, [t.grad for t in xu], (E_.grad if E_ is not None else None)

    gx, gW, gu, gE = vjp(tapped, W, untapped, E, dy)
    ax, aW, au, aE = vjp([t.abs() for t in tapped], W.abs(), [t.abs() for t in untapped],
                         E.abs() if E is not None else None, dy.abs())
    if r.residual is not None:
        w.pass_through(r.residual, r.y, dy_b)
    if prog.wgrad:
        Sdims = tuple(range(2, 2 + nd))
        for bp in r.bias_params:
            n = bp.numel()
            w.param(bp, 0, n, w.pgrad(w.after, bp), dy.sum((0,) + Sdims)[:n], dy.abs().sum((0,) + Sdims)[:n],
                    "colsum", "bias gradient")
        if r.tproj_off is not None:
            w.dtproj(r.tproj_off, dy.sum(Sdims), dy.abs().sum(Sdims), "dtproj slice")
        real = tuple(slice(0, s) for s in r.weight.shape)
        w.param(r.weight, 0, r.weight.numel(), w.pgrad(w.after, r.weight), gW[real], aW[real], "wgrad",
                "weight gradient")
        if r.extra_weight is not None:
            co, ce = r.extra_weight.shape[0], r.extra_weight.shape[1]
            sh = r.extra_weight.shape
            w.param(r.extra_weight, 0, r.extra_weight.numel(), w.pgrad(w.after, r.extra_weight),
                    gE[:co, :ce].reshape(sh), aE[:co, :ce].reshape(sh), "wgrad", "extra (folded skip) weight gradient")
    if not r.need_dgrad:
        return
    srcs_t = [t for t, tp in r.sources if tp]
    srcs_u = [t for t, tp in r.sources if not tp]
    ptrs = [prog.grads[id(t)].data_ptr() for t in srcs_t + srcs_u]
    assert len(set(ptrs)) == len(ptrs), f"{w.where}: two sources share one gradient buffer"
    c0 = 0
    for t, g_, a_ in zip(srcs_t, gx, ax):
        C = t.shape[-1]
        w.emit(t, cl(g_), cl(a_), "gemm", f"dgrad of source channels {c0}:{c0 + C}")
        c0 += C
    e0 = 0
    for t, g_, a_ in zip(srcs_u, gu, au):
        C = t.shape[-1]
        w.emit(t, cl(g_), cl(a_), "gemm", f"folded-skip dgrad of source channels {e0}:{e0 + C}")
        e0 += C


def gn_parts(w, r):
    """fp64 xhat, z, rstd of a GnRec from the recorded input and the engine's statistics."""
    x = f64(r.x.t).reshape(B, -1, r.x.C)
    S, C, G = x.shape[1], r.x.C, r.groups
    st, cpg = r.x.stats, r.x.cpg
    assert st.shape[1] * cpg == C, (st.shape, cpg, C)
    cg = C // G
    s = st.view(B, G, cg // cpg, 2).sum(2)
    n = cg * S
    mean = s[..., 0] / n
    var = s[..., 1] / n - mean * mean
    rstd = (var + r.eps).rsqrt()
    xh = ((x.view(B, S, G, cg) - mean[:, None, :, None]) * rstd[:, None, :, None]).reshape(B, S, C)
    gamma = f64(r.gamma[r.c_off:r.c_off + C])
    beta = f64(r.beta[r.c_off:r.c_off + C])
    return x, xh, xh * gamma + beta, rstd, gamma, beta, S, C, G, cg


def check_gn(w, r):
    prog = w.prog
    x, xh, z, rstd, gamma, beta, S, C, G, cg = gn_parts(w, r)
    a = F.silu(z) if r.silu else z
    rb = torch.zeros_like(a)
    if r.tproj_off is not None:
        rb = f64(w.tproj[:, r.tproj_off:r.tproj_off + C])[:, None, :].expand_as(a)
    res = f64(r.residual).reshape(B, S, C) if r.residual is not None else torch.zeros_like(a)
    Ay = (xh * gamma).abs() + beta.abs() + rb.abs() + res.abs()
    w.check("forward restated from the record", "fwd_gn", r.y.reshape(B, S, C), a + rb + res, Ay)
    dy_b = w.grad(w.before, r.y)
    dy = f64(dy_b).reshape(B, S, C)
    du = dy * dsilu(z) if r.silu else dy
    gdu = gamma * du
    gv = lambda t: t.view(B, S, G, cg)
    m1 = gv(gdu).mean((1, 3), keepdim=True)
    m2 = gv(gdu * xh).mean((1, 3), keepdim=True)
    r4 = rstd[:, None, :, None]
    dx = (r4 * (gv(gdu) - m1 - gv(xh) * m2)).reshape(B, S, C)
    Adx = (r4 * (gv(gdu).abs() + gv(gdu).abs().mean((1, 3), keepdim=True)
                 + gv(xh).abs() * gv(gdu * xh).abs().mean((1, 3), keepdim=True))).reshape(B, S, C)
    if r.residual is not None:
        w.pass_through(r.residual, r.y, dy_b)
    if prog.wgrad:
        dg, Adg = (du * xh).sum((0, 1)), (du * xh).abs().sum((0, 1))
        db, Adb = du.sum((0, 1)), du.abs().sum((0, 1))
        if r.gparam is not None:
            n = r.gparam.numel()
            w.param(r.gparam, 0, n, w.pgrad(w.after, r.gparam), dg[:n], Adg[:n], "gn_sum", "gamma gradient")
            w.param(r.bparam, 0, n, w.pgrad(w.after, r.bparam), db[:n], Adb[:n], "gn_sum", "beta gradient")
        else:
            sl = slice(r.c_off, r.c_off + C)
            w.param(r.gamma, r.c_off, r.c_off + C, w.pgrad(w.after, r.gamma)[sl], dg, Adg, "gn_sum",
                    "gamma gradient")
            w.param(r.beta, r.c_off, r.c_off + C, w.pgrad(w.after, r.beta)[sl], db, Adb, "gn_sum",
                    "beta gradient")
    if r.tproj_off is not None:
        w.dtproj(r.tproj_off, dy.sum(1), dy.abs().sum(1), "dtproj slice (row bias)")
    shp = tuple(r.x.t.shape)
    w.emit(r.x.t, dx.reshape(shp), Adx.reshape(shp), "gn_dx", "GroupNorm dx")
    if r.gparam is not None:
        assert not bool(w.grad(w.after, r.x.t)[..., r.gparam.numel():].any()), \
            f"{w.where}: gradient in the padding channels of the normalised input"


def check_attention(w, r):
    blk = r.blk
    C, h, n, npad = r.x.C, r.heads, r.n, r.npad
    d = C // h
    scale = float(d) ** -0.5
    hn = f64(r.hn).reshape(B, n, C)
    qkv = f64(r.qkv).reshape(B, n, 3 * C)
    q, k, v = (qkv.view(B, n, 3, h, d)[:, :, i] for i in range(3))
    kT = f64(r.kvT)[:, :C, :n].reshape(B, h, d, n)
    vT = f64(r.kvT)[:, C:, :n].reshape(B, h, d, n)
    Pm = f64(r.Pm)
    P = Pm[..., :n]
    O = f64(r.O).reshape(B, n, C)
    Wq, bq = wbf(blk.qkv.weight).reshape(3 * C, C), f64(blk.qkv.bias)
    Wp, bp = wbf(blk.proj.weight).reshape(C, C), f64(blk.proj.bias)
    xres = f64(r.x.t).reshape(B, n, C)
    # forward, stage by stage on the stored intermediates
    w.check("qkv restated", "gemm", qkv, hn @ Wq.t() + bq, hn.abs() @ Wq.abs().t() + bq.abs())
    w.check("kvT restated", "gemm", f64(r.kvT)[:, :, :n], torch.einsum("bnc,oc->bon", hn, Wq[C:]) + bq[C:, None],
            torch.einsum("bnc,oc->bon", hn.abs(), Wq[C:].abs()) + bq[C:, None].abs())
    Sx = torch.einsum("bihe,bjhe->bhij", q, k) * scale
    w.check("softmax P restated", "fwd_softmax", P, torch.softmax(Sx, -1), torch.softmax(Sx, -1))
    assert not bool(r.Pm[..., n:].any()), f"{w.where}: P has values in its padding columns"
    Or = torch.einsum("bhij,bhej->bihe", P, vT).reshape(B, n, C)
    Ao = torch.einsum("bhij,bhej->bihe", P, vT.abs()).reshape(B, n, C)
    w.check("O restated", "gemm", O, Or, Ao)
    w.check("out restated", "gemm", f64(r.out).reshape(B, n, C), O @ Wp.t() + bp + xres,
            O.abs() @ Wp.abs().t() + bp.abs() + xres.abs())
    # backward
    dout_b = w.grad(w.before, r.out)
    dout = f64(dout_b).reshape(B, n, C)
    w.pass_through(r.x.t, r.out, dout_b)
    w.param(blk.proj.bias, 0, C, w.pgrad(w.after, blk.proj.bias), dout.sum((0, 1)), dout.abs().sum((0, 1)),
            "colsum", "proj bias gradient")
    w.param(blk.proj.weight, 0, C * C, w.pgrad(w.after, blk.proj.weight).reshape(C, C),
            torch.einsum("bno,bnc->oc", dout, O), torch.einsum("bno,bnc->oc", dout.abs(), O.abs()), "wgrad",
            "proj weight gradient")
    w.check("dO", "gemm", f64(r.dO).reshape(B, n, C), dout @ Wp, dout.abs() @ Wp.abs())
    dO = f64(r.dO).reshape(B, n, h, d)
    w.check("dP", "gemm_f32", f64(r.dP)[..., :n], torch.einsum("bihe,bjhe->bhij", dO, v),
            torch.einsum("bihe,bjhe->bhij", dO.abs(), v.abs()))
    dP = f64(r.dP)[..., :n]
    rs = (P * dP).sum(-1, keepdim=True)
    w.check("dS (softmax backward)", "softmax", f64(r.dS)[..., :n], scale * P * (dP - rs),
            scale * P * (dP.abs() + (P * dP.abs()).sum(-1, keepdim=True)))
    assert not bool(r.dS[..., n:].any()), f"{w.where}: dS has values in its padding columns"
    dS = f64(r.dS)[..., :n]
    dqkv = f64(r.dqkv).reshape(B, n, 3, h, d)
    w.check("dq", "gemm", dqkv[:, :, 0], torch.einsum("bhij,bhej->bihe", dS, kT),
            torch.einsum("bhij,bhej->bihe", dS.abs(), kT.abs()))
    w.check("dk", "rowsum", dqkv[:, :, 1], torch.einsum("bhij,bihe->bjhe", dS, q),
            torch.einsum("bhij,bihe->bjhe", dS.abs(), q.abs()))
    w.check("dv", "rowsum", dqkv[:, :, 2], torch.einsum("bhij,bihe->bjhe", P, dO),
            torch.einsum("bhij,bihe->bjhe", P, dO.abs()))
    dq3 = dqkv.reshape(B, n, 3 * C)
    w.param(blk.qkv.bias, 0, 3 * C, w.pgrad(w.after, blk.qkv.bias), dq3.sum((0, 1)), dq3.abs().sum((0, 1)),
            "colsum", "qkv bias gradient")
    w.param(blk.qkv.weight, 0, 3 * C * C, w.pgrad(w.after, blk.qkv.weight).reshape(3 * C, C),
            torch.einsum("bno,bnc->oc", dq3, hn), torch.einsum("bno,bnc->oc", dq3.abs(), hn.abs()), "wgrad",
            "qkv weight gradient")
    shp = tuple(r.hn.shape)
    w.emit(r.hn, (dq3 @ Wq).reshape(shp), (dq3.abs() @ Wq.abs()).reshape(shp), "gemm", "dgrad of the norm output")


def check_time(w, r):
    dz = f64(w.before[-2])
    Adz = dz.abs()
    if r.act == 1:
        s = dsilu(f64(r.zproj))
        dz, Adz = dz * s, Adz * s.abs()
    cond, W_all = f64(r.cond), f64(r.W_all)
    o = 0
    for blk in r.blocks:
        for p, ref, A in ((blk.time_mlp.weight, dz.t() @ cond, Adz.t() @ cond.abs()),
                          (blk.time_mlp.bias, dz.sum(0), Adz.sum(0))):
            rows = p.shape[0]
            w.param(p, 0, p.numel(), w.pgrad(w.after, p), ref[o:o + rows], A[o:o + rows], "time",
                    "block projection gradient")
        o += blk.time_mlp.weight.shape[0]
    dc, Adc = dz @ W_all, Adz @ W_all.abs()

    def mlp(dout, Adout, la, lb, x_in, z_mid, h_mid, tag):
        hm, zm, xi = f64(h_mid), f64(z_mid), f64(x_in)
        w.param(lb.weight, 0, lb.weight.numel(), w.pgrad(w.after, lb.weight), dout.t() @ hm,
                Adout.t() @ hm.abs(), "time", f"{tag} second linear weight")
        w.param(lb.bias, 0, lb.bias.numel(), w.pgrad(w.after, lb.bias), dout.sum(0), Adout.sum(0), "time",
                f"{tag} second linear bias")
        Wb = f64(lb.weight)
        s = dsilu(zm)
        dzm, Adzm = (dout @ Wb) * s, (Adout @ Wb.abs()) * s.abs()
        w.param(la.weight, 0, la.weight.numel(), w.pgrad(w.after, la.weight), dzm.t() @ xi,
                Adzm.t() @ xi.abs(), "time", f"{tag} first linear weight")
        w.param(la.bias, 0, la.bias.numel(), w.pgrad(w.after, la.bias), dzm.sum(0), Adzm.sum(0), "time",
                f"{tag} first linear bias")

    mlp(dc, Adc, r.l1, r.l2, r.sin, r.z1, r.h1, "time_mlp")
    if r.slice is not None:
        s_ = r.slice
        mlp(dc, Adc, s_["s0"], s_["s2"], s_["z_in"], s_["zz"], s_["zh"], "slice_mlp")


def check_window(w, r):
    (sh, sw), (dh, dw), (nh, nw) = r.src_off, r.dst_off, r.size
    src_win = (slice(None), slice(sh, sh + nh), slice(sw, sw + nw))
    dst_win = (slice(None), slice(dh, dh + nh), slice(dw, dw + nw))
    assert torch.equal(r.dst[dst_win], r.src[src_win]), f"{w.where}: forward window copy differs"
    outside = torch.ones(r.dst.shape[1:3], dtype=torch.bool, device=r.dst.device)
    outside[dh:dh + nh, dw:dw + nw] = False
    assert not bool(r.dst[:, outside].any()), f"{w.where}: forward window copy wrote outside the window"
    dy = w.grad(w.before, r.dst)
    contrib = torch.zeros(r.src.shape, dtype=torch.float64, device=dy.device)
    contrib[src_win] = dy[dst_win].double()
    first = id(r.src) not in w.touched
    w.emit(r.src, contrib, contrib.abs(), "add", "window adjoint")
    if first:
        assert torch.equal(w.grad(w.after, r.src).double(), contrib), f"{w.where}: window adjoint is not a copy"


def check_resize(w, r):
    src = nc(r.src)
    size = tuple(r.dst.shape[1:3])
    up = lambda x: F.interpolate(x, size=size, mode="bilinear", align_corners=False)
    with torch.no_grad():
        w.check("forward restated", "resize", r.dst, cl(up(src)), cl(up(src.abs())))
    dy = nc(w.grad(w.before, r.dst))

    def adj(g):
        x = torch.zeros_like(src).requires_grad_()
        with torch.enable_grad():
            up(x).backward(g)
        return x.grad

    w.emit(r.src, cl(adj(dy)), cl(adj(dy.abs())), "resize", "bilinear adjoint")


CHECKERS = {"ConvRec": check_conv, "GnRec": check_gn, "AttnRec": check_attention, "TimeRec": check_time,
            "WindowRec": check_window, "ResizeRec": check_resize}


# ------------------------------------------------------------------------------------ the walk
def walk_records(prog, name, run_forward):
    run_forward()
    torch.cuda.synchronize()
    g = torch.Generator(device="cuda").manual_seed(1234)
    prog.dout_in.copy_(torch.randn(prog.dout_in.shape, generator=g, device="cuda"))
    S = prog.dout_in[0, 0].numel()
    prog._bwd_head(S)
    assert len(prog.bwd_ranges) == len(prog.tape)
    w = Walk(prog, name)
    nxt = 0
    state = w.snap()
    for i in reversed(range(len(prog.tape))):
        rec, (lo, hi) = prog.tape[i], prog.bwd_ranges[i]
        assert lo == nxt, "record op ranges must tile the launch list in backward order"
        nxt = hi
        prog.run_backward(lo, hi)
        torch.cuda.synchronize()
        w.before, w.after = state, w.snap()
        w.rec_index, w.kind = i, kind_of(rec)
        w.where = f"{name} record {i} {type(rec).__name__}({w.kind}) {getattr(rec, 'name', '')!r}"
        w.bufs_written, w.cols_at = set(), len(w.cols)
        CHECKERS[type(rec).__name__](w, rec)
        w.untouched()
        state = w.after
    assert nxt == len(prog.bwd_ops)
    return w, state


def check_program_wide(w, final):
    prog = w.prog
    # every tracked parameter written, each element by exactly one record; the op after which
    # plan_segments() treats it as final is the end of the last record that writes it
    for pid, p in w.params.items():
        assert pid in w.written, f"{w.name}: no record writes the gradient of a parameter of shape {tuple(p.shape)}"
        rngs = sorted(w.written[pid])
        pos = 0
        for a, b, _ in rngs:
            assert a == pos, f"{w.name}: parameter {tuple(p.shape)} elements [{pos}, {a}) unwritten or overlapping"
            pos = b
        assert pos == p.numel(), f"{w.name}: parameter {tuple(p.shape)} written up to {pos} of {p.numel()}"
        last = min(k for _, _, k in rngs)   # tape index: the backward pass reaches it last
        assert prog._g_last_op[pid] == prog.bwd_ranges[last][1], \
            f"{w.name}: parameter {tuple(p.shape)} is final after op {prog.bwd_ranges[last][1]}, " \
            f"recorded as {prog._g_last_op[pid]}"
        # after its last record nothing changes it (checked record by record); pgrad holds it
        off, n = prog._g_off[pid]
        assert torch.equal(prog.pgrad[pid].reshape(-1).view(torch.int32), final[-1][off:off + n].view(torch.int32))
    assert set(prog._g_off) == set(w.params), f"{w.name}: gradient slices of untracked parameters"
    if prog.dtproj is not None:
        pos = 0
        for a, b in sorted(w.cols):
            assert a == pos, f"{w.name}: dtproj columns [{pos}, {a}) unwritten or written twice"
            pos = b
        assert pos == prog.dtproj.shape[1], f"{w.name}: dtproj written up to column {pos}"


BUCKETS = [1 << 10, 64 << 10, 1 << 20, None]   # None: one bucket for the whole arena


def check_segments(prog):
    S = prog.dout_in[0, 0].numel()
    n_ops = len(prog.bwd_ops)
    for b in BUCKETS:
        segs = prog.plan_segments(b if b is not None else prog._garena_used * 4)
        assert segs[0][0] == 0 and segs[0][2] == 0 and segs[-1][1] == n_ops and segs[-1][3] == prog._garena_used
        for s0, s1 in zip(segs, segs[1:]):
            assert s0[1] == s1[0] and s0[3] == s1[2], segs
        prog._bwd_head(S)
        snaps = []
        for lo, hi, a_lo, a_hi in segs:
            prog.run_backward(lo, hi)
            torch.cuda.synchronize()
            snaps.append(prog.garena[a_lo:a_hi].clone())
        for (lo, hi, a_lo, a_hi), s in zip(segs, snaps):
            assert torch.equal(s.view(torch.int32), prog.garena[a_lo:a_hi].view(torch.int32)), \
                f"bucket {b}: arena [{a_lo}, {a_hi}) changed after segment ops [{lo}, {hi})"
        print(f"  segments at bucket {b}: {len(segs)}")
    prog.bwd_segments = []


@pytest.mark.parametrize("fusion", FUSIONS)
@pytest.mark.parametrize("name", PROGRAMS)
def test_backward_records(name, fusion):
    prog, _, run_forward = program(name, fusion)
    try:
        w, final = walk_records(prog, name, run_forward)
        check_program_wide(w, final)
        check_segments(prog)
        if fusion == "fused":
            assert prog._final, "the fused path defers parameter-gradient gathers"
        else:
            assert not prog._final and not any(h is not None and h[0] is not None
                                               for h in prog._gn_writer.values())
    finally:
        if fusion != "fused":
            _CACHE.pop((name, fusion), None)


def test_window_adjoint_with_offsets():
    """The programs' windows start at (0, 0) on both sides (pad at the end, crop from the start),
    so their records cannot tell the source offset from the destination offset.  Two windows of
    one source with distinct offsets on a bare backward list: the adjoint copies each window back
    to where it came from, the second one added with one rounding, and nothing outside them."""
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.backward import BackwardMixin, WindowRec
    _lib.require_device()
    bw = BackwardMixin()
    bw._binit()
    bw.device, bw.B = "cuda", 2
    g = torch.Generator().manual_seed(3)
    src = torch.zeros(2, 9, 11, 64, dtype=torch.bfloat16, device="cuda")
    dst1 = torch.zeros(2, 6, 8, 64, dtype=torch.bfloat16, device="cuda")
    dst2 = torch.zeros(2, 10, 12, 64, dtype=torch.bfloat16, device="cuda")
    dy1 = torch.randn(dst1.shape, generator=g).to(torch.bfloat16).cuda()
    dy2 = torch.randn(dst2.shape, generator=g).to(torch.bfloat16).cuda()
    bw.tape = [WindowRec(src, dst1, (1, 2), (2, 1), (4, 5)), WindowRec(src, dst2, (3, 0), (0, 4), (6, 7))]
    bw.build_backward({id(dst1): dy1, id(dst2): dy2})
    bw.run_backward()
    torch.cuda.synchronize()
    ref = torch.zeros(src.shape, dtype=torch.float64, device="cuda")
    ref[:, 3:9, 0:7] += dy2[:, 0:6, 4:11].double()     # the later record runs first
    ref[:, 1:5, 2:7] += dy1[:, 2:6, 1:6].double()
    got = bw.grads[id(src)].double()
    assert bool(((got - ref).abs() <= U16 * ref.abs()).all()), float((got - ref).abs().max())
    assert not bool(got[ref == 0].any())


def test_programs_cover_every_record_path():
    """The programs above produce every record type, every ConvRec kind and every special path."""
    seen = set()
    for name in PROGRAMS:
        prog = program(name, "fused")[0]
        for r in prog.tape:
            t = type(r).__name__
            seen.add(t)
            if t == "ConvRec":
                seen.add(f"kind:{r.kind}")
                for f in ("unpack", "unpack_extra", "extra_weight", "residual", "tproj_off", "dgrad_dy", "wfull"):
                    if getattr(r, f) is not None:
                        seen.add(f"conv.{f}")
                assert r.w_rows is None
            elif t == "GnRec":
                for f in ("residual", "tproj_off", "gparam"):
                    if getattr(r, f) is not None:
                        seen.add(f"gn.{f}")
                if r.c_off:
                    seen.add("gn.c_off")
            elif t == "TimeRec":
                seen.add(f"time.act{r.act}")
                if r.slice is not None:
                    seen.add("time.slice")
        if any(h is not None and h[0] is not None for h in prog._gn_writer.values()):
            seen.add("fused colsum")
        if getattr(prog, "z64", None) is not None:
            seen.add("input gradient")
    want = {"ConvRec", "GnRec", "AttnRec", "TimeRec", "WindowRec", "ResizeRec",
            "kind:conv", "kind:down", "kind:up", "kind:matrix",
            "conv.unpack", "conv.unpack_extra", "conv.extra_weight", "conv.residual", "conv.tproj_off",
            "conv.dgrad_dy", "conv.wfull", "gn.residual", "gn.tproj_off", "gn.gparam", "gn.c_off",
            "time.act0", "time.act1", "time.slice", "fused colsum", "input gradient"}
    assert want <= seen, sorted(want - seen)
