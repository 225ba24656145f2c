"""The tcgen05 GEMM kernels (csrc/gemm_tc.cu, csrc/gemm_wgrad.cu) element by element against
float64 references of the same operation on the same bf16-rounded operands, across schedules,
tile shapes and epilogue options.

tests/test_gpu_gemm.py checks whole-tensor rel-L2 <= 4e-3, which dilutes an error confined to one
tile of a 300-tile plan below its threshold.  Here every element is held to its own bound, every
output starts as NaN inside a sentinel-filled buffer (a missed store or a store outside the tensor
fails), and each failure names the output class, the box, the n-tile and, for stream-K plans,
the CTA ranges that share the tile.

Error model and tolerances.  Write r for the fp64 result of the bf16-rounded operands plus the
epilogue's fp32 terms, and A for the same sum over absolute values
(A = conv(|a|, |w|) + |bias| + |row bias| + |residual|).  The kernel's sources of error are the
fp32 accumulation inside tcgen05 and across the stream-K fold (bounded by a multiple of A, not of
|r|: cancellation does not shrink it) and the final rounding of the stored value:

* outputs:  |y - r| <= 2^-8 |r| + BETA A   (bf16 output; 2^-8 is one bf16 ulp, round-to-nearest
  is half of it) and |y - r| <= 2^-24 |r| + BETA A (fp32 output).
* GroupNorm partial sums (fp32 per-thread partials of the un-rounded accumulators, fp64 atomics):
  |sum - sum r| <= BETA_S sum A and |sumsq - sum r^2| <= BETA_S sum A |r| per (sample, group).
* weight gradients: |dw - dw0 - g| <= BETA_W sum |dy| |a| + 2^-23 (|dw0| + |g|) per element, g the
  fp64 sum over positions of dy a; the second term is the fp32 rounding of the red.global.add into
  a non-zero dw0.

The deterministic fp32 bound K 2^-24 is useless at K = 27 * 1024, so the BETAs are measured:
every case records max((|y - r| - 2^-8 |r|) / A) (and the analogues), and each BETA is 4x the
worst measured value.  Measured on one B200 at its 1000 W power limit, every case of this file:

* BETA   = 1.21e-6: worst 3.02e-7 (down plans; conv 2.6e-7, cfg4 top level 2.9e-7, epilogue
  2.3e-7, stream-K schedules 1.4e-7, up 1.2e-7, matrix 8.2e-8, thin_in_conv 3.6e-8).
* BETA_S = 8.9e-7:  worst 2.21e-7 (down plans; epilogue 2.1e-7, cfg4 1.7e-7, conv 1.2e-7).
* BETA_W = 1.96e-6: worst 4.88e-7 (stride-1 with concat and folded skip; down 2.6e-7, up 2.5e-7,
  attention product 1.6e-7).

For bf16 outputs err / bound reaches 0.99: round-to-nearest alone comes to 2^-8 |r| just
above a power of two, so the rounding term of the bound is tight and BETA A is what the
accumulation adds on top.  The WORST table (printed with -s) lists the measured betas, the worst
err / bound per family and the least factor by which the bound flags a plausible bug.

Sensitivity: for each conv family the bound is shown to flag, by a factor >= 10 on at least one
element, the loss of any single (tap, 64-channel slab) contribution, a row bias read for the
neighbouring sample and the residual of the neighbouring box.
"""
import itertools
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BETA = 1.21e-6   # outputs, per unit of A
BETA_S = 8.9e-7   # GroupNorm partial sums
BETA_W = 1.96e-6  # weight gradients
SENS = 10.0      # a plausible bug must exceed the bound by this factor on some element

WORST = {}     # key -> worst measured value (printed at the end of the module, run with -s)
LEAST = {}     # key -> least detection factor of a plausible bug


def note(key, value):
    WORST[key] = max(WORST.get(key, -math.inf), float(value))


def note_min(key, value):
    LEAST[key] = min(LEAST.get(key, math.inf), float(value))


@pytest.fixture(scope="module", autouse=True)
def _print_worst():
    yield
    if WORST:
        print("\n[gemm kernels] worst measured values")
        for k in sorted(WORST):
            print(f"  {k:44s} {WORST[k]: .3e}")
        for k in sorted(LEAST):
            print(f"  {k:44s} {LEAST[k]: .3e}")


@pytest.fixture(scope="module")
def P():
    from mri_image_generation_b200 import _lib, plan
    _lib.require_device()
    return plan


def sms(P):
    return P.gemm_workspace("cuda").n_ctas


# ------------------------------------------------------------------------------ guarded outputs
_PAD = 256          # elements before and after the tensor (512 B / 1 KB: 128-byte aligned offset)
_SENT = {torch.bfloat16: (torch.int16, 0x5A5A), torch.float32: (torch.int32, 0x5A5A5A5A)}


class Guarded:
    """A contiguous tensor inside a larger buffer whose head and tail hold a sentinel pattern."""

    def __init__(self, shape, dtype, device="cuda"):
        n = int(np.prod(shape))
        self.n = n
        self.dtype = dtype
        self.buf = torch.empty(n + 2 * _PAD, dtype=dtype, device=device)
        self.y = self.buf[_PAD:_PAD + n].view(shape)
        self.reset()

    def reset(self):
        it, pat = _SENT[self.dtype]
        self.buf.view(it).fill_(pat)
        self.y.fill_(float("nan"))

    def sentinels_ok(self):
        it, pat = _SENT[self.dtype]
        bits = self.buf.view(it)
        return bool((bits[:_PAD] == pat).all() and (bits[_PAD + self.n:] == pat).all())


# ------------------------------------------------------------------------------ schedule (Python)
def launch_grid(pl, G):
    """The grid mri_gemm_launch picks (gemm_tc.cu): min(tiles, G), or for a stream-K plan with
    fewer tiles than SMs, shares of >= max(8, n_kb / 4) k-steps."""
    tiles, n_kb = pl.grid(), pl.n_kb
    grid = min(tiles, G)
    if pl._args.sched and tiles < G:
        ms = max((n_kb + 3) // 4, 8)
        grid = min(max(tiles * n_kb // ms, tiles), G)
    return grid


def make_sched(pl, G):
    """make_sched / range_a of gemm_tc.cu restated: q, rem, GA and the phase-A unit ranges."""
    n_tiles, n_kb = pl.grid(), pl.n_kb
    grid = launch_grid(pl, G)
    s = dict(grid=grid, n_tiles=n_tiles, n_kb=n_kb, sched=pl._args.sched)
    if not pl._args.sched:
        s.update(q=0, rem=0, GA=0, ranges=[])
        return s
    q = n_tiles // grid
    rem = n_tiles - q * grid
    units = rem * n_kb
    ms = max((n_kb + 3) // 4, 8)
    ga = units // ms
    GA = (1 if rem > 0 else 0) if ga < 1 else min(ga, grid)
    ranges = [(units * r // GA, units * (r + 1) // GA) for r in range(GA)]
    s.update(q=q, rem=rem, GA=GA, ranges=ranges)
    return s


def straddles(s):
    """Some phase-A range is the tail of one tile and the head of the next."""
    n_kb = s["n_kb"]
    return any(u0 // n_kb != (u1 - 1) // n_kb and u0 % n_kb != 0 for u0, u1 in s["ranges"] if u1 > u0)


def tile_of(pl, cls, xs, ch):
    a = pl._args
    tix = [xs[i] // pl.box[i] for i in range(4)]
    f = pl.tile_fast_dim
    od = [f] + [k for k in range(4) if k != f]
    b, mul = 0, 1
    for k in range(4):
        b += tix[od[k]] * mul
        mul *= pl.tiles[od[k]]
    boxes = int(np.prod(pl.tiles))
    gpc = -(-boxes // 2) if a.swap_ab else boxes
    group = b // 2 if a.swap_ab else b
    return tix, (cls * gpc + group) * pl.n_tiles_n + ch // pl.block_n


def describe(pl, G, cls, xs, ch):
    tix, tile = tile_of(pl, cls, xs, ch)
    s = make_sched(pl, G)
    head = (f"class {cls}, box {tuple(tix)} (position {tuple(xs)}), n-tile {ch // pl.block_n} "
            f"(channel {ch}), tile {tile} of {s['n_tiles']}, grid {s['grid']}, sched {s['sched']}")
    n_kb = s["n_kb"]
    if not s["sched"]:
        r = next(r for r in range(s["grid"]) if s["n_tiles"] * (r + 1) // s["grid"] > tile)
        return head + f": whole tile of CTA {r}"
    if tile < s["rem"]:
        parts = []
        for r, (u0, u1) in enumerate(s["ranges"]):
            a, b = max(u0, tile * n_kb), min(u1, (tile + 1) * n_kb)
            if a < b:
                parts.append(f"CTA {r} k-steps {a - tile * n_kb}..{b - 1 - tile * n_kb}")
        return head + f": phase-A tile {tile}, " + ", ".join(parts)
    r = (tile - s["rem"]) // s["q"]
    return head + f": phase-B tile of CTA {r}"


# ------------------------------------------------------------------------------ checks
def bound_of(r, A, f32):
    return (2.0 ** -24 if f32 else 2.0 ** -8) * r.abs() + BETA * A


def check_out(fam, pl, G, y, r, A, where, f32=False, guard=None, tag=""):
    """Elementwise bound on y against (r, A) of the same shape.  where(flat index) -> (cls, xs, ch)
    or None."""
    y64 = y.double()
    fin = torch.isfinite(y64)
    if not bool(fin.all()):
        i = int((~fin).reshape(-1).nonzero()[0])
        loc = where(i) if where else None
        msg = describe(pl, G, *loc) if loc else f"flat index {i}"
        raise AssertionError(f"{fam}{tag}: {int((~fin).sum())} elements never stored; first at {msg}")
    if guard is not None:
        assert guard.sentinels_ok(), f"{fam}{tag}: store outside the output tensor"
    rnd = 2.0 ** -24 if f32 else 2.0 ** -8
    err = (y64 - r).abs()
    Ac = A.clamp_min(1e-300)
    note(f"beta {fam}", ((err - rnd * r.abs()) / Ac).max())
    ratio = err / bound_of(r, A, f32).clamp_min(1e-300)
    note(f"ratio {fam}", ratio.max())
    if float(ratio.max()) > 1.0:
        i = int(ratio.reshape(-1).argmax())
        loc = where(i) if where else None
        msg = describe(pl, G, *loc) if loc else f"flat index {i}"
        bad = int((ratio > 1).sum())
        raise AssertionError(
            f"{fam}{tag}: {bad} elements outside the bound; worst {float(ratio.reshape(-1)[i]):.2f}x "
            f"(y {float(y64.reshape(-1)[i]):.6g}, ref {float(r.reshape(-1)[i]):.6g}, "
            f"A {float(A.reshape(-1)[i]):.3g}) at {msg}")


def check_stats(fam, stats, r, A, groups):
    """stats [N, G, 2] fp64 vs (r, A) channels-last [N, ..., C]."""
    N, C = r.shape[0], r.shape[-1]
    rr = r.reshape(N, -1, groups, C // groups)
    aa = A.reshape(N, -1, groups, C // groups)
    s0, s1 = rr.sum((1, 3)), (rr * rr).sum((1, 3))
    b0, b1 = aa.sum((1, 3)), (aa * rr.abs()).sum((1, 3))
    e0 = (stats[..., 0] - s0).abs() / b0
    e1 = (stats[..., 1] - s1).abs() / b1
    note(f"beta_s {fam}", max(float(e0.max()), float(e1.max())))
    assert float(e0.max()) <= BETA_S, (fam, "sum", float(e0.max()), e0.argmax().item())
    assert float(e1.max()) <= BETA_S, (fam, "sumsq", float(e1.max()), e1.argmax().item())


def sensitivity(fam, contribs, r, A, f32=False):
    """contribs: iterable of (label, delta tensor broadcastable to r): each must exceed the bound
    by SENS on at least one element."""
    bnd = bound_of(r, A, f32)
    worst = math.inf
    for label, d in contribs:
        det = float((d.abs() / bnd.clamp_min(1e-300)).max())
        worst = min(worst, det)
        assert det >= SENS, f"{fam}: the bound cannot see {label} (x{det:.2f})"
    note_min(f"sensitivity {fam}", worst)


# ------------------------------------------------------------------------------ references
def nhwc(t):
    nd = t.dim() - 2
    return t.permute(0, *range(2, 2 + nd), 1).contiguous()


def nchw(t):
    nd = t.dim() - 2
    return t.permute(0, nd + 1, *range(1, nd + 1)).contiguous()


def bf(t):
    return t.to(torch.bfloat16)


def f64conv(fn, *args, **kw):
    try:
        return fn(*args, **kw)
    except RuntimeError:       # an fp64 shape the GPU library refuses: compute it on the CPU
        return fn(*[a.cpu() if torch.is_tensor(a) else a for a in args], **kw).cuda()


def tap_contribs(x, w, kind):
    """Per (tap, 64-channel slab) contributions [N, Co, *out] of a convolution: kind 'conv'
    (stride 1, pad k // 2), 'down' (k 4, stride 2, pad 1), 'up' (transposed, k 4, stride 2,
    pad 1; w [Ci, Co, *k])."""
    nd = x.dim() - 2
    N, Ci = x.shape[:2]
    ns = Ci // 64
    sp = x.shape[2:]
    k = w.shape[2]
    if kind == "up":
        Co = w.shape[1]
        for tap in itertools.product(range(k), repeat=nd):
            wt = w[(slice(None), slice(None)) + tap].reshape(ns, 64, Co)
            c = torch.einsum("nsc...,sco->sno...", x.reshape(N, ns, 64, *sp), wt)
            full = torch.zeros(ns, N, Co, *[2 * e + 2 for e in sp], dtype=x.dtype, device=x.device)
            idx = (slice(None),) * 3 + tuple(slice(t, t + 2 * e, 2) for t, e in zip(tap, sp))
            full[idx] = c
            out = full[(slice(None),) * 3 + tuple(slice(1, 1 + 2 * e) for e in sp)]
            for s in range(ns):
                yield f"tap {tap} slab {s}", out[s]
        return
    Co = w.shape[0]
    stride, pad = (1, k // 2) if kind == "conv" else (2, 1)
    xp = F.pad(x, [pad] * 2 * nd)
    osp = [(e + 2 * pad - k) // stride + 1 for e in sp]
    for tap in itertools.product(range(k), repeat=nd):
        idx = (slice(None),) * 2 + tuple(slice(t, t + stride * o, stride) for t, o in zip(tap, osp))
        xs = xp[idx]
        wt = w[(slice(None), slice(None)) + tap].reshape(Co, ns, 64)
        c = torch.einsum("nsc...,osc->sno...", xs.reshape(N, ns, 64, *osp), wt)
        for s in range(ns):
            yield f"tap {tap} slab {s}", c[s]


def conv_where(y_shape):
    """flat index of a channels-last [N, *sp, C] output -> (class, (x1..x4), channel)."""
    def f(i):
        idx = np.unravel_index(i, y_shape)
        n, spc, ch = idx[0], list(idx[1:-1]), idx[-1]
        xs = list(reversed(spc)) + [n]
        xs += [0] * (4 - len(xs))
        return 0, tuple(int(v) for v in xs), int(ch)
    return f


def up_where(y_shape):
    nd = len(y_shape) - 2

    def f(i):
        idx = np.unravel_index(i, y_shape)
        n, spc, ch = idx[0], list(idx[1:-1]), idx[-1]
        rho = [int(v) % 2 for v in reversed(spc)]       # w first
        cls = 0
        for b in rho:
            cls = cls * 2 + b
        xs = [int(v) // 2 for v in reversed(spc)] + [n]
        xs += [0] * (4 - len(xs))
        return cls, tuple(int(v) for v in xs), int(ch)
    return f


def run(pl, G, sched, guard, stats=None, swap=None):
    pl.sched = sched
    if swap is not None:
        pl.swap_ab = swap
    guard.reset()
    if stats is not None:
        stats.zero_()
    pl.materialize("cuda")
    pl.launch()
    torch.cuda.synchronize()
    return make_sched(pl, G)


def scheds_for(pl):
    """Every plan with K loops of >= 8 k-steps goes through both schedules."""
    return (0, 1) if pl.n_kb >= 8 else (0,)


# ============================================================================ 1-2. stride-1 conv_plan
# id, nd, sp, N, source channels, folded skip channels, Cout, options
CONV_CASES = [
    ("3d_c128_swap", 3, (8, 12, 10), 2, [128], 0, 128, {}),
    ("3d_bn16", 3, (8, 8, 8), 1, [128], 0, 16, {}),
    ("3d_bn32", 3, (6, 8, 7), 2, [64], 0, 32, {}),
    # boxes of two samples, three boxes, the last one half empty
    ("3d_cout64_n5", 3, (3, 3, 5), 5, [64], 0, 64, dict(bias=True, rowbias=True, cpg=8)),
    ("2d_two_src_256", 2, (24, 24), 3, [64, 64], 0, 256, {}),
    ("2d_three_src_skip", 2, (20, 20), 8, [64, 64, 64], 64, 128, {}),
    ("3d_1x1_1024", 3, (10, 12, 10), 2, [512], 0, 1024, dict(k=1)),
    ("3d_c512", 3, (10, 12, 10), 2, [256], 0, 512, {}),
    ("3d_n8_boxes_pair_samples", 3, (10, 12, 10), 8, [128], 0, 256, dict(rowbias=True, residual=True, cpg=32)),
    ("2d_n8_boxes_pair_samples", 2, (6, 10), 8, [64], 0, 32, dict(rowbias=True, cpg=8)),
    ("3d_xreuse0", 3, (12, 32, 16), 2, [128], 0, 128, dict(xreuse=0)),
    ("3d_xreuse1_tfd0", 3, (12, 32, 16), 2, [128], 0, 128, dict(xreuse=1, tfd=0)),
    ("3d_xreuse1_tfd1", 3, (12, 32, 16), 2, [128], 0, 128, dict(xreuse=1, tfd=1)),
    ("3d_xreuse2", 3, (12, 32, 16), 2, [128], 64, 128, dict(xreuse=2)),
    ("2d_xreuse2_concat", 2, (48, 24), 3, [64, 64], 0, 128, dict(xreuse=2)),
    ("3d_odd_boxes_lone", 3, (5, 16, 8), 1, [128], 0, 128, dict(xreuse=1)),
    ("3d_swap_off", 3, (8, 12, 10), 2, [128], 0, 128, dict(swap=False, xreuse=0)),
    ("2d_swap_off_192", 2, (30, 30), 3, [192], 0, 128, dict(swap=False, xreuse=0)),
]

# epilogue options on a swap-mode (128 channels) and a plain-tile (32 channels) convolution
EPI_OPTS = [
    dict(bias=True), dict(rowbias=True), dict(residual=True), dict(cpg=8), dict(cpg=16),
    dict(cpg=32), dict(cpg=64), dict(cpg=4), dict(out_f32=True), dict(out_f32=True, cpg=16),
    dict(bias=True, rowbias=True, residual=True, cpg=16),
]


def conv_inputs(nd, sp, N, cins, skip, cout, k, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    acts = [bf(torch.randn(N, *sp, c, device="cuda", generator=g)) for c in cins]
    cin = sum(cins)
    w = torch.randn(cout, cin, *([k] * nd), device="cuda", generator=g) / (cin * k ** nd) ** 0.5
    ws = torch.randn(cout, skip, *([1] * nd), device="cuda", generator=g) / max(skip, 1) ** 0.5 if skip else None
    return acts, w, ws, g


def conv_reference(nd, acts, w, ws, skip_src, bias, rb, res, k):
    """r and A, channels-last fp64, plus the inputs the sensitivity check needs (NCHW fp64)."""
    conv = F.conv3d if nd == 3 else F.conv2d
    x = torch.cat([nchw(a.double()) for a in acts], 1)
    w64 = bf(w).double()
    r = f64conv(conv, x, w64, padding=k // 2)
    A = f64conv(conv, x.abs(), w64.abs(), padding=k // 2)
    xs = ws64 = None
    if ws is not None:
        xs = nchw(skip_src.double())
        ws64 = bf(ws).double()
        r = r + f64conv(conv, xs, ws64)
        A = A + f64conv(conv, xs.abs(), ws64.abs())
    r, A = nhwc(r), nhwc(A)
    N, C = r.shape[0], r.shape[-1]
    bshape = (N,) + (1,) * nd + (C,)
    if bias is not None:
        r = r + bias.double().reshape(1, *([1] * nd), C)
        A = A + bias.double().abs().reshape(1, *([1] * nd), C)
    if rb is not None:
        r = r + rb[:, :C].double().reshape(bshape)
        A = A + rb[:, :C].double().abs().reshape(bshape)
    if res is not None:
        r = r + res.double()
        A = A + res.double().abs()
    return r, A, (x, w64, xs, ws64)


def conv_case(P, nd, sp, N, cins, skip, cout, opts, seed, fam):
    G = sms(P)
    k = opts.get("k", 3)
    acts, w, ws, g = conv_inputs(nd, sp, N, cins, skip, cout, k, seed)
    f32 = opts.get("out_f32", False)
    bias = torch.randn(cout, device="cuda", generator=g) if opts.get("bias") else None
    rb_ld = cout + 8
    rb = torch.randn(N, rb_ld, device="cuda", generator=g) if opts.get("rowbias") else None
    res = bf(torch.randn(N, *sp, cout, device="cuda", generator=g)) if opts.get("residual") else None
    cpg = opts.get("cpg", 0)
    stats = torch.zeros(N, cout // cpg, 2, dtype=torch.float64, device="cuda") if cpg else None
    srcs = [P.ConvSource(a) for a in acts]
    if skip:
        srcs.append(P.ConvSource(acts[0][..., :skip].contiguous(), taps=False))
    wm = P.pack_conv_weight(w, splits=cins, extra=[ws] if skip else ())
    guard = Guarded((N, *sp, cout), torch.float32 if f32 else torch.bfloat16)
    pl = P.conv_plan(srcs, wm, guard.y, k, bias=bias, rowbias=rb, rowbias_ld=rb_ld if rb is not None else 0,
                     residual=res, stats=stats, stats_cpg=cpg, xreuse=opts.get("xreuse"), out_f32=f32)
    # the case is in the class it exists for
    if "xreuse" in opts:
        assert pl.xreuse == opts["xreuse"], (pl.xreuse, pl.box)
    if "swap" in opts:
        pl.swap_ab = opts["swap"]
    if "tfd" in opts:
        pl.tile_fast_dim = opts["tfd"]
    assert pl.block_n == (128 if cout % 64 == 0 else (32 if cout % 32 == 0 else 16))
    assert pl.pick_swap() == (pl.block_n == 128 and not f32 and opts.get("swap", True))
    r, A, (x, w64, xs, ws64) = conv_reference(nd, acts, w, ws, srcs[-1].x if skip else None, bias, rb, res, k)
    where = conv_where(guard.y.shape)
    for sched in scheds_for(pl):
        s = run(pl, G, sched, guard, stats)
        check_out(fam, pl, G, guard.y, r, A, where, f32, guard, tag=f" sched {sched}")
        if stats is not None:
            check_stats(fam, stats, r, A, cout // cpg)
    return pl, r, A, (x, w64, xs, ws64, rb, res)


def conv_sensitivity(fam, pl, r, A, x, w64, xs, ws64, rb, res, f32=False, kind="conv"):
    rc, Ac = nchw(r), nchw(A)
    contribs = tap_contribs(x, w64, kind)
    if xs is not None:
        contribs = itertools.chain(contribs, (("skip " + l, d) for l, d in tap_contribs(xs, ws64, "conv")))
    sensitivity(fam, contribs, rc, Ac, f32)
    extra = []
    nd = r.dim() - 2
    N, C = r.shape[0], r.shape[-1]
    if rb is not None and N > 1:
        rbd = rb[:, :C].double()
        d = rbd[(torch.arange(N, device="cuda") + 1) % N] - rbd
        extra.append(("row bias of the neighbouring sample", d.reshape(N, *([1] * nd), C)))
    if res is not None:
        rs = res.double()
        # the first box dim with more than one box; x_i is channels-last dim nd - i (x_nd+1 = the
        # sample dim 0); up plans tile the input, whose boxes are twice as wide in the output
        i = next(i for i in range(4) if pl.tiles[i] > 1)
        dim = nd - i if i < nd else 0
        d = torch.roll(rs, shifts=pl.box[i] * (2 if kind == "up" and i < nd else 1), dims=dim) - rs
        extra.append(("residual of the neighbouring box", d))
    sensitivity(fam, extra, r, A, f32)


@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_conv_stride1(P, case):
    name, nd, sp, N, cins, skip, cout, opts = case
    pl, r, A, inp = conv_case(P, nd, sp, N, cins, skip, cout, opts, seed=sum(map(ord, name)), fam="conv")
    if name == "3d_odd_boxes_lone":
        assert pl.pick_swap() and int(np.prod(pl.tiles)) % 2 == 1     # one swap tile holds a lone box
    if "boxes_pair_samples" in name:
        assert pl.box[pl.sample_dim - 1] > 1                          # boxes span several samples
    if name == "3d_cout64_n5":
        assert int(np.prod(pl.tiles)) % 2 == 1 and any(e % b for e, b in zip(pl.ext, pl.box))
    conv_sensitivity("conv", pl, r, A, *inp)


@pytest.mark.parametrize("cout", [128, 32])
@pytest.mark.parametrize("opts", EPI_OPTS, ids=lambda o: "-".join(f"{k}{'' if v is True else v}" for k, v in o.items()))
def test_conv_epilogue(P, cout, opts):
    f32 = opts.get("out_f32", False)
    if opts.get("cpg", 0) > cout or (opts.get("cpg") == 4 and (cout != 128 or f32)):
        pytest.skip("statistics groups of 4 channels exist in swap mode only")
    N = 3
    pl, r, A, inp = conv_case(P, 3, (6, 8, 10), N, [128], 0, cout, opts, seed=7 + cout, fam="epilogue")
    assert pl.pick_swap() == (cout == 128 and not f32)
    conv_sensitivity("epilogue", pl, r, A, *inp, f32=f32)


# ============================================================================ 3. down / up plans
DOWN_UP = [
    ("down", 3, (8, 12, 8), 2, 128, 256, dict(bias=True, cpg=32)),
    ("down", 2, (32, 48), 2, 64, 64, dict(bias=True, cpg=8)),
    ("down", 3, (8, 12, 8), 2, 128, 128, dict(out_f32=True, cpg=16)),
    ("down", 2, (16, 24), 3, 128, 128, dict(residual=True)),
    ("up", 3, (4, 6, 4), 2, 128, 64, dict(bias=True, cpg=8)),
    ("up", 2, (16, 24), 2, 128, 128, dict(bias=True, cpg=16)),
    ("up", 3, (4, 6, 4), 2, 128, 128, dict(residual=True)),      # dgrad of a stride-2 conv
    ("up", 2, (16, 24), 2, 128, 128, dict(residual=True)),
    ("up", 3, (4, 6, 4), 2, 128, 128, dict(out_f32=True, cpg=16)),
]


@pytest.mark.parametrize("case", DOWN_UP, ids=lambda c: f"{c[0]}{c[1]}d-{c[4]}-{c[5]}-{'-'.join(c[6])}")
def test_down_up(P, case):
    kind, nd, sp, N, cin, cout, opts = case
    G = sms(P)
    g = torch.Generator(device="cuda").manual_seed(cin + cout + nd)
    f32 = opts.get("out_f32", False)
    a = bf(torch.randn(N, *sp, cin, device="cuda", generator=g))
    osp = [e // 2 for e in sp] if kind == "down" else [2 * e for e in sp]
    if kind == "down":
        w = torch.randn(cout, cin, *([4] * nd), device="cuda", generator=g) / (cin * 4 ** nd) ** 0.5
        wm = P.pack_conv_weight(w)
    else:
        w = torch.randn(cin, cout, *([4] * nd), device="cuda", generator=g) / (cin * 2 ** nd) ** 0.5
        wm = P.pack_convT_weight(w)
    bias = torch.randn(cout, device="cuda", generator=g) if opts.get("bias") else None
    res = bf(torch.randn(N, *osp, cout, device="cuda", generator=g)) if opts.get("residual") else None
    cpg = opts.get("cpg", 0)
    stats = torch.zeros(N, cout // cpg, 2, dtype=torch.float64, device="cuda") if cpg else None
    guard = Guarded((N, *osp, cout), torch.float32 if f32 else torch.bfloat16)
    mk = P.down_conv_plan if kind == "down" else P.up_conv_plan
    pl = mk(a, wm, guard.y, bias=bias, stats=stats, stats_cpg=cpg, residual=res, out_f32=f32)
    assert pl.n_class == (1 if kind == "down" else 2 ** nd)
    if res is not None and kind == "up":
        offs = {m.view.offset for m in pl.r_maps}
        assert len(offs) == 2 ** nd          # one residual offset per output class
    x = nchw(a.double())
    w64 = bf(w).double()
    fn = (F.conv3d if nd == 3 else F.conv2d) if kind == "down" else \
        (F.conv_transpose3d if nd == 3 else F.conv_transpose2d)
    r = nhwc(f64conv(fn, x, w64, stride=2, padding=1))
    A = nhwc(f64conv(fn, x.abs(), w64.abs(), stride=2, padding=1))
    if bias is not None:
        r, A = r + bias.double(), A + bias.double().abs()
    if res is not None:
        r, A = r + res.double(), A + res.double().abs()
    where = (conv_where if kind == "down" else up_where)(guard.y.shape)
    fam = kind
    for sched in scheds_for(pl):
        run(pl, G, sched, guard, stats)
        check_out(fam, pl, G, guard.y, r, A, where, f32, guard, tag=f" sched {sched}")
        if stats is not None:
            check_stats(fam, stats, r, A, cout // cpg)
    conv_sensitivity(fam, pl, r, A, x, w64, None, None, None, res, f32=f32, kind=kind)


# ============================================================================ 4. matrix plans
def matrix_check(fam, P, pl, G, guard, r, A, f32, slabs, where=None, stats=None, groups=0):
    for sched in scheds_for(pl):
        run(pl, G, sched, guard, stats)
        check_out(fam, pl, G, guard.y, r, A, where, f32, guard, tag=f" sched {sched}")
        if stats is not None:
            check_stats(fam, stats, r, A, groups)
    sensitivity(fam, slabs, r, A, f32)


def slab_contribs(a, b, eq):
    """einsum eq over the K slabs of 64 (a, b: K last)."""
    K = a.shape[-1]
    for k0 in range(0, K, 64):
        yield f"k-slab {k0 // 64}", torch.einsum(eq, a[..., k0:k0 + 64], b[..., k0:k0 + 64])


@pytest.mark.parametrize("n", [200, 333])
def test_matrix_qkT_fp32(P, n):
    G = sms(P)
    B, heads, d = 2, 4, 128
    C = heads * d
    g = torch.Generator(device="cuda").manual_seed(n)
    qk = bf(torch.randn(B, n, 2 * C, device="cuda", generator=g))
    npad = (n + 7) // 8 * 8
    guard = Guarded((B, heads, n, npad), torch.float32)
    S = guard.y
    a = P.TView(qk, (d, n, heads, B, 1), (1, 2 * C, d, n * 2 * C, B * n * 2 * C))
    b = P.TView(qk, (d, n, heads, B), (1, 2 * C, d, n * 2 * C), offset=C)
    o = P.TView(S, (npad, n, heads, B, 1), (1, npad, n * npad, heads * n * npad, B * heads * n * npad))
    pl = P.matrix_plan(a, (128, 1, 1, 1), b, o, K=d, n_total=npad, block_n=128,
                       ext=(n, heads, B, 1), tiles=(-(-n // 128), heads, B, 1), bz_sel=(3, 4), out_f32=True)
    assert n % 128 and not pl.pick_swap()
    q = qk[:, :, :C].double().reshape(B, n, heads, d).permute(0, 2, 1, 3)
    k = qk[:, :, C:].double().reshape(B, n, heads, d).permute(0, 2, 1, 3)
    kp = torch.zeros(B, heads, npad, d, dtype=torch.float64, device="cuda")
    kp[:, :, :n] = k
    r = q @ kp.transpose(-1, -2)
    A = q.abs() @ kp.abs().transpose(-1, -2)

    def where(i):
        bb, h, m, j = np.unravel_index(i, S.shape)
        return 0, (int(m), int(h), int(bb), 0), int(j)
    matrix_check("matrix", P, pl, G, guard, r, A, True, slab_contribs(q, kp, "bhmk,bhnk->bhmn"), where)


@pytest.mark.parametrize("d", [64, 128])
def test_matrix_pv(P, d):
    G = sms(P)
    B, heads, n = 2, 2, 520
    C = heads * d
    npad = (n + 7) // 8 * 8
    g = torch.Generator(device="cuda").manual_seed(d)
    Pm = bf(torch.rand(B, heads, n, npad, device="cuda", generator=g) / n)
    Pm[..., n:] = 0
    kvT = bf(torch.randn(B, 2 * C, npad, device="cuda", generator=g))
    sz = 2 * C * npad
    guard = Guarded((B, n, C), torch.bfloat16)
    O = guard.y
    pa = P.TView(Pm, (npad, n, heads, B, 1), (1, npad, n * npad, heads * n * npad, B * heads * n * npad))
    vb = P.TView(kvT, (npad, d, heads, B), (1, npad, d * npad, sz), offset=C * npad)
    oo = P.TView(O, (d, n, heads, B, 1), (1, C, d, n * C, B * n * C))
    pl = P.matrix_plan(pa, (128, 1, 1, 1), vb, oo, K=npad, n_total=d, block_n=min(d, 128),
                       ext=(n, heads, B, 1), tiles=(-(-n // 128), heads, B, 1), bz_sel=(3, 4))
    assert pl.block_n == d and pl.n_kb >= 8
    p64 = Pm.double()
    v = kvT[:, C:].double().reshape(B, heads, d, npad)
    r = torch.einsum("bhmk,bhdk->bmhd", p64, v).reshape(B, n, C)
    A = torch.einsum("bhmk,bhdk->bmhd", p64.abs(), v.abs()).reshape(B, n, C)

    def where(i):
        bb, m, c = np.unravel_index(i, O.shape)
        return 0, (int(m), int(c) // d, int(bb), 0), int(c) % d
    slabs = ((l, c.permute(0, 2, 1, 3).reshape(B, n, C)) for l, c in slab_contribs(p64, v, "bhmk,bhdk->bhmd"))
    matrix_check("matrix", P, pl, G, guard, r, A, False, slabs, where)


@pytest.mark.parametrize("rows_mult", [2, 1])      # kvT (2C rows) and vT (C rows)
def test_matrix_bias_m(P, rows_mult):
    G = sms(P)
    B, C, n = 2, 256, 200
    npad = (n + 7) // 8 * 8
    R = rows_mult * C
    g = torch.Generator(device="cuda").manual_seed(R)
    wkv = bf(torch.randn(R, C, device="cuda", generator=g) / C ** 0.5)
    bkv = torch.randn(R, device="cuda", generator=g)
    hn = bf(torch.randn(B, n, C, device="cuda", generator=g))
    guard = Guarded((B, R, npad), torch.bfloat16)
    kvT = guard.y
    a = P.TView(wkv, (C, R, 1, 1, 1), (1, C, R * C, R * C, R * C))
    b = P.TView(hn, (C, n, B, 1), (1, C, n * C, B * n * C))
    sz = R * npad
    o_views = [P.TView(kvT, (npad, R, 1, 1, 1), (1, npad, sz, sz, sz), offset=bi * sz) for bi in range(B)]
    pl = P.matrix_plan(a, (128, 1, 1, 1), b, o_views[0], K=C, n_total=npad, block_n=128,
                       ext=(R, 1, 1, 1), tiles=(R // 128, 1, 1, 1), bz_sel=(1, 0), bias_m=bkv)
    pl.o_maps = [P.MapSpec(v, pl.o_maps[0].box, pl.o_maps[0].swizzle) for v in o_views]
    pl.ktable = pl.ktable.repeat(B, axis=0)
    assert pl.n_class == B and not pl.pick_swap()
    h = torch.zeros(B, npad, C, dtype=torch.float64, device="cuda")
    h[:, :n] = hn.double()
    w64 = wkv.double()
    r = torch.einsum("rc,bjc->brj", w64, h) + bkv.double()[None, :, None]
    A = torch.einsum("rc,bjc->brj", w64.abs(), h.abs()) + bkv.double().abs()[None, :, None]

    def where(i):
        bb, m, j = np.unravel_index(i, kvT.shape)
        return int(bb), (int(m), 0, 0, 0), int(j)
    slabs = list(slab_contribs(w64[None].expand(B, R, C), h, "brc,bjc->brj"))
    slabs.append(("bias_m of the neighbouring row", (bkv.roll(1) - bkv).double()[None, :, None]))
    matrix_check("matrix", P, pl, G, guard, r, A, False, slabs, where)


@pytest.mark.parametrize("nd,sp,cout", [(2, (24, 20), 1), (2, (24, 20), 3), (3, (6, 8, 10), 4)])
def test_out_conv_tap_gemm(P, nd, sp, cout):
    """The thin out_conv's GEMM over taps: Y[q][tap * cout + co] = W[tap][co] . a[q]."""
    G = sms(P)
    N, cin = 2, 128
    taps = 3 ** nd
    n_y = -(-taps * cout // 16) * 16 if taps * cout <= 48 else -(-taps * cout // 64) * 64
    g = torch.Generator(device="cuda").manual_seed(n_y)
    a = bf(torch.randn(N, *sp, cin, device="cuda", generator=g))
    w = torch.randn(cout, cin, *([3] * nd), device="cuda", generator=g) / cin ** 0.5
    wm = P.pack_tap_weight(w, n_y)
    guard = Guarded((N, *sp, n_y), torch.bfloat16)
    pl = P.conv_plan([P.ConvSource(a)], wm, guard.y, 1)
    assert pl.block_n == {16: 16, 32: 32}.get(n_y, 128)
    wmat = wm.double()                                       # [n_y, cin]
    r = torch.einsum("n...c,oc->n...o", a.double(), wmat)
    A = torch.einsum("n...c,oc->n...o", a.double().abs(), wmat.abs())
    # the reference weight rows really are the taps of w
    assert torch.equal(wmat[:taps * cout].reshape(taps, cout, cin),
                       bf(w).double().reshape(cout, cin, taps).permute(2, 0, 1))
    slabs = slab_contribs(a.double(), wmat, "n...c,oc->n...o")
    matrix_check("tap_gemm", P, pl, G, guard, r, A, False, slabs, conv_where(guard.y.shape))


# ============================================================================ 5. schedules
def sched_matrix(P, T, n_kb, seed, swap=False, stats=False):
    """A plain [T * 128, K] x [K, 128] plan whose tile count is chosen against the grid."""
    M, K, Nn = T * 128 * (2 if swap else 1), n_kb * 64, 128
    g = torch.Generator(device="cuda").manual_seed(seed)
    am = bf(torch.randn(M, K, device="cuda", generator=g))
    bm = bf(torch.randn(Nn, K, device="cuda", generator=g) / K ** 0.5)
    bias = torch.randn(Nn, device="cuda", generator=g)
    guard = Guarded((M, Nn), torch.bfloat16)
    st = torch.zeros(1, 8, 2, dtype=torch.float64, device="cuda") if stats else None
    a = P.TView(am, (K, M, 1, 1, 1), (1, K, M * K, M * K, M * K))
    b = P.TView(bm, (K, Nn, 1, 1), (1, K, Nn * K, Nn * K))
    o = P.TView(guard.y, (Nn, M, 1, 1, 1), (1, Nn, M * Nn, M * Nn, M * Nn))
    pl = P.matrix_plan(a, (128, 1, 1, 1), b, o, K=K, n_total=Nn, block_n=128, ext=(M, 1, 1, 1),
                       tiles=(M // 128, 1, 1, 1), bias=bias, stats=st, stats_cpg=16 if stats else 0)
    pl.swap_ab = swap
    a64, b64 = am.double(), bm.double()
    r = a64 @ b64.T + bias.double()
    A = a64.abs() @ b64.abs().T + bias.double().abs()

    def where(i):
        m, c = divmod(int(i), Nn)
        return 0, (m, 0, 0, 0), c
    return pl, guard, st, r, A, where


def sched_cases(G):
    """(id, tiles, n_kb, property) against a grid of G CTAs."""
    return [
        ("tiles_lt_grid", max(G // 2, 1), 16, "share"),
        ("rem1", G + 1, 8, "rem1"),
        ("rem_G-1", 2 * G - 1, 16, "remG-1"),
        ("straddle", G + 5, 12, "straddle"),
        ("exact_multiple", 2 * G, 8, "exact"),
    ]


def sched_case_check(P, G, case, seed, swap=False):
    name, T, n_kb, prop = case
    pl, guard, st, r, A, where = sched_matrix(P, T, n_kb, seed, swap=swap, stats=True)
    assert pl.grid() == T and pl.n_kb == n_kb
    worst = 0.0
    for sched in (0, 1):
        s = run(pl, G, sched, guard, st)
        if sched == 1:
            if prop == "share":
                assert pl.grid() < G and s["grid"] > pl.grid() and s["q"] == 0, s
            elif prop == "rem1":
                assert s["rem"] == 1, s
            elif prop == "remG-1":
                assert s["rem"] == G - 1, s
            elif prop == "straddle":
                assert s["rem"] > 0 and straddles(s), s
            elif prop == "exact":
                assert s["rem"] == 0 and s["q"] >= 1, s
        check_out("sched", pl, G, guard.y, r, A, where, False, guard, tag=f" {name} sched {sched}")
        check_stats("sched", st, r[None], A[None], 8)
        worst = max(worst, float(((guard.y.double() - r).abs() / bound_of(r, A, False)).max()))
    return worst


@pytest.mark.parametrize("idx", range(5), ids=[c[0] for c in sched_cases(148)])
def test_schedule_tile_counts(P, idx):
    G = sms(P)
    sched_case_check(P, G, sched_cases(G)[idx], seed=idx)


def test_schedule_swap_tiles(P):
    """Stream-K with swap-mode tiles (two boxes per tile), a straddling phase-A range."""
    G = sms(P)
    pl, guard, st, r, A, where = sched_matrix(P, G + 5, 12, 99, swap=True)
    assert pl.pick_swap() and pl.grid() == G + 5
    for sched in (0, 1):
        s = run(pl, G, sched, guard)
        if sched:
            assert straddles(s), s
        check_out("sched", pl, G, guard.y, r, A, where, False, guard, tag=f" swap sched {sched}")


def test_cfg4_top_level(P):
    """The one full-size case: 1 x 128 x 40 x 48 x 40 -> 128, 3^3 (stream-K by default)."""
    G = sms(P)
    acts, w, _, g = conv_inputs(3, (40, 48, 40), 1, [128], 0, 128, 3, 40)
    bias = torch.randn(128, device="cuda", generator=g)
    stats = torch.zeros(1, 8, 2, dtype=torch.float64, device="cuda")
    guard = Guarded((1, 40, 48, 40, 128), torch.bfloat16)
    pl = P.conv_plan([P.ConvSource(acts[0])], P.pack_conv_weight(w), guard.y, 3, bias=bias,
                     stats=stats, stats_cpg=16)
    assert pl.pick_swap() and pl.xreuse == 1 and pl.tile_fast_dim == 2
    assert pl.pick_sched(G) == 1 and pl.grid() % G != 0
    r, A, _ = conv_reference(3, acts, w, None, None, bias, None, None, 3)
    for sched in (0, 1):
        run(pl, G, sched, guard, stats)
        check_out("cfg4", pl, G, guard.y, r, A, conv_where(guard.y.shape), False, guard, tag=f" sched {sched}")
        check_stats("cfg4", stats, r, A, 8)


# ============================================================================ 6. repeat and replay
def test_repeat_and_graph_replay(P):
    G = sms(P)
    pl, guard, st, r, A, where = sched_matrix(P, G + 5, 12, 5, stats=True)
    pl.sched = 1
    pl.materialize("cuda")
    outs, sts = [], []
    for _ in range(3):
        st.zero_()
        pl.launch()
        torch.cuda.synchronize()
        outs.append(guard.y.clone())
        sts.append(st.clone())
    check_out("replay", pl, G, guard.y, r, A, where, False, guard)
    guard.reset()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            st.zero_()
            pl.launch()
    torch.cuda.current_stream().wait_stream(stream)
    for _ in range(3):
        guard.y.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        outs.append(guard.y.clone())
        sts.append(st.clone())
    for o, s_ in zip(outs[1:], sts[1:]):
        assert torch.equal(o.view(torch.int16), outs[0].view(torch.int16))   # fixed fold order
        assert torch.allclose(s_, sts[0], rtol=1e-12, atol=0)
    assert guard.sentinels_ok()
    check_stats("replay", st, r[None], A[None], 8)


def test_two_stream_k_plans_back_to_back(P):
    """The second plan starts on the flags the first left behind (self-resetting)."""
    G = sms(P)
    p1 = sched_matrix(P, G + 5, 12, 11)
    p2 = sched_matrix(P, max(G // 2, 1), 16, 12)
    conv = conv_inputs(3, (8, 12, 10), 2, [128], 0, 128, 3, 13)
    g3 = Guarded((2, 8, 12, 10, 128), torch.bfloat16)
    pl3 = P.conv_plan([P.ConvSource(conv[0][0])], P.pack_conv_weight(conv[1]), g3.y, 3)
    for pl in (p1[0], p2[0], pl3):
        pl.sched = 1
        pl.materialize("cuda")
    for _ in range(2):
        for pl, gd in ((p1[0], p1[1]), (p2[0], p2[1]), (pl3, g3)):
            gd.reset()
        p1[0].launch()
        p2[0].launch()
        pl3.launch()
        p1[0].launch()
        torch.cuda.synchronize()
        for pl, guard, _, r, A, where in (p1, p2):
            check_out("back_to_back", pl, G, guard.y, r, A, where, False, guard)
        r3, A3, _ = conv_reference(3, conv[0], conv[1], None, None, None, None, None, 3)
        check_out("back_to_back", pl3, G, g3.y, r3, A3, conv_where(g3.y.shape), False, g3)


# ============================================================================ 7. narrowed grid
def _child():
    """Runs in a process with MRI_GEMM_SMS set: the stream-K cases at that grid width."""
    from mri_image_generation_b200 import _lib, plan as P
    _lib.require_device()
    G = sms(P)
    out = {"G": G}
    for i, case in enumerate(sched_cases(G)):
        out[case[0]] = sched_case_check(P, G, case, seed=50 + i)
    out["beta"] = WORST.get("beta sched")
    print("CHILD_RESULT " + json.dumps(out))


@pytest.mark.parametrize("n", [8, 37, 147])
def test_narrowed_grid(P, n):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, MRI_GEMM_SMS=str(n))
    env["PYTHONPATH"] = os.pathsep.join([root, os.path.join(root, "tests")] +
                                        ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), "--child"]
    r = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    tail = (r.stdout + r.stderr)[-4000:]
    assert r.returncode == 0, tail
    line = [l for l in r.stdout.splitlines() if l.startswith("CHILD_RESULT ")]
    assert line, tail
    res = json.loads(line[-1][len("CHILD_RESULT "):])
    assert res["G"] == min(n, torch.cuda.get_device_properties(0).multi_processor_count), res
    for k, v in res.items():
        if k not in ("G", "beta"):
            note(f"ratio sched (MRI_GEMM_SMS={n})", v)
            assert v <= 1.0, (k, v)
    if res["beta"] is not None:
        note("beta sched", res["beta"])


# ============================================================================ 8. WgradPlan
def wgrad_check(fam, wg, dw, dw0, gref, mag):
    wg.materialize("cuda")
    wg.launch()
    torch.cuda.synchronize()
    d = dw.double() - dw0.double()
    assert torch.isfinite(d).all()
    err = (d - gref).abs()
    rnd = 2.0 ** -23 * (dw0.double().abs() + gref.abs())
    note(f"beta_w {fam}", ((err - rnd) / mag.clamp_min(1e-300)).max())
    ratio = err / (rnd + BETA_W * mag).clamp_min(1e-300)
    note(f"ratio_w {fam}", ratio.max())
    if float(ratio.max()) > 1:
        i = np.unravel_index(int(ratio.argmax()), ratio.shape)
        raise AssertionError(f"{fam}: dw outside the bound x{float(ratio.max()):.2f} at (class, row, col) "
                             f"{tuple(int(v) for v in i)}, k-table entry {int(i[2]) // 64}")


def packed_grad(P, fn, inputs, w, dy):
    """fp64 weight gradient and its magnitude sum |dy| |a| through autograd."""
    w1 = w.clone().requires_grad_(True)
    (g,) = torch.autograd.grad(fn(inputs, w1), w1, dy)
    w2 = w.abs().clone().requires_grad_(True)
    (m,) = torch.autograd.grad(fn([t.abs() for t in inputs], w2), w2, dy.abs())
    return g, m


@pytest.mark.parametrize("nd,sp,N", [(3, (8, 12, 10), 2), (2, (48, 24), 3), (3, (5, 16, 8), 1)])
@pytest.mark.parametrize("xgroup", ["1", "0"])
@pytest.mark.parametrize("splits", ["1", "2", "pick", "total"])
def test_wgrad_stride1_concat_skip(P, monkeypatch, nd, sp, N, xgroup, splits):
    monkeypatch.setenv("MRI_WGRAD_XGROUP", xgroup)
    g = torch.Generator(device="cuda").manual_seed(N * 10 + nd)
    C1, C2, Co = 64, 128, 128
    a1 = bf(torch.randn(N, *sp, C1, device="cuda", generator=g))
    a2 = bf(torch.randn(N, *sp, C2, device="cuda", generator=g))
    dy = bf(torch.randn(N, *sp, Co, device="cuda", generator=g))
    w = torch.randn(Co, C1 + C2, *([3] * nd), device="cuda", generator=g) * 0.05
    ws = torch.randn(Co, C1, *([1] * nd), device="cuda", generator=g) * 0.1
    wm = P.pack_conv_weight(w, splits=[C1, C2], extra=[ws])
    y = torch.zeros(N, *sp, Co, dtype=torch.bfloat16, device="cuda")
    fwd = P.conv_plan([P.ConvSource(a1), P.ConvSource(a2), P.ConvSource(a1, taps=False)], wm, y, 3)
    total_mt = int(np.prod(fwd.tiles))
    dw0 = torch.randn(1, Co, wm.shape[1], device="cuda", generator=g)
    dw = dw0.clone()
    wg = P.WgradPlan(fwd, dy, dw, Co)
    wg.splits = {"1": 1, "2": 2, "pick": 0, "total": total_mt}[splits]
    runs = wg.runs()
    want_xg = (xgroup == "1" and fwd.xreuse == 1 and fwd.box[0] == 8 and fwd.box[1] == 16
               and int(np.prod(fwd.box)) == 128)
    if (nd, sp) == (2, (48, 24)):
        assert fwd.xreuse == 1 and fwd.box[:2] == (8, 16)      # the case for the xgroup mode
    assert any(xg for _, _, xg in runs) == want_xg, runs
    conv = F.conv3d if nd == 3 else F.conv2d
    x1, x2 = nchw(a1.double()), nchw(a2.double())
    dyn = nchw(dy.double())
    gw, mw = packed_grad(P, lambda ins, ww: conv(torch.cat(ins, 1), ww, padding=1), [x1, x2],
                         bf(w).double(), dyn)
    gs, ms = packed_grad(P, lambda ins, ww: conv(ins[0], ww), [x1], bf(ws).double(), dyn)
    gref = torch.cat([_pack64(gw, [C1, C2]), gs.reshape(Co, C1)], 1)[None]
    mag = torch.cat([_pack64(mw, [C1, C2]), ms.reshape(Co, C1)], 1)[None]
    wgrad_check("wgrad_conv", wg, dw, dw0, gref, mag)


def _pack64(w, splits):
    """pack_conv_weight's column order [source][tap][channel] in fp64 (no rounding)."""
    cout, cin = w.shape[:2]
    wt = w.reshape(cout, cin, -1)
    cols, c0 = [], 0
    for ci in splits:
        cols.append(wt[:, c0:c0 + ci, :].permute(0, 2, 1).reshape(cout, -1))
        c0 += ci
    return torch.cat(cols, 1)


def _packT64(w):
    """pack_convT_weight's layout [class][Cout][combo, Cin] in fp64."""
    cin, cout = w.shape[:2]
    nd = w.dim() - 2
    classes = list(itertools.product((0, 1), repeat=nd))
    out = torch.zeros(len(classes), cout, (2 ** nd) * cin, dtype=w.dtype, device=w.device)
    for ci, rho in enumerate(classes):
        col = 0
        for combo in itertools.product((0, 1), repeat=nd):
            ks = [(1, 3)[combo[i]] if rho[i] == 0 else (0, 2)[combo[i]] for i in range(nd)]
            out[ci, :, col:col + cin] = w[(slice(None), slice(None)) + tuple(reversed(ks))].t()
            col += cin
    return out


@pytest.mark.parametrize("kind,nd,sp,N", [("down", 3, (8, 12, 8), 2), ("down", 2, (32, 48), 2),
                                          ("up", 3, (4, 6, 4), 2), ("up", 2, (16, 24), 2)])
@pytest.mark.parametrize("splits", ["1", "2", "pick", "total"])
def test_wgrad_strided(P, kind, nd, sp, N, splits):
    g = torch.Generator(device="cuda").manual_seed(nd * 7 + N)
    C, Cd = 128, 128
    a = bf(torch.randn(N, *sp, C, device="cuda", generator=g))
    osp = [e // 2 for e in sp] if kind == "down" else [2 * e for e in sp]
    dy = bf(torch.randn(N, *osp, Cd, device="cuda", generator=g))
    y = torch.zeros(N, *osp, Cd, dtype=torch.bfloat16, device="cuda")
    x = nchw(a.double())
    dyn = nchw(dy.double())
    if kind == "down":
        w = bf(torch.randn(Cd, C, *([4] * nd), device="cuda", generator=g) * 0.05)
        fwd = P.down_conv_plan(a, P.pack_conv_weight(w.float()), y)
        conv = F.conv3d if nd == 3 else F.conv2d
        gw, mw = packed_grad(P, lambda ins, ww: conv(ins[0], ww, stride=2, padding=1), [x], w.double(), dyn)
        gref, mag = _pack64(gw, [C])[None], _pack64(mw, [C])[None]
    else:
        w = bf(torch.randn(C, Cd, *([4] * nd), device="cuda", generator=g) * 0.05)
        fwd = P.up_conv_plan(a, P.pack_convT_weight(w.float()), y)
        ct = F.conv_transpose3d if nd == 3 else F.conv_transpose2d
        gw, mw = packed_grad(P, lambda ins, ww: ct(ins[0], ww, stride=2, padding=1), [x], w.double(), dyn)
        gref, mag = _packT64(gw), _packT64(mw)
        # the fp64 packing matches the product's packing
        assert torch.equal(_packT64(w.double()).to(torch.bfloat16), P.pack_convT_weight(w.float()))
    assert fwd.n_class == (1 if kind == "down" else 2 ** nd)
    dw0 = torch.randn(fwd.n_class, Cd, fwd.n_kb * 64, device="cuda", generator=g)
    dw = dw0.clone()
    wg = P.WgradPlan(fwd, dy, dw, Cd)
    wg.splits = {"1": 1, "2": 2, "pick": 0, "total": int(np.prod(fwd.tiles))}[splits]
    wgrad_check(f"wgrad_{kind}", wg, dw, dw0, gref, mag)


@pytest.mark.parametrize("splits", ["pick", "1"])
def test_wgrad_attention_product(P, splits):
    """dW[cls][i][c] = sum_m lhs[cls][m][i] rhs[b][m][h d + c] (backward.py's explicit dy_views)."""
    g = torch.Generator(device="cuda").manual_seed(3)
    B, heads, n, d = 2, 2, 300, 128
    npad = (n + 7) // 8 * 8
    C = heads * d
    rhs_ld = 3 * C
    rhs = bf(torch.randn(B, n, rhs_ld, device="cuda", generator=g))
    rhs_off = C
    lhs = bf(torch.randn(B * heads, n, npad, device="cuda", generator=g))
    n_tiles = -(-n // 128)
    mpad = -(-n // 128) * 128
    ncls = B * heads
    a_maps, dy_views, kts = [], [], []
    for b in range(B):
        for h in range(heads):
            cls = b * heads + h
            av = P.TView(rhs, (d, n, 1, 1, 1), (1, rhs_ld, n * rhs_ld, n * rhs_ld, n * rhs_ld),
                         offset=b * n * rhs_ld + rhs_off + h * d)
            a_maps.append(P.MapSpec(av, (P.BLOCK_K, 128, 1, 1, 1), 3))
            dy_views.append(P.TView(lhs, (npad, n, 1, 1, 1), (1, npad, n * npad, n * npad, n * npad),
                                    offset=cls * n * npad))
            kts.append([[cls, c0, 0, 0, 0, 0, c0, 0] for c0 in range(0, d, P.BLOCK_K)])
    fake = P.GemmPlan(a_maps=a_maps, b_map=None, o_maps=[], ktable=np.asarray(kts, dtype=np.int32),
                      tiles=(n_tiles, 1, 1, 1), box=(128, 1, 1, 1), ext=(n, 1, 1, 1),
                      block_n=128, n_total=d)
    dw0 = torch.randn(ncls, mpad, d, device="cuda", generator=g)
    dw = dw0.clone()
    wg = P.WgradPlan(fake, lhs, dw, n, dy_views=dy_views)
    wg.splits = 1 if splits == "1" else 0
    L = lhs.double()[..., :n]                                              # [cls, m, i]
    R = rhs.double()[..., rhs_off:rhs_off + C].reshape(B, n, heads, d).permute(0, 2, 1, 3).reshape(ncls, n, d)
    gref = torch.zeros(ncls, mpad, d, dtype=torch.float64, device="cuda")
    mag = torch.zeros_like(gref)
    gref[:, :n] = torch.einsum("kmi,kmc->kic", L, R)
    mag[:, :n] = torch.einsum("kmi,kmc->kic", L.abs(), R.abs())
    wgrad_check("wgrad_attn", wg, dw, dw0, gref, mag)


# ============================================================================ 9. thin_in_conv
@pytest.mark.parametrize("sp,cin,cout", [((8, 12, 8), 3, 128), ((5, 7, 9), 3, 64), ((40, 48, 40), 3, 128),
                                         ((37, 50), 1, 64), ((128, 128), 1, 64), ((16, 24), 4, 128),
                                         ((240, 240), 1, 64)])
def test_thin_in_conv(P, sp, cin, cout):
    from mri_image_generation_b200 import ops
    nd = len(sp)
    B = 2
    g = torch.Generator(device="cuda").manual_seed(sum(sp) + cin + cout)
    x = torch.randn(B, cin, *sp, device="cuda", generator=g)
    w = torch.randn(cout, cin, *([3] * nd), device="cuda", generator=g) * 0.2
    bias = torch.randn(cout, device="cuda", generator=g)
    wp = torch.zeros(cout, 4, *([3] * nd), device="cuda")
    wp[:, :cin] = w
    packed = P.pack_conv_weight(wp)
    w128 = torch.zeros(cout, 128, dtype=torch.bfloat16, device="cuda")
    w128[:, :packed.shape[1]] = packed
    S = int(np.prod(sp))
    guard = Guarded((B, S, cout), torch.bfloat16)
    stats = torch.zeros(B, 8, 2, dtype=torch.float64, device="cuda")
    sp3 = (1,) * (3 - nd) + tuple(sp)
    ops.thin_in_conv(x, w128, bias, guard.y, stats, B, cin, sp3[0], sp3[1], sp3[2], nd, cout)
    torch.cuda.synchronize()
    conv = F.conv3d if nd == 3 else F.conv2d
    x64, w64 = bf(x).double(), bf(w).double()
    r = f64conv(conv, x64, w64, padding=1) + bias.double().reshape(1, -1, *([1] * nd))
    A = f64conv(conv, x64.abs(), w64.abs(), padding=1) + bias.double().abs().reshape(1, -1, *([1] * nd))
    r = r.reshape(B, cout, S).transpose(1, 2)
    A = A.reshape(B, cout, S).transpose(1, 2)
    y = guard.y
    assert torch.isfinite(y.double()).all() and guard.sentinels_ok()
    err = (y.double() - r).abs()
    note("beta thin_in_conv", ((err - 2.0 ** -8 * r.abs()) / A).max())
    ratio = err / bound_of(r, A, False)
    note("ratio thin_in_conv", ratio.max())
    if float(ratio.max()) > 1:
        b_, s_, c_ = np.unravel_index(int(ratio.argmax()), ratio.shape)
        raise AssertionError(f"thin_in_conv: x{float(ratio.max()):.2f} at sample {b_}, position {s_} "
                             f"(128-position tile {s_ // 128}), channel {c_}")
    check_stats("thin_in_conv", stats, r, A, 8)


if __name__ == "__main__" and sys.argv[1:] == ["--child"]:
    _child()
