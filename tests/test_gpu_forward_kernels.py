"""The forward kernels that are not GEMMs, one at a time, each against a float64 torch reference
of the same operation computed on the same bf16 / fp32 operands the kernel reads: the fused
attention kernel (csrc/attn_flash.cu), GroupNorm statistics and apply (csrc/norm_act.cu), the row
softmax, the small linears and the layout kernels (csrc/embed_layout.cu) and the split-precision
glue (csrc/split_precision.cu).

The model tests compare whole tensors (rel-L2), which hides a wrong value confined to one
128-query tile, to one sample segment of a gn_apply block that straddles samples, or to one
32-column group of the attention output.  Here every element is held to its own bound.  Every
output starts as NaN inside a buffer whose head and tail hold a sentinel (a missed store or a store
outside the tensor fails); padding columns the kernel must not read are NaN (or, where the
contract needs them finite, as v^T's are for attention, large finite values); padding columns the
kernel must zero are checked to be exactly 0 and those it must leave alone to keep their sentinel.
Inputs have distinct statistics per sample, per group and per head, so a read from a neighbour is
far outside the bound.

Error model.  r is the fp64 result and A the element's sum of absolute terms.  A bf16 output obeys
|y - r| <= 2^-8 |r| + BETA A (2^-8 |r| covers round-to-nearest of the stored value), an fp32 output
2^-24 in place of 2^-8, and a split (hi, lo) output holds hi + lo to 2^-16.  Each BETA is 4x the
worst max((|y - r| - 2^-8 |r|) / A) (resp. 2^-24, 2^-16) measured on one B200 at its 1000 W power
limit, over every case of this file; where that worst value is negative (the softmaxes) BETA is 0
and the rounding term alone bounds every element.  The WORST table (printed at the end of the
module with -s) lists the measured values; the constants below record them.  Error sources:

* attn_flash: P = ex2.approx((s - m_ref) c) is rounded to bf16 before the second MMA and the row
  sum l is taken over the rounded values, so each p_k carries a relative error <= 2^-9 (plus
  ex2.approx's 2^-22), which moves y by <= 2^-9 sum_k p_k |v_k - r| / sum_k p_k <= 2^-8 sum p |v|
  / sum p.  The logits are fp32 sums of d products (tcgen05 accumulation), error <= d 2^-24
  L_k with L_k = scale sum_i |q_i| |k_ki|, which moves y by sum_k p_k L_k |v_k - r| d 2^-24.
  A = sum_k p_k |v_k| / sum p + 2^-16 d sum_k p_k L_k |v_k - r| / sum p, so that with BETA near
  2^-8 the second term stands for the logit bound.  Measured: see ATTN_BETA.
* gn_apply: scale / shift are fp32 products of fp64 statistics (rsqrtf: 2 ulp), one fp32 FMA per
  element, SiLU through 0.5 tanh.approx(u / 2) + 0.5 (relative error 2^-11 of tanh, so
  <= 2^-12 |u| on silu), then fp32 adds of the row bias and the residual.
  A = |gamma x rstd| + |gamma mean rstd| + |beta| + |rowbias| + |residual| (the shift cancels
  against x * scale when |mean| >> std, and its rounding does not).
* gn_stats: fp32 per-thread partials of a few hundred terms, folded in fp64:
  |sum - r| <= BETA_S sum |x| and |sumsq - r| <= BETA_S sum x^2 per (sample, fine group).
* softmax_rows: __expf (ex2.approx of x log2 e: relative 2^-22 plus 2^-24 |x| from the product),
  fp32 row sum, reciprocal; A = r (1 + |x|) with x = scale s - max, plus an absolute floor of
  2^-126 where ex2.approx.ftz flushes to 0.
* linear: the fp32 summation bound (ceil(in_f / 32) + 6) 2^-24 (sum |x W| + |bias|) of the
  per-lane FMA chains and the 5-step shuffle tree (x 1.1 through SiLU), plus 8 ulp of the SiLU
  (expf, IEEE division) and one rounding for the addend: a deterministic bound, not measured.
* im2col4, tap_gather, nchw_to_nhwc, nhwc_to_nchw, split3, bf16_residual_nchw: bit-exact
  (tap_gather against an fp32 sum in the kernel's own order: bias, then the taps kd, kh, kw).
* gn_split: v in fp32 as gn_apply without the approximations (expf, IEEE division): hi = bf16(v),
  lo = bf16(v - hi) exactly, segment 3 = segment 1, |hi + lo - r| <= 2^-16 |r| + BETA A.
* stats_f32: fp64 sums of fp32 values, |err| <= BETA_S sum |x| (resp. sum x^2), BETA_S of the
  order of 2^-53 times the terms per thread.
* softmax_rows_split: expf (IEEE-accurate to a few ulp) and an fp32 row sum, far below the 2^-16
  of the (hi, lo) pair; A and the 2^-126 floor as for softmax_rows.
"""
import json
import math
import os
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
from test_gpu_backward_kernels import GN_CONFIGS, gn_stats_ref   # noqa: E402

EPS = 1e-5
U8, U16, U24 = 2.0 ** -8, 2.0 ** -16, 2.0 ** -24

# BETA per family: 4x the worst value measured on one B200 at its 1000 W power limit (module
# docstring; DESIGN.md section 4).  0 where the worst measured value is negative: the rounding
# term alone bounds every element.
ATTN_BETA = 1.08e-2                  # worst 2.70e-3
GN_BETA = {False: 3.1e-7,            # worst 7.85e-8
           True: 1.32e-5}            # worst 3.29e-6 (tanh.approx)
GN_BETA_S = 1.1e-5                   # worst 2.74e-6 (batch 16 at the cfg4 top level)
SM_BETA = 0.0                        # worst -6.0e-7
SPLIT_BETA = 3.5e-7                  # worst 8.72e-8
SPLIT32_BETA = 7.7e-7                # worst 1.92e-7
SMS_BETA = 0.0                       # worst -1.2e-7
SF32_BETA = 7.8e-15                  # worst 1.94e-15

WORST = {}   # family -> worst measured value (printed at the end of the module, run with -s)


def note(key, value):
    WORST[key] = max(WORST.get(key, -math.inf), float(value))


@pytest.fixture(scope="module", autouse=True)
def _print_worst():
    yield
    if WORST:
        print("\n[forward kernels] worst measured values")
        for k in sorted(WORST):
            print(f"  {k:48s} {WORST[k]: .3e}")


@pytest.fixture(scope="module")
def ops():
    from mri_image_generation_b200 import _lib, ops
    _lib.require_device()
    return ops


def bf16(t):
    return t.to(torch.bfloat16)


# ------------------------------------------------------------------------------ guarded outputs
_PAD = 256
_SENT = {torch.bfloat16: (torch.int16, 0x5A5A), torch.float32: (torch.int32, 0x5A5A5A5A),
         torch.float64: (torch.int64, 0x5A5A5A5A5A5A5A5A)}
_INT = {torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.float64: torch.int64}


class Guarded:
    """A contiguous tensor inside a larger buffer whose head and tail hold a sentinel pattern;
    the tensor itself starts as NaN (fill=None: as the sentinel)."""

    def __init__(self, shape, dtype, fill=float("nan"), tail=_PAD, device="cuda"):
        self.n = math.prod(shape)
        self.dtype, self.tail = dtype, tail
        self.buf = torch.empty(self.n + _PAD + tail, dtype=dtype, device=device)
        it, pat = _SENT[dtype]
        self.buf.view(it).fill_(pat)
        self.y = self.buf[_PAD:_PAD + self.n].view(shape)
        if fill is not None:
            self.y.fill_(fill)

    def bits(self):
        return self.y.view(_INT[self.dtype])

    def guards_ok(self):
        it, pat = _SENT[self.dtype]
        b = self.buf.view(it)
        return bool((b[:_PAD] == pat).all() and (b[_PAD + self.n:] == pat).all())


def same_bits(a, b):
    return torch.equal(a.contiguous().view(_INT[a.dtype]), b.contiguous().view(_INT[b.dtype]))


# ============================================================================ 1. attn_flash_kernel
ATTN_NS = [1, 7, 8, 100, 127, 128, 129, 255, 256, 257, 1200]
ATTN_HEADS = [1, 2, 4, 8]
ATTN_REGIMES = ["randn", "grow", "mixed", "onehot", "qzero"]


def _attn_cases():
    """(d, n, heads, batch): both head widths at every n, the head counts and batches rotating,
    then the test-size 3D UNet's bottleneck (n 8, d 64, 4 heads) and the cfg4 bench bottleneck
    (40x48x40 latent after two down-samplings: n 1200, d 128, 4 heads) at batch 1 and 3."""
    cases = []
    for di, d in enumerate((64, 128)):
        for i, n in enumerate(ATTN_NS):
            cases.append((d, n, ATTN_HEADS[(i + 2 * di) % 4], (1, 3)[(i + di) % 2]))
    cases += [(64, 8, 4, 2), (128, 1200, 4, 1), (128, 1200, 4, 3)]
    return cases


ATTN_CASES = _attn_cases()


def attn_inputs(B, n, heads, d, regime, seed):
    """fp64 q, k, v [B, n, heads * d] of one logit regime, with distinct (scale, offset) per
    (sample, head); returned bf16-rounded.
      randn   no rescale after tile 0 (|logits| ~ 3);
      grow    keys grow along the sequence: the row maximum rises by > 8 / log2(e) per key tile;
      mixed   as grow, but odd queries are scaled down 50x, so inside every warp rows that grow
              sit next to rows that do not (the warp takes the TMEM rescale path; they use a = 1);
      onehot  scale s in [100, 400] on the last valid key (in the ragged last tile), every other
              logit of the row at least ~20 below it: near one-hot rows;
      qzero   every third query is 0 (uniform attention: the mean of v over the n keys)."""
    g = torch.Generator().manual_seed(seed)
    f64 = dict(generator=g, dtype=torch.float64)
    shp = (B, n, heads, d)
    qs = 1 + torch.rand(B, 1, heads, 1, **f64)
    q = torch.randn(*shp, **f64) * qs
    k = torch.randn(*shp, **f64)
    mu = -2 + 4 * torch.rand(B, 1, heads, 1, **f64)
    sd = torch.exp(math.log(0.25) + math.log(16) * torch.rand(B, 1, heads, 1, **f64))
    v = mu + sd * torch.randn(*shp, **f64)
    scale = d ** -0.5
    if regime in ("grow", "mixed"):
        # scale * max_k q.k ~ 2.5 qs ramp over a tile: + >= 10 per tile of 128 keys
        ramp = 1 + 4 * torch.arange(n, dtype=torch.float64) / 128
        k = k * ramp.view(1, n, 1, 1)
        if regime == "mixed":
            q[:, 1::2] *= 0.02
    elif regime == "onehot":
        u = torch.randn(B, 1, heads, d, **f64)
        u = u / u.norm(dim=-1, keepdim=True)
        a = 16.0
        b = (100 + 300 * torch.rand(B, n, heads, 1, **f64)) / (scale * a)
        q = b * u + torch.randn(*shp, **f64)
        k[:, n - 1:n] = a * u
    elif regime == "qzero":
        q[:, ::3] = 0
    return (bf16(t.reshape(B, n, heads * d)) for t in (q, k, v))


def attn_reference(q, k, v, heads, d):
    """fp64 softmax(q k^T scale) v on the bf16 operands, and A (module docstring): [B, n, C]."""
    B, n, C = q.shape
    qd, kd, vd = (t.double().view(B, n, heads, d).transpose(1, 2) for t in (q, k, v))
    scale = float(torch.tensor(d ** -0.5, dtype=torch.float32))
    s = (qd @ kd.transpose(-1, -2)) * scale
    p = torch.softmax(s, -1)                                   # [B, h, n, n]
    r = p @ vd
    L = (qd.abs() @ kd.abs().transpose(-1, -2)) * scale       # sum_i |q_i| |k_ki| scale
    A = p @ vd.abs()
    # sum_k p_k L_k |v_k - r|: expand |v_k - r| <= |v_k| + |r| to keep it one matmul per term
    pl = p * L
    A = A + 2.0 ** -16 * d * (pl @ vd.abs() + pl.sum(-1, keepdim=True) * r.abs())
    back = lambda t: t.transpose(1, 2).reshape(B, n, C)
    return back(r), back(A)


def attn_launch(q, k, v, heads, d, ld_out=None, vpad=3.0e4):
    """Lay q, k, v out as the engine does (qkv token-major [B, n, 3C], v^T [B, C, npad] with
    columns [n, npad) = vpad: finite, as the kernel's contract needs), run mri_attn_flash_launch
    into a guarded output of row pitch ld_out, return (Guarded, launch, args)."""
    import ctypes as C_
    from mri_image_generation_b200 import _lib, plan as PL
    B, n, C = q.shape
    ld_out = ld_out or C
    npad = (n + 7) // 8 * 8
    qkv = torch.cat([q, k, v], -1).cuda().contiguous()
    vT = torch.full((B, C, npad), vpad, dtype=torch.bfloat16, device="cuda")
    vT[:, :, :n] = v.cuda().transpose(1, 2)
    # rows q0 + row >= n of the last sample would land in the tail: 128 rows of it
    out = Guarded((B, n, ld_out), torch.bfloat16, fill=None, tail=128 * ld_out + _PAD)
    out.y[..., :C] = float("nan")
    maps = PL.encode_maps([
        PL.MapSpec(PL.TView(qkv, (3 * C, n, B), (1, 3 * C, n * 3 * C)), (64, 128, 1), 3),
        PL.MapSpec(PL.TView(vT, (npad, C, B), (1, npad, C * npad)), (64, d, 1), 3)], "cuda")
    a = _lib.MriAttnArgs()
    a.qk_map, a.vt_map, a.out = maps.data_ptr(), maps.data_ptr() + 128, out.y.data_ptr()
    a.batch, a.heads, a.n, a.d, a.C = B, heads, n, d, C
    a.k_col0, a.v_row0, a.ld_out = C, 0, ld_out
    a.scale = float(d) ** -0.5
    lib = _lib.load()
    keep = (qkv, vT, maps)

    def launch():
        _lib.check(lib.mri_attn_flash_launch(C_.byref(a), _lib.current_stream_ptr()), "attn_flash")

    launch.keep = keep
    return out, launch, a


def attn_check(out, q, k, v, heads, d, what):
    B, n, C = q.shape
    torch.cuda.synchronize()
    assert out.guards_ok(), f"{what}: a store outside the output (rows >= n or past the buffer)"
    y = out.y[..., :C]
    if out.y.shape[-1] > C:
        assert (out.y[..., C:].view(torch.int16) == _SENT[torch.bfloat16][1]).all(), \
            f"{what}: columns [C, ld_out) were written"
    r, A = attn_reference(q.cuda(), k.cuda(), v.cuda(), heads, d)
    yd = y.double()
    assert torch.isfinite(yd).all(), f"{what}: {int((~torch.isfinite(yd)).sum())} non-finite outputs"
    err = (yd - r).abs()
    note("attn beta", ((err - U8 * r.abs()) / A).max())
    ratio = err / (U8 * r.abs() + ATTN_BETA * A)
    if float(ratio.max()) > 1:
        b, i, c = (int(t) for t in torch.unravel_index(ratio.argmax(), ratio.shape))
        raise AssertionError(
            f"{what}: x{float(ratio.max()):.2f} over the bound at sample {b}, query {i} (tile {i // 128}, "
            f"warp {(i % 128) // 32}), head {c // d}, column {c % d} (32-column group {(c % d) // 32}): "
            f"y {float(yd[b, i, c]):.6g}, r {float(r[b, i, c]):.6g}")
    return r


@pytest.mark.parametrize("d,n,heads,B", ATTN_CASES)
@pytest.mark.gpu
def test_attn_flash(ops, d, n, heads, B):
    for ri, regime in enumerate(ATTN_REGIMES):
        q, k, v = attn_inputs(B, n, heads, d, regime, seed=n * 131 + d * 7 + heads + ri)
        out, launch, _ = attn_launch(q, k, v, heads, d)
        launch()
        r = attn_check(out, q, k, v, heads, d, f"{regime} d={d} n={n} heads={heads} B={B}")
        if regime == "qzero":        # zero rows: the mean of v over exactly the n keys
            mean = v.cuda().double().mean(1)
            assert torch.allclose(r[:, ::3], mean[:, None].expand_as(r[:, ::3]), rtol=1e-12, atol=1e-12)
        if regime == "onehot":       # the maximum sits on the last valid key, in the last key tile
            qd, kd = q.double().view(B, n, heads, d), k.double().view(B, n, heads, d)
            s = torch.einsum("bqhd,bkhd->bhqk", qd, kd) * d ** -0.5
            assert (s.argmax(-1) == n - 1).all() and s.amax(-1).min() > 90


@pytest.mark.gpu
def test_attn_flash_wide_output_rows(ops):
    """ld_out > C: columns [C, ld_out) keep their sentinel, rows >= n of the last query tile are
    not written (the tail of the buffer keeps its sentinel), for both head widths."""
    for d, heads, n in ((64, 2, 129), (128, 3, 100)):
        q, k, v = attn_inputs(3, n, heads, d, "mixed", seed=d + n)
        out, launch, _ = attn_launch(q, k, v, heads, d, ld_out=heads * d + 24)
        launch()
        attn_check(out, q, k, v, heads, d, f"ld_out > C, d={d}")


@pytest.mark.gpu
def test_attn_flash_deterministic_and_graph_replay(ops):
    """Two launches give the same bits, and a CUDA-graph replay (the engine replays this kernel
    inside its graphs) gives the eager launch's bits: cfg4's bottleneck, keys growing."""
    B, n, heads, d = 2, 1200, 4, 128
    q, k, v = attn_inputs(B, n, heads, d, "mixed", seed=5)
    out, launch, _ = attn_launch(q, k, v, heads, d)
    launch()
    attn_check(out, q, k, v, heads, d, "cfg4 eager")
    first = out.y.clone()
    out.y.fill_(float("nan"))
    launch()
    torch.cuda.synchronize()
    assert same_bits(out.y, first), "two launches differ"
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    out.y.fill_(float("nan"))
    g.replay()
    torch.cuda.synchronize()
    assert same_bits(out.y, first), "graph replay differs from the eager launch"
    assert out.guards_ok()


@pytest.mark.parametrize("B,n,heads,d", [(2, 37, 2, 64), (1, 300, 4, 128)])
def test_attn_reference_on_cpu(B, n, heads, d):
    """The fp64 reference equals torch's attention, every regime builds what it claims, and a key
    mask one key too wide (key n reads v^T padding) is far outside the bound (CPU only)."""
    import torch.nn.functional as F
    for regime in ATTN_REGIMES:
        q, k, v = attn_inputs(B, n, heads, d, regime, seed=n + d)
        r, A = attn_reference(q, k, v, heads, d)
        qd, kd, vd = (t.double().view(B, n, heads, d).transpose(1, 2) for t in (q, k, v))
        want = F.scaled_dot_product_attention(qd, kd, vd, scale=float(torch.tensor(d ** -0.5)))
        assert torch.allclose(r, want.transpose(1, 2).reshape(B, n, -1), rtol=1e-10, atol=1e-10)
        assert (A >= r.abs() * (1 - 1e-12)).all()
        # the off-by-one mask: an extra key with logit 0 and value 3e4
        k1 = torch.cat([kd, torch.zeros_like(kd[:, :, :1])], 2)
        v1 = torch.cat([vd, torch.full_like(vd[:, :, :1], 3.0e4)], 2)
        bad = F.scaled_dot_product_attention(qd, k1, v1, scale=float(torch.tensor(d ** -0.5)))
        bad = bad.transpose(1, 2).reshape(B, n, -1)
        ratio = (bad - r).abs() / (U8 * r.abs() + ATTN_BETA * A)
        if regime in ("randn", "mixed", "qzero"):   # elsewhere the extra key's weight is < e^-30
            assert ratio.max() > 10, regime
    q, k, v = attn_inputs(B, n, heads, d, "grow", seed=1)
    s = torch.einsum("bqc,bkc->bqk", q.double()[..., :d], k.double()[..., :d]) * d ** -0.5
    if n > 128:
        assert (s[..., 128:256].amax(-1) - s[..., :128].amax(-1)).median() > 8 / math.log2(math.e)


# ============================================================================ 2. gn_stats + gn_apply
def gn_rows_step(C):
    vpr = C // 8
    return (256 // vpr) * vpr // vpr


def gn_partition(samples, spatial, C, bps):
    """mri_gn_apply's launch restated: blocks = 148 * bps, rows_per rounded up to 4 * rows_step,
    then as many blocks as that takes.  Returns (blocks, rows_per)."""
    total = samples * spatial
    quantum = 4 * gn_rows_step(C)
    blocks = 148 * bps
    rows_per = -(-total // blocks)
    rows_per = -(-rows_per // quantum) * quantum
    return -(-total // rows_per), rows_per


def gn_block_samples(samples, spatial, C, bps):
    """Per block: (first flat row, samples touched, starts mid-sample)."""
    blocks, rows_per = gn_partition(samples, spatial, C, bps)
    out = []
    for b in range(blocks):
        g0 = b * rows_per
        g1 = min(g0 + rows_per, samples * spatial)
        out.append((g0, (g1 - 1) // spatial - g0 // spatial + 1, g0 % spatial != 0))
    return out


def default_bps(residual):
    """The occupancy mri_gn_apply finds (4 blocks per SM, 3 with a residual stream), unless
    MRI_GN_BLOCKS_PER_SM overrides it."""
    env = int(os.environ.get("MRI_GN_BLOCKS_PER_SM", "0") or 0)
    return env if env > 0 else (3 if residual else 4)


def _gn_cases():
    """(C, groups, stats_cpg, N, S): every configuration at 3 samples of a row count that is not a
    multiple of 4 * rows_step, at one row, and at many small samples (a block spans several and
    starts mid-sample); then 300 samples x 5 rows, the cfg4 top level (1 x 40*48*40 x 128) and
    batch 16 at that level."""
    cases = []
    for (C, G, s) in GN_CONFIGS:
        rs = gn_rows_step(C)
        cases.append((C, G, s, 3, 7 * rs * 4 + 2 * rs + 1))
        cases.append((C, G, s, 1, 1))
        cases.append((C, G, s, 40, 3 * rs + 1))
    cases += [(128, 8, 16, 300, 5), (32, 8, 4, 300, 3), (64, 8, 8, 150, 7),
              (128, 8, 16, 1, 40 * 48 * 40), (128, 8, 16, 16, 40 * 48 * 40)]
    return cases


GN_CASES = _gn_cases()
GN_CHILD_CASES = [(128, 8, 16, 300, 5), (32, 8, 4, 300, 3), (64, 16, 4, 40, 13), (192, 8, 24, 7, 333),
                  (512, 64, 8, 40, 5), (2048, 8, 256, 5, 77)]


def gn_x(N, S, C, G, seed):
    """bf16 x [N, S, C] with a distinct (mean, std) per (sample, group)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    cpg = C // G
    mu = -2 + 4 * torch.rand(N, 1, G, 1, generator=g, device="cuda")
    sd = torch.exp(math.log(0.25) + math.log(16) * torch.rand(N, 1, G, 1, generator=g, device="cuda"))
    return bf16((mu + sd * torch.randn(N, S, G, cpg, generator=g, device="cuda")).reshape(N, S, C))


def gn_apply_reference(x, G, gamma, beta, silu, rb, res):
    """fp64 act(GroupNorm(x)) + rowbias + residual and its A (module docstring)."""
    N, S, C = x.shape
    xd = x.double().view(N, S, G, C // G)
    mean = xd.mean((1, 3), keepdim=True)
    rstd = (xd.var((1, 3), unbiased=False, keepdim=True) + EPS).rsqrt()
    gm, bt = gamma.double().view(1, 1, G, -1), beta.double().view(1, 1, G, -1)
    u = ((xd - mean) * rstd * gm + bt).view(N, S, C)
    A = ((xd * rstd * gm).abs() + (mean * rstd * gm).abs() + bt.abs()).view(N, S, C)
    r = u * torch.sigmoid(u) if silu else u
    if rb is not None:
        r = r + rb[:, None]
        A = A + rb.abs()[:, None]
    if res is not None:
        r = r + res.double()
        A = A + res.double().abs()
    return r, A


def gn_case_check(ops, C, G, scpg, N, S, seed):
    """gn_stats against fp64 sums, then every <silu, residual> instantiation of gn_apply, with
    and without row bias (pitch C + 24, NaN past C), fed exact fp64 statistics."""
    x = gn_x(N, S, C, G, seed)
    gref = torch.Generator(device="cuda").manual_seed(seed + 1)
    gamma = 1 + 0.5 * torch.randn(C, generator=gref, device="cuda")
    beta = 0.5 * torch.randn(C, generator=gref, device="cuda")
    stats = gn_stats_ref(x, scpg).contiguous()

    # gn_stats accumulates into its output: start from known values inside a guarded buffer
    st = Guarded(tuple(stats.shape), torch.float64, fill=None)
    st0 = torch.randn(stats.shape, generator=gref, device="cuda", dtype=torch.float64)
    st.y.copy_(st0)
    ops.gn_stats(x, st.y, N, S, C, scpg)
    torch.cuda.synchronize()
    assert st.guards_ok(), "gn_stats wrote outside its [N, C / stats_cpg, 2] output"
    xr = x.double().view(N, S, C // scpg, scpg)
    mag = torch.stack([xr.abs().sum((1, 3)), (xr * xr).sum((1, 3))], -1)
    e = ((st.y - st0) - stats).abs() / mag.clamp_min(1e-300)
    note("gn_stats beta_s", e.max())
    if float(e.max()) > GN_BETA_S:
        n, f, w = (int(t) for t in torch.unravel_index(e.argmax(), e.shape))
        raise AssertionError(f"gn_stats: (sample {n}, fine group {f}) {('sum', 'sumsq')[w]} "
                             f"|err| / bound {float(e.max()) / GN_BETA_S:.2f}")

    rbld = C + 24
    rb_full = torch.full((N, rbld), float("nan"), device="cuda")
    rb_full[:, :C] = 3 * torch.randn(N, 1, generator=gref, device="cuda") + torch.randn(N, C, generator=gref, device="cuda")
    res = bf16(2 * torch.randn(N, 1, 1, generator=gref, device="cuda") +
               torch.randn(N, S, C, generator=gref, device="cuda"))
    for silu in (False, True):
        for with_res in (False, True):
            for with_rb in (False, True):
                rb = rb_full if with_rb else None
                y = Guarded((N, S, C), torch.bfloat16)
                ops.gn_apply(x, y.y, stats, gamma, beta, N, S, C, G, scpg, EPS, silu,
                             rowbias=rb, rowbias_ld=rbld if with_rb else 0,
                             residual=res if with_res else None)
                torch.cuda.synchronize()
                what = f"gn_apply C={C} G={G} scpg={scpg} N={N} S={S} silu={silu} residual={with_res} rowbias={with_rb}"
                assert y.guards_ok(), f"{what}: store outside the output"
                r, A = gn_apply_reference(x, G, gamma, beta, silu, rb_full[:, :C].double() if with_rb else None,
                                          res if with_res else None)
                yd = y.y.double()
                assert torch.isfinite(yd).all(), f"{what}: {int((~torch.isfinite(yd)).sum())} non-finite"
                err = (yd - r).abs()
                note(f"gn_apply beta (silu={silu})", ((err - U8 * r.abs()) / A).max())
                ratio = (err / (U8 * r.abs() + GN_BETA[silu] * A)).view(N, S, G, C // G)
                blk = ratio.amax((1, 3))                       # per (sample, group)
                if float(blk.max()) > 1:
                    n, gi = divmod(int(blk.argmax()), G)
                    s = int(ratio[n, :, gi].amax(-1).argmax())
                    bps = default_bps(with_res)
                    _, rows_per = gn_partition(N, S, C, bps)
                    bad = int((blk > 1).sum())
                    raise AssertionError(
                        f"{what}: {bad} (sample, group) blocks over the bound; worst sample {n}, group {gi} "
                        f"x{float(blk.max()):.2f}, row {s} owned by block {(n * S + s) // rows_per} "
                        f"(rows_per {rows_per} at {bps} blocks per SM)")


@pytest.mark.parametrize("C,G,scpg,N,S", GN_CASES)
@pytest.mark.gpu
def test_gn_stats_and_apply(ops, C, G, scpg, N, S):
    gn_case_check(ops, C, G, scpg, N, S, seed=C * 7 + G + N * 31 + S)


@pytest.mark.parametrize("bps", [1, 3])
@pytest.mark.gpu
def test_gn_apply_other_partitions(ops, bps):
    """MRI_GN_BLOCKS_PER_SM (read once per process) moves every block boundary: the
    partition-sensitive cases again in a child process at 1 and at 3 blocks per SM."""
    root = os.path.dirname(HERE)
    env = dict(os.environ, MRI_GN_BLOCKS_PER_SM=str(bps))
    env["PYTHONPATH"] = os.pathsep.join([root, HERE] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), "--child"]
    r = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    tail = (r.stdout + r.stderr)[-4000:]
    assert r.returncode == 0, tail
    line = [l for l in r.stdout.splitlines() if l.startswith("CHILD_RESULT ")]
    assert line, tail
    res = json.loads(line[-1][len("CHILD_RESULT "):])
    for k, v in res.items():
        note(f"{k} (MRI_GN_BLOCKS_PER_SM={bps})", v)


def _child():
    from mri_image_generation_b200 import _lib, ops as ops_
    _lib.require_device()
    for i, (C, G, s, N, S) in enumerate(GN_CHILD_CASES):
        gn_case_check(ops_, C, G, s, N, S, seed=900 + i)
    print("CHILD_RESULT " + json.dumps({k: v for k, v in WORST.items() if k.startswith("gn_apply")}))


def test_gn_partition_restated_on_cpu():
    """The Python restatement covers every row once, and the parametrization holds blocks that
    start mid-sample and blocks that span >= 3 samples at every blocks-per-SM count used."""
    for bps in (1, 3, 4):
        spans3 = mid = False
        for cases in (GN_CASES, GN_CHILD_CASES):
            for (C, G, s, N, S) in cases:
                blocks, rows_per = gn_partition(N, S, C, bps)
                assert rows_per % (4 * gn_rows_step(C)) == 0 and blocks <= 148 * bps
                assert (blocks - 1) * rows_per < N * S <= blocks * rows_per
                for (_, ns, m) in gn_block_samples(N, S, C, bps):
                    spans3 |= ns >= 3
                    mid |= m
        assert spans3 and mid, bps
    blocks, rows_per = gn_partition(300, 5, 128, 4)
    assert (blocks, rows_per) == (24, 64)          # 12.8 samples per block
    assert gn_partition(1, 40 * 48 * 40, 128, 4) == (400, 192)
    # gn_stats_ref (the sums gn_apply is fed) against a plain loop
    x = bf16(torch.randn(2, 5, 16, generator=torch.Generator().manual_seed(0)))
    st = gn_stats_ref(x, 4)
    assert torch.allclose(st[1, 2, 1], (x[1, :, 8:12].double() ** 2).sum(), rtol=1e-12)


# ============================================================================ 3a. softmax_rows
SM_LDP = [256, 257, 512, 513, 1280, 1281, 2048]      # every template boundary of mri_softmax_rows


def sm_class(ld_p):
    """The softmax_rows_kernel instantiation (values per lane) mri_softmax_rows picks for ld_p."""
    per_lane = (ld_p + 31) // 32
    return next(k for k in (8, 16, 40, 64) if per_lane <= k)


def softmax_case(rows, cols, ld_s, seed):
    """fp32 S [rows, ld_s], NaN past cols; logits of row-dependent spread (1 .. 60)."""
    g = torch.Generator().manual_seed(seed)
    spread = 1 + 59 * torch.rand(rows, 1, generator=g)
    S = torch.full((rows, ld_s), float("nan"))
    S[:, :cols] = spread * torch.randn(rows, cols, generator=g) + 10 * torch.randn(rows, 1, generator=g)
    return S


def softmax_reference(S, cols, scale):
    x = S[:, :cols].double() * float(torch.tensor(scale, dtype=torch.float32))
    x = x - x.amax(-1, keepdim=True)
    r = torch.softmax(x, -1)
    return r, r * (1 + x.abs())


@pytest.mark.parametrize("ld_p", SM_LDP)
@pytest.mark.gpu
def test_softmax_rows(ops, ld_p):
    for rows, cols, extra_s in ((13, ld_p - 5, 3), (21, ld_p, 0), (3, ld_p // 2 + 1, 40)):
        scale = 0.125
        S = softmax_case(rows, cols, cols + extra_s, seed=ld_p * 3 + rows).cuda()
        P = Guarded((rows, ld_p), torch.bfloat16)
        ops.softmax_rows(S, P.y, rows, cols, cols + extra_s, ld_p, scale)
        torch.cuda.synchronize()
        what = f"softmax_rows rows={rows} cols={cols} ld_p={ld_p}"
        assert P.guards_ok(), what
        assert (P.bits()[:, cols:] == 0).all(), f"{what}: padding columns of P must be exactly 0"
        r, A = softmax_reference(S, cols, scale)
        y = P.y[:, :cols].double()
        assert torch.isfinite(y).all(), what
        err = (y - r).abs()
        note("softmax_rows beta", ((err - U8 * r - 2.0 ** -126) / A).max())
        ratio = err / (U8 * r + SM_BETA * A + 2.0 ** -126)
        if float(ratio.max()) > 1:
            i, c = (int(t) for t in torch.unravel_index(ratio.argmax(), ratio.shape))
            raise AssertionError(f"{what}: x{float(ratio.max()):.2f} at row {i}, column {c} (lane {c % 32})")


# ============================================================================ 3b. linear
LINEAR_SHAPES = [(64, 256), (256, 64), (64, 2304), (256, 1024), (1024, 256), (256, 4608), (1, 1024),
                 (256, 3712), (1, 256), (64, 3712), (37, 13), (100, 1), (1000, 7), (45, 257)]


def linear_reference(x, W, bias, act, addend):
    xd, Wd = x.double(), W.double()
    z = xd @ Wd.t()
    mag = xd.abs() @ Wd.abs().t()
    if bias is not None:
        z = z + bias.double()
        mag = mag + bias.double().abs()
    in_f = W.shape[1]
    bound = (-(-in_f // 32) + 6) * U24 * mag
    if act == 1:
        bound = 1.1 * bound
        z = z * torch.sigmoid(z)
        bound = bound + 8 * U24 * z.abs()
    if addend is not None:
        z = z + addend.double()
    return z, bound + 2 * U24 * z.abs() + 1e-36


@pytest.mark.parametrize("batch", [1, 8, 9, 17, 33])
@pytest.mark.parametrize("in_f,out_f", LINEAR_SHAPES)
@pytest.mark.gpu
def test_linear(ops, in_f, out_f, batch):
    g = torch.Generator().manual_seed(in_f * 13 + out_f + batch)
    x = (torch.randn(batch, 1, generator=g) * 2 + torch.randn(batch, in_f, generator=g)).cuda()
    W = (torch.randn(out_f, in_f, generator=g) / math.sqrt(in_f)).cuda()
    bias = torch.randn(out_f, generator=g).cuda()
    addend = (5 * torch.randn(batch, 1, generator=g) + torch.randn(batch, out_f, generator=g)).cuda()
    for act, with_add, with_bias in ((0, False, True), (1, True, True), (1, False, False), (0, True, False)):
        y = Guarded((batch, out_f), torch.float32)
        b, ad = (bias if with_bias else None), (addend if with_add else None)
        ops.linear(x, W, b, y.y, act=act, addend=ad)
        torch.cuda.synchronize()
        what = f"linear {batch}x{in_f}->{out_f} act={act} addend={with_add} bias={with_bias}"
        assert y.guards_ok(), what
        r, bound = linear_reference(x, W, b, act, ad)
        err = (y.y.double() - r).abs()
        note("linear |err| / fp32 summation bound", (err / bound).max())
        assert torch.isfinite(y.y).all() and (err <= bound).all(), \
            f"{what}: worst |err| / bound {float((err / bound).max()):.3e} at {divmod(int((err / bound).argmax()), out_f)}"


# ============================================================================ 3c. layout kernels
def _shift_stack(vol, k, ndim):
    """[n, D, H, W, c] -> list over taps (kd, kh, kw order) of (shifted values, in-bounds mask):
    the value at position o + tap - pad, zero (mask False) outside the volume."""
    n, D, H, W, c = vol.shape
    p = k // 2
    pd = p if ndim == 3 else 0
    pv = torch.zeros(n, D + 2 * pd, H + 2 * p, W + 2 * p, c, dtype=vol.dtype, device=vol.device)
    pv[:, pd:pd + D, p:p + H, p:p + W] = vol
    pm = torch.zeros(D + 2 * pd, H + 2 * p, W + 2 * p, dtype=torch.bool, device=vol.device)
    pm[pd:pd + D, p:p + H, p:p + W] = True
    out = []
    for kd in range(k if ndim == 3 else 1):
        for kh in range(k):
            for kw in range(k):
                out.append((pv[:, kd:kd + D, kh:kh + H, kw:kw + W], pm[kd:kd + D, kh:kh + H, kw:kw + W]))
    return out


LAYOUT_SHAPES = [((1, 5, 7), 2), ((1, 1, 6), 2), ((1, 9, 1), 2), ((3, 4, 5), 3), ((1, 4, 3), 3),
                 ((2, 1, 1), 3), ((4, 6, 5), 3)]


@pytest.mark.parametrize("sp,ndim", LAYOUT_SHAPES)
@pytest.mark.parametrize("cp", [4, 8])
@pytest.mark.gpu
def test_im2col4(ops, sp, ndim, cp):
    D, H, W = sp
    k, n = 3, 2
    taps = k ** ndim
    g = torch.Generator().manual_seed(D * 100 + H * 10 + W + cp)
    src = bf16(torch.randn(n, D * H * W, cp, generator=g)).cuda()
    for kpad in ((taps * cp + 63) // 64 * 64, (taps * cp + 7) // 8 * 8 + 8):
        dst = Guarded((n * D * H * W, kpad), torch.bfloat16)
        ops.im2col4(src, dst.y, n, cp, D, H, W, k, ndim, kpad)
        torch.cuda.synchronize()
        assert dst.guards_ok()
        want = torch.zeros(n, D, H, W, kpad, dtype=torch.bfloat16, device="cuda")
        for t, (vals, _) in enumerate(_shift_stack(src.view(n, D, H, W, cp), k, ndim)):
            want[..., t * cp:(t + 1) * cp] = vals
        assert same_bits(dst.y, want.view(-1, kpad)), f"im2col4 {sp} ndim={ndim} cp={cp} kpad={kpad}"


@pytest.mark.parametrize("sp,ndim", LAYOUT_SHAPES)
@pytest.mark.parametrize("cout", [1, 3, 4])
@pytest.mark.gpu
def test_tap_gather(ops, sp, ndim, cout):
    """out[o][co] = bias[co] + sum_tap Y[o + tap - pad][tap * cout + co] as an fp32 sum in the
    kernel's order; Y columns past taps * cout are NaN, out columns [cout, ldo) come back 0."""
    D, H, W = sp
    k, n = 3, 2
    taps = k ** ndim
    g = torch.Generator().manual_seed(D * 100 + H * 10 + W + cout)
    for ldy, ldo, with_bias in ((taps * cout + 5, 16, True), (taps * cout, cout, False)):
        y = torch.full((n, D * H * W, ldy), float("nan"))
        y[..., :taps * cout] = torch.randn(n, D * H * W, taps * cout, generator=g) * 3
        y = bf16(y).cuda()
        bias = torch.randn(cout, generator=g).cuda() if with_bias else None
        out = Guarded((n, D * H * W, ldo), torch.bfloat16)
        ops.tap_gather(y, out.y, bias, n, D, H, W, k, ndim, cout, ldy, ldo)
        torch.cuda.synchronize()
        what = f"tap_gather {sp} ndim={ndim} cout={cout} ldy={ldy} ldo={ldo}"
        assert out.guards_ok(), what
        acc = (bias.view(1, 1, 1, 1, cout) if with_bias else torch.zeros(cout, device="cuda")).expand(n, D, H, W, cout)
        acc = acc.float().contiguous()
        yv = y[..., :taps * cout].view(n, D, H, W, taps * cout)
        for t, (vals, m) in enumerate(_shift_stack(yv, k, ndim)):
            acc = torch.where(m[None, ..., None], acc + vals[..., t * cout:(t + 1) * cout].float(), acc)
        assert same_bits(out.y[..., :cout], bf16(acc).view(n, -1, cout)), what
        assert (out.bits()[..., cout:] == 0).all(), f"{what}: padding channels must be 0"


@pytest.mark.parametrize("n,S,C,ldc", [(1, 1, 1, 8), (2, 37, 3, 16), (3, 1000, 4, 4), (2, 5, 16, 64),
                                       (1, 2 * 48 * 40, 4, 64)])
@pytest.mark.gpu
def test_nchw_nhwc_converters(ops, n, S, C, ldc):
    g = torch.Generator().manual_seed(n + S + C + ldc)
    x = (torch.randn(n, C, S, generator=g) * 4).cuda()
    h = Guarded((n, S, ldc), torch.bfloat16)
    ops.nchw_to_nhwc(x, h.y, n, S, C, ldc)
    torch.cuda.synchronize()
    assert h.guards_ok()
    assert same_bits(h.y[..., :C], bf16(x.transpose(1, 2)))
    assert (h.bits()[..., C:] == 0).all(), "nchw_to_nhwc: padding channels must be 0"
    src = bf16(torch.randn(n, S, ldc, generator=g) * 4).cuda()
    src[..., C:] = float("nan")                # never read
    o = Guarded((n, C, S), torch.float32)
    ops.nhwc_to_nchw(src, o.y, n, S, C, ldc)
    torch.cuda.synchronize()
    assert o.guards_ok()
    assert same_bits(o.y, src[..., :C].float().transpose(1, 2))


# ============================================================================ 4. split-precision glue
def hi_lo(v):
    hi = bf16(v)
    return hi, bf16(v - hi.float())


GN_SPLIT_C = [(3, 3, 1), (4, 2, 2), (64, 8, 4), (96, 8, 4), (128, 8, 8), (192, 4, 24), (256, 8, 32),
              (384, 8, 16), (512, 8, 64)]          # (C, groups, stats_cpg)
GN_SPLIT_VARIANTS = [   # (stats, silu, rowbias pitch (0: none), residual, y, y32)
    (True, True, 5, False, True, False),
    (True, False, 0, True, False, True),          # SplitProgram.gn_f32: fp32 y + residual
    (True, True, 1, True, True, True),
    (False, False, 0, False, True, False),        # SplitProgram.raw
    (False, False, 5, True, True, True),
    (True, True, 0, False, True, True),
]


@pytest.mark.parametrize("N,S", [(3, 37), (2, 700)])
@pytest.mark.parametrize("C,G,scpg", GN_SPLIT_C)
@pytest.mark.gpu
def test_gn_split(ops, C, G, scpg, N, S):
    g = torch.Generator().manual_seed(C * 3 + N + S)
    cpg = C // G
    mu = -2 + 4 * torch.rand(N, 1, G, 1, generator=g)
    sd = torch.exp(math.log(0.25) + math.log(16) * torch.rand(N, 1, G, 1, generator=g))
    x = (mu + sd * torch.randn(N, S, G, cpg, generator=g)).reshape(N, S, C).cuda()
    gamma = (1 + 0.5 * torch.randn(C, generator=g)).cuda()
    beta = (0.5 * torch.randn(C, generator=g)).cuda()
    res = (3 * torch.randn(N, 1, 1, generator=g) + torch.randn(N, S, C, generator=g)).cuda()
    stats = gn_stats_ref(x, scpg).contiguous()
    xd = x.double().view(N, S, G, cpg)
    mean = xd.mean((1, 3), keepdim=True)
    rstd = (xd.var((1, 3), unbiased=False, keepdim=True) + EPS).rsqrt()
    gm, bt = gamma.double().view(1, 1, G, -1), beta.double().view(1, 1, G, -1)
    for (ws, silu, rbx, wres, wy, wy32) in GN_SPLIT_VARIANTS:
        what = f"gn_split C={C} N={N} S={S} stats={ws} silu={silu} rowbias={rbx} residual={wres} y={wy} y32={wy32}"
        if ws:
            u = ((xd - mean) * rstd * gm + bt).view(N, S, C)
            A = ((xd * rstd * gm).abs() + (mean * rstd * gm).abs() + bt.abs()).view(N, S, C)
            r = u * torch.sigmoid(u) if silu else u
        else:
            r, A = x.double(), x.double().abs()
        rbld = C + rbx - 1 if rbx else 0
        rb = None
        if rbx:
            rb = torch.full((N, rbld), float("nan"), device="cuda")
            rb[:, :C] = (2 * torch.randn(N, 1, generator=g) + torch.randn(N, C, generator=g)).cuda()
            r, A = r + rb[:, None, :C].double(), A + rb[:, None, :C].double().abs()
        if wres:
            r, A = r + res.double(), A + res.double().abs()
        y = Guarded((N, S, 3 * C), torch.bfloat16) if wy else None
        y32 = Guarded((N, S, C), torch.float32) if wy32 else None
        ops.gn_split(x, y.y if wy else None, stats if ws else None, gamma if ws else None,
                     beta if ws else None, N, S, C, G, scpg, EPS, silu, rowbias=rb, rowbias_ld=rbld,
                     residual=res if wres else None, y32=y32.y if wy32 else None)
        torch.cuda.synchronize()
        if wy32:
            assert y32.guards_ok(), what
            err = (y32.y.double() - r).abs()
            note("gn_split y32 beta", ((err - U24 * r.abs()) / A).max())
            ratio = err / (U24 * r.abs() + SPLIT32_BETA * A)
            assert ratio.max() <= 1, f"{what}: y32 x{float(ratio.max()):.2f} at {torch.unravel_index(ratio.argmax(), ratio.shape)}"
        if wy:
            assert y.guards_ok(), what
            hi, lo, hi3 = y.y[..., :C], y.y[..., C:2 * C], y.y[..., 2 * C:]
            assert same_bits(hi3, hi), f"{what}: segment 3 differs from segment 1"
            if wy32:                                   # the value the kernel formed is y32
                h2, l2 = hi_lo(y32.y)
                assert same_bits(hi, h2) and same_bits(lo, l2), f"{what}: (hi, lo) is not the split of y32"
            else:                                      # hi is the nearest bf16 of hi + lo
                ulp = torch.ldexp(torch.ones_like(hi.float()), torch.frexp(hi.float())[1] - 8)
                assert (lo.float().abs() <= 0.5 * ulp).all(), f"{what}: |lo| over half an ulp of hi"
            v = hi.double() + lo.double()
            err = (v - r).abs()
            note("gn_split hi+lo beta", ((err - U16 * r.abs()) / A).max())
            ratio = err / (U16 * r.abs() + SPLIT_BETA * A)
            assert ratio.max() <= 1, f"{what}: hi + lo x{float(ratio.max()):.2f} at {torch.unravel_index(ratio.argmax(), ratio.shape)}"


@pytest.mark.parametrize("N,S,G,cpg", [(2, 37, 512, 1), (3, 100, 1, 1), (1, 9, 1, 3), (2, 2368, 8, 16),
                                       (1, 3000, 4, 64), (5, 77, 32, 4), (2, 1000, 8, 64)])
@pytest.mark.gpu
def test_stats_f32(ops, N, S, G, cpg):
    """fp64 (sum, sum of squares) per (sample, group) of an fp32 channels-last tensor, added to
    the output.  Rows carry a strong trend, so visiting the wrong (row, channel) pairs shows."""
    C = G * cpg
    g = torch.Generator().manual_seed(N + S + G + cpg)
    x = (torch.linspace(-3, 5, S).view(1, S, 1) * torch.rand(N, 1, C, generator=g)
         + torch.randn(N, S, C, generator=g)).cuda()
    st = Guarded((N, G, 2), torch.float64, fill=None)
    st0 = torch.randn(N, G, 2, generator=g, dtype=torch.float64).cuda()
    st.y.copy_(st0)
    ops.stats_f32(x, st.y, N, S, C, G)
    torch.cuda.synchronize()
    assert st.guards_ok()
    xr = x.double().view(N, S, G, cpg)
    want = torch.stack([xr.sum((1, 3)), (xr * xr).sum((1, 3))], -1)
    mag = torch.stack([xr.abs().sum((1, 3)), (xr * xr).sum((1, 3))], -1)
    e = ((st.y - st0) - want).abs() / mag
    note("stats_f32 beta_s", e.max())
    assert e.max() <= SF32_BETA, f"worst (sample, group, sum|sumsq) {torch.unravel_index(e.argmax(), e.shape)}: {float(e.max()):.3e}"


def split3_expected(src_flat, dst_flat, outer, inner, width, so, si, do, di, seg, pattern, s_off, d_off):
    dev = src_flat.device
    o = torch.arange(outer, device=dev).view(-1, 1, 1)
    i = torch.arange(inner, device=dev).view(1, -1, 1)
    j = torch.arange(width, device=dev).view(1, 1, -1)
    sidx = (s_off + o * so + i * si + j).reshape(-1)
    didx = (d_off + o * do + i * di + j).reshape(-1)
    hi, lo = hi_lo(src_flat[sidx])
    want = dst_flat.clone()
    parts = (hi, lo, hi) if pattern == 0 else (hi, hi, lo)
    for p in range(3):
        want[didx + p * seg] = parts[p]
    return want, sidx


SPLIT3_CASES = [   # (outer, inner, width, src_outer_ld, src_inner_ld, dst_outer_ld, dst_inner_ld, seg, pattern, src_off, dst_off)
    # the engine's q / k splits (split_engine.py: B n rows of qkv [B, n, 3C] -> [B, n, heads, 3d])
    (2 * 37, 4, 64, 3 * 256, 64, 4 * 192, 192, 64, 0, 0, 0),
    (2 * 37, 4, 64, 3 * 256, 64, 4 * 192, 192, 64, 1, 256, 0),
    (3 * 8, 2, 128, 3 * 256, 128, 2 * 384, 384, 128, 1, 256, 0),
    # v^T [B C, npad] fp32 -> [B C, 3 npad], n valid keys
    (2 * 256, 1, 100, 128, 0, 3 * 128, 0, 128, 1, 0, 0),
    (3 * 64, 1, 1200, 1216, 0, 3 * 1216, 0, 1216, 1, 0, 0),
    # strides of its own, src_off / dst_off, seg > width
    (5, 3, 33, 200, 60, 400, 130, 41, 0, 7, 11),
    (7, 2, 9, 30, 11, 90, 40, 13, 1, 3, 5),
]


@pytest.mark.parametrize("case", SPLIT3_CASES)
@pytest.mark.gpu
def test_split3(ops, case):
    outer, inner, width, so, si, do, di, seg, pattern, s_off, d_off = case
    g = torch.Generator().manual_seed(sum(case))
    n_src = s_off + (outer - 1) * so + (inner - 1) * si + width + 16
    n_dst = d_off + (outer - 1) * do + (inner - 1) * di + 2 * seg + width + 16
    src = torch.full((n_src,), float("nan"), device="cuda")
    dst = Guarded((n_dst,), torch.bfloat16, fill=None)
    want, sidx = split3_expected(src, dst.y, outer, inner, width, so, si, do, di, seg, pattern, s_off, d_off)
    src[sidx] = (torch.randn(sidx.numel(), generator=g) * torch.exp(4 * torch.randn(sidx.numel(), generator=g))).cuda()
    want, _ = split3_expected(src, dst.y, outer, inner, width, so, si, do, di, seg, pattern, s_off, d_off)
    ops.split3(src, dst.y, outer, inner, width, so, si, do, di, seg, pattern, src_off=s_off, dst_off=d_off)
    torch.cuda.synchronize()
    assert dst.guards_ok()
    assert same_bits(dst.y, want), f"split3 {case}: {int((dst.bits() != want.view(torch.int16)).sum())} wrong elements"


@pytest.mark.parametrize("rows,cols,ld_s,seg,ld_p", [
    (2 * 4 * 100, 100, 128, 128, 3 * 128),            # the engine's strides (npad = rup(n, 64))
    (1 * 4 * 1200, 1200, 1216, 1216, 3 * 1216),
    (13, 64, 64, 64, 192),
    (9, 37, 44, 40, 3 * 40 + 10),                     # strides of its own
    (7, 1, 1, 1, 3)])
@pytest.mark.gpu
def test_softmax_rows_split(ops, rows, cols, ld_s, seg, ld_p):
    scale = 0.125
    S = softmax_case(rows, cols, ld_s, seed=rows + cols).cuda()
    P = Guarded((rows, ld_p), torch.bfloat16, fill=None)
    for p in range(3):
        P.y[:, p * seg:p * seg + cols] = float("nan")
    ops.softmax_rows_split(S, P.y, rows, cols, ld_s, ld_p, seg, scale)
    torch.cuda.synchronize()
    what = f"softmax_rows_split rows={rows} cols={cols} seg={seg} ld_p={ld_p}"
    assert P.guards_ok(), what
    untouched = torch.ones(ld_p, dtype=torch.bool, device="cuda")
    for p in range(3):
        untouched[p * seg:p * seg + cols] = False
    assert (P.bits()[:, untouched] == _SENT[torch.bfloat16][1]).all(), f"{what}: a padding column was written"
    hi, lo, hi3 = P.y[:, :cols], P.y[:, seg:seg + cols], P.y[:, 2 * seg:2 * seg + cols]
    assert same_bits(hi3, hi), f"{what}: segment 3 differs from segment 1"
    ulp = torch.ldexp(torch.ones_like(hi.float()), torch.frexp(hi.float())[1] - 8)
    assert (lo.float().abs() <= 0.5 * ulp).all(), what
    r, A = softmax_reference(S, cols, scale)
    err = (hi.double() + lo.double() - r).abs()
    note("softmax_rows_split beta", ((err - U16 * r - 2.0 ** -126) / A).max())
    ratio = err / (U16 * r + SMS_BETA * A + 2.0 ** -126)
    assert ratio.max() <= 1, f"{what}: x{float(ratio.max()):.2f} at {torch.unravel_index(ratio.argmax(), ratio.shape)}"


@pytest.mark.parametrize("B,per,stride,off", [(2, 3 * 8 * 12 * 8, 0, 0), (3, 1000, 2 * 1000 + 37, 5),
                                              (1, 7, 30, 9), (4, 4 * 2 * 48 * 40, 2 * 4 * 2 * 48 * 40 + 8, 16)])
@pytest.mark.gpu
def test_bf16_residual_nchw(ops, B, per, stride, off):
    g = torch.Generator().manual_seed(B + per)
    x = (torch.randn(B, per, generator=g) * torch.exp(3 * torch.randn(B, per, generator=g))).cuda()
    st = stride or 2 * per
    out = Guarded((off + B * st,), torch.float32, fill=None)
    ops.bf16_residual_nchw(x, out.y, B, per, out_sample_stride=stride, out_off=off)
    torch.cuda.synchronize()
    assert out.guards_ok()
    want = out.y.clone()
    for b in range(B):
        o = off + b * st
        want[o:o + per] = x[b] - bf16(x[b]).float()
        want[o + per:o + 2 * per] = x[b]
    assert same_bits(out.y, want)


# ============================================================================ 5. coverage
@pytest.mark.gpu
def test_parametrization_covers_what_the_models_run(ops, monkeypatch):
    """Every shape the inference programs of the test-size models hand to gn_apply, gn_split,
    softmax_rows, linear and the attention launch is in the parametrization above, and so are
    the cfg4 bench shapes (attention at n 1200, d 128, 4 heads; GroupNorm at C 128 / 256 / 512)."""
    import contextlib
    import io
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.vae import VAE3D
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet as UNet2D
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.unet import UNet as UNet25D

    seen = {k: set() for k in ("gn_apply", "gn_split", "softmax_rows", "linear", "attn")}

    def wrap(name, key):
        orig = getattr(ops, name)

        def rec(*a, **kw):
            seen[name].add(key(*a, **kw))
            return orig(*a, **kw)
        monkeypatch.setattr(ops, name, rec)

    wrap("gn_apply", lambda x, y, st, gm, bt, N, S, C, G, cpg, *a, **kw: (C, G, cpg))
    wrap("gn_split", lambda x, y, st, gm, bt, N, S, C, *a, **kw: C)
    wrap("softmax_rows", lambda S, P, rows, cols, ld_s, ld_p, scale: sm_class(ld_p))
    wrap("linear", lambda x, W, *a, **kw: (W.shape[1], W.shape[0]))

    dev = "cuda"
    progs = []
    with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
        progs.append(UNet3DModelWithAttention(3, base_channels=64, time_emb_dim=64).to(dev).eval()
                     .program(2, (8, 8, 8)))
        for precision in ("bf16", "split"):
            m2 = UNet2D(img_channels=1, base_channels=64, time_emb_dim=64).to(dev).eval()
            m2.precision = precision
            progs.append(m2.program(2, (32, 32), 1, 0))
            m25 = UNet25D(in_channels=20, out_channels=4, base_channels=64, time_emb_dim=64).to(dev).eval()
            m25.precision = precision
            progs.append(m25.program(2, (32, 32), 4, 16))
        vae = VAE3D(in_channels=4, base_channels=32, num_down=3, latent_channels=16).to(dev).eval()
        progs.append(vae._program("encode", torch.zeros(2, 4, 16, 24, 16, device=dev)))
        progs.append(vae._program("decode", torch.zeros(2, 16, 4, 6, 4, device=dev)))
        for prog in progs:
            prog.run()
            for a in getattr(prog, "_keep_alive", []):
                if isinstance(a, _lib.MriAttnArgs):
                    seen["attn"].add((a.n, a.d, a.heads))
    torch.cuda.synchronize()
    print("recorded:", {k: sorted(v) for k, v in seen.items()})
    assert seen["gn_apply"] and seen["gn_split"] and seen["linear"] and seen["attn"]
    cover = {
        "gn_apply": {(C, G, s) for (C, G, s, *_ ) in GN_CASES},
        "gn_split": {C for (C, _, _) in GN_SPLIT_C},
        "softmax_rows": {sm_class(ld) for ld in SM_LDP},
        "linear": set(LINEAR_SHAPES),
        "attn": {(n, d, h) for (d, n, h, _) in ATTN_CASES},
    }
    missing = {k: sorted(seen[k] - cover[k]) for k in seen if seen[k] - cover[k]}
    assert not missing, missing
    assert (1200, 128, 4) in cover["attn"] and {1, 3} <= {B for (d, n, h, B) in ATTN_CASES if (n, d, h) == (1200, 128, 4)}
    assert {(128, 8, 16), (256, 8, 32), (512, 8, 64)} <= cover["gn_apply"]
    assert (128, 8, 16, 1, 40 * 48 * 40) in GN_CASES and (128, 8, 16, 16, 40 * 48 * 40) in GN_CASES


if __name__ == "__main__" and sys.argv[1:] == ["--child"]:
    _child()
