"""The HBM-bound backward kernels (csrc/backward_ops.cu) one at a time, each against a float64
torch reference of the same operation computed on the same bf16 / fp32 inputs the kernel reads.

The whole-model gradient tests allow rel-L2 5e-2 per parameter, which hides e.g. a GroupNorm
backward that drops its group-mean terms or normalises with a neighbouring group's statistics
(1e-3 .. 2e-2 there).  Here every output the kernel overwrites starts as NaN (a missed write
fails), every padding column it must not read is NaN (a stray read leaks), and the inputs are
built so that plausible bugs are far outside the tolerances.

Tolerances, from the error sources each kernel has:

* GroupNorm(+SiLU) backward dx, per (sample, group) block and overall: rel-L2 <= 5e-3 =
  2^-8 (bf16 round-to-nearest of the stored dx, a bound per element) + 2^-10 (silu' built on the
  tanh.approx sigmoid, relative error 2^-11, amplified at most ~2x by 1 + u (1 - sigmoid)).
  Pass-A sums S0 = sum dy, S1 = sum du, S2 = sum du * xhat over each (sample, channel): rel-L2 over
  the [samples, C] array <= 2e-5 without SiLU (fp32 per-thread partial sums of at most a few
  hundred terms before the fp64 fold) and <= 2e-3 with it (the sigmoid error above, which does
  not average out in a sum).  The column sums (fused into gn_bwd_apply and the standalone
  ops.colsum) are fp32 per-thread partials of the bf16 values folded in fp64:
  |err| <= 1e-5 * sum |dx| per column.
* ops.gn_stats (forward statistics, 4 channels per group included) also sums fp32 partials per
  thread before its fp64 atomics: |err| <= 1e-5 * sum |x| (resp. sum x^2) per group, not 1e-12.
* softmax_bwd: per row rel-L2 <= 4e-3 (bf16 output rounding, bound 2^-8; the fp32 row dot
  product adds ~1e-5).
* linear_bwd: the standard fp32 summation bound n u sum |terms| per element, u = 2^-24, with
  n = 64 + ceil(out_f / 64) + 1 for dX (64-term fma chains per chunk, then one fp32 atomic per
  chunk) and n = batch + 1 for dW and db.
* silu / silu_bwd (fp32 expf, IEEE division): 8 ulp relative for silu and 2^-18 of the term
  magnitudes for silu_bwd (1 - sigmoid(v) cancels for v ~ 16, losing log2(v) bits), plus an
  absolute floor of 1e-36 where expf(-v) overflows (v < -88.7) and the result underflows.
* minsnr loss (fp32 sums per thread, then atomics): loss and per-sample MSE relative 1e-5;
  dpred elementwise relative 4e-6 (a handful of fp32 roundings).
* add_bf16, grad_finalize and the fp64 -> fp32 copy_cast: bit-exact.
"""
import math

import pytest
import torch
import torch.nn.functional as F

EPS = 1e-5
DX_TOL = 5e-3
SUM_TOL = {False: 2e-5, True: 2e-3}
COLSUM_TOL = 1e-5
SM_TOL = 4e-3

# (C, groups, channels per statistics group) -- the stats arrive as [N, C / stats_cpg, 2] partial
# sums, so stats_cpg < C / groups means several statistics groups fold into one norm group
GN_CONFIGS = [
    (32, 8, 4), (64, 16, 4),                   # the VAE's 4-channel groups (kFine); 64 = 32 padded
    (64, 8, 8), (128, 8, 16), (256, 8, 32), (512, 8, 64),   # GroupNorm(8, C) of the UNets
    (64, 4, 8), (128, 4, 16), (256, 4, 32), (512, 4, 64),   # GN(8, 2C) over a concatenation, run
                                                            # as GN(4, C) per half: 2 stats groups each
    (192, 8, 24), (384, 8, 48),                # 240 / 192 threads: a partial last warp (192)
    (512, 64, 8), (256, 64, 4),                # the 64-group bound of gn_bwd_apply
    (1024, 8, 128),
    (2048, 8, 256),                            # 256 vectors per row: one row per block step
]
SOFTMAX_COLS = [1, 31, 33, 150, 256, 257, 1200, 1280, 1281, 2048]


def _rows_step(C):
    vpr = C // 8
    return (256 // vpr) * vpr // vpr


def _gn_cases():
    """(C, groups, stats_cpg, N, S, add, colsum) -- each width at 1 row, fewer rows than one
    4-row-step batch, and a row count that is not a multiple of rows_step * 4, with the three
    ways the gradient is written (fresh, + a separate tensor, + in place) and both column sums."""
    cases = []
    for (C, G, scpg) in GN_CONFIGS:
        rs = _rows_step(C)
        cases.append((C, G, scpg, 3, 7 * rs * 4 + 2 * rs + 1, "none", True))
        cases.append((C, G, scpg, 1, 1, "separate", False))
        cases.append((C, G, scpg, 8, max(2, 4 * rs - 1), "inplace", True))
    cases.append((128, 8, 16, 1, 40 * 48 * 40, "inplace", True))     # cfg4/5 latent, top level
    cases.append((64, 8, 8, 300, 5, "separate", True))             # > 296 samples: one block each
    cases.append((32, 8, 4, 300, 3, "none", False))
    return cases


WORST = {}   # section -> worst measured error (printed at the end of the module, run with -s)


def note(section, value):
    WORST[section] = max(WORST.get(section, 0.0), float(value))


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300)).item()


def bf16(t):
    return t.to(torch.bfloat16)


def nan_like(shape, dtype, device):
    return torch.full(shape, float("nan"), dtype=dtype, device=device)


# ---------------------------------------------------------------- GroupNorm references (CPU or GPU)
def gn_inputs(N, S, C, G, device, seed=0):
    """bf16 x, dy with distinct (mean, scale) per (sample, group) and dy = a + b xhat + noise per
    group, fp32 gamma / beta.  Such a dy keeps large group means of gamma * du and
    gamma * du * xhat, so a backward that drops or misplaces them is far off."""
    g = torch.Generator().manual_seed(seed)
    cpg = C // G
    per_group = lambda lo, hi: (lo + (hi - lo) * torch.rand(N, 1, G, 1, generator=g, dtype=torch.float64))
    mu, sd = per_group(-2, 2), torch.exp(per_group(math.log(0.25), math.log(4)))
    x = bf16(mu + sd * torch.randn(N, S, G, cpg, generator=g, dtype=torch.float64)).reshape(N, S, C)
    xh, _ = gn_xhat(x.double(), G)
    a = torch.randn(N, 1, G, 1, generator=g, dtype=torch.float64).expand(N, 1, G, cpg).reshape(N, 1, C)
    b = torch.randn(N, 1, G, 1, generator=g, dtype=torch.float64).expand(N, 1, G, cpg).reshape(N, 1, C)
    dy = bf16(a + b * xh + 0.3 * torch.randn(N, S, C, generator=g, dtype=torch.float64))
    gamma = (1 + 0.5 * torch.randn(C, generator=g)).float()
    beta = (0.5 * torch.randn(C, generator=g)).float()
    return x.to(device), dy.to(device), gamma.to(device), beta.to(device)


def gn_stats_ref(x, stats_cpg):
    """fp64 (sum, sumsq) per (sample, statistics group): [N, C / stats_cpg, 2]."""
    N, S, C = x.shape
    xr = x.double().reshape(N, S, C // stats_cpg, stats_cpg)
    return torch.stack([xr.sum((1, 3)), (xr * xr).sum((1, 3))], -1)


def gn_xhat(x, G, eps=EPS, swap=False):
    """(x - mean) * rstd per (sample, group) in fp64; swap: with the statistics of group g ^ 1."""
    N, S, C = x.shape
    xr = x.reshape(N, S, G, C // G)
    mean = xr.mean((1, 3), keepdim=True)
    rstd = (xr.var((1, 3), unbiased=False, keepdim=True) + eps).rsqrt()
    if swap:
        gi = torch.arange(G, device=x.device) ^ 1
        mean, rstd = mean[:, :, gi], rstd[:, :, gi]
    return ((xr - mean) * rstd).reshape(N, S, C), rstd


def gn_bwd_autograd(x, dy, gamma, beta, G, silu, eps=EPS):
    """torch.autograd in fp64 through F.silu(F.group_norm(x)) (or F.group_norm alone): dx and the
    per-(sample, channel) sums S0 = sum dy, S1 = sum du (dbeta), S2 = sum du * xhat (dgamma)."""
    xd = x.double().permute(0, 2, 1).contiguous().requires_grad_(True)   # [N, C, S]
    xh = F.group_norm(xd, G, eps=eps)
    u = xh * gamma.double()[:, None] + beta.double()[:, None]
    u.retain_grad()
    y = F.silu(u) if silu else u
    dyd = dy.double().permute(0, 2, 1)
    y.backward(dyd)
    du = u.grad
    S0 = dyd.sum(-1)
    S1 = du.sum(-1)
    S2 = (du * xh.detach()).sum(-1)
    return xd.grad.permute(0, 2, 1), torch.stack([S0, S1, S2])


def gn_bwd_formula(x, dy, gamma, beta, G, silu, eps=EPS, drop_means=False, swap=False):
    """The fp64 formula gn_bwd_apply implements, dx = rstd (gamma du - m1 - xhat m2) with per
    (sample, group) m1 = mean(gamma du), m2 = mean(gamma du xhat).  drop_means / swap build the
    plausible wrong kernels the inputs must tell apart: no m1 / m2 terms, and every channel
    normalised with the statistics of group g ^ 1."""
    N, S, C = x.shape
    cpg = C // G
    xh, rstd = gn_xhat(x.double(), G, eps, swap)
    gm, bt = gamma.double(), beta.double()
    u = xh * gm + bt
    sg = torch.sigmoid(u)
    du = dy.double() * (sg * (1 + u * (1 - sg)) if silu else 1.0)
    gdu = (gm * du).reshape(N, S, G, cpg)
    xr = xh.reshape(N, S, G, cpg)
    m1 = gdu.mean((1, 3), keepdim=True)
    m2 = (gdu * xr).mean((1, 3), keepdim=True)
    if drop_means:
        m1, m2 = 0 * m1, 0 * m2
    return (rstd * (gdu - m1 - xr * m2)).reshape(N, S, C)


def block_errors(out, ref, G):
    """rel-L2 per (sample, group) block of [N, S, C] tensors: [N, G]."""
    N, S, C = ref.shape
    d = (out.double() - ref.double()).reshape(N, S, G, C // G)
    r = ref.double().reshape(N, S, G, C // G)
    return d.norm(dim=(1, 3)) / r.norm(dim=(1, 3)).clamp_min(1e-300)


@pytest.mark.parametrize("N,S,C,G,silu", [(2, 37, 32, 8, True), (3, 20, 64, 8, False),
                                           (2, 50, 64, 16, True), (1, 9, 192, 8, True)])
def test_gn_reference_helpers_on_cpu(N, S, C, G, silu):
    """The fp64 formula behind the wrong references equals torch.autograd, and the inputs put the
    plausible bugs > 10x the dx tolerance away (CPU only)."""
    x, dy, gamma, beta = gn_inputs(N, S, C, G, "cpu", seed=N * C + S)
    ref, sums = gn_bwd_autograd(x, dy, gamma, beta, G, silu)
    assert rel(gn_bwd_formula(x, dy, gamma, beta, G, silu), ref) < 1e-10
    xh, _ = gn_xhat(x.double(), G)
    u = xh * gamma.double() + beta.double()
    du = dy.double() * (torch.sigmoid(u) * (1 + u * (1 - torch.sigmoid(u))) if silu else 1.0)
    assert rel(sums[1], du.sum(1)) < 1e-10 and rel(sums[2], (du * xh).sum(1)) < 1e-10
    assert rel(sums[0], dy.double().sum(1)) < 1e-12
    for kw in (dict(drop_means=True), dict(swap=True)):
        assert rel(gn_bwd_formula(x, dy, gamma, beta, G, silu, **kw), ref) > 10 * DX_TOL, kw
    st = gn_stats_ref(x, C // G)
    assert torch.allclose(st[..., 0], x.double().reshape(N, S, G, C // G).sum((1, 3)), rtol=1e-12)


# ---------------------------------------------------------------- GPU fixtures
@pytest.fixture(scope="module")
def ops():
    from mri_image_generation_b200 import _lib, ops
    _lib.require_device()
    yield ops
    for k in sorted(WORST):
        print(f"worst {k}: {WORST[k]:.3e}")


def _mri_error():
    from mri_image_generation_b200 import _lib
    return _lib.MriError


# ---------------------------------------------------------------- 1. GroupNorm(+SiLU) backward
@pytest.mark.gpu
@pytest.mark.parametrize("silu", [True, False])
@pytest.mark.parametrize("C,G,scpg,N,S,add_mode,with_colsum", _gn_cases())
def test_gn_bwd_reduce_apply(ops, C, G, scpg, N, S, add_mode, with_colsum, silu):
    dev = "cuda"
    x, dy, gamma, beta = gn_inputs(N, S, C, G, dev, seed=C + G + N + S)
    stats = gn_stats_ref(x, scpg).contiguous()
    st_kernel = torch.zeros_like(stats)
    ops.gn_stats(x, st_kernel, N, S, C, scpg)
    xa = x.double().abs().reshape(N, S, C // scpg, scpg).sum((1, 3))
    note("gn_stats |err| / sum|x|", ((st_kernel[..., 0] - stats[..., 0]).abs() / xa).max())
    assert ((st_kernel[..., 0] - stats[..., 0]).abs() <= COLSUM_TOL * xa).all()
    assert ((st_kernel[..., 1] - stats[..., 1]).abs() <= COLSUM_TOL * stats[..., 1]).all()

    ref_dx, ref_sums = gn_bwd_autograd(x, dy, gamma, beta, G, silu)
    for kw in (dict(drop_means=True), dict(swap=True)):   # the inputs can tell the bugs apart
        wrong = gn_bwd_formula(x, dy, gamma, beta, G, silu, **kw)
        assert rel(wrong, ref_dx) > 10 * DX_TOL, kw

    sums = torch.zeros(3, N, C, dtype=torch.float64, device=dev)   # accumulated into
    ops.gn_bwd_reduce(x, dy, stats, gamma, beta, sums, N, S, C, G, scpg, EPS, silu)
    for q in range(3):
        e = rel(sums[q], ref_sums[q])
        note(f"gn_bwd_reduce S{q} rel-L2 (silu={silu})", e)
        assert e <= SUM_TOL[silu], f"S{q}: rel-L2 {e:.3e}"

    g = torch.Generator().manual_seed(7)
    add_val = bf16(torch.randn(N, S, C, generator=g) * ref_dx.float().std().cpu()).to(dev)
    if add_mode == "none":
        add, dx = None, nan_like((N, S, C), torch.bfloat16, dev)
    elif add_mode == "separate":
        add, dx = add_val, nan_like((N, S, C), torch.bfloat16, dev)
    else:                                 # in place: BackwardMixin.emit_grad's produce(g, g)
        dx = add_val.clone()
        add = dx
    cs0 = torch.randn(N, C, dtype=torch.float64, generator=g).to(dev)
    cs = cs0.clone() if with_colsum else None
    ops.gn_bwd_apply(x, dy, add, dx, stats, gamma, beta, sums, N, S, C, G, scpg, EPS, silu, colsum=cs)
    want = ref_dx + (add_val.double() if add_mode != "none" else 0)
    assert torch.isfinite(dx.float()).all()
    blk = block_errors(dx, want, G)
    n, gi = divmod(int(blk.argmax()), G)
    note("gn_bwd_apply dx rel-L2 per (sample, group)", blk.max())
    assert blk.max() <= DX_TOL, f"dx: worst (sample {n}, group {gi}) rel-L2 {blk.max():.3e}"
    assert rel(dx, want) <= DX_TOL

    written = dx.double().sum(1)                     # fp64 sum of the bf16 values written
    bound = COLSUM_TOL * dx.double().abs().sum(1) + 1e-300
    if with_colsum:
        note("colsum |err| / sum|dx|", ((cs - cs0 - written).abs() / bound).max() * COLSUM_TOL)
        assert ((cs - cs0 - written).abs() <= bound).all(), "fused colsum"
    cs2 = torch.full((N, C), -3.25, dtype=torch.float64, device=dev)
    ops.colsum(dx, cs2, N, S, C)
    note("colsum |err| / sum|dx|", ((cs2 + 3.25 - written).abs() / bound).max() * COLSUM_TOL)
    assert ((cs2 + 3.25 - written).abs() <= bound).all(), "ops.colsum must add to the buffer"


@pytest.mark.gpu
@pytest.mark.parametrize("silu", [True, False])
def test_gn_bwd_zero_padded_groups(ops, silu):
    """VAE3D's 32-channel level runs zero-padded to 64 channels as 16 groups of 4: x = gamma =
    beta = 0 over the padding.  dx must be exactly 0 there and finite everywhere."""
    dev, N, S, C, G = "cuda", 2, 300, 64, 16
    x, dy, gamma, beta = gn_inputs(N, S, C, G, dev, seed=11)
    x[..., 32:] = 0
    gamma[32:] = 0
    beta[32:] = 0
    stats = gn_stats_ref(x, 4).contiguous()
    sums = torch.zeros(3, N, C, dtype=torch.float64, device=dev)
    dx = nan_like((N, S, C), torch.bfloat16, dev)
    ops.gn_bwd_reduce(x, dy, stats, gamma, beta, sums, N, S, C, G, 4, EPS, silu)
    ops.gn_bwd_apply(x, dy, None, dx, stats, gamma, beta, sums, N, S, C, G, 4, EPS, silu)
    assert torch.isfinite(dx.float()).all()
    assert (dx[..., 32:].float() == 0).all()
    ref, _ = gn_bwd_autograd(x, dy, gamma, beta, G, silu)
    assert block_errors(dx[..., :32], ref[..., :32], 8).max() <= DX_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("C,G,scpg", [(128, 8, 16), (32, 8, 4)])
def test_gn_bwd_constant_group(ops, C, G, scpg):
    """A group holding one bf16-exact value (variance 0, rstd = 1 / sqrt(eps)) still matches."""
    dev, N, S = "cuda", 2, 50
    x, dy, gamma, beta = gn_inputs(N, S, C, G, dev, seed=12)
    cpg = C // G
    x[1, :, 2 * cpg:3 * cpg] = 1.5
    stats = gn_stats_ref(x, scpg).contiguous()
    sums = torch.zeros(3, N, C, dtype=torch.float64, device=dev)
    dx = nan_like((N, S, C), torch.bfloat16, dev)
    ops.gn_bwd_reduce(x, dy, stats, gamma, beta, sums, N, S, C, G, scpg, EPS, True)
    ops.gn_bwd_apply(x, dy, None, dx, stats, gamma, beta, sums, N, S, C, G, scpg, EPS, True)
    ref, _ = gn_bwd_autograd(x, dy, gamma, beta, G, True)
    blk = block_errors(dx, ref, G)
    assert blk.max() <= DX_TOL, blk


@pytest.mark.gpu
def test_gn_bwd_bad_configurations_raise(ops):
    MriError = _mri_error()
    dev = "cuda"

    def run(C, G, scpg, which):
        x = torch.zeros(1, 8, C, dtype=torch.bfloat16, device=dev)
        gm, bt = torch.ones(C, device=dev), torch.zeros(C, device=dev)
        st = torch.zeros(1, C // scpg, 2, dtype=torch.float64, device=dev)
        sums = torch.zeros(3, 1, C, dtype=torch.float64, device=dev)
        if which == "reduce":
            ops.gn_bwd_reduce(x, x, st, gm, bt, sums, 1, 8, C, G, scpg, EPS, True)
        else:
            ops.gn_bwd_apply(x, x, None, x.clone(), st, gm, bt, sums, 1, 8, C, G, scpg, EPS, True)

    with pytest.raises(MriError):
        run(520, 65, 8, "apply")          # gmean[2][64] in shared memory
    for which in ("reduce", "apply"):     # 12 channels per group: neither 4 nor a multiple of 8
        with pytest.raises(MriError):
            run(96, 8, 4, which)


@pytest.mark.gpu
def test_gn_bwd_reduce_65_groups(ops):
    """Pass A has no group limit (it works per channel): 65 groups of 8 reduce correctly."""
    dev, N, S, C, G = "cuda", 2, 33, 520, 65
    x, dy, gamma, beta = gn_inputs(N, S, C, G, dev, seed=13)
    stats = gn_stats_ref(x, 8).contiguous()
    sums = torch.zeros(3, N, C, dtype=torch.float64, device=dev)
    ops.gn_bwd_reduce(x, dy, stats, gamma, beta, sums, N, S, C, G, 8, EPS, True)
    _, ref = gn_bwd_autograd(x, dy, gamma, beta, G, True)
    for q in range(3):
        assert rel(sums[q], ref[q]) <= SUM_TOL[True], q


# ---------------------------------------------------------------- 2. softmax backward
def _softmax_case(rows, cols, ld_p, ld_dp, scale, dev, seed):
    g = torch.Generator().manual_seed(seed)
    logits = 2 * torch.randn(rows, cols, generator=g, dtype=torch.float64)
    Pv = bf16(torch.softmax(scale * logits, -1))
    dPv = (4 * torch.randn(rows, 1, generator=g) + torch.randn(rows, cols, generator=g)).float()
    P = nan_like((rows, ld_p), torch.bfloat16, "cpu")
    P[:, :cols] = Pv
    dP = nan_like((rows, ld_dp), torch.float32, "cpu")
    dP[:, :cols] = dPv
    pd, dpd = Pv.double(), dPv.double()
    ref = scale * pd * (dpd - (pd * dpd).sum(-1, keepdim=True))
    return P.to(dev), dP.to(dev), ref.to(dev)


def _check_softmax_rows(dS, ref, cols, scale, dP):
    assert (dS[:, cols:].float() == 0).all(), "padding columns of dS must be written as 0"
    out = dS[:, :cols].double()
    err = (out - ref).norm(dim=1)
    atol = 1e-6 * scale * dP[:, :cols].double().abs().amax(1)
    row_rel = err / ref.norm(dim=1).clamp_min(1e-300)
    worst = int(torch.argmax(torch.where(err <= atol, torch.zeros_like(row_rel), row_rel)))
    ok = err <= SM_TOL * ref.norm(dim=1) + atol
    note("softmax_bwd row rel-L2", torch.where(err <= atol, torch.zeros_like(row_rel), row_rel).max())
    assert ok.all(), f"{int((~ok).sum())} bad rows; worst row {worst} rel-L2 {row_rel[worst]:.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("cols", SOFTMAX_COLS)
@pytest.mark.parametrize("rows", [1, 7, 9])
def test_softmax_bwd(ops, rows, cols):
    dev, scale = "cuda", 0.125
    ld_p = (cols + 7) // 8 * 8
    for ld_dp in (ld_p, cols + 3):        # the engine's layout, and a dP stride of its own
        P, dP, ref = _softmax_case(rows, cols, ld_p, ld_dp, scale, dev, seed=rows * 4096 + cols)
        dS = nan_like((rows, ld_p), torch.bfloat16, dev)
        ops.softmax_bwd(P, dP, dS, rows, cols, ld_p, ld_dp, scale)
        _check_softmax_rows(dS, ref, cols, scale, dP)


@pytest.mark.gpu
def test_softmax_bwd_real_layer_and_wide_stride(ops):
    """cfg5's mid attention (B 2, 4 heads, 40x48x40 latent at two down-samplings = 1200 tokens),
    and ld_p beyond cols rounded up to 8: the extra padding columns come back as 0."""
    dev = "cuda"
    rows, cols = 2 * 4 * 1200, 1200
    scale = 1 / math.sqrt(128)
    P, dP, ref = _softmax_case(rows, cols, 1200, 1200, scale, dev, seed=5)
    dS = nan_like((rows, 1200), torch.bfloat16, dev)
    ops.softmax_bwd(P, dP, dS, rows, cols, 1200, 1200, scale)
    _check_softmax_rows(dS, ref, cols, scale, dP)
    for cols, ld_p in ((150, 200), (250, 264), (1281, 1320)):
        P, dP, ref = _softmax_case(9, cols, ld_p, cols + 1, 0.5, dev, seed=cols)
        dS = nan_like((9, ld_p), torch.bfloat16, dev)
        ops.softmax_bwd(P, dP, dS, 9, cols, ld_p, cols + 1, 0.5)
        _check_softmax_rows(dS, ref, cols, 0.5, dP)


@pytest.mark.gpu
def test_softmax_bwd_rejects_wide_rows(ops):
    P = torch.zeros(1, 2056, dtype=torch.bfloat16, device="cuda")
    dP = torch.zeros(1, 2056, device="cuda")
    with pytest.raises(_mri_error()):
        ops.softmax_bwd(P, dP, P.clone(), 1, 2050, 2056, 2056, 1.0)


# ---------------------------------------------------------------- 3. linear_bwd, silu, silu_bwd
LINEAR_SHAPES = [
    (64, 256), (256, 64), (64, 2304),          # 3D test model (time_emb_dim 64): time MLP, projections
    (256, 1024), (1024, 256), (256, 4608),     # cfg5 UNet3DModelWithAttention(base 128, t_dim 256)
    (1, 1024), (256, 3712),                    # 2D / 2.5D UNet: slice MLP input, block projections
    (1, 1), (257, 65), (256, 129),             # ragged 64-wide chunks and 256-wide tiles
]


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [1, 8, 64])
@pytest.mark.parametrize("in_f,out_f", LINEAR_SHAPES)
def test_linear_bwd(ops, in_f, out_f, batch):
    dev = "cuda"
    g = torch.Generator().manual_seed(in_f * 7 + out_f + batch)
    dZ = torch.randn(batch, out_f, generator=g).to(dev)
    X = torch.randn(batch, in_f, generator=g).to(dev)
    W = (0.05 * torch.randn(out_f, in_f, generator=g)).to(dev)
    dZd, Xd, Wd = dZ.double(), X.double(), W.double()
    u = 2.0 ** -24
    k_dx = 64 + -(-out_f // 64) + 1
    bound_dx = k_dx * u * (dZd.abs() @ Wd.abs())
    bound_dw = (batch + 1) * u * (dZd.abs().t() @ Xd.abs())
    bound_db = (batch + 1) * u * dZd.abs().sum(0)

    def check(t, ref, bound, what):
        e = (t.double() - ref).abs()
        note("linear_bwd |err| / summation bound", (e / (bound + 1e-300)).max())
        assert torch.isfinite(t).all() and (e <= bound + 1e-300).all(), \
            f"{what}: worst |err| / bound {(e / (bound + 1e-300)).max():.3e}"

    # (dX, dW, db): block projections and the second time-MLP layer
    dX, dW, db = (nan_like(s, torch.float32, dev) for s in ((batch, in_f), (out_f, in_f), (out_f,)))
    ops.linear_bwd(dZ, X, W, dX, dW, db)
    check(dX, dZd @ Wd, bound_dx, "dX")
    check(dW, dZd.t() @ Xd, bound_dw, "dW")
    check(db, dZd.sum(0), bound_db, "db")
    # (None, dW, db): the first time-MLP layer
    dW, db = nan_like((out_f, in_f), torch.float32, dev), nan_like((out_f,), torch.float32, dev)
    ops.linear_bwd(dZ, X, W, None, dW, db)
    check(dW, dZd.t() @ Xd, bound_dw, "dW")
    check(db, dZd.sum(0), bound_db, "db")
    # dW without db: nothing is written past dW
    buf = nan_like((out_f * in_f + out_f,), torch.float32, dev)
    dW = buf[:out_f * in_f].view(out_f, in_f)
    ops.linear_bwd(dZ, X, W, None, dW, None)
    check(dW, dZd.t() @ Xd, bound_dw, "dW")
    assert torch.isnan(buf[out_f * in_f:]).all()


def _silu_inputs(n):
    special = [0.0, 1e-30, -1e-30, 1e-40, -1e-40, 1e-45, -1e-45, 88.8, -88.8, 88.7, -88.7, 87.0,
               -87.0, 100.0, -100.0, 16.6, -1.2785, 1.0, -1.0]
    if n == 1:
        return torch.tensor([-1.5])
    z = torch.cat([torch.tensor(special), torch.linspace(-100, 100, n - len(special))])
    return z.float()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 1531])
def test_silu_and_silu_bwd(ops, n):
    dev = "cuda"
    z = _silu_inputs(n).to(dev)
    dy = torch.randn(n, generator=torch.Generator().manual_seed(n)).to(dev)
    y = nan_like((n,), torch.float32, dev)
    dz = nan_like((n,), torch.float32, dev)
    ops.silu(z, y)
    ops.silu_bwd(z, dy, dz)
    zd, dyd = z.double(), dy.double()
    sg = torch.sigmoid(zd)
    ref_y = zd * sg
    ref_dz = dyd * sg * (1 + zd * (1 - sg))
    mag_dz = dyd.abs() * sg * (1 + zd.abs() * (1 - sg))
    assert torch.isfinite(y).all() and torch.isfinite(dz).all()
    ey = (y.double() - ref_y).abs()
    edz = (dz.double() - ref_dz).abs()
    note("silu |err| / (|y| ulp)", (ey / (2.0 ** -24 * ref_y.abs() + 1e-36)).max())
    note("silu_bwd |err| / (2^-24 term magnitude)", (edz / (2.0 ** -24 * mag_dz + 1e-36)).max())
    ok_y = ey <= 8 * 2.0 ** -24 * ref_y.abs() + 1e-36
    ok_dz = edz <= 2.0 ** -18 * mag_dz + 1e-36
    assert ok_y.all(), list(zip(z[~ok_y].tolist(), y[~ok_y].tolist(), ref_y[~ok_y].tolist()))[:8]
    assert ok_dz.all(), list(zip(z[~ok_dz].tolist(), dz[~ok_dz].tolist(), ref_dz[~ok_dz].tolist()))[:8]


# ---------------------------------------------------------------- 4. min-SNR loss
@pytest.mark.gpu
@pytest.mark.parametrize("sched", ["linear", "cosine"])
@pytest.mark.parametrize("gamma", [5.0, 0.0])
@pytest.mark.parametrize("B,P", [(1, 1), (3, 7), (8, 3 * 40 * 48 * 40), (2, 400_003)])
def test_minsnr_loss_and_grad(ops, B, P, gamma, sched):
    """(2, 400003): per-sample size beyond loss_bwd_kernel's grid cap (1184 / B blocks of 256)."""
    from oracle import reference_oracle as O
    dev, T = "cuda", 1000
    betas = O.linear_betas(T) if sched == "linear" else O.cosine_betas(T)
    snr = O.schedule_buffers(betas)["snr"]
    g = torch.Generator().manual_seed(B * 31 + P)
    pred = torch.randn(B, P, generator=g)
    noise = torch.randn(B, P, generator=g)
    t = torch.tensor(([0, 1, T - 1] + torch.randint(0, T, (B,), generator=g).tolist())[:B] if B > 1
                     else [T - 1])
    pd = pred.double().requires_grad_(True)
    if gamma > 0:
        loss_ref = O.minsnr_loss({"snr": snr.double()}, pd, noise.double(), t, gamma)
    else:
        loss_ref = O.mse_loss(pd, noise.double())
    (grad_ref,) = torch.autograd.grad(loss_ref, pd)
    mse_ref = ((pred.double() - noise.double()) ** 2).mean(1)
    pred_c, noise_c, t_c, snr_c = pred.to(dev), noise.to(dev), t.to(dev), snr.to(dev)
    per = nan_like((B,), torch.float32, dev)
    loss = nan_like((1,), torch.float32, dev)
    ops.minsnr_loss(pred_c, noise_c, t_c, snr_c, gamma, per, loss)
    note("minsnr loss rel", abs(loss.item() - loss_ref.item()) / abs(loss_ref.item()))
    note("minsnr per-sample mse rel", ((per.cpu().double() - mse_ref).abs() / mse_ref).max())
    assert abs(loss.item() - loss_ref.item()) <= 1e-5 * abs(loss_ref.item())
    assert ((per.cpu().double() - mse_ref).abs() <= 1e-5 * mse_ref).all()
    for up in (1.0, 1.0 / B, 65536.0):
        dpred = nan_like((B, P), torch.float32, dev)
        upstream = torch.tensor([up], dtype=torch.float32, device=dev)
        ops.minsnr_loss_bwd(pred_c, noise_c, t_c, snr_c, gamma, upstream, dpred)
        want = float(torch.tensor(up, dtype=torch.float32)) * grad_ref.to(dev)
        err = (dpred.double() - want).abs()
        note("minsnr dpred rel", (err / want.abs().clamp_min(1e-300)).max())
        assert (err <= 4e-6 * want.abs()).all(), f"upstream {up}: worst rel {(err / want.abs()).max():.3e}"


# ---------------------------------------------------------------- 5. add_bf16, grad_finalize, copy_cast
@pytest.mark.gpu
@pytest.mark.parametrize("n", [8, 2048, 148 * 16 * 256 * 8 + 4104])
def test_add_bf16_bit_exact(ops, n):
    dev = "cuda"
    g = torch.Generator().manual_seed(n)
    a = bf16(torch.randn(n, generator=g) * 3).to(dev)
    b = bf16(torch.randn(n, generator=g)).to(dev)
    want = (a.float() + b.float()).bfloat16()
    out = nan_like((n,), torch.bfloat16, dev)
    ops.add_bf16(a, b, out)
    assert torch.equal(out.view(torch.int16), want.view(torch.int16))
    ops.add_bf16(a, b, a)                 # out is a: BackwardMixin.pass_grad
    assert torch.equal(a.view(torch.int16), want.view(torch.int16))


@pytest.mark.gpu
def test_add_bf16_rejects_ragged_length(ops):
    a = torch.zeros(12, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(_mri_error()):
        ops.add_bf16(a, a, a.clone())


@pytest.mark.gpu
def test_grad_finalize_one_launch(ops):
    """Gather segments (with -1 holes) and fp64 batch-sum segments in one table, one launch, built
    as BackwardMixin._final_table does; every dst sits between NaN guards that must survive."""
    from mri_image_generation_b200 import _lib
    dev = "cuda"
    g = torch.Generator().manual_seed(3)
    GUARD = 37
    keep, segs, blocks, checks = [], [], 0, []

    def dst_between_guards(n):
        buf = nan_like((n + 2 * GUARD,), torch.float32, dev)
        keep.append(buf)
        return buf, buf[GUARD:GUARD + n]

    def add_seg(dst, src, idx, batch, ld):
        nonlocal blocks
        sg = _lib.MriFinalSeg()
        sg.dst, sg.src = dst.data_ptr(), src.data_ptr()
        sg.idx = idx.data_ptr() if idx is not None else None
        sg.n, sg.block0, sg.batch, sg.ld = dst.numel(), blocks, batch, ld
        blocks += -(-dst.numel() // 2048)
        segs.append(sg)

    for n in (1, 2047, 2048, 2049, 100_000):
        m = n + 500
        src = torch.randn(m, generator=g).to(dev)
        idx = torch.randperm(m, generator=g)[:n].to(torch.int32)
        idx[torch.rand(n, generator=g) < 0.1] = -1
        if n > 1:
            idx[0], idx[-1] = -1, m - 1
        idx = idx.to(dev)
        buf, dst = dst_between_guards(n)
        keep += [src, idx]
        add_seg(dst, src, idx, 0, 0)
        want = torch.where(idx >= 0, src[idx.clamp_min(0).long()], torch.zeros_like(src[:1]))
        checks.append((f"gather n={n}", buf, n, want))
    for batch, n, ld in ((1, 3000, 3008), (3, 1, 64), (64, 2049, 2100), (3, 5000, 5001)):
        src = torch.randn(batch, ld, dtype=torch.float64, generator=g) * 10
        src[:, n:] = float("nan")         # columns past n are never read
        acc = torch.zeros(n, dtype=torch.float64)
        for b in range(batch):            # the kernel's order: b = 0, 1, ... in fp64
            acc = acc + src[b, :n]
        src = src.to(dev)
        buf, dst = dst_between_guards(n)
        keep.append(src)
        add_seg(dst, src, None, batch, ld)
        checks.append((f"batch-sum batch={batch} n={n}", buf, n, acc.float().to(dev)))

    arr = (_lib.MriFinalSeg * len(segs))(*segs)
    table = torch.frombuffer(bytearray(bytes(memoryview(arr))), dtype=torch.uint8).to(dev)
    _lib.check(_lib.load().mri_grad_finalize(table.data_ptr(), len(segs), blocks,
                                             _lib.current_stream_ptr()), "mri_grad_finalize")
    torch.cuda.synchronize()
    for what, buf, n, want in checks:
        got = buf[GUARD:GUARD + n]
        assert torch.equal(got, want), what
        assert torch.isnan(buf[:GUARD]).all() and torch.isnan(buf[GUARD + n:]).all(), what


@pytest.mark.gpu
def test_copy_cast_fp64_into_column_window(ops):
    """_bwd_bias_and_tproj / bwd_gn: dtproj[:, off:off + C] <- the fp64 column sums [B, C]."""
    dev = "cuda"
    g = torch.Generator().manual_seed(4)
    for B, C, W, off in ((2, 256, 2304, 512), (8, 128, 4608, 4480), (1, 64, 200, 0)):
        src = (torch.randn(B, C, dtype=torch.float64, generator=g) * 1e3).to(dev)
        dst = nan_like((B, W), torch.float32, dev)
        ops.copy_cast(src, dst[:, off:off + C])
        assert torch.equal(dst[:, off:off + C], src.float())
        assert torch.isnan(dst[:, :off]).all() and torch.isnan(dst[:, off + C:]).all()


# ---------------------------------------------------------------- 6. coverage guard
@pytest.mark.gpu
def test_parametrization_covers_what_the_models_run(ops):
    """Every GroupNorm and attention-softmax shape the training programs of the test-size models
    record is in the parametrization above; the full-size cfg4 / cfg5 UNet's GroupNorm widths
    (read off its constructor on the meta device) too."""
    import contextlib
    import io
    from mri_image_generation_b200.backward import AttnRec, GnRec
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet import UNet3DModel
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.vae import VAE3D
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet as UNet2D
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.unet import UNet as UNet25D

    gn_cover = {(C, G, s, silu) for (C, G, s) in GN_CONFIGS for silu in (True, False)}
    sm_class = lambda ld: 8 if ld <= 256 else (40 if ld <= 1280 else 64)   # mri_softmax_bwd
    sm_cover = {sm_class((c + 7) // 8 * 8) for c in SOFTMAX_COLS}
    dev = "cuda"
    progs = []
    with contextlib.redirect_stdout(io.StringIO()):
        progs.append(UNet3DModelWithAttention(3, base_channels=64, time_emb_dim=64).to(dev)
                     .program(2, (8, 8, 8), training=True))
        progs.append(UNet3DModel(3, base_channels=64, time_emb_dim=64).to(dev)
                     .program(1, (8, 12, 8), training=True))
        progs.append(UNet2D(img_channels=1, base_channels=64, time_emb_dim=64).to(dev)
                     .program(2, (32, 32), 1, 0, training=True))
        progs.append(UNet25D(in_channels=20, out_channels=4, base_channels=64, time_emb_dim=64).to(dev)
                     .program(2, (32, 32), 4, 16, training=True))
        vae = VAE3D(in_channels=4, base_channels=32, num_down=3, latent_channels=16).to(dev)
        progs.append(vae._program("encode", torch.zeros(2, 4, 16, 24, 16, device=dev), training=True))
        progs.append(vae._program("decode", torch.zeros(2, 16, 4, 6, 4, device=dev), training=True))
    missing, seen = set(), set()
    for prog in progs:
        for r in prog.tape:
            if isinstance(r, GnRec):
                key = (r.x.C, r.groups, r.x.cpg, bool(r.silu))
                seen.add(key)
                if key not in gn_cover:
                    missing.add(("gn",) + key)
            elif isinstance(r, AttnRec):
                seen.add(("attn", r.npad))
                if sm_class(r.npad) not in sm_cover:
                    missing.add(("attn", r.npad))
    print("recorded:", sorted(seen, key=str))
    assert any(isinstance(k[0], int) for k in seen)
    pairs = {(C, G) for (C, G, _) in GN_CONFIGS}
    with torch.device("meta"):
        big = UNet3DModelWithAttention(3, base_channels=128, channel_mults=(1, 2, 4), time_emb_dim=256)
    for m in big.modules():
        if isinstance(m, torch.nn.GroupNorm):
            C, G = m.num_channels, m.num_groups
            # a norm over a concatenation [x, skip] runs as GN(G / 2) over each half
            if (C, G) not in pairs and (C // 2, G // 2) not in pairs:
                missing.add(("cfg5 GroupNorm", C, G))
    assert not missing, sorted(missing, key=str)
