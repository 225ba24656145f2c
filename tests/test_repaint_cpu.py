"""RePaint resampling without a GPU: schedules.repaint_levels against a restatement of diffusers'
RePaintScheduler loop and its counting properties, argument checks (ValueError before x_T is
drawn), and the fp64 conditioning check of test_inpaint_cpu.py with resampling.

Measured (cosine T = 1000, B = 32, n = 1024, a = 1, d = 0.1, same x_T and generator seeds), error
of the regenerated half's mean against the posterior mean:
  replacement (inpaint today):        0.01459, ratio 91.3
  RePaint, jump_length 10, n_sample 2: 0.00795, ratio 167.5   (test: >= 120 and below replacement)
"""
import math

import pytest
import torch

from mri_image_generation_b200 import schedules
from test_inpaint_cpu import _diffusions, _SHAPE, _buffers, corr_eps, ddpm_loop, gaussian_problem, \
    region_error

T = 1000


def diffusers_levels(T, L, r):
    """diffusers' RePaintScheduler.set_timesteps with one timestep per training step, mapped to
    levels: the list holds the timestep of every move, and after the move at t the state is at
    level t - 1 (a reverse step at t lands there, and so does an undo from t - 1)."""
    jumps = {}
    for j in range(0, T - L, L):
        jumps[j] = r - 1
    ts, t = [], T
    while t >= 1:
        t = t - 1
        ts.append(t)
        if jumps.get(t, 0) > 0:
            jumps[t] = jumps[t] - 1
            for _ in range(L):
                t = t + 1
                ts.append(t)
    return [T - 1] + [t - 1 for t in ts]


CASES = [(1000, 10, 2), (1000, 10, 10), (1000, 10, 5), (12, 3, 3), (12, 1, 2), (12, 11, 2),
         (12, 12, 3), (12, 20, 4), (12, 5, 1), (7, 2, 3), (2, 1, 3), (1, 1, 2), (3, 2, 2)]


@pytest.mark.parametrize("T_, L, r", CASES)
def test_levels_match_the_scheduler_restatement(T_, L, r):
    assert schedules.repaint_levels(T_, L, r) == diffusers_levels(T_, L, r)


@pytest.mark.parametrize("T_, L, r", CASES)
def test_levels_properties(T_, L, r):
    lv = schedules.repaint_levels(T_, L, r)
    assert lv[0] == T_ - 1 and lv[-1] == -1
    assert all(abs(b - a) == 1 for a, b in zip(lv, lv[1:]))
    assert min(lv) == -1 and max(lv) == T_ - 1
    P = len(range(0, T_ - L, L))
    n_rev = sum(b < a for a, b in zip(lv, lv[1:]))
    n_undo = sum(b > a for a, b in zip(lv, lv[1:]))
    assert n_rev == T_ + (r - 1) * L * P
    assert n_undo == (r - 1) * L * P
    # an undo from level l reads alphas / betas[l + 1]: inside the table
    assert all(a <= T_ - 2 for a, b in zip(lv, lv[1:]) if b > a)
    if r == 1 or L >= T_:
        assert lv == list(range(T_ - 1, -2, -1))


def test_levels_counts_of_the_documented_settings():
    for r, calls in ((2, 1990), (5, 4960), (10, 9910)):
        lv = schedules.repaint_levels(1000, 10, r)
        assert sum(b < a for a, b in zip(lv, lv[1:])) == calls


@pytest.mark.parametrize("bad", [0, -1, 2.5, "10", None, True, 10.0])
def test_levels_reject_non_integers_and_values_below_one(bad):
    with pytest.raises(ValueError):
        schedules.repaint_levels(12, bad, 2)
    with pytest.raises(ValueError):
        schedules.repaint_levels(12, 3, bad)


# ------------------------------------------------------------------------------------ conditioning
def repaint_loop(buf, x_T, g, known, mask, levels):
    """fp64 restatement of the RePaint walk: a move l -> l - 1 is ddpm_loop's replacement step at
    i = l, a move l -> l + 1 is x = sqrt(alphas[l + 1]) x + sqrt(betas[l + 1]) z."""
    x = x_T.clone()
    for lv, nxt in zip(levels, levels[1:]):
        if nxt < lv:
            i = lv
            eps = corr_eps(x, buf["alphas_cumprod"][i])
            z = torch.randn(x.shape, generator=g, dtype=torch.float64)
            w = math.sqrt(buf["posterior_variance"][i]) if i > 0 else 0.0
            x = buf["sqrt_recip_alphas"][i] * (x - buf["betas"][i] / buf["sqrt_one_minus_alphas_cumprod"][i] * eps) + w * z
            nz = torch.randn(x.shape, generator=g, dtype=torch.float64)
            kn = known if i == 0 else (buf["sqrt_alphas_cumprod"][i - 1] * known
                                       + buf["sqrt_one_minus_alphas_cumprod"][i - 1] * nz)
            x = torch.where(mask, x, kn)
        else:
            z = torch.randn(x.shape, generator=g, dtype=torch.float64)
            x = buf["alphas"][lv + 1].sqrt() * x + buf["betas"][lv + 1].sqrt() * z
    return x


def test_repaint_conditions_more_strongly_than_replacement():
    buf = _buffers()
    known, mask, post = gaussian_problem(32, 1024, 0)
    x_T = torch.randn(known.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    free = ddpm_loop(buf, x_T, torch.Generator().manual_seed(2))
    repl = ddpm_loop(buf, x_T, torch.Generator().manual_seed(2), known, mask)
    plain = repaint_loop(buf, x_T, torch.Generator().manual_seed(2), known, mask,
                         schedules.repaint_levels(T, 10, 1))
    assert torch.equal(plain, repl)          # jump_n_sample = 1 is replacement
    rp = repaint_loop(buf, x_T, torch.Generator().manual_seed(2), known, mask,
                      schedules.repaint_levels(T, 10, 2))
    assert torch.equal(rp[~mask], known[~mask])
    e_free, e_repl, e_rp = (region_error(v, mask, post) for v in (free, repl, rp))
    print(f"unconditional {e_free:.4g}, replacement {e_repl:.4g} (ratio {e_free / e_repl:.1f}), "
          f"RePaint 10/2 {e_rp:.4g} (ratio {e_free / e_rp:.1f})")
    assert e_rp < e_repl
    assert e_free / e_rp >= 120


# ------------------------------------------------------------------------------------ argument checks
_BAD_JUMPS = [dict(jump_length=0, jump_n_sample=2), dict(jump_length=-3, jump_n_sample=2),
              dict(jump_length=2.5, jump_n_sample=2), dict(jump_length="10", jump_n_sample=2),
              dict(jump_length=None, jump_n_sample=2), dict(jump_length=10, jump_n_sample=0),
              dict(jump_length=10, jump_n_sample=-1), dict(jump_length=10, jump_n_sample=1.5),
              dict(jump_length=10, jump_n_sample=True), dict(jump_length=0, jump_n_sample=1)]


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
@pytest.mark.parametrize("bad", range(len(_BAD_JUMPS)))
def test_bad_jump_arguments_raise_before_any_draw(kind, bad):
    """ValueError, not the MriError these CPU objects raise when they draw x_T: the check comes
    first (tests/test_gpu_repaint.py checks that the CUDA generator is left untouched)."""
    d = _diffusions()[kind]
    with pytest.raises(ValueError):
        d.inpaint(torch.zeros(_SHAPE[kind]), torch.ones(1, dtype=torch.bool), **_BAD_JUMPS[bad])


@pytest.mark.parametrize("kind", ["3d", "2d", "25d"])
def test_valid_jump_arguments_on_cpu_raise_mri_error(kind):
    from mri_image_generation_b200 import _lib
    d = _diffusions()[kind]
    for kw in (dict(jump_length=10, jump_n_sample=2), dict(jump_length=3, jump_n_sample=1),
               dict(jump_length=100, jump_n_sample=5)):
        with pytest.raises(_lib.MriError):
            d.inpaint(torch.zeros(_SHAPE[kind]), torch.ones(1, dtype=torch.bool), **kw)
