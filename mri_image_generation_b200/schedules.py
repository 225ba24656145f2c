"""Noise schedules and the registered buffers of the diffusion wrappers (host logic, fp32 on
the CPU exactly as the reference builds them, then moved with the module).

linear:  slice_cond_2d_ddpm/diffusion.py:23-49, ddpm_25d_all_modalities/diffusion.py:22-47
cosine:  ddpm_3d_ldm/diffusion.py:23-56
These must stay bit-identical to the reference (checkpoints carry them; metrics.py:291-294
infers `timesteps` from betas.numel()), which tests/test_oracle_golden.py and tests/test_host_api.py check against
tests/golden/schedules.pt.
"""
import math
import numbers
from collections import OrderedDict

import torch


def linear_beta_schedule(timesteps: int, beta_start: float, beta_end: float) -> torch.Tensor:
    return torch.linspace(beta_start, beta_end, timesteps, dtype=torch.float32)


def cosine_beta_schedule(timesteps: int, s: float = 0.008) -> torch.Tensor:
    steps = timesteps + 1
    x = torch.linspace(0, timesteps, steps, dtype=torch.float32)
    alphas_cumprod = torch.cos(((x / timesteps) + s) / (1 + s) * math.pi * 0.5) ** 2
    alphas_cumprod = alphas_cumprod / alphas_cumprod[0]
    betas = 1 - (alphas_cumprod[1:] / alphas_cumprod[:-1])
    return torch.clamp(betas, 1e-8, 0.999)


def make_buffers(betas: torch.Tensor, with_snr: bool) -> "OrderedDict[str, torch.Tensor]":
    """Buffers in the reference's registration order (state_dict key order)."""
    alphas = 1.0 - betas
    alphas_cumprod = torch.cumprod(alphas, dim=0)
    alphas_cumprod_prev = torch.cat(
        [torch.tensor([1.0], dtype=torch.float32), alphas_cumprod[:-1]], dim=0)
    out = OrderedDict()
    out["betas"] = betas
    out["alphas"] = alphas
    out["alphas_cumprod"] = alphas_cumprod
    out["alphas_cumprod_prev"] = alphas_cumprod_prev
    out["sqrt_alphas_cumprod"] = torch.sqrt(alphas_cumprod)
    out["sqrt_one_minus_alphas_cumprod"] = torch.sqrt(1.0 - alphas_cumprod)
    out["sqrt_recip_alphas"] = torch.sqrt(1.0 / alphas)
    if with_snr:
        out["snr"] = alphas_cumprod / (1.0 - alphas_cumprod)
    posterior_variance = betas * (1.0 - alphas_cumprod_prev) / (1.0 - alphas_cumprod)
    out["posterior_variance"] = posterior_variance
    out["posterior_log_variance_clipped"] = torch.log(torch.clamp(posterior_variance, min=1e-20))
    return out


def dpmpp_timesteps(start_t: int, num_steps: int) -> list:
    """The points DPM-Solver++(2M) visits: round(linspace(start_t, 0, M + 1))[:-1] in integer
    arithmetic (halves round up), then -1 for sigma = 0.  With start_t = T - 1 this is the
    "linspace" timestep spacing of diffusers' multistep scheduler.  Needs 1 <= M <= start_t, which
    keeps the UNet timesteps distinct and >= 1."""
    M, s = int(num_steps), int(start_t)
    if not 1 <= M <= s:
        raise ValueError(f"need 1 <= num_steps <= start_t (got num_steps={M}, start_t={s})")
    return [(2 * s * (M - i) + M) // (2 * M) for i in range(M)] + [-1]


def repaint_levels(timesteps: int, jump_length: int, jump_n_sample: int) -> list:
    """The noise levels RePaint's resampling visits, one timestep per training step (the jump rule
    of diffusers' RePaintScheduler).  Level l means x ~ q_sample(x0, l); -1 means clean.  The list
    starts at T - 1, ends at -1 and moves by exactly 1: l -> l - 1 is a reverse step at t = l,
    l -> l + 1 an undo step (one step of forward noising).  After the reverse step at each jump
    point j in range(0, T - L, L), the sampler jumps back up L levels, r - 1 times in all, and
    each time walks down again: T + (r - 1) L P reverse and (r - 1) L P undo steps,
    P = len(range(0, T - L, L)).  r = 1, or L >= T, gives [T - 1, ..., 0, -1]."""
    T, L, r = timesteps, jump_length, jump_n_sample
    for name, v in (("timesteps", T), ("jump_length", L), ("jump_n_sample", r)):
        if isinstance(v, bool) or not isinstance(v, numbers.Integral) or v < 1:
            raise ValueError(f"{name} must be an integer >= 1 (got {v!r})")
    T, L, r = int(T), int(L), int(r)
    jumps = {j: r - 1 for j in range(0, T - L, L)}
    levels, t = [T - 1], T - 1
    while t >= 0:
        j = t
        t -= 1
        levels.append(t)
        if jumps.get(j, 0) > 0:
            jumps[j] -= 1
            levels.extend(range(t + 1, t + L + 1))
            t += L
    return levels


def dpmpp_2m_table(alphas_cumprod: torch.Tensor, timesteps):
    """DPM-Solver++(2M) (data prediction, midpoint second-order form) over the visited points
    t_0 > t_1 > ... > t_M; a final -1 means sigma = 0.  Returns (ts, coef): the M timesteps the
    UNet is evaluated at (int64) and one fp32 row (s, r, A, B, C) per step, for the update

        x0 = (x - s * eps) * r ;  x <- (A * x + B * x0) + C * (x0 - x0_prev)

    computed in fp64 from the fp32 alphas_cumprod and rounded once.  Row 0 is first order (C = 0);
    a step to sigma = 0 is first order and returns x0 (A, B, C = 0, 1, 0)."""
    ac = [float(v) for v in alphas_cumprod.detach().cpu().double().tolist()]
    T = len(ac)
    ts = [int(v) for v in timesteps]
    if len(ts) < 2:
        raise ValueError("DPM-Solver++ needs at least two timesteps")
    for i, t in enumerate(ts):
        if not (0 <= t <= T - 1 or (t == -1 and i == len(ts) - 1)):
            raise ValueError(f"timestep {t} outside [0, {T - 1}] (only the last may be -1)")
    if any(a <= b for a, b in zip(ts, ts[1:])):
        raise ValueError(f"timesteps must be strictly decreasing: {ts}")
    M = len(ts) - 1
    alpha = [math.sqrt(ac[t]) if t >= 0 else 1.0 for t in ts]
    sigma = [math.sqrt(1.0 - ac[t]) if t >= 0 else 0.0 for t in ts]
    lam = [math.log(alpha[i]) - math.log(sigma[i]) if ts[i] >= 0 else math.inf for i in range(M + 1)]
    rows = []
    for i in range(M):
        s, r = sigma[i], 1.0 / alpha[i]
        if ts[i + 1] < 0:
            rows.append((s, r, 0.0, 1.0, 0.0))
            continue
        h = lam[i + 1] - lam[i]
        phi = math.expm1(-h)
        A, B = sigma[i + 1] / sigma[i], -alpha[i + 1] * phi
        C = 0.0
        if i > 0:
            rho = (lam[i] - lam[i - 1]) / h
            C = -0.5 * alpha[i + 1] * phi / rho
        rows.append((s, r, A, B, C))
    return (torch.tensor(ts[:M], dtype=torch.int64),
            torch.tensor(rows, dtype=torch.float64).to(torch.float32))
