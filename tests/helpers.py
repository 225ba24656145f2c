"""Shared test helpers (tests only)."""
import hashlib
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def synthetic_state_dict(shapes, seed: int):
    """Must match oracle/make_golden.py::synthetic_state_dict."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, shp in shapes:
        w = torch.randn(*shp, generator=g) * 0.05
        if ("norm" in k) and k.endswith(".weight"):
            w = w + 1.0
        sd[k] = w
    return sd


def shapes_of(module):
    return [(k, tuple(v.shape)) for k, v in module.state_dict().items()]


def rel_l2(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def load_gold(name):
    return torch.load(os.path.join(GOLD, name), weights_only=False)


def sha16(t: torch.Tensor) -> str:
    return hashlib.sha256(t.numpy().tobytes()).hexdigest()[:16]


def float32_ulp(x: torch.Tensor) -> torch.Tensor:
    """Spacing of the float32 grid at |x| (float64)."""
    a = x.float().abs()
    return (torch.nextafter(a, torch.tensor(math.inf)) - a).double()


# torch's CPU sqrt and log kernels round faithfully but not correctly: which of the two float32
# neighbours of the exact result they return differs between torch builds.  Schedule buffers made
# with them are checked against the float64 value of the same formula; all others bit for bit.
LIBM_BUFFERS = {
    "sqrt_alphas_cumprod": lambda b: b["alphas_cumprod"].double().sqrt(),
    "sqrt_one_minus_alphas_cumprod": lambda b: (1.0 - b["alphas_cumprod"]).double().sqrt(),
    "sqrt_recip_alphas": lambda b: (1.0 / b["alphas"]).double().sqrt(),
    "posterior_log_variance_clipped": lambda b: b["posterior_variance"].clamp(min=1e-20).double().log(),
}


def check_schedule_against_gold(bufs, gold):
    """Diffusion buffers against the reference's (an entry of tests/golden/schedules.pt): the
    arithmetic-only buffers hash-identical, the sqrt / log ones within one float32 ulp of the exact
    result on those (hash-checked) inputs and of the reference's first and last values."""
    assert list(bufs) == list(gold["sha"])
    for k, v in bufs.items():
        if k not in LIBM_BUFFERS:
            assert sha16(v) == gold["sha"][k], k
            continue
        exact = LIBM_BUFFERS[k](bufs)
        ulp = float32_ulp(exact)
        assert ((v.double() - exact).abs() <= ulp).all(), k
        first, last = gold["first_last"][k]
        assert abs(v[0].item() - first) <= ulp[0].item() and abs(v[-1].item() - last) <= ulp[-1].item(), k
