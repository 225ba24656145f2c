#!/usr/bin/env python
"""Cost of the variational-bound evaluation (GPU only): ms per replay of the 'vb' step graph
(q_sample with the noise drawn in-kernel, the UNet, mri_vb_terms, step_advance) against the 'ddpm'
reverse-step graph on the same program, and end to end for calc_bpd_loop at T = 1000.

  cfg4  ddpm_3d_ldm         UNet3DModelWithAttention(3, base 128, mults 1-2-4) B=16 3x40x48x40
  cfg2  slice_cond_2d_ddpm  UNet(1, base 64, mults 1-2-4-8)                   B=64 1x240x240

Each step time is CUDA events around STEPS replays of one captured step graph (after warm-up
replays); the two graphs are timed in turn, REPS times alternating, and the median and the spread
((max - min) / median) are reported, with the vb / ddpm ratio run by run.  End to end is CUDA
events around the public call (T = 1000 replays, the fp64 finalisation), once for the first call
(which captures the 'vb' graph) and E2E_REPS times after.  Random-init weights: this measures the cost
of the evaluation only.  GPU name and power limit are read with a read-only nvidia-smi query in the
same run.

  python tools/likelihood_bench.py [--out profiles/<name>.json] [--steps 20] [--reps 3] [--e2e-reps 2]
"""
import argparse
import contextlib
import io
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from sampler_bench import events_ms, gpu_info, summary  # noqa: E402

T = 1000


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def step_times(diff, prog, x, steps, reps, warm=3):
    """ms per replay of the 'vb' and 'ddpm' step graphs on `prog` (both already captured)."""
    g = {k: prog._step_graphs[k][2] for k in ("vb", "ddpm")}
    rng = diff._rng(x.device)

    def reset(key):
        prog.t_in.fill_(T - 1)
        if key == "vb":
            prog._vb_bufs["x0"].copy_(x)
        else:
            prog.x_in.copy_(x)
        rng.load()

    def replays(key, n):
        for _ in range(n):
            g[key].replay()

    for key in g:
        reset(key)
        replays(key, warm)
    out = {k: [] for k in g}
    for _ in range(reps):
        for key in g:
            reset(key)
            out[key].append(events_ms(lambda: replays(key, steps)) / steps)
    res = {k: summary(v) for k, v in out.items()}
    res["vb_over_ddpm"] = summary([a / b for a, b in zip(out["vb"], out["ddpm"])])
    return res


def measure(diff, prog, x, bpd, steps, reps, e2e_reps):
    """Capture both graphs (the first calc_bpd_loop is timed: it includes the capture), time the
    replays, then calc_bpd_loop end to end."""
    out = {}
    call = lambda: out.update(bpd(x))
    first = events_ms(call)
    diff._reverse_loop(prog, x, T - 1, 3, "ddpm")
    r = {"ms_per_step": step_times(diff, prog, x, steps, reps)}
    e2e = summary([events_ms(call) for _ in range(e2e_reps)])
    e2e["first_call_ms"] = first
    e2e["samples_per_s"] = x.shape[0] / (e2e["median"] / 1e3)
    r["calc_bpd_loop_ms"] = e2e
    assert torch.isfinite(out["total_bpd"]).all()
    r["total_bpd_mean"] = float(out["total_bpd"].mean())
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--e2e-reps", type=int, default=2)
    ap.add_argument("--b4", type=int, default=16)
    ap.add_argument("--b2", type=int, default=64)
    args = ap.parse_args()
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet

    _lib.require_device()
    dev = torch.device("cuda", torch.cuda.current_device())
    res = {"gpu": gpu_info(dev.index), "timesteps": T, "steps_per_timing": args.steps, "reps": args.reps,
           "note": "evaluation cost only (random-init weights)"}
    with torch.no_grad():
        # ---- cfg4 ---------------------------------------------------------------------------------
        B, shape = args.b4, (40, 48, 40)
        torch.manual_seed(0)
        m = UNet3DModelWithAttention(in_channels=3, base_channels=128, channel_mults=(1, 2, 4),
                                     time_emb_dim=256, groups=8, num_heads=4).to(dev).eval()
        d = quiet(GaussianDiffusionLatent3D, m, 3, timesteps=T).to(dev)
        x = torch.randn(B, 3, *shape, device=dev)
        prog = m.program(B, shape)
        r = {"batch": B, "shape": [3, *shape]}
        r.update(measure(d, prog, x, d.calc_bpd_loop, args.steps, args.reps, args.e2e_reps))
        res["cfg4"] = r
        del m, d, x, prog
        torch.cuda.empty_cache()
        # ---- cfg2 ---------------------------------------------------------------------------------
        B, S = args.b2, 240
        torch.manual_seed(0)
        m = quiet(UNet, img_channels=1, base_channels=64, channel_mults=(1, 2, 4, 8),
                  time_emb_dim=256).to(dev).eval()
        d = quiet(GaussianDiffusion, m, S, channels=1, timesteps=T).to(dev)
        z = torch.rand(B, device=dev)
        x = torch.rand(B, 1, S, S, device=dev) * 2 - 1
        prog = m.program(B, (S, S), 1, 0)
        r = {"batch": B, "shape": [1, S, S]}
        r.update(measure(d, prog, x, lambda xs: d.calc_bpd_loop(xs, z), args.steps, args.reps,
                           args.e2e_reps))
        res["cfg2"] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
