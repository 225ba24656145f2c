#!/usr/bin/env python
"""Cost of undersampled k-space reconstruction (GPU only): ms per replay of the 'ddpm',
'ddpm+kspace', 'dpmpp' and 'dpmpp+kspace' step graphs on one program, the mri_kspace_merge
launches alone and their FLOP rate, and reconstruct_dpmpp(num_steps=20) end to end against
sample_dpmpp(num_steps=20).

  cfg2  slice_cond_2d_ddpm       UNet(1, base 64, mults 1-2-4-8)       B=64 1x240x240
  cfg3  ddpm_25d_all_modalities  UNet(20 -> 4, base 64, mults 1-2-4-8) B=32 4x192x192 (16 context)

Step times are CUDA events around STEPS replays of one captured graph after warm-up replays; the
four graphs are timed in turn, REPS times alternating, and the median and the spread
((max - min) / median) are reported, with the k-space step over the plain step run by run.  The
merge alone is CUDA events around MERGE_ITERS launches (in-kernel Philox draw).  Its FLOP count,
computed from shapes, is the multiply-adds the three passes need: per plane 2 H Wh W (forward rows,
real input) + 8 Wh H^2 (forward and inverse columns, complex) + 2 H W Wh (inverse rows, real part
only), Wh = W / 2 + 1, 2 FLOP each.  The column pass pads Wh to whole 16-column tiles and its
inverse half skips rows of a tile with no measured sample; the count credits neither.  The mask
is every fourth phase-encode row plus the four lowest, as an accelerated Cartesian scan measures.  Random-init weights: this
measures cost only.  GPU name and power limit are read with a read-only nvidia-smi query in the
same run.

  python tools/kspace_bench.py [--out profiles/<name>.json] [--steps 20] [--reps 5]
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

T = 1000
MERGE_ITERS = 200


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def gpu_info(dev):
    r = subprocess.run(["nvidia-smi", f"--id={dev}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, power, clk = [v.strip() for v in r.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk,
            "torch_name": torch.cuda.get_device_name(dev)}


def events_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def summary(v):
    med = statistics.median(v)
    return {"median": med, "spread": (max(v) - min(v)) / med, "runs": v}


def merge_flops(B, C, H, W):
    wh = W // 2 + 1
    return 2 * B * C * (2 * H * wh * W + 8 * wh * H * H + 2 * H * W * wh)


def line_mask(shape, dev):
    B, C, H, W = shape
    keep = torch.zeros(H, dtype=torch.bool)
    keep[::4] = True
    keep[[0, 1, H - 2, H - 1]] = True
    return keep.view(1, 1, H, 1).expand(shape).to(dev)


def step_times(diff, prog, x, kspace, kmask, steps, reps, warm=3):
    from mri_image_generation_b200 import ops
    zf, M = diff._kspace_inputs(kspace, kmask)
    table = diff._dpmpp_table(T - 1, steps)
    diff._reverse_loop(prog, x, T - 1, 3, "ddpm")
    diff._reverse_loop(prog, x, T - 1, 3, "dpmpp", table=table)
    diff._reverse_loop(prog, x, T - 1, 3, "ddpm", inpaint=(zf, M), kspace=True)
    diff._reverse_loop(prog, x, T - 1, 3, "dpmpp", table=table, inpaint=(zf, M), kspace=True)
    keys = ("ddpm", "dpmpp", "ddpm+kspace", "dpmpp+kspace")
    g = {k: prog._step_graphs[k][2] for k in keys}
    dpm = prog._dpmpp_bufs

    def reset():
        prog.x_in.copy_(x)
        prog.t_in.fill_(T - 1)
        dpm["k"].zero_()
        diff._rng(x.device).load()

    def replays(key, n):
        for _ in range(n):
            g[key].replay()

    for k in keys:
        reset()
        replays(k, warm)
    out = {k: [] for k in keys}
    for _ in range(reps):
        for k in keys:
            reset()
            out[k].append(events_ms(lambda: replays(k, steps)) / steps)
    assert torch.isfinite(prog.x_in).all()
    res = {k: summary(v) for k, v in out.items()}
    for k in ("ddpm", "dpmpp"):
        res[f"{k}+kspace"]["ratio_to_plain"] = summary([a / b for a, b in zip(out[f"{k}+kspace"], out[k])])

    # the merge alone: three launches, z drawn in the kernel
    rng = diff._rng(x.device)
    work = prog._inpaint_bufs["work"]
    xs = x.clone()
    t = torch.full((x.shape[0],), T - 1, dtype=torch.int64, device=x.device)

    def merges():
        for _ in range(MERGE_ITERS):
            ops.kspace_merge(xs, zf, M, t, -1, diff.sqrt_alphas_cumprod,
                             diff.sqrt_one_minus_alphas_cumprod, work=work, rng=rng)

    rng.load()
    merges()
    ms = [events_ms(merges) / MERGE_ITERS for _ in range(reps)]
    fl = merge_flops(*x.shape)
    res["merge_alone"] = dict(summary(ms), flop=fl,
                              tflops=fl / (statistics.median(ms) * 1e-3) / 1e12,
                              share_of_ddpm_step=statistics.median(ms) / res["ddpm"]["median"])
    return res


def end_to_end(fn, reps):
    fn()
    return summary([events_ms(fn) for _ in range(reps)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.diffusion import GaussianDiffusion as G25
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.unet import UNet as U25
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet

    _lib.require_device()
    dev = torch.device("cuda", torch.cuda.current_device())
    res = {"gpu": gpu_info(dev.index), "timesteps": T, "dpmpp_num_steps": args.steps, "reps": args.reps,
           "merge_iters": MERGE_ITERS, "mask": "every 4th phase-encode row + 4 lowest",
           "note": "cost only (random-init weights), not reconstruction quality"}
    with torch.no_grad():
        for name, B, C, S, cc in (("cfg2", 64, 1, 240, 0), ("cfg3", 32, 4, 192, 16)):
            torch.manual_seed(0)
            if cc == 0:
                m = quiet(UNet, img_channels=1, base_channels=64, channel_mults=(1, 2, 4, 8),
                          time_emb_dim=256).to(dev).eval()
                d = quiet(GaussianDiffusion, m, S, channels=1, timesteps=T).to(dev)
                ctx, kw = None, {}
            else:
                m = quiet(U25, in_channels=20, out_channels=4, base_channels=64, channel_mults=(1, 2, 4, 8),
                          time_emb_dim=256).to(dev).eval()
                d = quiet(G25, m, S, channels=4, timesteps=T).to(dev)
                ctx = torch.randn(B, cc, S, S, device=dev)
                kw = {"context": ctx}
            z = torch.rand(B, device=dev)
            x = torch.randn(B, C, S, S, device=dev)
            kspace = torch.fft.fft2(torch.randn(B, C, S, S, device=dev), norm="ortho")
            kmask = line_mask(x.shape, dev)
            prog = m.program(B, (S, S), C, cc)
            prog.z_in.copy_(z.reshape(-1, 1))
            if ctx is not None:
                prog.ctx_in.copy_(ctx)
            r = {"batch": B, "shape": [C, S, S],
                 "ms_per_step": step_times(d, prog, x, kspace, kmask, args.steps, args.reps)}
            r["reconstruct_dpmpp_ms"] = end_to_end(
                lambda: d.reconstruct_dpmpp(kspace, kmask, z_pos=z, num_steps=args.steps, **kw), args.reps)
            r["sample_dpmpp_ms"] = end_to_end(
                lambda: d.sample_dpmpp(B, z_pos=z, num_steps=args.steps, **kw), args.reps)
            res[name] = r
            del m, d, x, prog, ctx
            torch.cuda.empty_cache()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
