#!/usr/bin/env python
"""Cost of the three samplers (GPU only): ms per reverse step of the replayed step graph for
DDPM (ancestral), strided DDIM and DPM-Solver++(2M), the DDPM and DPM-Solver++ inpainting steps
(the same step plus mri_inpaint_merge, every element kept: the merge's worst case), ms per replay of
RePaint's undo graph (mri_repaint_undo + step_advance), and end to end for
sample_dpmpp(num_steps=20) and for inpaint() against inpaint(jump_length=10, jump_n_sample=2) at
T = 1000 (1000 against 1990 UNet calls; half of each sample regenerated, one run each).

  cfg4  ddpm_3d_ldm         UNet3DModelWithAttention(3, base 128, mults 1-2-4) B=16 3x40x48x40
  cfg2  slice_cond_2d_ddpm  UNet(1, base 64, mults 1-2-4-8)                   B=64 1x240x240

Each step time is CUDA events around STEPS replays of one captured step graph (after warm-up
replays); the step graphs are timed in turn, REPS times alternating, and the median and the
spread ((max - min) / median) are reported.  End to end is CUDA events around the public call
(x_T draw, table build and upload, 20 replays, result copy), REPS times.  Random-init weights:
this measures sampling cost only, not sample quality.  GPU name and power limit are read with a
read-only nvidia-smi query in the same run.

  python tools/sampler_bench.py [--out profiles/<name>.json] [--steps 20] [--reps 3]
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
DDIM_STRIDE = 50   # sample_ddim(num_steps=20) at T = 1000


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


def step_times(diff, prog, x, steps, reps, warm=3):
    """ms per replayed step of the DDPM, strided-DDIM, DPM-Solver++ and the two inpainting step
    graphs on `prog`."""
    # inpainting inputs: a known volume and a mask that keeps every element, the merge's most
    # expensive case (it reads x and known and writes x everywhere; a group of four regenerated
    # elements would be skipped)
    known = torch.randn_like(x)
    mask = torch.zeros(x.shape, dtype=torch.uint8, device=x.device)
    # one short run each captures the step graphs (and warms every shape)
    diff._reverse_loop(prog, x, T - 1, 3, "ddpm")
    diff._reverse_loop(prog, x, T - 1, 3, "ddim", stride=DDIM_STRIDE)
    diff._reverse_loop(prog, x, T - 1, 3, "dpmpp", table=diff._dpmpp_table(T - 1, steps))
    diff._reverse_loop(prog, x, T - 1, 3, "ddpm", inpaint=(known, mask))
    diff._reverse_loop(prog, x, T - 1, 3, "dpmpp", table=diff._dpmpp_table(T - 1, steps),
                       inpaint=(known, mask))
    # three reverse steps and one undo: captures the undo graph
    diff._reverse_loop(prog, x, T - 1, 3, "ddpm", inpaint=(known, mask),
                       levels=[T - 1, T - 2, T - 1, T - 2, T - 3])
    g = {k: prog._step_graphs[k][2] for k in ("ddpm", f"ddim/{DDIM_STRIDE}", "dpmpp", "ddpm+inpaint",
                                              "dpmpp+inpaint", "repaint-undo")}
    tprev, dpm = prog._tprev_buf, prog._dpmpp_bufs
    n_ddim = min(steps, (T - 1) // DDIM_STRIDE)   # t stays >= 0 over the timed replays

    def reset(key):
        prog.x_in.copy_(x)
        # the undo steps t up by one per replay and reads alphas[t + 1]: start low enough
        prog.t_in.fill_(T - 2 - steps if key == "repaint-undo" else T - 1)
        tprev.fill_(T - 1 - DDIM_STRIDE)
        dpm["k"].zero_()
        diff._rng(x.device).load()

    def replays(key, n):
        for _ in range(n):
            g[key].replay()

    plan = {"ddpm": ("ddpm", steps), "ddim": (f"ddim/{DDIM_STRIDE}", n_ddim), "dpmpp": ("dpmpp", steps),
            "ddpm+inpaint": ("ddpm+inpaint", steps), "dpmpp+inpaint": ("dpmpp+inpaint", steps),
            "repaint-undo": ("repaint-undo", steps)}
    for name, (key, n) in plan.items():
        reset(key)
        replays(key, min(warm, n))
    out = {k: [] for k in plan}
    for _ in range(reps):
        for name, (key, n) in plan.items():
            reset(key)
            out[name].append(events_ms(lambda: replays(key, n)) / n)
    assert torch.isfinite(prog.x_in).all()
    res = {k: summary(v) for k, v in out.items()}
    for k in ("ddpm", "dpmpp"):   # the inpainting step against the plain step, run by run
        ratios = [a / b for a, b in zip(out[f"{k}+inpaint"], out[k])]
        res[f"{k}+inpaint"]["ratio_to_plain"] = summary(ratios)
    return res


def end_to_end(fn, batch, reps):
    fn()   # warm: the graph already exists; this loads the table path once
    ms = [events_ms(fn) for _ in range(reps)]
    s = summary(ms)
    s["per_second"] = batch / (s["median"] / 1e3)
    return s


def repaint_end_to_end(inpaint, x):
    """ms of one inpaint() and one inpaint(jump_length=10, jump_n_sample=2) at T = 1000 on the step
    graphs step_times captured; half of each sample regenerated."""
    from mri_image_generation_b200 import schedules
    lv = schedules.repaint_levels(T, 10, 2)
    known = torch.randn_like(x)
    mask = torch.zeros(x.shape, dtype=torch.bool, device=x.device)
    mask[..., x.shape[-1] // 2:] = True
    plain = events_ms(lambda: inpaint(known, mask))
    rp = events_ms(lambda: inpaint(known, mask, jump_length=10, jump_n_sample=2))
    return {"inpaint_ms": plain, "repaint_10_2_ms": rp, "ratio": rp / plain,
            "unet_calls": {"inpaint": T, "repaint_10_2": sum(q < p for p, q in zip(lv, lv[1:]))}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
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
    res = {"gpu": gpu_info(dev.index), "timesteps": T, "dpmpp_num_steps": args.steps,
           "ddim_stride": DDIM_STRIDE, "reps": args.reps,
           "note": "sampling cost only (random-init weights), not sample quality"}
    with torch.no_grad():
        # ---- cfg4 ---------------------------------------------------------------------------------
        B, shape = args.b4, (40, 48, 40)
        torch.manual_seed(0)
        m = UNet3DModelWithAttention(in_channels=3, base_channels=128, channel_mults=(1, 2, 4),
                                     time_emb_dim=256, groups=8, num_heads=4).to(dev).eval()
        d = quiet(GaussianDiffusionLatent3D, m, 3, timesteps=T).to(dev)
        x = torch.randn(B, 3, *shape, device=dev)
        prog = m.program(B, shape)
        r = {"batch": B, "shape": [3, *shape], "ms_per_step": step_times(d, prog, x, args.steps, args.reps)}
        r["sample_dpmpp_ms"] = end_to_end(lambda: d.sample_dpmpp(B, shape, num_steps=args.steps), B, args.reps)
        r["volumes_per_s_dpmpp"] = r["sample_dpmpp_ms"]["per_second"]
        r["volumes_per_s_ddpm_1000_steps_derived"] = B / (T * r["ms_per_step"]["ddpm"]["median"] / 1e3)
        r["repaint_end_to_end"] = repaint_end_to_end(d.inpaint, x)
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
        x = torch.randn(B, 1, S, S, device=dev)
        prog = m.program(B, (S, S), 1, 0)
        prog.z_in.copy_(z.reshape(-1, 1))
        r = {"batch": B, "shape": [1, S, S], "ms_per_step": step_times(d, prog, x, args.steps, args.reps)}
        r["sample_dpmpp_ms"] = end_to_end(lambda: d.sample_dpmpp(B, z_pos=z, num_steps=args.steps), B,
                                          args.reps)
        r["slices_per_s_dpmpp"] = r["sample_dpmpp_ms"]["per_second"]
        r["slices_per_s_ddpm_1000_steps_derived"] = B / (T * r["ms_per_step"]["ddpm"]["median"] / 1e3)
        r["repaint_end_to_end"] = repaint_end_to_end(
            lambda known, mask, **kw: d.inpaint(known, mask, z_pos=z, **kw), x)
        res["cfg2"] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
