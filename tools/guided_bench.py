#!/usr/bin/env python
"""Cost of measurement-guided sampling of the 3D LDM (GPU only), at BASELINE cfg4's shapes:
UNet3DModelWithAttention(3, 128, (1, 2, 4)) on a 3x40x48x40 latent, VAE3D(4, 32, 3, 3) decoding it
to a 4x160x192x160 image, B = 1, 2, 4.

For each B:
  - ms per replay of the 'dpmpp' step graph and of the 'dpmpp+guided:kspace' one (CUDA events
    around STEPS replays after warm-up replays, REPS times alternating; median and spread);
  - the guided step's stages timed one by one with CUDA events (UNet forward, decoder forward,
    the k-space data term, decoder data-gradient backward, and the rest: x0, eps' and the update),
    each over STAGE_ITERS launches outside a graph, so their sum exceeds the replayed step by the
    launch gaps;
  - mri_dc_project3d alone: ms, the FLOPs and HBM bytes its five DFT passes need (computed from
    shapes below) and the achieved rates, with the share of the HBM bandwidth bound;
  - peak allocated memory of the guided run per volume (torch.cuda.max_memory_allocated), or the
    error when it does not fit.

FLOPs of the projector per (sample, channel) volume, Wh = W / 2 + 1, 2 FLOP per multiply-add:
forward rows 2 D H Wh W (real input), forward H 4 D Wh H^2, forward and inverse D 8 H Wh D^2,
inverse H 4 D Wh H^2, inverse rows 2 D H W Wh (real part only).  Bytes: u, x_zf and g (fp32), the
mask (uint8) and four round trips of the complex half spectrum (8 bytes a value).  The mask is
every fourth (D, H) phase-encode line plus the centre.  Random-init weights: cost only.  GPU name
and power limit are read with a read-only nvidia-smi query in the same run.

  python tools/guided_bench.py [--out profiles/<name>.json] [--steps 10] [--reps 3]
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
STAGE_ITERS = 5
PROJ_ITERS = 10
HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU
LAT = (40, 48, 40)
IMG = (160, 192, 160)


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


def proj_cost(B, C, D, H, W):
    wh = W // 2 + 1
    flop = 2 * B * C * (D * H * wh * W + 2 * D * wh * H * H + 4 * H * wh * D * D + 2 * D * wh * H * H
                        + D * H * W * wh)
    n = B * C * D * H * W
    byts = 12 * n + n + 4 * 2 * 8 * B * C * D * H * wh
    return flop, byts


def plane_mask(dev):
    D, H, W = IMG
    keep = torch.zeros(D, H, dtype=torch.bool)
    keep[::4, ::4] = True
    keep[D // 2 - 8:D // 2 + 8, H // 2 - 8:H // 2 + 8] = True
    keep[0, 0] = True
    return keep.view(1, 1, D, H, 1).to(dev)


def run_batch(diff, unet, vae, B, steps, reps, dev):
    from mri_image_generation_b200 import ops
    torch.cuda.reset_peak_memory_stats(dev)
    x_img = torch.randn(B, 4, *IMG, device=dev)
    y = torch.fft.fftn(x_img, dim=(-3, -2, -1), norm="ortho")
    m = plane_mask(dev)
    table = diff._dpmpp_table(T - 1, steps)
    # one guided call sets up the decoder program, the buffers and the captured graph
    diff.reconstruct_dpmpp(y, m, vae, num_steps=3)
    mem = torch.cuda.max_memory_allocated(dev)
    prog = unet.program(B, LAT)
    x = torch.randn(B, 3, *LAT, device=dev)
    diff._reverse_loop(prog, x, T - 1, 3, "dpmpp", table=table)
    keys = ("dpmpp", "dpmpp+guided:kspace")
    g = {k: prog._step_graphs[k][2] for k in keys}
    dpm = prog._dpmpp_bufs

    def reset():
        prog.x_in.copy_(x)
        prog.t_in.fill_(T - 1)
        dpm["k"].zero_()

    def replays(key, n):
        for _ in range(n):
            g[key].replay()

    for k in keys:
        reset()
        replays(k, 2)
    out = {k: [] for k in keys}
    for _ in range(reps):
        for k in keys:
            reset()
            out[k].append(events_ms(lambda: replays(k, steps)) / steps)
    res = {k: summary(v) for k, v in out.items()}
    res["guided_over_plain"] = summary([a / b for a, b in zip(out[keys[1]], out[keys[0]])])

    # stages of the guided step, one by one
    b = prog._guided_bufs
    dec = b["dec"]
    sa, s1m = diff.sqrt_alphas_cumprod, diff.sqrt_one_minus_alphas_cumprod
    C, ldc = prog.cout, prog.cout_pad
    reset()
    xp, eps = dpm["x0_prev"], b["eps"]

    def rest():
        ops.guided_x0(prog.x_in, prog.eps_nhwc, prog.t_in, sa, s1m, b["inv_s"], dec.x_in, eps_nhwc_ldc=ldc,
                      channels=C)
        ops.guided_eps(prog.eps_nhwc, dec.dz_out, b["gg"], b["lam"], b["inv_s"], prog.t_in, sa, s1m, eps,
                       eps_nhwc_ldc=ldc, channels=C)
        ops.dpmpp_step(prog.x_in, eps, xp, dpm["coef"], dpm["k"], prog.x_in)

    stages = {"unet": prog.run,
              "decoder_forward": lambda: (dec.run(), dec.finish_output()),
              "data_term": lambda: ops.dc_project3d(dec.out, b["zf"], b["mask"], dec.dout_in, b["gg"],
                                                    b["work"]),
              "decoder_backward": dec.run_input_backward,
              "rest": rest}
    st = {}
    for name, fn in stages.items():
        fn()

        def many(fn=fn):
            for _ in range(STAGE_ITERS):
                fn()
        st[name] = summary([events_ms(many) / STAGE_ITERS for _ in range(reps)])
    total = sum(v["median"] for v in st.values())
    for v in st.values():
        v["share"] = v["median"] / total
    res["stages_ms"] = st

    def projs():
        for _ in range(PROJ_ITERS):
            ops.dc_project3d(dec.out, b["zf"], b["mask"], dec.dout_in, b["gg"], b["work"])
    projs()
    ms = [events_ms(projs) / PROJ_ITERS for _ in range(reps)]
    med = statistics.median(ms)
    flop, byts = proj_cost(B, 4, *IMG)
    res["projector"] = dict(summary(ms), flop=flop, bytes=byts, tflops=flop / (med * 1e-3) / 1e12,
                            hbm_tb_per_s=byts / (med * 1e-3) / 1e12,
                            hbm_bound_share=byts / HBM_BYTES_PER_S / (med * 1e-3))
    res["peak_mem_gb_per_volume"] = mem / B / 1e9
    res["peak_mem_gb"] = mem / 1e9
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batches", default="1,2,4")
    args = ap.parse_args()
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.vae import VAE3D

    _lib.require_device()
    dev = torch.device("cuda", torch.cuda.current_device())
    res = {"gpu": gpu_info(dev.index), "timesteps": T, "dpmpp_num_steps": args.steps, "reps": args.reps,
           "latent": [3, *LAT], "image": [4, *IMG],
           "note": "cost only (random-init weights), not reconstruction quality"}
    with torch.no_grad():
        for B in [int(v) for v in args.batches.split(",")]:
            torch.manual_seed(0)
            unet = UNet3DModelWithAttention(3, 128, (1, 2, 4)).to(dev).eval()
            vae = VAE3D(4, 32, 3, 3).to(dev).eval()
            diff = quiet(GaussianDiffusionLatent3D, unet, 3, timesteps=T).to(dev)
            try:
                res[f"B{B}"] = run_batch(diff, unet, vae, B, args.steps, args.reps, dev)
            except torch.cuda.OutOfMemoryError as e:
                res[f"B{B}"] = {"error": f"out of memory: {str(e).splitlines()[0]}"}
            print(json.dumps({f"B{B}": res[f"B{B}"]}), flush=True)
            del unet, vae, diff
            torch.cuda.empty_cache()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
