#!/usr/bin/env python
"""Cost of keeping an EMA of the weights during training (GPU only), on the cfg5 training step of
`bench.py --mode train` (UNet3DModelWithAttention base 128, B = 8 latents of 3x40x48x40, q_sample +
forward + min-SNR loss + backward + fused Adam, one GPU).  Three arms on the same model and
optimizer, timed in turn REPS times alternating (median and spread (max - min) / median):

  none            Adam(...)
  ema             Adam(..., ema=EMA(unet, 0.9999)): one mri_ema_update launch inside step()
  averaged_model  Adam(...) then torch.optim.swa_utils.AveragedModel(unet,
                  multi_avg_fn=get_ema_multi_avg_fn(0.9999)).update_parameters(unet)

Each arm time is CUDA events around STEPS steps after WARM steps of that arm.  The mri_ema_update
launch alone (ema_update_kernel + the one-thread counter advance) is timed with CUDA events over
KERNEL_ITERS launches, and its rate is given against 3 x 4 x n_params bytes (read p and e, write e;
1.64 GB per update at cfg5, larger than the 126 MB L2).  GPU name and power limit are read with a
read-only nvidia-smi query in the same run.

  python tools/ema_bench.py [--out profiles/<name>.json] [--steps 20] [--reps 3] [--kernel-iters 200]
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
LATENT = (3, 40, 48, 40)
DECAY = 0.9999


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warm", type=int, default=4)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-iters", type=int, default=200)
    args = ap.parse_args()
    from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn

    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet_attention import UNet3DModelWithAttention
    from mri_image_generation_b200.optim import EMA, Adam

    _lib.require_device()
    dev = torch.device("cuda", torch.cuda.current_device())
    res = {"gpu": gpu_info(dev.index), "batch": args.batch, "latent": list(LATENT), "decay": DECAY,
           "steps_per_timing": args.steps, "reps": args.reps,
           "step": "q_sample (in-kernel Philox) + fwd + min-SNR loss + bwd + fused Adam (bench.py --mode train, 1 GPU)"}
    torch.manual_seed(0)
    model = UNet3DModelWithAttention(in_channels=3, base_channels=128, channel_mults=(1, 2, 4), time_emb_dim=256,
                                     groups=8, num_heads=4).to(dev).train()
    with contextlib.redirect_stdout(io.StringIO()):
        diff = GaussianDiffusionLatent3D(model, LATENT[0], timesteps=T).to(dev)
    ema = EMA(model, DECAY)
    opt = Adam(model.parameters(), lr=2e-4)
    avg = AveragedModel(model, multi_avg_fn=get_ema_multi_avg_fn(DECAY))
    avg.update_parameters(model)   # its first call only copies
    n_params = sum(p.numel() for p in model.parameters())
    torch.manual_seed(1234)
    z = torch.randn(args.batch, *LATENT, device=dev)

    def step(arm):
        t = torch.randint(1, T, (args.batch,), device=dev)
        opt.zero_grad(set_to_none=True)
        loss = diff.p_losses(z, t, cond=None, min_snr_gamma=5.0)
        loss.backward()
        opt.step()
        if arm == "averaged_model":
            avg.update_parameters(model)

    def run(arm, n):
        opt.ema = ema if arm == "ema" else None
        for _ in range(n):
            step(arm)

    arms = ("none", "ema", "averaged_model")
    for arm in arms:
        run(arm, args.warm)
    ms = {a: [] for a in arms}
    for _ in range(args.reps):
        for arm in arms:
            run(arm, args.warm)
            ms[arm].append(events_ms(lambda: run(arm, args.steps)) / args.steps)
    res["ms_per_step"] = {a: summary(v) for a, v in ms.items()}
    res["ratio_to_none"] = {a: summary([x / y for x, y in zip(ms[a], ms["none"])]) for a in arms[1:]}
    opt.ema = None

    # ---- the launch alone ------------------------------------------------------------------------
    lib = _lib.load()
    shadow, live = list(ema.module.parameters()), list(model.parameters())
    table, n, blocks = ema._table(shadow, live)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def launches(k):
        for _ in range(k):
            _lib.check(lib.mri_ema_update(table.data_ptr(), n, blocks, DECAY, 0, ema.num_updates.data_ptr(),
                                          None, stream), "mri_ema_update")

    launches(10)
    kms = [events_ms(lambda: launches(args.kernel_iters)) / args.kernel_iters for _ in range(args.reps)]
    nbytes = 3 * 4 * n_params
    k = summary(kms)
    k["bytes"] = nbytes
    k["GB_per_s"] = nbytes / (k["median"] * 1e-3) / 1e9
    k["launches_per_timing"] = args.kernel_iters
    res["mri_ema_update_ms"] = k
    res["n_params"] = n_params
    res["n_tensors"] = n
    avg_ms = [events_ms(lambda: avg.update_parameters(model)) for _ in range(args.reps)]
    res["averaged_model_update_parameters_ms"] = summary(avg_ms)
    res["note"] = ("random-init weights, synthetic latents; ms_per_step are device events around whole "
                   "steps, mri_ema_update_ms includes the one-thread counter advance")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
